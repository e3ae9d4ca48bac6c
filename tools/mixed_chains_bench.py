"""Step time of wide models whose chains differ in depth or activation (the per-unit form of the tensor-core path) at
batch 65 536, next to an equal-depth, single-activation model of the same embedded widths.

usage: mixed_chains_bench.py [STEPS] [--repeats R]
Pairs (RbQ10, N = 2^20 rows, Adam, mse):
  depth:      rb [512, 512, 512] with Q10 global            against  rb [384, 384, 384] + Q10 [128] (pass-through units)
  activation: rb [256, 256] tanh + Q10 [256, 256] tanh      against  rb [256, 256] relu + Q10 [256, 256] tanh
The two models of a pair run alternately.  Prints the GPU's name and power limit first, then one line per model and
repeat (device time of STEPS steps from CUDA events)."""
import argparse
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import easyhybrid_b200 as eh

B = 65536
PARAMS = dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0))


def synth(n, seed=42):
    rng = np.random.default_rng(seed)
    ta = (10 + 10 * rng.standard_normal(n)).astype(np.float32)
    sw = np.abs(50 + 20 * rng.standard_normal(n)).astype(np.float32)
    dsw = np.concatenate([[0.0], np.diff(sw)]).astype(np.float32)
    reco = ((3.0 + 0.02 * (sw - sw.mean())) * 2.0 ** (0.1 * (ta - 15.0)) + 0.1 * rng.standard_normal(n)).astype(np.float32)
    return dict(ta=ta, sw_pot=sw, dsw_pot=dsw, reco=reco)


def single(hidden):
    return eh.constructHybridModel({"rb": ["sw_pot", "dsw_pot"]}, ["ta"], ["reco"], eh.RbQ10, PARAMS, ["Q10"],
                                   hidden_layers={"rb": list(hidden)}, activation="tanh", scale_nn_outputs=True)


def two(hidden_rb, hidden_q10, act_rb, act_q10):
    return eh.constructHybridModel({"rb": ["sw_pot", "dsw_pot"], "Q10": ["ta"]}, ["ta"], ["reco"], eh.RbQ10, PARAMS, [],
                                   hidden_layers={"rb": list(hidden_rb), "Q10": list(hidden_q10)},
                                   activation={"rb": act_rb, "Q10": act_q10}, scale_nn_outputs=True)


PAIRS = {
    "depth": [("rb 3x512, Q10 global", lambda: single((512, 512, 512))),
              ("rb 3x384 + Q10 [128]", lambda: two((384, 384, 384), (128,), "tanh", "tanh"))],
    "activation": [("2x256 tanh + 2x256 tanh", lambda: two((256, 256), (256, 256), "tanh", "tanh")),
                   ("2x256 relu + 2x256 tanh", lambda: two((256, 256), (256, 256), "relu", "tanh"))],
}


def main():
    ap = argparse.ArgumentParser(description="step time of wide models whose chains differ in depth or activation")
    ap.add_argument("steps", nargs="?", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        print("gpu:", q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown")
    except (OSError, subprocess.SubprocessError):
        print("gpu: unknown")
    n = 1 << 20
    data = synth(n)
    for pair, models in PAIRS.items():
        sessions = []
        for label, mk in models:
            model = mk()
            xf, y = eh.prepare_data(model, data)
            sess = eh.FusedSession(model, training_loss="mse", agg="sum", opt=eh.Adam(0.001))
            sess.upload(0, xf, y)
            sess.set_params(model.initialparameters(np.random.default_rng(0)))
            sess.set_perm(np.random.default_rng(7).permutation(n))
            sess.run_steps(B, 0, 8)   # warm-up: module load, first launches
            sessions.append((label, sess))
        for r in range(args.repeats):   # the models of a pair alternate within each repeat
            for label, sess in sessions:
                losses = sess.run_steps(B, 8, args.steps)
                ms, launches, _ = sess.last_timing()
                us = 1e3 * ms / args.steps
                print(f"[{pair}] {label}: {sess.kernel_variant()}: {args.steps} steps, {us:.1f} us/step, "
                      f"{B / (us * 1e-6):.3e} samples/s, {launches // args.steps} launches/step, "
                      f"loss {losses[0]:.4f} -> {losses[-1]:.4f} (repeat {r})")
        for _, sess in sessions:
            sess.close()


if __name__ == "__main__":
    main()
