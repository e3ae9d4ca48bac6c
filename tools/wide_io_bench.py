"""Step time of wide models with many chain inputs / outputs at batch 65 536, next to the same model with 8 inputs.

usage: wide_io_bench.py [STEPS] [--inputs N] [--chains K] [--outputs O] [--hidden 512,512,512] [--repeats R]
The model: a traced process model of four parameters (rb, Q10, alpha, beta); N predictors in total, split over K chains
(MultiNN, one neural parameter per chain) or one chain predicting O neural parameters (K = 1); the other parameters are
global.  N = 2^20 rows, Adam, mse.  The same model with min(N, 8) inputs runs alternately as the reference shape (layer 1
and the layer-1 column sums scale with the input count).  Prints the GPU's name and power limit first, then one line
per shape and repeat (device time of STEPS steps from CUDA events)."""
import argparse
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import easyhybrid_b200 as eh

B = 65536
NAMES = ["rb", "Q10", "alpha", "beta"]
PARAMS = dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0), alpha=(0.5, -2.0, 2.0), beta=(0.2, -1.0, 1.0))


def four_param_pm(*, ta, dsw_pot, rb, Q10, alpha, beta, tref=15.0):
    return {"reco": rb * Q10 ** (0.1 * (ta - tref)) + alpha * np.tanh(0.05 * dsw_pot) + beta * np.sin(0.1 * ta)}


def synth(n, seed=42):
    rng = np.random.default_rng(seed)
    ta = (10 + 10 * rng.standard_normal(n)).astype(np.float32)
    sw = np.abs(50 + 20 * rng.standard_normal(n)).astype(np.float32)
    dsw = np.concatenate([[0.0], np.diff(sw)]).astype(np.float32)
    reco = ((3.0 + 0.02 * (sw - sw.mean())) * 2.0 ** (0.1 * (ta - 15.0)) + 0.3 * np.tanh(0.05 * dsw)
            + 0.1 * rng.standard_normal(n)).astype(np.float32)
    t = dict(ta=ta, sw_pot=sw, dsw_pot=dsw, reco=reco)
    for k in range(9):
        t["z%d" % k] = rng.standard_normal(n).astype(np.float32)
    return t


def make_model(inputs, chains, outputs, hidden):
    cols = (["sw_pot", "dsw_pot", "ta"] + ["z%d" % k for k in range(9)])[:inputs]
    if chains == 1:
        neural = NAMES[:outputs]
        preds = cols
        hl = list(hidden)
    else:
        neural = NAMES[:chains]
        per = [inputs // chains + (1 if c < inputs % chains else 0) for c in range(chains)]
        preds, o = {}, 0
        for c, name in enumerate(neural):
            preds[name] = cols[o:o + per[c]]
            o += per[c]
        hl = {name: list(hidden) for name in neural}
    glob = [p for p in NAMES if p not in neural]
    return eh.constructHybridModel(preds, ["ta", "dsw_pot"], ["reco"], four_param_pm, PARAMS, neural if chains == 1 else [],
                                   glob, hidden_layers=hl, activation="tanh", scale_nn_outputs=True)


def main():
    ap = argparse.ArgumentParser(description="step time of wide models with many chain inputs / outputs")
    ap.add_argument("steps", nargs="?", type=int, default=64)
    ap.add_argument("--inputs", type=int, default=12, help="chain inputs in total (1..12)")
    ap.add_argument("--chains", type=int, default=1, help="chains (1..4); with K > 1 every chain predicts one parameter")
    ap.add_argument("--outputs", type=int, default=4, help="neural parameters of a single chain (1..4; K = 1 only)")
    ap.add_argument("--hidden", default="512,512,512", help="hidden widths of every chain, comma separated")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    if not 1 <= args.chains <= 4 or not 1 <= args.outputs <= 4 or not args.chains <= args.inputs <= 12:
        ap.error("1..4 chains, 1..4 outputs, chains..12 inputs")
    hidden = [int(h) for h in args.hidden.split(",")]
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        print("gpu:", q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown")
    except (OSError, subprocess.SubprocessError):
        print("gpu: unknown")
    n = 1 << 20
    data = synth(n)
    shapes = [args.inputs] + ([min(args.inputs, 8)] if args.inputs > 8 else [])
    sessions = {}
    for p in shapes:
        model = make_model(p, args.chains, args.outputs, hidden)
        xf, y = eh.prepare_data(model, data)
        sess = eh.FusedSession(model, training_loss="mse", agg="sum", opt=eh.Adam(0.001))
        sess.upload(0, xf, y)
        sess.set_params(model.initialparameters(np.random.default_rng(0)))
        sess.set_perm(np.random.default_rng(7).permutation(n))
        sess.run_steps(B, 0, 8)   # warm-up: module load, first launches
        sessions[p] = sess
    nout = args.outputs if args.chains == 1 else args.chains
    for r in range(args.repeats):   # shapes alternate within each repeat
        for p, sess in sessions.items():
            losses = sess.run_steps(B, 8, args.steps)
            ms, launches, _ = sess.last_timing()
            us = 1e3 * ms / args.steps
            print(f"[inputs {p} chains {args.chains} outputs {nout} hidden {args.hidden}] {sess.kernel_variant()}: "
                  f"{args.steps} steps, {us:.1f} us/step, {B / (us * 1e-6):.3e} samples/s, {launches // args.steps} launches/step, "
                  f"loss {losses[0]:.4f} -> {losses[-1]:.4f} (repeat {r})")
    for sess in sessions.values():
        sess.close()


if __name__ == "__main__":
    main()
