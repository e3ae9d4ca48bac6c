"""Step time of chains with one wide hidden layer (the fused exact-fp32 kernel k_wide_one) at batch 65 536.

usage: one_hidden_bench.py [STEPS] [--repeats R]
Workloads (RbQ10, N = 2^20 rows, Adam, mse): [2-64-1], [2-512-1], two chains [1+2 -> 256+256 -> 2], and, as context,
the two-layer [2-512-512-1] step on the bf16 tensor-core path.  Prints one line per workload and repeat (device time of
STEPS steps from CUDA events) and the GPU's name and power limit first."""
import argparse
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import easyhybrid_b200 as eh

B = 65536


def synth(n, seed=42):
    rng = np.random.default_rng(seed)
    ta = (10 + 10 * rng.standard_normal(n)).astype(np.float32)
    sw = np.abs(50 + 20 * rng.standard_normal(n)).astype(np.float32)
    dsw = np.concatenate([[0.0], np.diff(sw)]).astype(np.float32)
    reco = ((3.0 + 0.02 * (sw - sw.mean())) * 2.0 ** (0.1 * (ta - 15.0)) + 0.1 * rng.standard_normal(n)).astype(np.float32)
    return dict(ta=ta, sw_pot=sw, dsw_pot=dsw, reco=reco)


def model_of(name):
    par = dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0))
    if name == "two-chain 1+2->256+256->2":
        return eh.constructHybridModel({"rb": ["sw_pot", "dsw_pot"], "Q10": ["ta"]}, ["ta"], ["reco"], eh.RbQ10, par, [],
                                       hidden_layers=[256], activation="tanh", scale_nn_outputs=True)
    hidden = {"2-64-1": [64], "2-512-1": [512], "2-512-512-1": [512, 512]}[name]
    return eh.constructHybridModel(["sw_pot", "dsw_pot"], ["ta"], ["reco"], eh.RbQ10, par, ["rb"], ["Q10"],
                                   hidden_layers=hidden, activation="tanh", scale_nn_outputs=True)


def main():
    ap = argparse.ArgumentParser(description="step time of one wide hidden layer")
    ap.add_argument("steps", nargs="?", type=int, default=512)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        print("gpu:", q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown")
    except (OSError, subprocess.SubprocessError):
        print("gpu: unknown")
    n = 1 << 20
    names = ["2-64-1", "2-512-1", "two-chain 1+2->256+256->2", "2-512-512-1"]
    data = synth(n)
    sessions = {}
    for name in names:
        model = model_of(name)
        xf, y = eh.prepare_data(model, data)
        sess = eh.FusedSession(model, training_loss="mse", agg="sum", opt=eh.Adam(0.001))
        sess.upload(0, xf, y)
        sess.set_params(model.initialparameters(np.random.default_rng(0)))
        sess.set_perm(np.random.default_rng(7).permutation(n))
        sess.run_steps(B, 0, 8)   # warm-up: module load, first launches
        sessions[name] = sess
    for r in range(args.repeats):   # workloads alternate within each repeat
        for name in names:
            sess = sessions[name]
            losses = sess.run_steps(B, 8, args.steps)
            ms, launches, _ = sess.last_timing()
            us = 1e3 * ms / args.steps
            print(f"[{name}] {sess.kernel_variant()}: {args.steps} steps, {us:.1f} us/step, {B / (us * 1e-6):.3e} samples/s, "
                  f"{launches // args.steps} launches/step, loss {losses[0]:.4f} -> {losses[-1]:.4f} (repeat {r})")
    for sess in sessions.values():
        sess.close()


if __name__ == "__main__":
    main()
