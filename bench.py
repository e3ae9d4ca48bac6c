#!/usr/bin/env python
"""bench.py -- training samples/s of the fused hybrid step (fwd + bwd + optimiser).

Workload (BASELINE.json configs[2], "C3"): RbQ10, MLP [2 -> 16 -> 16 -> 1] tanh,
scale_nn_outputs, global Q10, mse, Adam(0.01), N = 2^24 synthetic Q10-shaped samples resident
in HBM, batch 65536.  A "step" is one optimiser step on one batch.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

value      : samples/s, device-timed (CUDA events on the launching stream inside the library),
             data + index stream already resident in HBM.
e2e        : same metric through the C ABI with HOST batches: every step copies that batch
             (X, forcing, target; pinned host memory) host->device and reads the loss back.
roofline   : algorithmic bytes (16 B/sample) of one fused-step launch / its mean duration
             (per-launch CUDA events in profiling mode) vs the measured HBM peak.
cpu_baseline: the oracle (CPU restatement of the reference algorithm; the reference itself is
             Julia and cannot run in this image) on all host cores, bounded sample.
With --impl reference the same CPU implementation is what is timed.
--dump-outputs DIR: after the K timed steps, DIR/<name>.npy holds what they hand their caller (see dump_outputs);
             the inputs are seeded, so two builds run with the same arguments can be compared output for output.
Multi-GPU (torchrun, one rank per GPU): weak scaling, every rank owns its own 2^24-sample shard
and trains on per-GPU batches of 65536; gradients are combined once per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (the tree may be read-only)

B = 65536
N_PER_GPU = 1 << 24
BYTES_PER_SAMPLE = 16           # 4 (P + F + T) = 4 * (2 + 1 + 1), SURVEY.md section 8(d)
FMA_PER_SAMPLE = 880            # fwd + bwd of [2,16,16,1], SURVEY.md section 7.3


def synth(n, seed):
    rng = np.random.default_rng(seed)
    ta = (10 + 10 * rng.standard_normal(n, dtype=np.float32)).astype(np.float32)
    sw = np.abs(50 + 20 * rng.standard_normal(n, dtype=np.float32)).astype(np.float32)
    dsw = np.empty_like(sw)
    dsw[0] = 0
    dsw[1:] = sw[1:] - sw[:-1]
    rb = 3.0 + 0.02 * (sw - sw.mean())
    reco = (rb * np.exp2(0.1 * (ta - 15.0)) + 0.1 * rng.standard_normal(n, dtype=np.float32)).astype(np.float32)
    return (np.ascontiguousarray(np.stack([sw, dsw], 1)), {"ta": ta}), {"reco": reco}


def traced_model_leg(eh, device, xf, y, n, B):
    """The headline workload with its process model written as a user callable the library has no built-in form for (it is
    traced into a program): per-step time with the program interpreted per sample (compiled-in generic variant) and compiled
    into the kernels at run time (NVRTC; the compilation itself is outside the timed region).  Rank 0, one GPU."""
    def custom(*, ta, rb, Q10, tref=15.0):
        return {"reco": rb * Q10 ** (0.1 * (ta - tref)) + 0.0 * ta}
    model = eh.constructHybridModel(["sw_pot", "dsw_pot"], ["ta"], ["reco"], custom, dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0)),
                                    ["rb"], ["Q10"], hidden_layers=[16, 16], activation="tanh", scale_nn_outputs=True)
    out = {"workload": "C3 with the process model as a traced callable (rb * Q10^(0.1 (ta - 15)) + 0 * ta), batch %d" % B}
    for key, jit in (("interpreted", False), ("compiled_nvrtc", True)):
        t0 = time.perf_counter()
        sess = eh.FusedSession(model, opt=eh.Adam(0.01), device=device, jit=jit)
        t_create = time.perf_counter() - t0
        sess.upload(0, xf, y)
        sess.set_params(model.initialparameters(np.random.default_rng(0)))
        sess.set_perm(np.random.default_rng(7).permutation(n))
        sess.run_steps(B, 0, 32)
        K = 128
        losses = sess.run_steps(B, 32, K)
        ms, _, _ = sess.last_timing()
        out[key] = {"us_per_step": 1e3 * ms / K, "samples_per_s": K * B / (ms * 1e-3), "variant": sess.kernel_variant(),
                    "create_s": round(t_create, 2), "final_loss": float(losses[-1])}
        sess.close()
    return out


def wide_c5_leg(eh, device, rank=0, world=1, dist=None):
    """BASELINE config 5 (reported next to the headline, not instead of it): two-target Expo hybrid, hidden 3 x 512,
    bf16 tcgen05 GEMMs, PerTarget(nseLoss, mse), batch 65536 per GPU; tensor roofline of its hidden GEMMs.  With several
    ranks: data parallel (weak scaling), the 0.5 M-entry gradient all-reduced over NVLink peer memory every step."""
    n = 1 << 20
    rng = np.random.default_rng(2314 + rank)
    T = (rng.random(n, dtype=np.float32) * 40 - 10).astype(np.float32)
    SM = (rng.random(n, dtype=np.float32) * 0.8 + 0.1).astype(np.float32)
    resp = 1.1 * np.exp(-8.0 * (SM - 0.6) ** 2) * np.exp(0.07 * T)
    noise = 0.05 * float(resp.mean())
    data = dict(T=T, SM=SM, Resp_obs=(resp + noise * rng.standard_normal(n, dtype=np.float32)).astype(np.float32),
                Resp_obs2=(2.0 * resp + noise * rng.standard_normal(n, dtype=np.float32)).astype(np.float32))
    model = eh.constructHybridModel({"Resp0": ["SM"]}, ["T"], ["Resp_obs", "Resp_obs2"], eh.Expo_resp_model2,
                                    dict(k=(0.01, 0.0, 0.2), Resp0=(2.0, 0.0, 8.0)), ["k"],
                                    hidden_layers=[512, 512, 512], activation="tanh", scale_nn_outputs=False)
    xf, y = eh.prepare_data(model, data)
    sess = eh.FusedSession(model, training_loss=eh.PerTarget("nseLoss", "mse"), agg="sum", opt=eh.Adam(0.001), device=device)
    sess.upload(0, xf, y)
    sess.set_params(model.initialparameters(np.random.default_rng(0)))
    if world > 1:
        sess.comm_init(rank, world, dist)
    sess.set_perm(np.random.default_rng(7 + rank).permutation(n))
    if world > 1:
        sess.dp_exchange_batch_stats(B, dist)   # nseLoss: SS_tot of the GLOBAL batch
        dist.barrier()
    sess.run_steps(B, 0, 4)
    k = 32
    if world > 1:
        import torch
        dist.barrier()
        torch.cuda.synchronize()
    losses = sess.run_steps(B, 4, k)
    ms, launches, _ = sess.last_timing()
    if world > 1:
        import torch
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    sess.close()
    flop = 2.0 * 3 * 2 * B * 512 * 512 * k  # two 512 x 512 hidden matrices x (forward, backward-data, weight-gradient), per GPU
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("bf16_tflops_sustained", 0) or 0)
    tf = flop / (ms * 1e-3) / 1e12
    return {"workload": f"C5: two-target Expo hybrid [1-512-512-512-1] tanh, PerTarget(nseLoss, mse), Adam, batch 65536 per GPU, {world} GPU(s), N=2^20 per GPU",
            "value": world * k * B / (ms * 1e-3), "unit": "samples/s", "n_gpus": world, "scaling": "weak", "us_per_step": 1e3 * ms / k, "steps": k, "dtype": "bf16 (fp32 accumulate)",
            "gpu_launches_per_step": launches / k,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peak or None, "unit": "TFLOP/s",
                         "frac": (tf / peak) if peak else None,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peak else "unavailable",
                         "flops_counted": "hidden-layer GEMMs only (2 * 3 * 2 * B * 512 * 512 per step), per GPU"},
            "loss_first_last": [float(losses[0]), float(losses[-1])]}


def dump_outputs(d, sess, losses):
    """What the timed steps computed, as a caller of eh_run_steps receives it: the per-step losses of the timed call and,
    after its last step, the trained parameters and the Adam moments (float32, a few KB in all)."""
    os.makedirs(d, exist_ok=True)
    m, v, _ = sess.get_opt_state()
    for name, a in (("losses", losses), ("params", sess.get_params()), ("adam_m", m), ("adam_v", v)):
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float32))


def make_model(eh):
    return eh.constructHybridModel(["sw_pot", "dsw_pot"], ["ta"], ["reco"], eh.RbQ10,
                                   dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0)), ["rb"], ["Q10"],
                                   hidden_layers=[16, 16], activation="tanh", scale_nn_outputs=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, windows):
        """windows: [(t0, t1), ...] -- the timed regions (device-resident leg and the end-to-end legs)"""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()

        def inside(t):
            return any(t0 - 0.02 <= t <= t1 + 0.02 for (t0, t1) in windows)

        for (t, line) in self.rows:
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                if inside(t):
                    sm.append(float(p[0]))
                smax = float(p[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active") and inside(t):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "sampled_over": "the timed regions of the device-resident and end-to-end legs"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """DRAM bytes per optimiser step of the persistent kernel from the ncu capture of the CURRENT kernel
    (profiles/r2_kernel_metrics.json, written by tools/ncu_metrics_to_json.py from `ncu --set full`); None if absent"""
    try:
        m = json.load(open(os.path.join(ROOT, "profiles", "r2_kernel_metrics.json")))["k_epoch"]
        return (float(m["dram_bytes_read"]) + float(m["dram_bytes_write"])) / float(m["steps"]), m
    except (OSError, ValueError, KeyError):
        return None, None


def dp_parity_check(eh, dist, rank, world, local):
    """Outside the timed region: two data-parallel optimiser steps of batch 65536 per GPU on small shards; rank 0 runs
    the CPU oracle (test infrastructure, the checker) on the UNION batches and compares per-step loss (1e-5) and the
    trained Q10 (1e-4); all ranks must hold bit-identical parameters."""
    import hashlib
    n_local = 1 << 17
    model = make_model(eh)
    xf, y = synth(n_local, 9000 + rank)
    flat0 = model.initialparameters(np.random.default_rng(5))
    perm = np.random.default_rng(9100 + rank).permutation(n_local)
    sess = eh.FusedSession(model, opt=eh.Adam(0.01), device=local)
    sess.upload(0, xf, y)
    sess.set_params(flat0)
    sess.comm_init(rank, world, dist)
    sess.set_perm(perm)
    dist.barrier()
    losses = sess.run_steps(B, 0, 2)
    ps = sess.get_params()
    sess.close()
    digests = [None] * world
    dist.all_gather_object(digests, hashlib.sha1(ps.tobytes()).hexdigest())
    out = {"steps": 2, "global_batch": world * B}
    if rank == 0:
        from oracle import oracle as orc
        from easyhybrid_b200.dp import global_batch_indices
        shards = [synth(n_local, 9000 + r) for r in range(world)]
        perms = [np.random.default_rng(9100 + r).permutation(n_local) for r in range(world)]
        Xall = np.concatenate([sh[0][0] for sh in shards])
        fall = {"ta": np.concatenate([sh[0][1]["ta"] for sh in shards])}
        yall = {"reco": np.concatenate([sh[1]["reco"] for sh in shards])}
        o = orc.Oracle(model, opt=eh.Adam(0.01))
        ref = flat0.copy()
        want = []
        threads = max(orc.max_threads(), len(os.sched_getaffinity(0)))
        for k in range(2):
            gi = global_batch_indices(perms, [n_local] * world, B, k)
            L, g = o.loss_grad(ref, (Xall, fall), yall, gi, precision=64, nthreads=threads)
            want.append(L)
            o.opt_step(ref, g.astype(np.float32))
        rel = float(np.max(np.abs(np.asarray(losses, dtype=np.float64) - np.array(want)) / np.abs(want)))
        q10 = lambda p: 1.0 + 3.0 / (1.0 + np.exp(-float(p[-1])))
        dq = abs(q10(ps) - q10(ref)) / q10(ref)
        same = all(d == digests[0] for d in digests)
        out.update({"ok": bool(rel <= 1e-5 and dq <= 1e-4 and same), "max_rel_loss_err": rel, "q10_rel_err": float(dq),
                    "replicas_bit_identical": bool(same), "checker": "float64 oracle on the union batches (rank 0)"})
    return out


def strong_scaling_leg(eh, dist, rank, world, local, K):
    """SURVEY 8(d) C4, second reading: GLOBAL batch 65536 (strong scaling): every rank trains on 65536 / world samples per
    step; reported next to the weak-scaling headline."""
    import torch
    Bl = B // world
    n = 1 << 22
    model = make_model(eh)
    xf, y = synth(n, 4200 + rank)
    sess = eh.FusedSession(model, opt=eh.Adam(0.01), device=local)
    sess.upload(0, xf, y)
    sess.set_params(model.initialparameters(np.random.default_rng(0)))
    sess.comm_init(rank, world, dist)
    sess.set_perm(np.random.default_rng(77 + rank).permutation(n))
    sess.run_steps(Bl, 0, 8)
    dist.barrier()
    torch.cuda.synchronize()
    sess.run_steps(Bl, 8, K)
    ms, _, _ = sess.last_timing()
    t = torch.tensor([ms], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    sess.close()
    return {"scaling": "strong", "global_batch": B, "per_gpu_batch": Bl, "n_gpus": world, "steps": K,
            "value": K * B / (ms * 1e-3), "unit": "samples/s", "us_per_step": 1e3 * ms / K}


def cpu_baseline(eh, model, seconds=12.0, max_steps=4000):
    """oracle on all host cores, bounded sample of the same workload (batch 65536 out of 2^22 samples)"""
    from oracle import oracle as orc
    n = 1 << 22
    xf, y = synth(n, 1234)
    o = orc.Oracle(model, opt=eh.Adam(0.01))
    flat = model.initialparameters(np.random.default_rng(0))
    rng = np.random.default_rng(1)
    # all host cores: torchrun exports OMP_NUM_THREADS=1 to its workers, which would silently make this a 1-core number
    threads = max(orc.max_threads(), len(os.sched_getaffinity(0)))
    o.train_steps(flat, xf, y, rng.permutation(n)[: 2 * B], B, nthreads=threads)  # warm-up
    steps, t0 = 0, time.perf_counter()
    while steps < max_steps and time.perf_counter() - t0 < seconds:
        k = 4
        o.train_steps(flat, xf, y, rng.permutation(n)[: k * B], B, nthreads=threads)
        steps += k
    dt = time.perf_counter() - t0
    return {"value": steps * B / dt, "unit": "samples/s", "cores": threads, "kind": "port",
            "sample": f"{steps} steps of batch {B} drawn from 2^22 synthetic samples, {dt:.1f} s, "
                      "C oracle (CPU restatement of the reference algorithm; Julia reference not runnable here)"}, steps, dt


def run_reference(args):
    import easyhybrid_b200 as eh
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model = make_model(eh)
    cb, steps, dt = cpu_baseline(eh, model, seconds=max(5.0, min(60.0, 0.5 * (args.steps + args.warmup))),
                                 max_steps=max(8, args.steps))
    line = {"impl": "reference", "metric": "training samples/sec (fwd+bwd+Adam)", "value": cb["value"],
            "unit": "samples/s", "n_gpus": args.gpus, "steps": steps, "warmup": 2, "ms_per_step": 1e3 * dt / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C3: RbQ10 [2-16-16-1] tanh, mse, Adam(0.01), batch 65536 (CPU: bounded sample of 2^22)"},
            "cpu_baseline": cb, "gpu_launches": 0,
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=256)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--n", type=int, default=N_PER_GPU)
    ap.add_argument("--no-wide", action="store_true", help="skip the extra C5 (wide MLP, tcgen05) leg")
    ap.add_argument("--flags", type=int, default=0, help="EH_FLAG_* bits (1 = no CUDA graph, 2 = no PDL)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the timed steps to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_
        torch.cuda.set_device(local)
        # torch.distributed is plumbing only (IPC-handle exchange, barriers, max over ranks);
        # the per-step gradient exchange is the library's own NVLink peer-memory kernel
        dist_.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_

    import easyhybrid_b200 as eh
    W = max(args.warmup, 3)
    K = args.steps
    model = make_model(eh)
    n = args.n
    xf, y = synth(n, 42 + rank)
    sess = eh.FusedSession(model, opt=eh.Adam(0.01), device=local, flags=args.flags)
    sess.upload(0, xf, y)
    flat = model.initialparameters(np.random.default_rng(0))
    sess.set_params(flat)
    if world > 1:
        sess.comm_init(rank, world, dist)
    perm = np.random.default_rng(7 + rank).permutation(n)
    sess.set_perm(perm)
    nb = n // B

    def barrier():
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident throughput ("value") ----
    sess.run_steps(B, 0, W)
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.1)
    barrier()
    t0 = time.perf_counter()
    losses = sess.run_steps(B, W, K)
    t1 = time.perf_counter()
    barrier()
    windows = [(t0, t1)]
    dev_ms, launches, _ = sess.last_timing()
    if dist is not None:
        import torch
        t = torch.tensor([dev_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
    value = world * K * B / (dev_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sess, losses)

    # ---- roofline of the dominant kernel ----
    # The timed region is ONE launch of the persistent kernel k_epoch (all K steps, exchange included):
    # algorithmic bytes of that launch = K * B * 16 B per GPU, duration = the CUDA-event time above.
    peak, peak_src = measured_peaks()
    traffic_per_step, traffic_meta = measured_traffic()
    per_gpu_sps = K * B / (dev_ms * 1e-3)
    achieved = per_gpu_sps * BYTES_PER_SAMPLE / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                # dram__bytes_read + write of k_epoch per step from the ncu --set full capture of the current kernel
                # (profiles/r2_kernel_metrics.json), scaled to this launch's K steps; None when the capture is absent
                "traffic": (traffic_per_step * K) if traffic_per_step is not None else None,
                "traffic_source": ("profiles/r2_kernel_metrics.json (ncu --set full, git %s, %s steps)" % (traffic_meta.get("git"), traffic_meta.get("steps"))) if traffic_meta else None,
                "traffic_algorithmic": float(K) * B * BYTES_PER_SAMPLE,
                "peak_source": peak_src,
                "kernel": "k_epoch (persistent: fused fwd+process+loss+bwd, grid exchange, Adam; one launch = K steps)",
                "kernel_us_per_step": 1e3 * dev_ms / K,
                "binding_roof": {"name": "fp32 issue / shared-memory operand bandwidth (see DESIGN.md section 4)",
                                 "fma_per_sample": FMA_PER_SAMPLE,
                                 "achieved_tfma_s": per_gpu_sps * FMA_PER_SAMPLE / 1e12,
                                 "peak_tfma_s": 148 * 128 * 1.965e9 / 1e12}}
    if world == 1:
        # the one-launch-per-step form of the same computation (k_step), per-launch CUDA events
        sess.set_profiling(True)
        kp = min(K, 256)
        sess.run_steps(B, 0, 8)
        sess.run_steps(B, 8, kp)
        _, _, k1_ms = sess.last_timing()
        sess.set_profiling(False)
        roofline["k_step_us_per_launch"] = 1e3 * k1_ms / kp

    # ---- end to end through the C ABI with host batches ----
    e2e = None
    if not args.no_e2e:
        pool = 16
        hb = []
        for i in range(pool):
            sl = slice(i * B, (i + 1) * B)
            hb.append(sess.host_batch(sess.pinned(xf[0][sl]), [sess.pinned(xf[1]["ta"][sl])], [sess.pinned(y["reco"][sl])]))
        ke = min(K, 2048)
        el = sess.pinned(np.zeros(ke + 8, dtype=np.float32))
        for i in range(8):
            sess.step_host_async(hb[i % pool], el, i)
        sess.sync()
        barrier()
        te0 = time.perf_counter()
        for i in range(ke):
            sess.step_host_async(hb[i % pool], el, i)
        sess.sync()
        te1 = time.perf_counter()
        barrier()
        windows.append((te0, te1))
        dt = te1 - te0
        if dist is not None:
            import torch
            t = torch.tensor([dt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": world * ke * B / dt, "unit": "samples/s", "h2d_bytes_per_step": B * BYTES_PER_SAMPLE,
               "d2h_bytes_per_step": 4, "steps": ke, "api": "eh_step_host_async + eh_sync (page-locked host batches are read in place over PCIe by the packer kernel on four streams; every 16 batches one persistent launch runs their 16 optimiser steps; losses land in page-locked host memory)"}
        # the path train() takes: dataset staged once, every epoch call ships the host permutation (8 B/sample)
        # host->device and the per-step losses back
        kr = min(K, nb)
        perm_pinned = sess.pinned(perm[: kr * B].astype(np.int64) + 1)  # the host's 1-based permutation, page-locked
        sess.epoch(perm_pinned[: 4 * B], B, one_based=True)
        sess.epoch(perm_pinned, B, one_based=True)
        barrier()
        tr0 = time.perf_counter()
        reps = max(1, min(8, K // kr))
        for _ in range(reps):
            sess.epoch(perm_pinned, B, one_based=True)
        tr1 = time.perf_counter()
        barrier()
        windows.append((tr0, tr1))
        dtr = tr1 - tr0
        if dist is not None:
            import torch
            t = torch.tensor([dtr], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtr = float(t.item())
        e2e["resident_dataset"] = {"value": world * reps * kr * B / dtr, "unit": "samples/s",
                                   "h2d_bytes_per_step": 8 * B, "d2h_bytes_per_step": 4, "steps": reps * kr,
                                   "api": "eh_epoch(page-locked host permutation, streamed in segments behind the training) on the dataset staged once by eh_upload"}

    clocks = sampler.stop(windows)
    wide = None
    if not args.no_wide:
        try:
            wide = wide_c5_leg(eh, local, rank, world, dist)
        except Exception as e:  # the extra leg must never take the headline line down
            wide = {"error": str(e)[:200]}
    traced = None
    if not args.no_wide and rank == 0 and world == 1:
        try:
            traced = traced_model_leg(eh, local, xf, y, n, B)
        except Exception as e:
            traced = {"error": str(e)[:200]}
    dp_parity = strong = None
    if os.environ.get("EH_BENCH_DEBUG"):
        print("[bench] rank %d: headline + e2e + wide legs done" % rank, file=sys.stderr, flush=True)
    if world > 1:
        try:
            dp_parity = dp_parity_check(eh, dist, rank, world, local)
        except Exception as e:
            dp_parity = {"ok": False, "error": str(e)[:200]}
        try:
            strong = strong_scaling_leg(eh, dist, rank, world, local, K)
        except Exception as e:
            strong = {"error": str(e)[:200]}

    if rank == 0:
        line = {"metric": "training samples/sec (fwd+bwd+Adam)", "value": value, "unit": "samples/s", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "C3: RbQ10 [2-16-16-1] tanh, scale_nn_outputs, mse, Adam(0.01), "
                                       f"N=2^{int(np.log2(n))} per GPU resident, batch {B} per GPU",
                           "l2": "inputs larger than L2 (268 MB of records gathered through a random permutation)",
                           "parallelism": f"dp{world}"},
                "roofline": roofline, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
                "final_loss": float(losses[-1])}
        if wide is not None:
            line["extra"] = {"c5_wide_mlp": wide}
        if traced is not None:
            line.setdefault("extra", {})["traced_process_model"] = traced
        if dp_parity is not None:
            line["dp_parity_ok"] = bool(dp_parity.get("ok", False))
            line["dp_parity"] = dp_parity
        if strong is not None:
            line.setdefault("extra", {})["c4_strong_scaling"] = strong
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(eh, model)[0]
        out = json.dumps(line)
        if os.environ.get("EH_BENCH_DEBUG"):
            print("[bench] rank 0 writes %d bytes to fd %d (isatty %s)" % (len(out), sys.stdout.fileno(), sys.stdout.isatty()), file=sys.stderr, flush=True)
        print(out, flush=True)   # (flushed here: a block-buffered line was lost at interpreter exit under torchrun)
    sess.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
