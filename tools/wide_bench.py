"""C5 workload driver: multi-target Expo hybrid, hidden 3x512, PerTarget(nseLoss, mse), batch 65536 (SURVEY 8d).

usage: wide_bench.py [STEPS] [--loss nseLoss,mse] [--weight-l2 LAMBDA]
--loss: one training loss per target (comma separated), e.g. kgeLoss,mse; --weight-l2: add the extra loss
LAMBDA * weight_l2(ps).  Without them the workload is the C5 one and the printed line is unchanged."""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import easyhybrid_b200 as eh

B = 65536


def synth(n, seed=2314):
    rng = np.random.default_rng(seed)
    T = (rng.random(n, dtype=np.float32) * 40 - 10).astype(np.float32)
    SM = (rng.random(n, dtype=np.float32) * 0.8 + 0.1).astype(np.float32)
    resp = 1.1 * np.exp(-8.0 * (SM - 0.6) ** 2) * np.exp(0.07 * T)
    obs = (resp + rng.standard_normal(n, dtype=np.float32) * 0.05 * resp.mean()).astype(np.float32)
    obs2 = (2.0 * resp + rng.standard_normal(n, dtype=np.float32) * 0.05 * resp.mean()).astype(np.float32)
    return dict(T=T, SM=SM, Resp_obs=obs, Resp_obs2=obs2)


def make_model():
    return eh.constructHybridModel({"Resp0": ["SM"]}, ["T"], ["Resp_obs", "Resp_obs2"], eh.Expo_resp_model2,
                                   dict(k=(0.01, 0.0, 0.2), Resp0=(2.0, 0.0, 8.0)), ["k"],
                                   hidden_layers=[512, 512, 512], activation="tanh", scale_nn_outputs=False)


def main():
    ap = argparse.ArgumentParser(description="C5 step time on the tensor-core path")
    ap.add_argument("steps", nargs="?", type=int, default=32)
    ap.add_argument("--loss", default="nseLoss,mse", help="training loss per target, comma separated")
    ap.add_argument("--weight-l2", type=float, default=0.0, metavar="LAMBDA", help="extra loss LAMBDA * weight_l2(ps)")
    args = ap.parse_args()
    log2n = int(os.environ.get("EH_WIDE_LOG2N", "20"))
    steps = args.steps
    losses_per_target = [x.strip() for x in args.loss.split(",")]
    if len(losses_per_target) not in (1, 2):
        ap.error("--loss: one loss for both targets or one per target")
    training_loss = losses_per_target[0] if len(losses_per_target) == 1 else eh.PerTarget(*losses_per_target)
    extra = eh.WeightL2(args.weight_l2) if args.weight_l2 else None
    default = args.loss == "nseLoss,mse" and not args.weight_l2
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = 1 << log2n
    model = make_model()
    xf, y = eh.prepare_data(model, synth(n, 2314 + rank))
    sess = eh.FusedSession(model, training_loss=training_loss, agg="sum", opt=eh.Adam(0.001), device=local, extra_loss=extra)
    sess.upload(0, xf, y)
    sess.set_params(model.initialparameters(np.random.default_rng(0)))
    if world > 1:
        sess.comm_init(rank, world, dist)
    sess.set_perm(np.random.default_rng(7 + rank).permutation(n))
    if world > 1:
        sess.dp_exchange_batch_stats(B, dist)
        dist.barrier()
    sess.run_steps(B, 0, 4)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    losses = sess.run_steps(B, 4, steps)
    t1 = time.perf_counter()
    ms, launches, _ = sess.last_timing()
    if world > 1:
        import torch
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    flop = 2.0 * 3 * 2 * B * 512 * 512 * world   # 2 hidden matrices x (fwd, bwd-data, wgrad), all ranks
    if rank == 0:
        print(f"wide C5 x{world}: {steps} steps, {1e3 * ms / steps:.1f} us/step (device, max over ranks), "
              f"{world * B * steps / (ms * 1e-3):.3e} samples/s, {flop * steps / (ms * 1e-3) / 1e12:.1f} TFLOP/s in the hidden GEMMs, "
              f"wall {1e3 * (t1 - t0):.1f} ms, loss {losses[0]:.4f} -> {losses[-1]:.4f}"
              + ("" if default else f" [loss {args.loss}" + (f", weight_l2 {args.weight_l2:g}" if args.weight_l2 else "") + "]"))
    sess.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
