"""Worker for the data-parallel test of a twelve-input / three-output wide model: `torchrun --nproc-per-node 2
tests/dp_worker_wide_io.py`.

Every rank trains its shard of a MultiNN model of three [128]-unit chains with four predictors each (the fused exact-fp32
kernel k_wide_one) in data-parallel mode; the flat gradient is all-reduced over NVLink peer memory.  Rank 0 checks that
all replicas hold bit-identical parameters, that the first step's loss is the float64 oracle's union-batch loss to 1e-5
and that the per-step losses follow the oracle trained on the union batches."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import easyhybrid_b200 as eh
    from easyhybrid_b200.dp import global_batch_indices
    from oracle import oracle as orc
    import test_gpu_wide_io as wio

    model = wio.m_three_chains(eh, (128,))
    nl, B, steps = 4096, 1024, 8
    shards = [eh.prepare_data(model, wio.table(nl, seed=400 + r)) for r in range(world)]
    perms = [np.random.default_rng(500 + r).permutation(nl) for r in range(world)]
    X = np.concatenate([s[0][0] for s in shards])
    f = {k: np.concatenate([s[0][1][k] for s in shards]) for k in shards[0][0][1]}
    yall = {t: np.concatenate([s[1][t] for s in shards]) for t in model.targets}
    o = orc.Oracle(model, training_loss="mse", opt=eh.Adam(0.001))
    flat = model.initialparameters(np.random.default_rng(6))
    xf, y = shards[rank]
    sess = eh.FusedSession(model, training_loss="mse", opt=eh.Adam(0.001), device=local)
    assert sess.kernel_variant() == "wide/fp32-one-hidden", sess.kernel_variant()
    sess.upload(0, xf, y)
    sess.set_params(flat)
    sess.comm_init(rank, world, dist)
    sess.set_perm(perms[rank])
    sess.dp_exchange_batch_stats(B, dist)
    dist.barrier()
    losses = sess.run_steps(B, 0, steps)
    ps = sess.get_params()
    allps = [None] * world
    dist.all_gather_object(allps, ps.tobytes())
    if rank == 0:
        assert all(b == allps[0] for b in allps), "replicas diverged (twelve inputs, three outputs)"
        gi = global_batch_indices(perms, [nl] * world, B, 0)
        L64, _ = o.loss_grad(flat, (X, f), yall, gi, precision=64)
        assert abs(losses[0] - L64) <= 1e-5 * abs(L64), (losses[0], L64)
        ref = flat.copy()
        want = []
        for s in range(steps):
            gi = global_batch_indices(perms, [nl] * world, B, s % (nl // B))
            want.append(o.train_steps(ref, (X, f), yall, gi, world * B)[0])
        np.testing.assert_allclose(losses, np.array(want), rtol=2e-4)
        np.testing.assert_allclose(ps, ref, rtol=0, atol=2e-4 * max(1.0, float(np.abs(ref).max())))
        print("DP_WIDE_IO_OK", losses[:3], want[:3])
    sess.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
