"""Worker for the data-parallel test of a wide model whose chains differ in depth and activation: `torchrun
--nproc-per-node 2 tests/dp_worker_wide_mixed.py`.

Every rank trains its shard of a MultiNN model (rb: [256, 256] relu, Q10: [64] tanh, alpha global) on the bf16
tensor-core path in its per-unit form; the flat gradient is all-reduced over NVLink peer memory.  Rank 0 checks that all
replicas hold bit-identical parameters and that the per-step losses follow the float64 oracle trained on the union
batches at the bf16 tolerance (5e-2 per step)."""
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
    import test_gpu_wide_mixed_chains as mix

    model = mix.m_custom(eh, ((256, 256), (64,)), ("relu", "tanh"))
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
    assert sess.kernel_variant() == mix.PU, sess.kernel_variant()
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
        assert all(b == allps[0] for b in allps), "replicas diverged (chains of different depth and activation)"
        ref = flat.copy()
        want = []
        for s in range(steps):
            gi = global_batch_indices(perms, [nl] * world, B, s % (nl // B))
            want.append(o.train_steps(ref, (X, f), yall, gi, world * B)[0])
        np.testing.assert_allclose(losses, np.array(want), rtol=5e-2)
        print("DP_WIDE_MIXED_OK", losses[:3], want[:3])
    sess.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
