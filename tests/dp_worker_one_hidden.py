"""Worker for the data-parallel test of one wide hidden layer: `torchrun --nproc-per-node 2 tests/dp_worker_one_hidden.py`.

Every rank trains its shard of a [256]-unit, two-target chain (the fused exact-fp32 kernel k_wide_one) in data-parallel
mode; the flat gradient is all-reduced over NVLink peer memory.  Rank 0 checks that all replicas hold bit-identical
parameters, that the first step's loss is the float64 oracle's union-batch loss to 1e-5 and that the per-step losses
follow the oracle trained on the union batches.  Then both ranks check that kgeLoss and weight_l2 are refused."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def expo2(n, seed):
    rg = np.random.default_rng(seed)
    T = rg.random(n) * 40 - 10
    SM = rg.random(n) * 0.8 + 0.1
    resp = 1.1 * np.exp(-8.0 * (SM - 0.6) ** 2) * np.exp(0.07 * T)
    return {k: v.astype(np.float32) for k, v in dict(
        T=T, SM=SM, Resp_obs=resp + rg.standard_normal(n) * 0.05 * resp.mean(),
        Resp_obs2=2.0 * resp + rg.standard_normal(n) * 0.05 * resp.mean()).items()}


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import easyhybrid_b200 as eh
    from easyhybrid_b200 import _abi
    from easyhybrid_b200.dp import global_batch_indices
    from oracle import oracle as orc

    model = eh.constructHybridModel({"Resp0": ["SM"]}, ["T"], ["Resp_obs", "Resp_obs2"], eh.Expo_resp_model2,
                                    dict(k=(0.01, 0.0, 0.2), Resp0=(2.0, 0.0, 8.0)), ["k"],
                                    hidden_layers=[256], activation="tanh", scale_nn_outputs=False)
    nl, B, steps = 4096, 1024, 8
    shards = [eh.prepare_data(model, expo2(nl, 400 + r)) for r in range(world)]
    perms = [np.random.default_rng(500 + r).permutation(nl) for r in range(world)]
    X = np.concatenate([s[0][0] for s in shards])
    f = {"T": np.concatenate([s[0][1]["T"] for s in shards])}
    yall = {t: np.concatenate([s[1][t] for s in shards]) for t in model.targets}
    loss = eh.PerTarget("nseLoss", "mse")
    o = orc.Oracle(model, training_loss=loss, opt=eh.Adam(0.001))
    flat = model.initialparameters(np.random.default_rng(6))
    xf, y = shards[rank]
    sess = eh.FusedSession(model, training_loss=loss, opt=eh.Adam(0.001), device=local)
    assert sess.kernel_variant().startswith("wide/"), sess.kernel_variant()
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
        assert all(b == allps[0] for b in allps), "replicas diverged (one hidden layer)"
        gi = global_batch_indices(perms, [nl] * world, B, 0)
        L64, g64 = o.loss_grad(flat, (X, f), yall, gi, precision=64)
        assert abs(losses[0] - L64) <= 1e-5 * abs(L64), (losses[0], L64)
        ref = flat.copy()
        want = []
        for s in range(steps):
            gi = global_batch_indices(perms, [nl] * world, B, s % (nl // B))
            want.append(o.train_steps(ref, (X, f), yall, gi, world * B)[0])
        np.testing.assert_allclose(losses, np.array(want), rtol=2e-4)
        assert abs(float(ps[-1]) - float(ref[-1])) <= 2e-4, (ps[-1], ref[-1])
        print("DP_ONE_HIDDEN_OK", losses[:3], want[:3])
    sess.close()
    for what in ("kgeLoss", "weight_l2"):
        if what == "kgeLoss":
            s2 = eh.FusedSession(model, training_loss="kgeLoss", device=local)
        else:
            s2 = eh.FusedSession(model, extra_loss=eh.WeightL2(0.3), device=local)
        try:
            s2.comm_init(rank, world, dist)
            raise AssertionError(f"{what} was accepted in data-parallel mode")
        except eh.EasyHybridCudaError as e:
            assert e.status == _abi.EH_EUNSUPPORTED, str(e)
        s2.close()
    if rank == 0:
        print("DP_ONE_HIDDEN_REFUSALS_OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
