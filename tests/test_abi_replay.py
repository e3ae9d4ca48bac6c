"""The drop-in boundary driven FROM C (SURVEY 7.1-9: "a recorded-call C harness").

tests/abi_replay.c replays the call sequence of the reference-side binding (julia/EasyHybridCUDA.jl: eh_create ->
eh_upload -> eh_set_params -> eh_loss_grad -> eh_epoch per epoch -> eh_get_params / eh_get_opt_state -> eh_eval, then
the per-step form eh_step_host on host batches) against include/easyhybrid_cuda.h with plain gcc -- no Python, no
ctypes, no torch between the caller and the library.  The harness writes its inputs and results to files; this test
checks the results against the CPU checker on exactly those inputs.

CPU part: the harness compiles as C against the header, links against the library, and -- with no GPU visible -- fails
loudly instead of falling back."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "easyhybrid.jl_b200")


def _build(tmp_path):
    exe = str(tmp_path / "abi_replay")
    subprocess.check_call(["gcc", "-O1", "-Wall", "-Werror", "-std=c99", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "abi_replay.c"), "-o", exe, "-L", PKG, "-l:libeasyhybrid_cuda.so",
                           "-Wl,-rpath," + PKG, "-lm"])
    return exe


def test_replay_harness_builds_as_c_and_fails_loudly_without_a_gpu(tmp_path):
    exe = _build(tmp_path)
    # the harness sees no device (CUDA_VISIBLE_DEVICES empty), also on a machine that has a GPU
    r = subprocess.run([exe, str(tmp_path / "out")], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 3 and "no CPU fallback" in r.stderr, (r.returncode, r.stderr)


def _parse(path):
    out = {}
    for line in open(path):
        k, *v = line.split()
        out[k] = v[0] if k == "variant" else np.array([float(x) for x in v])
    return out


@pytest.mark.gpu
def test_c_replay_matches_the_checker(tmp_path, eh, orc):
    exe = _build(tmp_path)
    stem = str(tmp_path / "replay")
    r = subprocess.run([exe, stem], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    raw = open(stem + ".bin", "rb").read()
    n, nval, B, nepochs, nflat = np.frombuffer(raw, dtype=np.int64, count=5)
    off = 40
    ntot = n + nval
    X = np.frombuffer(raw, dtype=np.float32, count=2 * ntot, offset=off).reshape(ntot, 2); off += 8 * ntot
    ta = np.frombuffer(raw, dtype=np.float32, count=ntot, offset=off); off += 4 * ntot
    reco = np.frombuffer(raw, dtype=np.float32, count=ntot, offset=off); off += 4 * ntot
    flat0 = np.frombuffer(raw, dtype=np.float32, count=nflat, offset=off).copy(); off += 4 * nflat
    perm = np.frombuffer(raw, dtype=np.int64, count=n * nepochs, offset=off) - 1
    got = _parse(stem + ".txt")
    assert got["variant"].startswith("ffma2/PmRbQ10"), got["variant"]
    assert int(got["nflat"][0]) == nflat

    from conftest import rbq10_model
    model = rbq10_model(eh)
    xf, y = (X[:n], {"ta": ta[:n]}), {"reco": reco[:n]}
    o = orc.Oracle(model, opt=eh.Adam(0.01))
    nt = orc.max_threads()
    # compute_loss + gradient on the first batch
    L64, g64 = o.loss_grad(flat0, xf, y, perm[:B], precision=64, nthreads=nt)
    assert abs(got["loss0"][0] - L64) <= 1e-5 * abs(L64), (got["loss0"], L64)
    assert np.abs(got["grad0"] - g64).max() <= 1e-5 * np.abs(g64).max()
    # run_epoch! twice (a fresh permutation per epoch; the last batch of each epoch is partial)
    ref = flat0.copy()
    want = np.concatenate([o.train_steps(ref, xf, y, perm[e * n:(e + 1) * n], int(B), nthreads=nt) for e in range(nepochs)])
    np.testing.assert_allclose(got["epoch_losses"], want, rtol=1e-4)
    assert int(got["steps"][0]) == len(want)
    assert abs(got["params"][-1] - ref[-1]) <= 1e-4        # phi (Q10 logit); theta is compared through the losses
    # the per-step host-batch form walks the same trajectory
    np.testing.assert_allclose(got["host_losses"], got["epoch_losses"], rtol=2e-6)
    np.testing.assert_allclose(got["host_params"], got["params"], rtol=0, atol=2e-6)
    # evaluate_epoch on the validation split: n valid, SSE (shifted sums, include/easyhybrid_cuda.h EH_EVAL_STATS)
    yv = reco[n:]
    yhat = o.forward(got["params"].astype(np.float32), (X[n:], {"ta": ta[n:]}), precision=64, nthreads=nt)
    yhat = np.asarray(yhat, dtype=np.float64)[0]
    m = ~np.isnan(yv)
    assert int(got["val_stats"][0]) == int(m.sum())
    sse = float(((yhat[m] - yv[m].astype(np.float64)) ** 2).sum())
    assert abs(got["val_stats"][6] - sse) <= 1e-4 * sse, (got["val_stats"], sse)
    np.testing.assert_allclose(got["val_yhat_head"], yhat[:8], rtol=1e-4)
