"""One hidden layer wider than 32 units (33..512, one to four chains) on the fused exact-fp32 kernel k_wide_one against the
float64 oracle.

k_wide_one runs the forward, the loss seeds, the backward and the gradient sums per sample on-chip in fp32 with the exact
path's activation formulas, so the exact path's tolerances apply (DESIGN.md section 8), not the bf16 ones of
test_gpu_wide.py: loss within 1e-5 relative, gradient max-abs error <= 1e-5 max|g64|, trajectories within 2e-4 per step."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import make_expo2, make_synth, rbq10_model, truth_trajectory

pytestmark = pytest.mark.gpu

RTOL_LOSS = 1e-5
RTOL_GRAD = 1e-5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def expo2_one(eh, width, activation="tanh"):
    return eh.constructHybridModel({"Resp0": ["SM"]}, ["T"], ["Resp_obs", "Resp_obs2"], eh.Expo_resp_model2,
                                   dict(k=(0.01, 0.0, 0.2), Resp0=(2.0, 0.0, 8.0)), ["k"],
                                   hidden_layers=[width], activation=activation)


def two_chain(eh, h_rb, h_q10):
    return eh.constructHybridModel({"rb": ["sw_pot", "dsw_pot"], "Q10": ["ta"]}, ["ta"], ["reco"], eh.RbQ10,
                                   dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0)), [],
                                   hidden_layers={"rb": [h_rb], "Q10": [h_q10]}, activation="tanh", scale_nn_outputs=True)


def traced(eh, width):
    def custom(*, ta, dsw_pot, rb, Q10, alpha, tref=15.0):
        return {"reco": rb * Q10 ** (0.1 * (ta - tref)) + alpha * np.tanh(0.05 * dsw_pot)}

    return eh.constructHybridModel(["sw_pot", "dsw_pot"], ["ta", "dsw_pot"], ["reco"], custom,
                                   dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0), alpha=(0.5, -2.0, 2.0)), ["rb"], ["Q10", "alpha"],
                                   hidden_layers=[width], activation="tanh", scale_nn_outputs=True)


def _loss(eh, loss):
    return eh.PerTarget("nseLoss", "mse") if loss == "PT-nse-mse" else loss


# (id, model, data, training loss, agg, extra loss)
CASES = [
    ("rbq10-64-tanh", lambda eh: rbq10_model(eh, hidden=(64,)), lambda: make_synth(2048), "mse", "sum", None),
    ("rbq10-512-sigmoid-scale-bn", lambda eh: rbq10_model(eh, hidden=(512,), activation="sigmoid", bn=True),
     lambda: make_synth(2048), "mse", "sum", None),
    ("rbq10-300-relu", lambda eh: rbq10_model(eh, hidden=(300,), activation="relu"), lambda: make_synth(2048), "mse", "mean", None),
    ("rbq10-96-swish-mae", lambda eh: rbq10_model(eh, hidden=(96,), activation="swish"), lambda: make_synth(2048), "mae", "sum", None),
    ("expo2-256-pertarget-nan", lambda eh: expo2_one(eh, 256), lambda: make_expo2(2048, nan_frac=0.05), "PT-nse-mse", "sum", None),
    ("traced-128", lambda eh: traced(eh, 128), lambda: make_synth(2048), "mse", "sum", None),
    ("two-chain-48-40", lambda eh: two_chain(eh, 48, 40), lambda: make_synth(2048, nan_frac=0.03), "mse", "sum", None),
    ("rbq10-64-kge", lambda eh: rbq10_model(eh, hidden=(64,)), lambda: make_synth(2048), "kgeLoss", "sum", None),
    ("expo2-128-rmse-two-targets", lambda eh: expo2_one(eh, 128), lambda: make_expo2(2048), "rmse", "mean", None),
    ("rbq10-128-weight-l2", lambda eh: rbq10_model(eh, hidden=(128,)), lambda: make_synth(2048), "mse", "sum", dict(lam=0.3)),
]


def _session(eh, orc, model, loss, agg="sum", xl=None, opt=None):
    kw = {} if opt is None else dict(opt=opt)
    sess = eh.FusedSession(model, training_loss=loss, agg=agg, extra_loss=xl, **kw)
    assert sess.kernel_variant() == "wide/fp32-one-hidden", sess.kernel_variant()
    return sess, orc.Oracle(model, training_loss=loss, agg=agg, extra_loss=xl, **kw)


@pytest.mark.parametrize("name,mk,mkdata,loss,agg,l2", CASES, ids=[c[0] for c in CASES])
def test_one_hidden_loss_grad_against_oracle(eh, orc, name, mk, mkdata, loss, agg, l2):
    model = mk(eh)
    loss = _loss(eh, loss)
    xl = eh.WeightL2(**l2) if l2 else None
    xf, y = eh.prepare_data(model, mkdata(), drop_missing_rows=False)
    n = xf[0].shape[0]
    rng = np.random.default_rng(17)
    flat = model.initialparameters(rng)
    flat += (0.05 * rng.standard_normal(flat.size)).astype(np.float32)
    sess, o = _session(eh, orc, model, loss, agg, xl)
    sess.upload(0, xf, y)
    sess.set_params(flat)
    for B in (n, 517, 12):
        idx = rng.permutation(n)[:B]
        L, g = sess.loss_grad(idx)
        L64, g64 = o.loss_grad(flat, xf, y, idx, precision=64)
        assert abs(L - L64) <= RTOL_LOSS * abs(L64), (name, B, L, L64)
        err = float(np.abs(g.astype(np.float64) - g64).max())
        assert err <= RTOL_GRAD * float(np.abs(g64).max()), (name, B, err / float(np.abs(g64).max()))
    sess.close()


def test_one_hidden_adam_trajectory_step_and_eval(eh, orc):
    """25 Adam steps through sess.epoch follow the oracle's own trajectory; one sess.step; then evaluation: predictions,
    neural parameters and metric statistics"""
    model = rbq10_model(eh, hidden=(256,), bn=False)
    n, B = 4096, 512
    xf, y = eh.prepare_data(model, make_synth(n, nan_frac=0.02), drop_missing_rows=False)
    rng = np.random.default_rng(23)
    flat = model.initialparameters(rng)
    sess, o = _session(eh, orc, model, "mse", opt=eh.Adam(0.01))
    sess.upload(0, xf, y)
    sess.set_params(flat)
    perm = np.concatenate([rng.permutation(n) for _ in range(4)])[: 25 * B]
    got = sess.epoch(perm, B)
    ref = flat.copy()
    want = o.train_steps(ref, xf, y, perm, B)
    assert got[-1] < got[0], got
    np.testing.assert_allclose(got, want, rtol=2e-4)
    ps = sess.get_params()
    np.testing.assert_allclose(ps, ref, rtol=0, atol=2e-4 * max(1.0, float(np.abs(ref).max())))
    # one more step on its own
    idx = rng.permutation(n)[:B]
    L = sess.step(idx)
    L64, _ = o.loss_grad(ref, xf, y, idx, precision=64)
    assert abs(L - L64) <= 1e-5 * abs(L64), (L, L64)
    o.train_steps(ref, xf, y, idx, B)
    ps = sess.get_params()
    yhat, stats, par = sess.eval(0, want_yhat=True, want_params=True)
    yo, po = o.forward(ps, xf, precision=64, want_params=True)
    np.testing.assert_allclose(yhat, yo, rtol=2e-5, atol=2e-5 * float(np.abs(yo).max()))
    rb = model.parameters.names.index("rb")
    np.testing.assert_allclose(par[rb], po[rb], rtol=2e-5, atol=2e-5 * float(np.abs(po[rb]).max()))
    yy = y["reco"].astype(np.float64)
    m = ~np.isnan(yy)
    assert stats[0, 0] == m.sum()
    mse = float(np.mean((yo[0][m] - yy[m]) ** 2))
    assert abs(stats[0, 6] / stats[0, 0] - mse) <= 1e-4 * mse, (stats[0, 6] / stats[0, 0], mse)
    sess.close()


def test_one_hidden_epoch_is_bit_reproducible(eh):
    """the same epoch twice at batch 65 536: bit-identical losses and parameters"""
    model = rbq10_model(eh, hidden=(512,))
    n, B = 3 * 65536, 65536
    xf, y = eh.prepare_data(model, make_synth(n, seed=7))
    flat = model.initialparameters(np.random.default_rng(31))
    perm = np.random.default_rng(32).permutation(n)
    out = []
    for _ in range(2):
        sess = eh.FusedSession(model, training_loss="mse", opt=eh.Adam(0.001))
        assert sess.kernel_variant() == "wide/fp32-one-hidden"
        sess.upload(0, xf, y)
        sess.set_params(flat)
        losses = sess.epoch(perm, B)
        out.append((losses.tobytes(), sess.get_params().tobytes()))
        sess.close()
    assert out[0] == out[1]


def test_one_hidden_host_batches_walk_the_resident_epoch(eh, orc):
    """ragged host batches (700, 700, 400) through step_host_async give the resident epoch's losses and parameters"""
    model = rbq10_model(eh, hidden=(128,))
    xf, y = eh.prepare_data(model, make_synth(1800, nan_frac=0.03), drop_missing_rows=False)
    n, B = xf[0].shape[0], 700
    rng = np.random.default_rng(29)
    flat = model.initialparameters(rng)
    sess, _ = _session(eh, orc, model, "mse", opt=eh.Adam(0.01))
    sess.upload(0, xf, y)
    sess.set_params(flat)
    perm = rng.permutation(n)
    got = sess.epoch(perm, B)
    assert got.shape == (3,)
    p_epoch = sess.get_params()
    sess.set_params(flat)
    sess.set_opt_state(None, None, 0)
    losses = sess.pinned(np.zeros(3, dtype=np.float32))
    keep = []
    for k in range(3):
        idx = perm[k * B:(k + 1) * B]
        hb = sess.host_batch(sess.pinned(xf[0][idx]), [sess.pinned(xf[1]["ta"][idx])], [sess.pinned(y["reco"][idx])])
        keep.append(hb)
        sess.step_host_async(hb, losses, k)
    sess.sync()
    np.testing.assert_allclose(np.asarray(losses), got, rtol=1e-5)
    np.testing.assert_allclose(sess.get_params(), p_epoch, rtol=0, atol=1e-5)
    sess.close()


def test_train_api_with_one_wide_hidden_layer(eh):
    """train(model, data; ...) with hidden_layers = [128]: the validation loss falls and Q10 (true value 2) is recovered"""
    model = rbq10_model(eh, hidden=(128,), activation="tanh", bn=True)
    out = eh.train(model, make_synth(6000), nepochs=12, batchsize=300, opt=eh.Adam(0.01), loss_types=["mse", "r2"])
    assert out is not None and len(out.train_history) == 13
    assert out.val_history[-1]["mse"]["sum"] < out.val_history[0]["mse"]["sum"] * 0.1
    assert abs(out.train_diffs["Q10"] - 2.0) < 0.25


def test_one_hidden_routing(eh, monkeypatch):
    """33..512 units in one layer take the fused kernel; 32 keeps its exact register-tile variant; a narrow traced one-layer
    model sent away from the register-tile kernels is still refused; two layers of swish are still refused"""
    for h in (33, 64, 512):
        sess = eh.FusedSession(rbq10_model(eh, hidden=(h,)))
        assert sess.kernel_variant() == "wide/fp32-one-hidden", (h, sess.kernel_variant())
        sess.close()
    sess = eh.FusedSession(rbq10_model(eh, hidden=(32,)))
    assert not sess.kernel_variant().startswith("wide/"), sess.kernel_variant()
    sess.close()
    with pytest.raises(eh.EasyHybridCudaError):
        eh.FusedSession(rbq10_model(eh, hidden=(513,)))
    with pytest.raises(eh.EasyHybridCudaError):
        eh.FusedSession(rbq10_model(eh, hidden=(64, 64), activation="swish"))
    monkeypatch.setenv("EH_NO_SMALL_PROGRAM", "1")
    with pytest.raises(eh.EasyHybridCudaError) as ei:
        eh.FusedSession(traced(eh, 16))
    assert "no fused kernel" in str(ei.value), str(ei.value)


def test_one_hidden_data_parallel_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29631", os.path.join(ROOT, "tests", "dp_worker_one_hidden.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "DP_ONE_HIDDEN_OK" in r.stdout and "DP_ONE_HIDDEN_REFUSALS_OK" in r.stdout, \
        r.stdout[-2000:] + r.stderr[-4000:]
