"""Wide models with 9..12 chain inputs and 3..4 chain outputs (1..4 chains) against the float64 oracle.

Such models need a hidden layer wider than 32 units; narrower ones keep the limits of the exact register-tile kernels
(<= 8 inputs, <= 2 outputs without run-time compilation).  One hidden layer runs on the fused exact-fp32 kernel
k_wide_one at the exact path's tolerances (loss 1e-5 relative, gradient max-abs 1e-5 max|g64|, trajectories 2e-4 per
step); two or more on the bf16 tensor-core path at the tolerances of test_gpu_wide.py (loss 2e-2 relative, per parameter
block cosine >= 0.995 and norm within 3e-2)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import make_synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXACT_LOSS, EXACT_GRAD = 1e-5, 1e-5
BF16_LOSS, COS_MIN, RTOL_NORM = 2e-2, 0.995, 3e-2
ONE, TC = "wide/fp32-one-hidden", "wide/bf16-tcgen05"
PARAMS3 = dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0), alpha=(0.5, -2.0, 2.0))
PARAMS4 = dict(PARAMS3, beta=(0.2, -1.0, 1.0))
Z = ["z%d" % k for k in range(9)]


def custom_pm(*, ta, dsw_pot, rb, Q10, alpha, tref=15.0):
    return {"reco": rb * Q10 ** (0.1 * (ta - tref)) + alpha * np.tanh(0.05 * dsw_pot)}


def four_param_pm(*, ta, dsw_pot, rb, Q10, alpha, beta, tref=15.0):
    return {"reco": rb * Q10 ** (0.1 * (ta - tref)) + alpha * np.tanh(0.05 * dsw_pot) + beta * np.sin(0.1 * ta)}


def table(n, nan_frac=0.0, seed=9):
    """the synthetic RbQ10 table (conftest.make_synth) with the traced models' extra term and nine noise predictors"""
    t = make_synth(n, seed=seed + 33)
    t["reco"] = (t["reco"] + 0.3 * np.tanh(0.05 * t["dsw_pot"]) + 0.1 * np.sin(0.1 * t["ta"])).astype(np.float32)
    rng = np.random.default_rng(seed)
    for k in Z:
        t[k] = rng.standard_normal(n).astype(np.float32)
    if nan_frac:
        t["reco"] = np.where(rng.random(n) < nan_frac, np.nan, t["reco"]).astype(np.float32)
    return t


def m_inputs(eh, n_in, hidden, activation="tanh", bn=False, scale=True):
    """one chain of n_in (10..12) predictors, rb neural, Q10 / alpha global"""
    preds = ["sw_pot", "dsw_pot", "ta"] + Z[: n_in - 3]
    return eh.constructHybridModel(preds, ["ta", "dsw_pot"], ["reco"], custom_pm, PARAMS3, ["rb"], ["Q10", "alpha"],
                                   hidden_layers=list(hidden), activation=activation, scale_nn_outputs=scale, input_batchnorm=bn)


def m_three_neural(eh, hidden):
    """SingleNN: one chain of three predictors predicts rb, Q10 and alpha (three chain outputs)"""
    return eh.constructHybridModel(["sw_pot", "dsw_pot", "ta"], ["ta", "dsw_pot"], ["reco"], custom_pm, PARAMS3,
                                   ["rb", "Q10", "alpha"], [], hidden_layers=list(hidden), activation="tanh",
                                   scale_nn_outputs=True)


def m_twelve_four(eh, hidden, scale=True):
    """SingleNN: twelve predictors, four neural parameters (P = 12, NOUT = 4)"""
    return eh.constructHybridModel(["sw_pot", "dsw_pot", "ta"] + Z, ["ta", "dsw_pot"], ["reco"], four_param_pm, PARAMS4,
                                   ["rb", "Q10", "alpha", "beta"], [], hidden_layers=list(hidden), activation="tanh",
                                   scale_nn_outputs=scale)


def m_three_chains(eh, hidden, activation="tanh"):
    """MultiNN: three chains of four predictors (P = 12, NOUT = 3)"""
    preds = {"rb": ["sw_pot", "dsw_pot", "z0", "z1"], "Q10": ["ta", "z2", "z3", "z4"], "alpha": ["dsw_pot", "z5", "z6", "z7"]}
    return eh.constructHybridModel(preds, ["ta", "dsw_pot"], ["reco"], custom_pm, PARAMS3, [],
                                   hidden_layers={k: list(hidden) for k in preds}, activation=activation, scale_nn_outputs=True)


def m_four_chains(eh, hidden, activation="tanh"):
    """MultiNN: four chains of three predictors with a four-parameter traced model (P = 12, NOUT = 4)"""
    preds = {"rb": ["sw_pot", "dsw_pot", "z0"], "Q10": ["ta", "z1", "z2"], "alpha": ["dsw_pot", "z3", "z4"],
             "beta": ["ta", "z5", "z6"]}
    return eh.constructHybridModel(preds, ["ta", "dsw_pot"], ["reco"], four_param_pm, PARAMS4, [],
                                   hidden_layers={k: list(hidden) for k in preds}, activation=activation, scale_nn_outputs=True)


def _blocks(model):
    """(name, slice) of every parameter block of the flat vector, chain after chain, then phi"""
    out, off = [], 0
    for c, shapes in enumerate(model.layer_shapes()):
        for li, (o, i) in enumerate(shapes):
            out.append((f"c{c}W{li + 1}", slice(off, off + o * i)))
            off += o * i
            out.append((f"c{c}b{li + 1}", slice(off, off + o)))
            off += o
    if model.num_params() > off:
        out.append(("phi", slice(off, model.num_params())))
    return out


def _setup(eh, orc, model, loss="mse", agg="sum", xl=None, opt=None, variant=None, n=2048, nan_frac=0.0, seed=17):
    kw = {} if opt is None else dict(opt=opt)
    xf, y = eh.prepare_data(model, table(n, nan_frac), drop_missing_rows=False)
    rng = np.random.default_rng(seed)
    flat = model.initialparameters(rng)
    flat += (0.05 * rng.standard_normal(flat.size)).astype(np.float32)
    sess = eh.FusedSession(model, training_loss=loss, agg=agg, extra_loss=xl, **kw)
    if variant:
        assert sess.kernel_variant() == variant, sess.kernel_variant()
    sess.upload(0, xf, y)
    sess.set_params(flat)
    return sess, orc.Oracle(model, training_loss=loss, agg=agg, extra_loss=xl, **kw), xf, y, flat, rng


ONE_CASES = [
    ("ten-inputs-256-sigmoid-bn-nse", lambda eh: m_inputs(eh, 10, (256,), "sigmoid", bn=True), "nseLoss", None, 0.0),
    ("twelve-inputs-96-swish-mae", lambda eh: m_inputs(eh, 12, (96,), "swish"), "mae", None, 0.0),
    ("three-neural-128-scale", lambda eh: m_three_neural(eh, (128,)), "mse", None, 0.0),
    ("four-chains-64-nan", lambda eh: m_four_chains(eh, (64,)), "mse", None, 0.04),
    ("four-chains-64-kge", lambda eh: m_four_chains(eh, (64,)), "kgeLoss", None, 0.0),
    ("twelve-inputs-128-weight-l2", lambda eh: m_inputs(eh, 12, (128,)), "mse", dict(lam=0.3), 0.0),
]


@pytest.mark.parametrize("name,mk,loss,l2,nan", ONE_CASES, ids=[c[0] for c in ONE_CASES])
def test_one_hidden_io_loss_grad_against_oracle(eh, orc, name, mk, loss, l2, nan):
    model = mk(eh)
    xl = eh.WeightL2(**l2) if l2 else None
    sess, o, xf, y, flat, rng = _setup(eh, orc, model, loss, xl=xl, variant=ONE, nan_frac=nan)
    n = xf[0].shape[0]
    for B in (n, 517, 12):
        idx = rng.permutation(n)[:B]
        L, g = sess.loss_grad(idx)
        L64, g64 = o.loss_grad(flat, xf, y, idx, precision=64)
        assert abs(L - L64) <= EXACT_LOSS * abs(L64), (name, B, L, L64)
        err = float(np.abs(g.astype(np.float64) - g64).max())
        assert err <= EXACT_GRAD * float(np.abs(g64).max()), (name, B, err / float(np.abs(g64).max()))
    sess.close()


TC_CASES = [
    ("ten-inputs-2x256-tanh-bn", lambda eh: m_inputs(eh, 10, (256, 256), "tanh", bn=True), "mse"),
    ("three-chains-2x128", lambda eh: m_three_chains(eh, (128, 128)), "mse"),
    ("four-chains-3x64-relu-kge", lambda eh: m_four_chains(eh, (64, 64, 64), "relu"), "kgeLoss"),
    ("twelve-inputs-four-outputs-3x512-scale", lambda eh: m_twelve_four(eh, (512, 512, 512)), "mse"),
]


def _check_bf16(eh, orc, model, loss, name):
    sess, o, xf, y, flat, rng = _setup(eh, orc, model, loss, variant=TC, seed=3)
    n = xf[0].shape[0]
    for B in (n, 512, 128):
        idx = rng.permutation(n)[:B]
        L, g = sess.loss_grad(idx)
        L64, g64 = o.loss_grad(flat, xf, y, idx, precision=64)
        assert abs(L - L64) <= BF16_LOSS * abs(L64), (name, B, L, L64)
        for bname, sl in _blocks(model):
            a, b = g[sl].astype(np.float64), g64[sl].astype(np.float64)
            nb = np.linalg.norm(b)
            if nb < 1e-12:
                continue
            cos = float(a @ b / (np.linalg.norm(a) * nb))
            assert cos >= COS_MIN, (name, B, bname, cos)
            assert abs(np.linalg.norm(a) - nb) <= RTOL_NORM * nb, (name, B, bname, np.linalg.norm(a), nb)
    sess.close()


@pytest.mark.parametrize("name,mk,loss", TC_CASES, ids=[c[0] for c in TC_CASES])
def test_tensor_core_io_loss_grad_against_oracle(eh, orc, name, mk, loss):
    _check_bf16(eh, orc, mk(eh), loss, name)


def test_tensor_core_twelve_inputs_without_persistent_gemms(eh, orc, monkeypatch):
    """the non-persistent backward-data GEMM (EH_WIDE_NO_PERSIST=1) computes the 12-input column sums too"""
    monkeypatch.setenv("EH_WIDE_NO_PERSIST", "1")
    _check_bf16(eh, orc, m_three_chains(eh, (128, 128)), "mse", "three-chains-no-persist")


def test_one_hidden_io_adam_trajectory_and_eval(eh, orc):
    """25 Adam steps of the four-chain / four-output model on k_wide_one follow the oracle within 2e-4 per step;
    evaluated predictions and neural parameters match o.forward"""
    model = m_four_chains(eh, (64,))
    sess, o, xf, y, flat, rng = _setup(eh, orc, model, opt=eh.Adam(0.01), variant=ONE, n=4096, nan_frac=0.02, seed=23)
    n, B = xf[0].shape[0], 512
    perm = np.concatenate([rng.permutation(n) for _ in range(4)])[: 25 * B]
    got = sess.epoch(perm, B)
    ref = flat.copy()
    want = o.train_steps(ref, xf, y, perm, B)
    assert got[-1] < got[0], got
    np.testing.assert_allclose(got, want, rtol=2e-4)
    ps = sess.get_params()
    # (Adam moves an entry whose gradient is at noise level by up to eta per step in either direction: the parameters
    # are held to 1e-3, the losses above to 2e-4)
    np.testing.assert_allclose(ps, ref, rtol=0, atol=1e-3 * max(1.0, float(np.abs(ref).max())))
    yhat, stats, par = sess.eval(0, want_yhat=True, want_params=True)
    yo, po = o.forward(ps, xf, precision=64, want_params=True)
    np.testing.assert_allclose(yhat, yo, rtol=2e-5, atol=2e-5 * float(np.abs(yo).max()))
    for name in ("rb", "Q10", "alpha", "beta"):
        k = model.parameters.names.index(name)
        np.testing.assert_allclose(par[k], po[k], rtol=2e-5, atol=2e-5 * float(np.abs(po[k]).max()), err_msg=name)
    sess.close()


def test_tensor_core_io_trajectory_and_eval(eh, orc):
    """30 Adam steps of a ten-input [256, 256] model on the tensor-core path: losses within 5e-2 per step, phi within
    2e-2; evaluated predictions and rb against o.forward"""
    model = m_inputs(eh, 10, (256, 256), "tanh", bn=True)
    sess, o, xf, y, flat, rng = _setup(eh, orc, model, opt=eh.Adam(0.001), variant=TC, n=4096, seed=11)
    n, B = xf[0].shape[0], 1024
    perm = np.concatenate([rng.permutation(n) for _ in range(8)])[: 30 * B]
    got = sess.epoch(perm, B)
    ref = flat.copy()
    want = o.train_steps(ref, xf, y, perm, B)
    assert got[-1] < got[0], got
    assert np.allclose(got, want, rtol=5e-2), (got, want)
    ps = sess.get_params()
    for k in (-1, -2):
        assert abs(float(ps[k]) - float(ref[k])) <= 2e-2 * max(1.0, abs(float(ref[k]))), (k, ps[k], ref[k])
    yhat, _, par = sess.eval(0, want_yhat=True, want_params=True)
    yo, po = o.forward(ps, xf, precision=64, want_params=True)
    assert np.allclose(yhat, yo, rtol=3e-2, atol=3e-2 * float(np.abs(yo).max()))
    rb = model.parameters.names.index("rb")
    assert np.allclose(par[rb], po[rb], rtol=3e-2, atol=3e-2 * float(np.abs(po[rb]).max()))
    sess.close()


@pytest.mark.parametrize("path", ["one-hidden", "tensor-core"])
def test_io_epoch_is_bit_reproducible(eh, path):
    """the same epoch twice: bit-identical losses and parameters"""
    model = m_twelve_four(eh, (256,) if path == "one-hidden" else (256, 256))
    n, B = 3 * 16384, 16384
    xf, y = eh.prepare_data(model, table(n, seed=7))
    flat = model.initialparameters(np.random.default_rng(31))
    perm = np.random.default_rng(32).permutation(n)
    out = []
    for _ in range(2):
        sess = eh.FusedSession(model, training_loss="mse", opt=eh.Adam(0.001))
        assert sess.kernel_variant() == (ONE if path == "one-hidden" else TC)
        sess.upload(0, xf, y)
        sess.set_params(flat)
        losses = sess.epoch(perm, B)
        out.append((losses.tobytes(), sess.get_params().tobytes()))
        sess.close()
    assert out[0] == out[1]


@pytest.mark.parametrize("path", ["one-hidden", "tensor-core"])
def test_io_host_batches_walk_the_resident_epoch(eh, orc, path):
    """ragged host batches (700, 700, 400) through step_host_async give the resident epoch's losses and parameters
    bit for bit"""
    model = m_three_chains(eh, (128,) if path == "one-hidden" else (128, 128))
    sess, _, xf, y, flat, rng = _setup(eh, orc, model, opt=eh.Adam(0.01), variant=ONE if path == "one-hidden" else TC,
                                       n=1800, nan_frac=0.03, seed=29)
    n, B = xf[0].shape[0], 700
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
        hb = sess.host_batch(sess.pinned(xf[0][idx]), [sess.pinned(xf[1][f][idx]) for f in ("ta", "dsw_pot")],
                             [sess.pinned(y["reco"][idx])])
        keep.append(hb)
        sess.step_host_async(hb, losses, k)
    sess.sync()
    np.testing.assert_array_equal(np.asarray(losses), got)
    np.testing.assert_array_equal(sess.get_params(), p_epoch)
    sess.close()


def test_train_api_with_three_wide_chains(eh):
    """train(model, data; ...) with three chains of [128, 128] (twelve inputs): the validation loss falls"""
    model = m_three_chains(eh, (128, 128))
    out = eh.train(model, table(6000), nepochs=10, batchsize=300, opt=eh.Adam(0.003), loss_types=["mse", "r2"])
    assert out is not None and len(out.train_history) == 11
    assert out.val_history[-1]["mse"]["sum"] < out.val_history[0]["mse"]["sum"] * 0.5


def test_io_routing(eh, monkeypatch):
    """9..12 inputs / 3..4 outputs take the wide kernels once a layer is wider than 32; 13 inputs, five outputs and swish
    on two layers are still refused, and so is a narrow three-output model without run-time compilation"""
    cases = [(m_inputs(eh, 10, (256,)), ONE), (m_inputs(eh, 12, (96,), "swish"), ONE), (m_three_neural(eh, (128,)), ONE),
             (m_four_chains(eh, (64,)), ONE), (m_inputs(eh, 10, (256, 256)), TC), (m_three_chains(eh, (128, 128)), TC),
             (m_four_chains(eh, (64, 64, 64), "relu"), TC), (m_twelve_four(eh, (512, 512, 512)), TC)]
    for model, want in cases:
        sess = eh.FusedSession(model)
        assert sess.kernel_variant() == want, (want, sess.kernel_variant())
        sess.close()
    # 13 inputs: four chains of 4 + 3 + 3 + 3
    preds13 = {"rb": ["sw_pot", "dsw_pot", "z0", "z7"], "Q10": ["ta", "z1", "z2"], "alpha": ["dsw_pot", "z3", "z4"],
               "beta": ["ta", "z5", "z6"]}
    m13 = eh.constructHybridModel(preds13, ["ta", "dsw_pot"], ["reco"], four_param_pm, PARAMS4, [],
                                  hidden_layers={k: [64] for k in preds13}, activation="tanh")

    def five_param_pm(*, ta, dsw_pot, rb, Q10, alpha, beta, gamma, tref=15.0):
        return {"reco": rb * Q10 ** (0.1 * (ta - tref)) + alpha * np.tanh(0.05 * dsw_pot) + beta * np.sin(0.1 * ta) + gamma}

    m5 = eh.constructHybridModel(["sw_pot", "dsw_pot", "ta"], ["ta", "dsw_pot"], ["reco"], five_param_pm,
                                 dict(PARAMS4, gamma=(0.0, -1.0, 1.0)), ["rb", "Q10", "alpha", "beta", "gamma"], [],
                                 hidden_layers=[128])
    for bad in (m13, m5, m_inputs(eh, 12, (64, 64), "swish")):
        with pytest.raises(eh.EasyHybridCudaError):
            eh.FusedSession(bad)
    # the three-output [24, 20] model of test_jit.py is still refused without run-time compilation
    monkeypatch.setenv("EH_JIT", "0")
    m24 = eh.constructHybridModel(["sw_pot", "dsw_pot", "ta"], ["ta", "dsw_pot"], ["reco"], custom_pm, PARAMS3,
                                  ["rb", "Q10", "alpha"], [], hidden_layers=[24, 20], activation="tanh",
                                  scale_nn_outputs=True, input_batchnorm=True)
    with pytest.raises(eh.EasyHybridCudaError) as ei:
        eh.FusedSession(m24)
    assert "no fused kernel" in str(ei.value), str(ei.value)


def test_io_data_parallel_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29637", os.path.join(ROOT, "tests", "dp_worker_wide_io.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "DP_WIDE_IO_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
