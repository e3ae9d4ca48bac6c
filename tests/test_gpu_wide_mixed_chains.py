"""MultiNN models whose chains differ in depth or activation, with some layer wider than 32 units, on the bf16 tensor-core
path (variant wide/bf16-tcgen05-per-unit) against the float64 oracle.

A chain of depth d_k < NH carries its last hidden layer up to layer NH on pass-through units (weight 1 from the unit below,
bias 0, identity activation: exact in bf16); every hidden unit has its own activation.  Tolerances are those of
test_gpu_wide.py: loss 2e-2 relative, per parameter block cosine >= 0.995 and norm within 3e-2."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import make_expo2
import test_gpu_wide_io as wio

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF16_LOSS, COS_MIN, RTOL_NORM = 2e-2, 0.995, 3e-2
PU, TC = "wide/bf16-tcgen05-per-unit", "wide/bf16-tcgen05"
RBQ10 = dict(rb=(3.0, 0.0, 13.0), Q10=(2.0, 1.0, 4.0))


def m_rbq10(eh, hidden, acts=("tanh", "tanh")):
    """RbQ10 with one chain per parameter: rb over (sw_pot, dsw_pot), Q10 over ta"""
    return eh.constructHybridModel({"rb": ["sw_pot", "dsw_pot"], "Q10": ["ta"]}, ["ta"], ["reco"], eh.RbQ10, RBQ10, [],
                                   hidden_layers={"rb": list(hidden[0]), "Q10": list(hidden[1])},
                                   activation={"rb": acts[0], "Q10": acts[1]}, scale_nn_outputs=True)


def m_custom(eh, hidden, acts=("tanh", "relu"), bn=False):
    """the traced custom_pm of test_gpu_wide_io.py: rb and Q10 from their own chains, alpha global"""
    return eh.constructHybridModel({"rb": ["sw_pot", "dsw_pot"], "Q10": ["ta", "sw_pot"]}, ["ta", "dsw_pot"], ["reco"],
                                   wio.custom_pm, wio.PARAMS3, ["alpha"],
                                   hidden_layers={"rb": list(hidden[0]), "Q10": list(hidden[1])},
                                   activation={"rb": acts[0], "Q10": acts[1]}, scale_nn_outputs=True, input_batchnorm=bn)


def m_expo2(eh, hidden=((128, 128), (64, 64, 64, 64)), bn=True):
    """Expo with two targets, Resp0 and k each from a chain (depths 2 and 4), input BatchNorm"""
    return eh.constructHybridModel({"Resp0": ["SM"], "k": ["SM", "T"]}, ["T"], ["Resp_obs", "Resp_obs2"], eh.Expo_resp_model2,
                                   dict(k=(0.01, 0.0, 0.2), Resp0=(2.0, 0.0, 8.0)), [],
                                   hidden_layers={"Resp0": list(hidden[0]), "k": list(hidden[1])},
                                   activation={"Resp0": "tanh", "k": "sigmoid"}, scale_nn_outputs=True, input_batchnorm=bn)


def m_four_depths(eh, width=64):
    """four chains of three predictors and depths 1, 2, 3, 4 feeding a traced four-parameter model (P = 12, NOUT = 4)"""
    preds = {"rb": ["sw_pot", "dsw_pot", "z0"], "Q10": ["ta", "z1", "z2"], "alpha": ["dsw_pot", "z3", "z4"],
             "beta": ["ta", "z5", "z6"]}
    hidden = {k: [width] * (d + 1) for d, k in enumerate(preds)}
    acts = {"rb": "relu", "Q10": "tanh", "alpha": "sigmoid", "beta": "tanh"}
    return eh.constructHybridModel(preds, ["ta", "dsw_pot"], ["reco"], wio.four_param_pm, wio.PARAMS4, [],
                                   hidden_layers=hidden, activation=acts, scale_nn_outputs=True)


def table_for(model, n, nan_frac=0.0):
    """the Expo table for the Expo models, else the RbQ10 table with the traced models' extra columns"""
    return make_expo2(n, nan_frac=nan_frac) if "Resp_obs" in model.targets else wio.table(n, nan_frac)


def _setup(eh, orc, model, loss="mse", xl=None, opt=None, n=2048, nan_frac=0.0, seed=3):
    kw = {} if opt is None else dict(opt=opt)
    xf, y = eh.prepare_data(model, table_for(model, n, nan_frac), drop_missing_rows=False)
    rng = np.random.default_rng(seed)
    flat = model.initialparameters(rng)
    flat += (0.05 * rng.standard_normal(flat.size)).astype(np.float32)
    sess = eh.FusedSession(model, training_loss=loss, extra_loss=xl, **kw)
    assert sess.kernel_variant() == PU, sess.kernel_variant()
    sess.upload(0, xf, y)
    sess.set_params(flat)
    return sess, orc.Oracle(model, training_loss=loss, extra_loss=xl, **kw), xf, y, flat, rng


def _check_bf16(eh, orc, model, loss, name, xl=None, nan_frac=0.0):
    sess, o, xf, y, flat, rng = _setup(eh, orc, model, loss, xl=xl, nan_frac=nan_frac)
    n = xf[0].shape[0]
    for B in (n, 512, 128):
        idx = rng.permutation(n)[:B]
        L, g = sess.loss_grad(idx)
        L64, g64 = o.loss_grad(flat, xf, y, idx, precision=64)
        assert abs(L - L64) <= BF16_LOSS * abs(L64), (name, B, L, L64)
        for bname, sl in wio._blocks(model):
            a, b = g[sl].astype(np.float64), g64[sl].astype(np.float64)
            nb = np.linalg.norm(b)
            if nb < 1e-12:
                continue
            cos = float(a @ b / (np.linalg.norm(a) * nb))
            assert cos >= COS_MIN, (name, B, bname, cos)
            assert abs(np.linalg.norm(a) - nb) <= RTOL_NORM * nb, (name, B, bname, np.linalg.norm(a), nb)
    sess.close()


CASES = [
    # depths 2 and 1: Q10's 64 units ride on pass-through units in layer 2
    ("rbq10-2x256-tanh-and-64-tanh", lambda eh: m_rbq10(eh, ((256, 256), (64,))), "mse", None, 0.0),
    ("equal-depth-relu-and-tanh-nan", lambda eh: m_rbq10(eh, ((128, 128), (128, 128)), ("relu", "tanh")), "mse", None, 0.05),
    # layers 2 and 3 hold 384 + 128 pass-through units = 512, the width limit
    ("3x384-tanh-and-128-sigmoid", lambda eh: m_rbq10(eh, ((384, 384, 384), (128,)), ("tanh", "sigmoid")), "mse", None, 0.0),
    ("expo2-pertarget-bn-depths-2-and-4", m_expo2, "PT", None, 0.0),
    ("kge-depths-2-and-1", lambda eh: m_custom(eh, ((256, 256), (64,)), ("relu", "tanh")), "kgeLoss", None, 0.0),
    ("weight-l2-depths-3-and-1", lambda eh: m_custom(eh, ((128, 128, 128), (96,)), ("tanh", "relu")), "mse", dict(lam=0.3), 0.0),
    ("traced-four-chains-depths-1-to-4", m_four_depths, "mse", None, 0.0),
]


@pytest.mark.parametrize("name,mk,loss,l2,nan", CASES, ids=[c[0] for c in CASES])
def test_mixed_chains_loss_grad_against_oracle(eh, orc, name, mk, loss, l2, nan):
    if loss == "PT":
        loss = eh.PerTarget("nseLoss", "mse")
    _check_bf16(eh, orc, mk(eh), loss, name, xl=eh.WeightL2(**l2) if l2 else None, nan_frac=nan)


def test_mixed_chains_without_persistent_gemms(eh, orc, monkeypatch):
    """the non-persistent forward / backward-data GEMMs (EH_WIDE_NO_PERSIST=1) take the per-unit activations too, the
    twelve-input layer-1 column sums included"""
    monkeypatch.setenv("EH_WIDE_NO_PERSIST", "1")
    _check_bf16(eh, orc, m_four_depths(eh), "mse", "four-depths-no-persist")


def test_mixed_chains_trajectory_and_eval(eh, orc):
    """30 Adam steps of a model with chains of depth 2 (relu) and 1 (tanh): losses within 5e-2 per step, phi within
    2e-2; evaluated predictions and rb against o.forward"""
    model = m_custom(eh, ((256, 256), (64,)), ("relu", "tanh"), bn=True)
    sess, o, xf, y, flat, rng = _setup(eh, orc, model, opt=eh.Adam(0.001), n=4096, seed=11)
    n, B = xf[0].shape[0], 1024
    perm = np.concatenate([rng.permutation(n) for _ in range(8)])[: 30 * B]
    got = sess.epoch(perm, B)
    ref = flat.copy()
    want = o.train_steps(ref, xf, y, perm, B)
    assert got[-1] < got[0], got
    assert np.allclose(got, want, rtol=5e-2), (got, want)
    ps = sess.get_params()
    assert abs(float(ps[-1]) - float(ref[-1])) <= 2e-2 * max(1.0, abs(float(ref[-1]))), (ps[-1], ref[-1])
    yhat, _, par = sess.eval(0, want_yhat=True, want_params=True)
    yo, po = o.forward(ps, xf, precision=64, want_params=True)
    assert np.allclose(yhat, yo, rtol=3e-2, atol=3e-2 * float(np.abs(yo).max()))
    rb = model.parameters.names.index("rb")
    assert np.allclose(par[rb], po[rb], rtol=3e-2, atol=3e-2 * float(np.abs(po[rb]).max()))
    sess.close()


def test_mixed_chains_epoch_is_bit_reproducible(eh):
    """the same epoch twice: bit-identical losses and parameters"""
    model = m_four_depths(eh)
    n, B = 3 * 16384, 16384
    xf, y = eh.prepare_data(model, wio.table(n, seed=7))
    flat = model.initialparameters(np.random.default_rng(31))
    perm = np.random.default_rng(32).permutation(n)
    out = []
    for _ in range(2):
        sess = eh.FusedSession(model, training_loss="mse", opt=eh.Adam(0.001))
        assert sess.kernel_variant() == PU
        sess.upload(0, xf, y)
        sess.set_params(flat)
        losses = sess.epoch(perm, B)
        out.append((losses.tobytes(), sess.get_params().tobytes()))
        sess.close()
    assert out[0] == out[1]


def test_mixed_chains_host_batches_walk_the_resident_epoch(eh, orc):
    """ragged host batches (700, 700, 400) through step_host_async give the resident epoch's losses and parameters
    bit for bit"""
    model = m_custom(eh, ((128, 128, 128), (96,)), ("tanh", "sigmoid"))
    sess, _, xf, y, flat, rng = _setup(eh, orc, model, opt=eh.Adam(0.01), n=1800, nan_frac=0.03, seed=29)
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


def test_train_api_with_per_parameter_hidden_layers_and_activation(eh):
    """train(model, data; ...) with hidden_layers / activation dicts (rb [128, 128] tanh, Q10 [64] sigmoid): the
    validation loss falls"""
    model = m_custom(eh, ((128, 128), (64,)), ("tanh", "sigmoid"), bn=True)
    out = eh.train(model, wio.table(6000), nepochs=10, batchsize=300, opt=eh.Adam(0.003), loss_types=["mse", "r2"])
    assert out is not None and len(out.train_history) == 11
    assert out.val_history[-1]["mse"]["sum"] < out.val_history[0]["mse"]["sum"] * 0.5


def test_mixed_chains_routing(eh, monkeypatch):
    """chains that differ in depth or activation take the per-unit form once a layer is wider than 32 units; equal
    chains keep wide/bf16-tcgen05; swish, one hidden layer, different input_batchnorm, a layer over 512 units with
    pass-through units, and narrow models without run-time compilation are still refused"""
    for _, mk, _, _, _ in CASES:
        sess = eh.FusedSession(mk(eh))
        assert sess.kernel_variant() == PU, sess.kernel_variant()
        sess.close()
    for model in (m_rbq10(eh, ((128, 128), (128, 128))), m_custom(eh, ((256, 256), (64, 64)), ("tanh", "tanh"))):
        sess = eh.FusedSession(model)
        assert sess.kernel_variant() == TC, sess.kernel_variant()
        sess.close()
    bn_mixed = m_custom(eh, ((128, 128), (64,)), ("tanh", "relu"))
    bn_mixed.chains[1]["input_batchnorm"] = True
    refused = [
        (m_custom(eh, ((128, 128), (64,)), ("tanh", "swish")), "no fused kernel"),
        (m_custom(eh, ((128, 128), (64, 64)), ("swish", "swish")), "no fused kernel"),
        (m_custom(eh, ((64,), (64,)), ("tanh", "relu")), "no fused kernel"),
        (bn_mixed, "input_batchnorm"),
        (m_rbq10(eh, ((256, 448), (128,))), "no fused kernel"),   # layer 2: 448 + 128 pass-through units
    ]
    for model, msg in refused:
        with pytest.raises(eh.EasyHybridCudaError) as ei:
            eh.FusedSession(model)
        assert msg in str(ei.value), str(ei.value)
    # narrow chains (every layer <= 32) keep the exact-fp32 route and its refusal without run-time compilation
    monkeypatch.setenv("EH_JIT", "0")
    with pytest.raises(eh.EasyHybridCudaError) as ei:
        eh.FusedSession(m_custom(eh, ((16, 12), (8,)), ("relu", "tanh")))
    assert "run-time compilation" in str(ei.value), str(ei.value)


def test_mixed_chains_data_parallel_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29641", os.path.join(ROOT, "tests", "dp_worker_wide_mixed.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "DP_WIDE_MIXED_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
