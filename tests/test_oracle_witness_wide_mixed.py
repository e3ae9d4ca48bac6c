"""The float64 oracle against the independent torch float64 witness (tests/witness.py) for the shapes of
test_gpu_wide_mixed_chains.py, at small widths: chains that differ in depth (pass-through units in the embedding) or in
activation, with NaN targets, input BatchNorm, PerTarget(nseLoss, mse), kgeLoss, weight_l2 and four chains of depths 1..4
over twelve inputs.  The GPU tests of those shapes trust the oracle; this is the oracle's own check."""
import numpy as np
import pytest

import test_gpu_wide_mixed_chains as mix
from witness import objective

CASES = [
    ("rbq10-depths-2-and-1", lambda eh: mix.m_rbq10(eh, ((6, 5), (4,))), 0.0, "mse", None),
    ("equal-depth-relu-and-tanh-nan", lambda eh: mix.m_rbq10(eh, ((5, 5), (4, 4)), ("relu", "tanh")), 0.05, "mse", None),
    ("depths-3-and-1-tanh-and-sigmoid", lambda eh: mix.m_rbq10(eh, ((6, 6, 6), (4,)), ("tanh", "sigmoid")), 0.0, "mse", None),
    ("expo2-pertarget-bn-depths-2-and-4", lambda eh: mix.m_expo2(eh, ((5, 4), (3, 3, 3, 3))), 0.0, "PT", None),
    ("kge-depths-2-and-1", lambda eh: mix.m_custom(eh, ((6, 5), (4,)), ("relu", "tanh")), 0.0, "kgeLoss", None),
    ("weight-l2-depths-3-and-1", lambda eh: mix.m_custom(eh, ((5, 5, 5), (4,)), ("tanh", "relu")), 0.0, "mse", 0.3),
    ("four-chains-depths-1-to-4", lambda eh: mix.m_four_depths(eh, width=4), 0.03, "mse", None),
]


@pytest.mark.parametrize("name,mk,nan,loss,lam", CASES, ids=[c[0] for c in CASES])
def test_wide_mixed_oracle_vs_autograd(eh, orc, name, mk, nan, loss, lam):
    model = mk(eh)
    if loss == "PT":
        loss = eh.PerTarget("nseLoss", "mse")
    xl = eh.WeightL2(lam=lam) if lam else None
    xf, y = eh.prepare_data(model, mix.table_for(model, 300, nan), drop_missing_rows=False)
    rng = np.random.default_rng(7)
    flat = model.initialparameters(rng)
    flat += (0.05 * rng.standard_normal(flat.size)).astype(np.float32)
    n = xf[0].shape[0]
    idx = rng.permutation(n)[: n - 37]
    o = orc.Oracle(model, training_loss=loss, agg="sum", extra_loss=xl)
    Lw, gw = objective(model, flat, xf, y, idx, training_loss=loss, agg="sum", extra_loss=xl)
    L64, g64 = o.loss_grad(flat, xf, y, idx, precision=64)
    assert L64 == pytest.approx(Lw, rel=1e-10), name
    assert np.abs(g64 - gw).max() <= 1e-9 * np.abs(gw).max(), name
