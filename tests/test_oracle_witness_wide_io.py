"""The float64 oracle against the independent torch float64 witness (tests/witness.py) for the shapes of
test_gpu_wide_io.py that no other witness test covers: twelve chain inputs over four chains with four chain outputs, and
one chain with three outputs.  The GPU tests of those shapes trust the oracle; this is the oracle's own check."""
import numpy as np
import pytest

import test_gpu_wide_io as wio
from witness import objective

CASES = [
    ("four-chains-twelve-inputs-nan", lambda eh: wio.m_four_chains(eh, (6,)), 0.05, "mse"),
    ("four-chains-twelve-inputs-two-layers-kge", lambda eh: wio.m_four_chains(eh, (5, 4), "relu"), 0.0, "kgeLoss"),
    ("three-outputs-one-chain", lambda eh: wio.m_three_neural(eh, (7,)), 0.03, "mse"),
    ("twelve-inputs-four-outputs", lambda eh: wio.m_twelve_four(eh, (6, 5)), 0.0, "mae"),
]


@pytest.mark.parametrize("name,mk,nan,loss", CASES, ids=[c[0] for c in CASES])
def test_wide_io_oracle_vs_autograd(eh, orc, name, mk, nan, loss):
    model = mk(eh)
    xf, y = eh.prepare_data(model, wio.table(300, nan), drop_missing_rows=False)
    rng = np.random.default_rng(7)
    flat = model.initialparameters(rng)
    flat += (0.05 * rng.standard_normal(flat.size)).astype(np.float32)
    n = xf[0].shape[0]
    idx = rng.permutation(n)[: n - 37]
    o = orc.Oracle(model, training_loss=loss, agg="sum")
    Lw, gw = objective(model, flat, xf, y, idx, training_loss=loss, agg="sum")
    L64, g64 = o.loss_grad(flat, xf, y, idx, precision=64)
    assert L64 == pytest.approx(Lw, rel=1e-10), name
    assert np.abs(g64 - gw).max() <= 1e-9 * np.abs(gw).max(), name
