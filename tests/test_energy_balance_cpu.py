"""plan.energy_balance: the global balance of a partition from per-rank energy records (pure numpy, no GPU)."""
import numpy as np
import pytest

import saa_b200  # noqa: F401
from saa_b200 import plan as splan


def _records(seed, steps, tn):
    rng = np.random.default_rng(seed)
    r = np.zeros(len(steps), dtype=splan.ENERGY_DTYPE)
    r["step"], r["tn"] = steps, tn
    for f in splan.ENERGY_FIELDS[2:]:
        r[f] = rng.standard_normal(len(steps))
    return r


def test_additive_fields_are_summed_in_ascending_rank_order():
    steps, tn = np.array([0, 5, 10]), np.array([0.0, 0.5, 1.0])
    recs = [_records(q, steps, tn) for q in range(3)]
    # values whose sum depends on the order: 1 + 1e-16 + -1 vs other orders
    recs[0]["coupling"][:] = 1.0
    recs[1]["coupling"][:] = 1e-16
    recs[2]["coupling"][:] = -1.0
    b = splan.energy_balance(recs)
    assert np.array_equal(b["step"], steps) and np.array_equal(b["tn"], tn)
    for f in splan.ENERGY_FIELDS[2:]:
        assert np.array_equal(b[f], (recs[0][f] + recs[1][f]) + recs[2][f]), f
    assert np.all(b["coupling"] == (1.0 + 1e-16) + -1.0)


def test_total_and_residual():
    steps, tn = np.array([0, 1]), np.array([0.0, 0.1])
    r = np.zeros(2, dtype=splan.ENERGY_DTYPE)
    r["step"], r["tn"] = steps, tn
    r["kinetic_half"] = [1.0, 2.0]
    r["coupling"] = [3.0, 4.0]
    r["energy_at_arm"] = 4.0
    r["work_external"] = [0.0, 2.5]
    r["work_damping"] = [0.0, 0.5]
    b = splan.energy_balance([r])
    assert b.dtype == splan.BALANCE_DTYPE
    assert np.array_equal(b["total"], [4.0, 6.0])
    assert np.array_equal(b["residual"], [0.0, 0.0])          # 6 - 4 - 2.5 + 0.5
    r["work_damping"][1] = 1.0
    assert splan.energy_balance([r])["residual"][1] == 0.5


@pytest.mark.parametrize("field", ["step", "tn"])
def test_records_of_different_steps_are_refused(field):
    steps, tn = np.array([0, 5]), np.array([0.0, 0.5])
    a, b = _records(0, steps, tn), _records(1, steps, tn)
    b[field][1] = b[field][1] + 1
    with pytest.raises(ValueError, match="rank 1"):
        splan.energy_balance([a, b])
    with pytest.raises(ValueError):
        splan.energy_balance([a, b[:1]])
