"""`fast_monte_carlo_b200.helpers` (the reference's sim_helpers.py on the engine)."""
import importlib.util
import os
import sys

import numpy as np
import pytest

from conftest import NO_REFERENCE, REFERENCE, has_reference
from fast_monte_carlo_b200 import helpers


@pytest.mark.skipif(not has_reference("sim_helpers.py"), reason=NO_REFERENCE)
def test_softmax_equals_reference():
    import oracle.fake_xgboost as fx
    saved = sys.modules.get("xgboost")
    sys.modules["xgboost"] = fx                        # sim_helpers imports xgboost at module level
    try:
        spec = importlib.util.spec_from_file_location("sim_helpers_ref", os.path.join(REFERENCE, "sim_helpers.py"))
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
    finally:
        if saved is None:
            sys.modules.pop("xgboost", None)
        else:
            sys.modules["xgboost"] = saved
    rng = np.random.default_rng(0)
    for dt in (np.float32, np.float64):
        z = (rng.normal(0, 3, (500, 4)) / 1.3).astype(dt)
        assert np.array_equal(helpers.softmax(z), ref.softmax(z))


@pytest.mark.gpu
def test_pass_outcome_model_and_quantile_yards(engine, oracle, models_s2):
    from test_pack import _rows
    rows = _rows(3000, 21)
    m = helpers.PassOutcomeModel(engine, "pass_stage2", temperature=1.7)          # best_iteration 241 of the forest
    assert m.best_it == 241 and m.n_classes == 3
    got = m.predict_proba(rows)
    cols = [g.column_of("Unknown") for g in models_s2["pass_stage2"].groups] + [-1, -1]
    margin = oracle.predict("pass_stage2", rows, np.tile(np.array(cols[:2]), (rows.shape[0], 1)), 3, 0, 242 * 3)
    want = helpers.softmax(margin.astype(np.float32) / 1.7)
    assert got.dtype == np.float32 and np.array_equal(got, want) and np.allclose(got.sum(axis=1), 1.0, atol=1e-6)
    full = helpers.PassOutcomeModel(engine, "pass_stage2", best_iteration=10_000).predict_proba(rows[:10])
    assert not np.array_equal(full, got[:10])                                    # the iteration range matters
    qy = helpers.QuantileYards(engine, "run_yards")
    colr = [g.column_of("Unknown") for g in models_s2["run_yards"].groups] + [-1, -1]
    q = oracle.predict("run_yards", rows[:5], np.tile(np.array(colr[:2]), (5, 1)), 3)
    assert np.array_equal(qy.quantiles(rows[:5]), q)
    for i in range(5):
        rng_a, rng_b = np.random.default_rng(i), np.random.default_rng(i)
        y = qy.sample(rows[i], -4.0, 40.0, noise=0.5, rng=rng_a)
        u = rng_b.random()
        q10, q50, q90 = q[i]
        w = q10 + (q50 - q10) * (u / 0.5) if u < 0.5 else q50 + (q90 - q50) * ((u - 0.5) / 0.5)
        assert y == float(np.clip(w + rng_b.normal(0, 0.5), -4.0, 40.0))
