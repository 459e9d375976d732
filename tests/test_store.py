"""Literal score tables and sim_store-layout bundles written at scale (SURVEY 8f row 2), host only."""
import importlib.util
import json
import os

import numpy as np
import pandas as pd
import pytest

from conftest import NO_REFERENCE, REFERENCE, has_reference
from fast_monte_carlo_b200 import outputs, store


def _scores(n, seed=0):
    rng = np.random.default_rng(seed)
    a = 7 * rng.integers(0, 8, n) + 3 * rng.integers(0, 4, n)
    b = 7 * rng.integers(0, 7, n) + 3 * rng.integers(0, 5, n)
    return np.stack([a, b], axis=1).astype(np.int32)


@pytest.mark.parametrize("ext", ["parquet", "csv"])
@pytest.mark.parametrize("n", [0, 1, 10_001])
def test_scores_table_equals_sims_frame(tmp_path, ext, n):
    sc = _scores(n, 3)
    path = str(tmp_path / f"scores_a_b_wk1_sims.{ext}")
    assert outputs.write_scores_table(path, "A State", "B Tech", sc, chunk_rows=4096) == n
    got = pd.read_parquet(path) if ext == "parquet" else pd.read_csv(path)
    want = outputs.sims_frame("A State", "B Tech", sc)
    assert list(got.columns) == ["team", "opp", "pts", "opp_pts"] and len(got) == n
    if n:
        assert (got["team"].astype(str).to_numpy() == want["team"].to_numpy()).all()
        assert (got["opp"].astype(str).to_numpy() == want["opp"].to_numpy()).all()
        assert np.array_equal(got["pts"].to_numpy(), want["pts"].to_numpy())
        assert np.array_equal(got["opp_pts"].to_numpy(), want["opp_pts"].to_numpy())


def test_bundle_layout_and_signature(tmp_path):
    sc = _scores(5000, 4)
    meta = {"teams": ["A", "B"], "n": 2500, "seed": 11, "engine": "fmc-b200"}
    sig = store.save_sim_bundle(str(tmp_path / "run"), "A", "B", sc, meta, seed=11, chunk_rows=1024)
    assert sig == store.make_signature(meta) and len(sig) == 64
    games, players, m = store.load_sim_bundle(str(tmp_path / "run"))
    assert list(games.columns) == store.GAMES_COLUMNS and len(games) == 5000
    assert np.array_equal(games["sim_id"].to_numpy(), np.arange(5000))
    assert np.array_equal(games["margin"].to_numpy(), (games["pts"] - games["opp_pts"]).to_numpy())
    assert np.array_equal(games["total"].to_numpy(), (games["pts"] + games["opp_pts"]).to_numpy())
    assert (games["seed"] == 11).all() and m["signature"] == sig and len(players) == 0
    # canonical-JSON signature of the reference (sim_store.py:6-8)
    import hashlib
    assert sig == hashlib.sha256(json.dumps(meta, sort_keys=True, separators=(",", ":")).encode()).hexdigest()


@pytest.mark.skipif(not has_reference("edge_finder.py"), reason=NO_REFERENCE)
def test_unmodified_edge_finder_reads_the_parquet(tmp_path, monkeypatch):
    spec = importlib.util.spec_from_file_location("edge_finder_ref", os.path.join(REFERENCE, "edge_finder.py"))
    ef = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ef)
    sc = _scores(6000, 5)
    base = "kansasstate_iowastate_wk1_sims"
    outputs.write_scores_table(str(tmp_path / f"scores_{base}.parquet"), "Kansas State", "Iowa State", sc)
    monkeypatch.chdir(tmp_path)
    got = ef.game_market_odds(base, team="Kansas State", opp="Iowa State", spread=-3.5, total=52.5)
    h = outputs.histogram_from_scores(sc)
    want = outputs.game_market_odds_from_hist(h, "Kansas State", "Iowa State", spread=-3.5, total=52.5)
    for k in ("p_cover", "p_notcover", "push_rate", "mean_margin", "median_margin"):
        assert got["spread"][k] == pytest.approx(want["spread"][k], abs=1e-9)
    for k in ("p_over", "p_under", "mean_total", "median_total"):
        assert got["total"][k] == pytest.approx(want["total"][k], abs=1e-9)
