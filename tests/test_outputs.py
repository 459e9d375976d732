"""Host-side output contract: sims_df layout, summary, and the histogram adapter against the
UNMODIFIED edge_finder.py (when the reference is mounted) and against a direct restatement."""
import importlib.util
import os

import numpy as np
import pandas as pd
import pytest

from conftest import NO_REFERENCE, REFERENCE, has_reference
from fast_monte_carlo_b200 import outputs


def _scores(n, seed=0):
    rng = np.random.default_rng(seed)
    a = 7 * rng.integers(0, 8, n) + 3 * rng.integers(0, 4, n)
    b = 7 * rng.integers(0, 7, n) + 3 * rng.integers(0, 5, n)
    return np.stack([a, b], axis=1).astype(np.int32)


def test_sims_frame_layout():
    sc = _scores(10)
    df = outputs.sims_frame("A U", "B St", sc)
    assert list(df.columns) == ["team", "opp", "pts", "opp_pts"] and len(df) == 10
    assert list(df["team"][:4]) == ["A U", "B St", "A U", "B St"]        # rows alternate A-first / B-first
    assert list(df["pts"][:2]) == [sc[0, 0], sc[1, 1]] and list(df["opp_pts"][:2]) == [sc[0, 1], sc[1, 0]]


def test_summary_matches_reference_definition():
    sc = _scores(2000, 1)
    df = outputs.sims_frame("A", "B", sc)
    s = outputs.summary_frame(df)
    # FMC:1681-1687 restated literally
    want = df.groupby("team").agg(
        mean_pts=("pts", "mean"), sd_pts=("pts", "std"), mean_opp=("opp_pts", "mean"), sd_opp=("opp_pts", "std"),
        win_rate=("pts", lambda x: (x.values > df.loc[x.index, "opp_pts"].values).mean()))
    pd.testing.assert_frame_equal(s, want)
    h = outputs.histogram_from_scores(sc)
    s2 = outputs.summary_from_hist(h, "A", "B")
    np.testing.assert_allclose(s2.to_numpy(), want.to_numpy(), rtol=1e-12)


def _direct(df, team, opp, spread, total):
    sub = df[(df["team"] == team) & (df["opp"] == opp)]
    margin = (sub["pts"] - sub["opp_pts"]).to_numpy()
    totals = (sub["pts"] + sub["opp_pts"]).to_numpy()
    return dict(p_cover=float(np.mean(margin > -spread)), p_notcover=float(np.mean(margin < -spread)),
                push=float(np.mean(np.isclose(margin, -spread))), mean_margin=float(np.mean(margin)),
                median_margin=float(np.median(margin)), p_over=float(np.mean(totals > total)),
                mean_total=float(np.mean(totals)), median_total=float(np.median(totals)))


@pytest.mark.parametrize("n", [1001, 4000])
def test_histogram_adapter_equals_direct(n):
    sc = _scores(n, 2)
    df = outputs.sims_frame("A", "B", sc)
    h = outputs.histogram_from_scores(sc)
    for team, opp, is_a in (("A", "B", True), ("B", "A", False)):
        for spread, total in ((-3.5, 55.5), (7.0, 49.0), (0.0, 52.0)):
            got = outputs.game_market_odds_from_hist(h, team, opp, team_is_a=is_a, spread=spread, total=total)
            d = _direct(df, team, opp, spread, total)
            assert got["spread"]["p_cover"] == round(d["p_cover"], 6)
            assert got["spread"]["p_notcover"] == round(d["p_notcover"], 6)
            assert got["spread"]["push_rate"] == round(d["push"], 6)
            assert abs(got["spread"]["mean_margin"] - d["mean_margin"]) < 1e-9
            assert got["spread"]["median_margin"] == d["median_margin"]
            assert got["total"]["p_over"] == round(d["p_over"], 6)
            assert abs(got["total"]["mean_total"] - d["mean_total"]) < 1e-9
            assert got["total"]["median_total"] == d["median_total"]


@pytest.mark.skipif(not has_reference("edge_finder.py"), reason=NO_REFERENCE)
def test_unmodified_edge_finder_reads_our_files(tmp_path):
    """Gate G9: edge_finder.game_market_odds / moneyline_from_sims on a materialised scores_*.csv
    equal the histogram adapter."""
    spec = importlib.util.spec_from_file_location("edge_finder_ref", os.path.join(REFERENCE, "edge_finder.py"))
    ef = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ef)
    from fast_monte_carlo_b200.priors import csv_base_from
    sc = _scores(3000, 3)
    df = outputs.sims_frame("Kansas State", "Iowa State", sc)
    base = csv_base_from("Kansas State", "Iowa State", 1)
    df.to_csv(tmp_path / f"scores_{base}", index=False)
    stem = base[:-4]
    h = outputs.histogram_from_scores(sc)
    want = ef.game_market_odds(stem, "Kansas State", "Iowa State", spread=-3.5, total=58.5, directory=str(tmp_path))
    got = outputs.game_market_odds_from_hist(h, "Kansas State", "Iowa State", spread=-3.5, total=58.5)
    for k in ("spread", "total"):
        for kk, v in want[k].items():
            if isinstance(v, float):
                assert abs(got[k][kk] - v) < 1e-9, (k, kk)
            else:
                assert got[k][kk] == v, (k, kk)
    want = ef.game_market_odds(stem, "Iowa State", "Kansas State", spread=3.5, total=58.5, directory=str(tmp_path))
    got = outputs.game_market_odds_from_hist(h, "Iowa State", "Kansas State", team_is_a=False, spread=3.5, total=58.5)
    assert got["spread"]["p_cover"] == want["spread"]["p_cover"] and got["total"]["median_total"] == want["total"]["median_total"]
    ml = ef.moneyline_from_sims(stem, "Kansas State", "Iowa State", directory=str(tmp_path))
    assert outputs.moneyline_from_hist(h, "Kansas State", "Iowa State") == ml
