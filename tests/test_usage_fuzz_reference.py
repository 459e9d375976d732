"""Host usage loaders against the UNMODIFIED reference on random inputs (runs only where FMC_REFERENCE_DIR names
the original project).  `usage.build_focus_usage_tables` / `usage.load_usage_table` must return the
reference's tables bit for bit: names, order, float64 shares, track sets."""
import numpy as np
import pandas as pd
import pytest

from conftest import NO_REFERENCE, has_reference
from fast_monte_carlo_b200 import usage

pytestmark = pytest.mark.skipif(not has_reference("fast_monte_carlo_cfb.py"), reason=NO_REFERENCE)


@pytest.fixture(scope="module")
def ref():
    from oracle import ref_harness as rh
    return rh.load_reference()


def _random_sheet(rng, path):
    teams = ["Kansas State", "Iowa State", " Texas ", "UTSA"]
    rows = []
    for t in teams:
        for stat in ("pass_yards", "rush_yards", "rec_yards", "Pass_Yards ", "other_stat"):
            n = int(rng.integers(0, 6))
            mode = rng.choice(["frac_low", "frac_high", "percent", "zeros", "mixed"])
            for i in range(n):
                if mode == "frac_low":
                    u = rng.uniform(0.01, 0.9 / max(n, 1))
                elif mode == "frac_high":
                    u = rng.uniform(0.2, 0.9)
                elif mode == "percent":
                    u = rng.uniform(1.0, 60.0)
                elif mode == "zeros":
                    u = 0.0
                else:
                    u = rng.choice([np.nan, -0.2, 0.0, 0.3, 1.4, 25.0])
                name = f"Player {int(rng.integers(0, 4))}" if rng.random() < 0.3 else f" P{t.strip()[:2]}{stat[:2]}{i} "
                rows.append(dict(team=t, player=name, pos=rng.choice(["qb", "RB", "wr"]), usage=u, stat=stat,
                                 yards=float(rng.integers(10, 300)) + 0.5))
    pd.DataFrame(rows, columns=["team", "player", "pos", "usage", "stat", "yards"]).to_csv(path, index=False)


def test_focus_tables_equal_reference(ref, tmp_path):
    rng = np.random.default_rng(2025)
    for it in range(25):
        p = str(tmp_path / f"sheet_{it}.csv")
        _random_sheet(rng, p)
        want = ref._build_focus_usage_tables(p)
        got = usage.build_focus_usage_tables(p)
        assert set(got) == set(want), it
        for team in want:
            for key, col in (("qb_df", "passer_name"), ("ru_df", "rusher_name"), ("tg_df", "receiver_name")):
                a, b = want[team][key], got[team][key]
                assert list(a.columns) == list(b.columns) == [col, "share"], (it, team, key)
                assert [str(x) for x in a[col]] == [str(x) for x in b[col]], (it, team, key)
                assert np.array_equal(a["share"].to_numpy(dtype=np.float64), b["share"].to_numpy(dtype=np.float64)), (it, team, key)
            for key in ("track_pass", "track_rush", "track_rec"):
                assert want[team][key] == got[team][key], (it, team, key)
    assert usage.build_focus_usage_tables(str(tmp_path / "missing.csv")) == ref._build_focus_usage_tables(str(tmp_path / "missing.csv")) == {}


def test_usage_files_equal_reference(ref, tmp_path):
    rng = np.random.default_rng(7)
    for it in range(20):
        n = int(rng.integers(0, 12))
        df = pd.DataFrame(dict(offense=rng.choice(["Ohio State", "Michigan"], n), year=rng.choice([2024, 2025], n),
                               rusher_name=[f"R{int(rng.integers(0, 9))}" for _ in range(n)],
                               share=rng.choice([np.nan, -1.0, 0.0, 0.25, 3.0, 17.0], n)))
        p = str(tmp_path / f"usage_{it}.csv")
        df.to_csv(p, index=False)
        for team in ("Ohio State", "Michigan", "Nobody"):
            for col in ("rusher_name", "passer_name"):
                want = ref._load_usage_table(p, team, 2025, col)
                got = usage.load_usage_table(p, team, 2025, col)
                assert (want is None) == (got is None), (it, team, col)
                if want is not None:
                    assert want[col].tolist() == got[col].tolist()
                    assert np.array_equal(want["share"].to_numpy(float), got["share"].to_numpy(float), equal_nan=True)
    assert usage.load_usage_table(str(tmp_path / "nope.csv"), "Ohio State", 2025, "rusher_name") is None
