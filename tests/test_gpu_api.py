"""The reference-facing Python entry points on the GPU."""
import os

import numpy as np
import pandas as pd
import pytest

from fast_monte_carlo_b200 import api, outputs, priors

pytestmark = pytest.mark.gpu


def test_simulate_upcoming_matchup_drop_in(engine, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    base = api.csv_base_from("Kansas State", "Iowa State", 1)
    sims_df, players_df, summary, A, B, meta = api.simulate_upcoming_matchup(
        "Kansas State", "Iowa State", year=2025, week=1, sp_path=priors.packaged_priors_path(), n=500,
        show_progress=False, collect_players=True, save_csv=base, processes=4, seed=11, engine=engine)
    assert list(sims_df.columns) == ["team", "opp", "pts", "opp_pts"] and len(sims_df) == 1000
    assert list(sims_df["team"][:2]) == ["Kansas State", "Iowa State"]
    assert list(players_df.columns) == api.PLAYER_COLS
    assert list(summary.columns) == ["mean_pts", "sd_pts", "mean_opp", "sd_opp", "win_rate"]
    assert set(summary.index) == {"Kansas State", "Iowa State"}
    assert (A.sp_rating, A.sp_offense, A.sp_defense) == (15.6, 35.7, 20.0) and B.name == "Iowa State"
    assert {"sim_time_sec", "io_time_sec", "total_time_sec", "sims"} <= set(meta) and meta["sims"] == 500
    on_disk = pd.read_csv(tmp_path / f"scores_{base}")
    assert on_disk.equals(sims_df.reset_index(drop=True).astype(on_disk.dtypes.to_dict()))
    assert os.path.exists(tmp_path / f"players_{base}")
    # parquet route: the chunked writer fed straight from the engine's score array (SURVEY 8f row 2)
    pq_base = base.replace(".csv", ".parquet")
    sims2, *_ = api.simulate_upcoming_matchup(
        "Kansas State", "Iowa State", sp_path=priors.packaged_priors_path(), n=500, show_progress=False,
        save_csv=pq_base, seed=11, engine=engine)
    pq = pd.read_parquet(tmp_path / f"scores_{pq_base}")
    assert (pq["team"].astype(str) == sims2["team"]).all() and np.array_equal(pq["pts"], sims2["pts"])
    assert np.array_equal(pq["opp_pts"], sims2["opp_pts"]) and sims2.equals(sims_df)
    # reproducible for a given seed; histogram adapter agrees with the table
    again, _ = api.simulate_matchup(A, B, n=500, seed=11, engine=engine)
    assert again.equals(sims_df)
    h = api.LAST_RUN["hist"]
    got = outputs.summary_from_hist(h, "Kansas State", "Iowa State")
    np.testing.assert_allclose(got.loc[summary.index].to_numpy(), summary.to_numpy(), rtol=1e-12)


def test_unknown_team_raises(engine):
    with pytest.raises(ValueError, match="not found in provided SP\\+ table"):
        api.simulate_upcoming_matchup("Nowhere Tech", "Iowa State", sp_path=priors.packaged_priors_path(), n=1,
                                      engine=engine)


def test_simulate_slate_matches_per_matchup_runs(engine):
    """One launch for a slate == the matchups simulated one by one (same seed => same games, since the Philox
    counter carries the matchup index only through the per-matchup game ids... and the matchup id)."""
    pairs = [("Kansas State", "Iowa State"), ("UTSA", "Ohio State"), ("Texas", "Michigan")]
    res = api.simulate_slate(pairs, n=400, seed=7, engine=engine,
                             markets={("Kansas State", "Iowa State"): {"spread": -3.5, "total": 55.5}})
    assert res["_counters"]["games"] == 3 * 800
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    from fast_monte_carlo_b200.engine import MatchupSpec
    for m, (a, b) in enumerate(pairs):
        e = res[(a, b)]
        assert e["games"] == 800 and e["hist"].shape == (2, 128, 128)
        assert int(e["hist"][0].sum()) == 400 and int(e["hist"][1].sum()) == 400
        assert set(e["summary"].index) == {a, b}
        assert 0.0 <= e["moneyline"]["team"]["p_win"] <= 1.0
    assert res[("Kansas State", "Iowa State")]["markets"]["spread"]["samples"] == 400
    assert res[("UTSA", "Ohio State")]["markets"] is None
    # the slate's first matchup is the same stream of games as a single-matchup launch (matchup index 0)
    engine.set_matchups([MatchupSpec("Kansas State", "Iowa State", priors.lookup_sp_flex("Kansas State", sp),
                                     priors.lookup_sp_flex("Iowa State", sp), 800, 0, 800, 0)])
    single = engine.simulate_host(7)
    assert np.array_equal(single["hist"][0].astype(np.int64), res[("Kansas State", "Iowa State")]["hist"])
    with pytest.raises(ValueError):
        api.simulate_slate([("Nowhere Tech", "Iowa State")], n=1, engine=engine)


def test_bench_json_line_contract(tmp_path):
    """`python bench.py` (small size) prints ONE JSON line with every key of the driver's contract."""
    import json, subprocess, sys
    from conftest import ROOT
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--games", "200000", "--steps", "2", "--warmup", "3",
                        "--cpu-games", "300", "--e2e-steps", "2", "--tree-states", str(1 << 20), "--roofline-steps", "1"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline",
              "memo", "tree_eval"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["gpu_launches"] == 2 and d["scaling"] == "weak"
    assert d["value"] > 1e7 and d["e2e"]["value"] > 1e6 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    rf = d["roofline"]
    # the walk is bound by the L1 data pipe (cache-resident node tables), not by HBM: a fraction of a true peak
    assert rf["bound"] == "l1-data-pipe" and rf["unit"] == "Gwavefront/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert 0.0 < rf["frac"] <= 1.2 and rf["algorithmic"]["gbs"] > 0 and rf["gathered"]["gbs"] > 0
    assert 0.0 < rf["gather_probe"]["frac_of_coherent_probe"] < 1.0
    te = d["tree_eval"]
    assert te["states_per_sec"] > 1e6 and te["roofline"]["bound"] == "l1-data-pipe" and 0.0 < te["roofline"]["frac"] <= 1.2
    assert d["memo"]["mode"] == "on" and 0.0 < d["memo"]["hit_rate"] < 1.0
    assert len(d["e2e"]["step_seconds"]) == 2
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and "sample" in cb
    assert set(("sm_mhz", "sm_max_mhz", "reasons")) <= set(d["clocks"])
    assert "workload" in d["config"] and "model" not in d["config"]


def test_bench_dump_outputs_equal_the_oracle(tmp_path):
    """`bench.py --dump-outputs` writes the last timed step's games: scores, boxes and event counters are the C
    oracle's games of the same seed, and the histogram is that of the dumped scores."""
    import subprocess, sys
    from conftest import ROOT
    from test_gpu_players import _box_equal_philox
    import bench
    n = 4000
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--players", "--games", str(n), "--steps", "2",
                        "--warmup", "1", "--e2e-steps", "1", "--no-roofline", "--no-tree-eval", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    got = {p.stem: np.load(p) for p in out.iterdir()}
    assert sorted(got) == ["counters", "hist", "players", "scores"]
    assert got["scores"].dtype == np.float32 and got["scores"].shape == (n, 2)
    assert all(got[k].dtype == np.float64 for k in ("counters", "hist", "players"))
    assert got["hist"].shape == (1, 2, 128, 128) and got["counters"].shape == (15,) and got["counters"][0] == n
    assert np.array_equal(got["hist"][0], outputs.histogram_from_scores(got["scores"].astype(np.int64)))
    ref, _, _ = bench.cpu_run(bench.load_models("synthetic"), n, "synthetic", players=True)
    assert np.array_equal(got["scores"], ref["scores"])
    _box_equal_philox(got["players"], ref["players"])
    assert got["counters"][1:14].tolist() == list(ref["counters"].values())


def test_simulate_upcoming_matchup_players(engine, oracle, models_s2, tmp_path, monkeypatch):
    """collect_players=True with a focus sheet: players_df / players_<base>.csv carry the reference's rows, and
    they equal the oracle's on the same Philox seed."""
    from conftest import GOLDEN
    from fast_monte_carlo_b200 import usage
    monkeypatch.chdir(tmp_path)
    base = api.csv_base_from("Kansas State", "Iowa State", 1)
    sheet = os.path.join(GOLDEN, "players_focus.csv")
    sims_df, players_df, summary, A, B, meta = api.simulate_upcoming_matchup(
        "Kansas State", "Iowa State", sp_path=priors.packaged_priors_path(), n=400, show_progress=False,
        collect_players=True, save_csv=base, seed=21, engine=engine, focus_csv=sheet)
    assert list(players_df.columns) == api.PLAYER_COLS and len(sims_df) == 800
    assert set(players_df["role"]) == {"QB", "Rusher", "Receiver"} and "__Other__" not in set(players_df["player"])
    assert set(players_df["start"]) == {"A", "B"} and players_df["sim"].max() <= 799
    us = (usage.resolve_team(A, models_s2), usage.resolve_team(B, models_s2))
    ref = oracle.simulate(oracle.make_config(models_s2, A.sp, B.sp), 800, seed=21, usage=oracle.make_usage(us),
                          n_slots=max(len(u.slots) for u in us))
    want = usage.player_rows(ref["players"], 0, ("Kansas State", "Iowa State"), us)
    assert len(want) == len(players_df)
    for c in api.PLAYER_COLS:
        if c.endswith("_yds"):
            assert np.allclose(players_df[c].to_numpy(float), want[c].to_numpy(float), atol=1e-6), c
        else:
            assert players_df[c].tolist() == want[c].tolist(), c
    on_disk = pd.read_csv(tmp_path / f"players_{base}")
    assert len(on_disk) == len(players_df) and list(on_disk.columns) == api.PLAYER_COLS
    odds = usage.player_prop_odds_from_box(api.LAST_RUN["player_box"], ("Kansas State", "Iowa State"), us,
                                           "Kansas State", "Taylen Green", "pass_yards", 150.5)
    assert odds["samples"] > 700 and 0.0 < odds["p_over"] < 1.0
    # without the sheet the same call is the shipped configuration: nobody is tracked
    _, empty, *_ = api.simulate_upcoming_matchup("Kansas State", "Iowa State", sp_path=priors.packaged_priors_path(),
                                                 n=50, show_progress=False, seed=21, engine=engine)
    assert len(empty) == 0 and list(empty.columns) == api.PLAYER_COLS
