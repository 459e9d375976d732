"""Per-player path on the CPU: the host usage tables and the C oracle against fixtures produced by the
UNMODIFIED reference (tests/golden/make_golden_players.py: synthetic focus sheet -> the reference's
`_build_focus_usage_tables`, `simulate_game` under injected draws, `flatten_player_box_rows`)."""
import json
import os

import numpy as np
import pandas as pd
import pytest

from conftest import GOLDEN, NO_REFERENCE, REFERENCE, has_reference

from fast_monte_carlo_b200 import priors, usage


@pytest.fixture(scope="module")
def gold():
    t = np.load(os.path.join(GOLDEN, "ref_players.npz"))
    return dict(t=t, meta=json.loads(str(t["meta"])), teams=json.loads(str(t["teams"])),
                cols=json.loads(str(t["player_cols"])), rows=json.loads(str(t["player_rows"])))


@pytest.fixture(scope="module")
def contexts(gold):
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    return {name: priors.build_team_context_from_sp_flex(name, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
            for name in gold["teams"]}


def test_usage_tables_match_reference(gold, contexts):
    """Share tables (names, order, float64 bits) and track sets of the reference's own loader."""
    for name, ref in gold["teams"].items():
        tc = contexts[name]
        for key, df, col in (("qb", tc.qb_share, "passer_name"), ("ru", tc.rush_share, "rusher_name"),
                             ("tg", tc.target_share, "receiver_name")):
            assert [str(x) for x in df[col]] == ref[key][0], (name, key)
            assert np.array_equal(np.asarray(df["share"].values, dtype=np.float64), np.asarray(ref[key][1])), (name, key)
        assert sorted(tc.track_pass) == ref["track_pass"]
        assert sorted(tc.track_rush) == ref["track_rush"]
        assert sorted(tc.track_rec) == ref["track_rec"]
        assert [tc.sp_rating, tc.sp_offense, tc.sp_defense] == ref["sp"]


def test_resolve_team_columns(models, contexts):
    ksu = usage.resolve_team(contexts["Kansas State"], models)
    assert ksu.role["pass"].names == ["Taylen Green", "Zach Gibson", "__Other__"]
    assert [s for s in ksu.role["pass"].slot] == [0, 1, -1]                 # `__Other__` is never tracked
    g = models["pass_stage1"].group("passer_name")
    assert ksu.role["pass"].col["pass_stage1"] == [g.column_of("Taylen Green"), g.column_of("Zach Gibson"), -1]
    # the receiver remainder is fed to the models as "Unknown" (FMC:1066); an unseen name lights nothing
    tg = models["pass_yards"].group("target_name")
    assert ksu.role["rec"].names[-1] == "__Other__"
    assert ksu.role["rec"].col["pass_yards"][-1] == tg.column_of("Unknown") >= 0
    assert ksu.role["rec"].col["pass_yards"][ksu.role["rec"].names.index("Nobody Known")] == -1
    assert usage.resolve_team(contexts["UTSA"], models).trivial
    assert [usage.ROLE_LABEL[r] for r, _ in ksu.slots] == ["QB", "QB", "Rusher", "Rusher", "Rusher", "Receiver", "Receiver", "Receiver"]


def test_py_round1():
    x = np.array([1.15, 2.25, 0.05, 7.349999, 12.45, -0.15, 3.0, 1e-9, 104.65])
    assert usage.py_round1(x).tolist() == [round(float(v), 1) for v in x]
    rng = np.random.default_rng(0)
    y = np.round(rng.random(20000) * 60, 2)
    assert usage.py_round1(y).tolist() == [round(float(v), 1) for v in y]


def _frame(rows, cols):
    df = pd.DataFrame(rows, columns=cols)
    return df.sort_values(["sim", "team", "role", "player"], kind="stable").reset_index(drop=True)


def test_oracle_players_match_reference(models, oracle, gold, contexts):
    """Trajectories bit for bit, and the reference's players table row for row."""
    t, meta = gold["t"], gold["meta"]
    stream = oracle.make_stream(len(meta), int(t["stream_seed"]))
    frames = []
    for g, m in enumerate(meta):
        ta, tb = contexts[m["team_a"]], contexts[m["team_b"]]
        us = [usage.resolve_team(ta, models), usage.resolve_team(tb, models)]
        n_slots = max(len(u.slots) for u in us)
        cfg = oracle.make_config(models, ta.sp, tb.sp)
        r = oracle.simulate(cfg, 1, game0=g, stream=stream[g:g + 1], trace=True, threads=1,
                            usage=oracle.make_usage(us), n_slots=n_slots)
        n = int(t["iters"][g])
        assert r["iters"][0] == n, g
        assert np.array_equal(r["trace"][0, :n], t["traces"][g, :n]), g
        first = g & 1
        assert (r["scores"][0, first], r["scores"][0, first ^ 1]) == tuple(t["scores"][g])
        frames.append(usage.player_rows(r["players"], g, (m["team_a"], m["team_b"]), us))
    got = pd.concat(frames, ignore_index=True)
    want = _frame(gold["rows"], gold["cols"])
    got = _frame(got.values.tolist(), gold["cols"])
    assert len(got) == len(want) > 50
    for c in gold["cols"]:
        assert got[c].tolist() == want[c].tolist(), c


def test_oracle_trivial_usage_equals_plain_run(models, oracle):
    """One "Unknown" per role and nothing tracked is the shipped configuration: same games as without usage."""
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ta = priors.build_team_context_from_sp_flex("Kansas State", 2025, 1, sp, usage_dir=GOLDEN)
    tb = priors.build_team_context_from_sp_flex("Iowa State", 2025, 1, sp, usage_dir=GOLDEN)
    us = [usage.resolve_team(ta, models), usage.resolve_team(tb, models)]
    assert us[0].trivial and us[1].trivial
    cfg = oracle.make_config(models, ta.sp, tb.sp)
    a = oracle.simulate(cfg, 64, seed=5)
    b = oracle.simulate(cfg, 64, seed=5, usage=oracle.make_usage(us), n_slots=0)
    assert np.array_equal(a["scores"], b["scores"]) and np.array_equal(a["iters"], b["iters"])


@pytest.mark.skipif(not has_reference("edge_finder.py"), reason=NO_REFERENCE)
def test_unmodified_edge_finder_reads_our_players_file(models, oracle, contexts, tmp_path, monkeypatch):
    """`players_<base>.csv` written from the per-game box is what edge_finder.player_prop_odds /
    scan_props_for_matchup expect (edge_finder.py:131-231, 340-390), and the box adapter returns the same odds."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("edge_finder_ref", os.path.join(REFERENCE, "edge_finder.py"))
    ef = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ef)
    monkeypatch.chdir(tmp_path)                      # edge_finder drops a scratch `testings.csv` into the cwd
    ta, tb = contexts["Kansas State"], contexts["Iowa State"]
    us = [usage.resolve_team(ta, models), usage.resolve_team(tb, models)]
    n = 600
    r = oracle.simulate(oracle.make_config(models, ta.sp, tb.sp), n, seed=3, usage=oracle.make_usage(us),
                        n_slots=max(len(u.slots) for u in us))
    names = ("Kansas State", "Iowa State")
    df = usage.player_rows(r["players"], 0, names, us)
    assert list(df.columns) == gold_cols() and len(df) > 5 * n
    base = priors.csv_base_from("Kansas State", "Iowa State", 1)
    stem = base[:-4]
    from fast_monte_carlo_b200 import outputs
    outputs.sims_frame(*names, r["scores"]).to_csv(tmp_path / f"scores_{base}", index=False)
    df.to_csv(tmp_path / f"players_{base}", index=False)
    for team, player, stat, line in (("Kansas State", "Taylen Green", "pass_yards", 180.5),
                                     ("Kansas State", "Blake Watson", "rush_yards", 35.5),
                                     ("Iowa State", "Carson Hansen", "rec_yards", 40.5),
                                     ("Iowa State", "Levi Williams", "pass_td", 1.5),
                                     ("kansas state", "benjamin brahmer", "rec", 3.0)):
        want = ef.player_prop_odds(stem, team, player, stat, line, directory=str(tmp_path))
        got = usage.player_prop_odds_from_box(r["players"], names, us, team, player, stat, line)
        assert set(want) == set(got)
        for k, v in want.items():
            if isinstance(v, float):
                assert abs(got[k] - v) < 1e-9, (player, k, got[k], v)
            else:
                assert got[k] == v, (player, k)
    sheet = os.path.join(GOLDEN, "players_focus.csv")
    props = ef.scan_props_for_matchup(stem, "Kansas State", "Iowa State", prop_sheet_path=sheet, directory=str(tmp_path),
                                      min_abs_edge_pct=0.0)
    assert len(props) >= 10 and {"Taylen Green", "Bo Nix"} <= set(props["player"])
    ours = usage.scan_props_from_hist(usage.player_hist_from_box(r["players"], us), names, us, sheet)
    assert len(ours) == len(props)
    a = props.sort_values(["team", "player", "stat", "line"]).reset_index(drop=True)
    b = ours.sort_values(["team", "player", "stat", "line"]).reset_index(drop=True)
    for c in a.columns:
        if a[c].dtype.kind == "f":
            assert np.allclose(a[c].to_numpy(), b[c].to_numpy(), rtol=1e-9, atol=1e-9), c
        else:
            assert a[c].tolist() == b[c].tolist(), c
    with pytest.raises(ValueError):
        usage.player_prop_odds_from_box(r["players"], names, us, "Kansas State", "Nobody Here", "rush_yards", 10.5)


def gold_cols():
    from fast_monte_carlo_b200.api import PLAYER_COLS
    return PLAYER_COLS


def test_prop_odds_from_histograms_equal_from_rows(models, oracle, contexts):
    """The per-player histograms (the form ranks merge with one all-reduce) answer every prop question exactly
    like the per-game box / `players_*` rows do."""
    ta, tb = contexts["Kansas State"], contexts["Iowa State"]
    us = [usage.resolve_team(ta, models), usage.resolve_team(tb, models)]
    n = 1500
    r = oracle.simulate(oracle.make_config(models, ta.sp, tb.sp), n, seed=8, usage=oracle.make_usage(us),
                        n_slots=max(len(u.slots) for u in us))
    names = ("Kansas State", "Iowa State")
    h = usage.player_hist_from_box(r["players"], us)
    assert h.shape == (2, 8, usage.PH_BINS)
    for t in (0, 1):
        for s, (role, nm) in enumerate(us[t].slots):
            rec = r["players"][:, t, s]
            seen = int(((rec[:, 1] > 0) | (rec[:, 5] > 0)).sum())
            assert int(h[t, s, :usage.PH_YDS_BINS].sum()) == seen
            for stat, (rl, fld) in usage._STAT_FIELD.items():
                if rl != role or seen == 0:
                    continue
                for line in (0.5, 2.5, 3.0, 40.5, 62.4, 180.5):
                    a = usage.player_prop_odds_from_box(r["players"], names, us, names[t], nm, stat, line)
                    b = usage.player_prop_odds_from_hist(h, names, us, names[t], nm, stat, line)
                    assert set(a) == set(b)
                    for k, v in a.items():
                        if isinstance(v, float):
                            assert abs(b[k] - v) <= 1e-9 * max(1.0, abs(v)), (nm, stat, line, k, b[k], v)
                        else:
                            assert b[k] == v, (nm, stat, line, k)


def test_usage_capacity_errors(models):
    """Table limits of the kernels are reported by name, before anything is launched."""
    rush = models["run_yards"].group("rusher_name").categories
    known = [n for n in rush if n not in ("Unknown",)][:9]
    tc = priors.TeamContext("X", 2025, 1, 1.0, 2.0, 3.0,
                            rush_share=pd.DataFrame({"rusher_name": known, "share": [1.0 / 9] * 9}))
    with pytest.raises(ValueError, match="rush names that the models have one-hot columns for"):
        usage.resolve_team(tc, models)
    many = [f"Walk On {i}" for i in range(33)]
    tc = priors.TeamContext("X", 2025, 1, 1.0, 2.0, 3.0,
                            rush_share=pd.DataFrame({"rusher_name": many, "share": [1.0] * 33}))
    with pytest.raises(ValueError, match="usage entries"):
        usage.resolve_team(tc, models)
    ok = priors.TeamContext("X", 2025, 1, 1.0, 2.0, 3.0,
                            rush_share=pd.DataFrame({"rusher_name": many[:32], "share": [1.0] * 32}))
    assert usage.name_rows(usage.resolve_team(ok, models).role["rush"]) == [-1] * 32     # unknown names need no row
    bad = priors.TeamContext("X", 2025, 1, 1.0, 2.0, 3.0,
                             rush_share=pd.DataFrame({"rusher_name": ["A", "B"], "share": [0.0, 0.0]}))
    with pytest.raises(ValueError, match="shares"):
        usage.resolve_team(bad, models)


def test_oracle_players_adversarial_streams(models, oracle, gold, contexts):
    """The reference's own player-mode games under ADVERSARIAL draws (tests/streams.py): u = 0 must pick the first
    usage entry with a positive share (zero-share entries are skipped), u just below 1 the last entry, +-4 sigma
    yardage, 112-112 shoot-outs -- trajectories bit for bit and the players table row for row."""
    from streams import adversarial_stream
    t = gold["t"]
    meta = json.loads(str(t["adv_meta"]))
    stream = adversarial_stream(len(meta), int(t["adv_stream_seed"]))
    frames = []
    for g, m in enumerate(meta):
        ta, tb = contexts[m["team_a"]], contexts[m["team_b"]]
        us = [usage.resolve_team(ta, models), usage.resolve_team(tb, models)]
        cfg = oracle.make_config(models, ta.sp, tb.sp)
        r = oracle.simulate(cfg, 1, game0=g, stream=stream[g:g + 1], trace=True, threads=1,
                            usage=oracle.make_usage(us), n_slots=max(len(u.slots) for u in us))
        n = int(t["adv_iters"][g])
        assert r["iters"][0] == n, (g, m["pattern"])
        assert np.array_equal(r["trace"][0, :n], t["adv_traces"][g, :n]), (g, m["pattern"])
        f = g & 1
        assert (r["scores"][0, f], r["scores"][0, f ^ 1]) == tuple(t["adv_scores"][g])
        frames.append(usage.player_rows(r["players"], g, (m["team_a"], m["team_b"]), us))
    got = _frame(pd.concat(frames, ignore_index=True).values.tolist(), gold["cols"])
    want = _frame(json.loads(str(t["adv_player_rows"])), gold["cols"])
    assert len(got) == len(want) > 10
    for c in gold["cols"]:
        assert got[c].tolist() == want[c].tolist(), c
