"""Overtime on the B200 (fmc_simulate_overtime, the overtime instantiations of both simulation kernels): the overtime
oracle game by game (Philox games with the memo off, on and persistent, player mode, the scripted streams, live starts
at 0:00 and late in the fourth quarter), overtime on against off at the same seed, the histogram against the per-game
rows, and the API."""
import os

import numpy as np
import pytest

import overtime_scripts as osc
from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import api, outputs, priors, usage
from fast_monte_carlo_b200.engine import GameState, MatchupSpec, OvertimeRules
from test_gpu_players import _box_equal_philox
from test_gpu_segments import memo_engines  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

RULES = OvertimeRules()
ORACLE_COUNTERS = ("plays", "iters", "pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg", "punt", "go")
NP = outputs.OT_MAX_PERIODS + 1


@pytest.fixture(scope="module")
def oto(models_s2):
    import oracle_overtime
    oracle_overtime.load_models(models_s2)
    return oracle_overtime


def _oracle(oto, cfg, n, chunk=5000, **kw):
    parts = [oto.simulate(cfg, min(chunk, n - lo), game0=lo, **kw) for lo in range(0, n, chunk)]
    out = {k: np.concatenate([p[k] for p in parts]) for k in ("scores", "iters", "periods")}
    out["counters"] = {k: sum(p["counters"][k] for p in parts) for k in ORACLE_COUNTERS}
    if kw.get("trace"):
        out["trace"] = np.concatenate([p["trace"] for p in parts])
    if kw.get("usage") is not None:
        out["players"] = np.concatenate([p["players"] for p in parts])
    return out


def hist_from_rows(scores, periods, games):
    """[2][OT_MAX_PERIODS + 1][3] of per-game final scores and overtime periods, game ids `games`."""
    h = np.zeros((2, NP, 3), dtype=np.int64)
    r = np.where(scores[:, 0] > scores[:, 1], 0, np.where(scores[:, 1] > scores[:, 0], 1, 2))
    np.add.at(h, (np.asarray(games) & 1, periods, r), 1)
    return h


def _check_against_oracle(got, ref, games, counters=True):
    assert np.array_equal(got["scores"], ref["scores"])
    assert np.array_equal(got["iters"], ref["iters"])
    assert np.array_equal(got["ot_periods"].astype(np.int64), ref["periods"])
    assert np.array_equal(got["ot_hist"][0].astype(np.int64), hist_from_rows(ref["scores"], ref["periods"], games))
    if counters:
        assert {k: got["counters"][k] for k in ORACLE_COUNTERS} == ref["counters"]
    assert got["counters"]["ot_games"] == int((ref["periods"] > 0).sum())
    assert got["counters"]["ot_periods"] == int(ref["periods"].sum())


# ---- 1. Philox games from the kickoff, game by game ------------------------------------------------------------------
@pytest.mark.parametrize("memo", ["on", "off", "persistent"])
def test_overtime_equals_the_oracle(memo_engines, oracle, models_s2, oto, memo):
    e = memo_engines[memo]
    n = 20_000
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    got = e.simulate_host(20251018, want_iters=True, overtime=RULES, want_ot_periods=True, want_ot_hist=True)
    ref = _oracle(oto, oracle.make_config(models_s2, KSU, ISU), n, seed=20251018)
    _check_against_oracle(got, ref, np.arange(n))
    assert 200 < got["counters"]["ot_games"] < 2000
    if memo != "off":
        assert got["counters"]["memo_hits"] > 0


@pytest.mark.parametrize("memo", ["on", "off"])
def test_overtime_traces(memo_engines, oracle, models_s2, oto, memo):
    """Trace rows bit for bit under injected draws (Philox traces may differ in the last bit of a yard line: a normal
    draw in the AS241 tail goes through `log`, where the device and glibc may round differently)."""
    e = memo_engines[memo]
    n = 3000
    stream = oracle.make_stream(n, 99)
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    got = e.simulate_host(0, stream=stream, want_iters=True, want_trace=True, overtime=OvertimeRules(8, 90),
                          want_ot_periods=True, want_ot_hist=True)
    ref = oto.simulate(oracle.make_config(models_s2, KSU, ISU), n, stream=stream, trace=True, max_periods=8, snap_clock=90)
    _check_against_oracle(got, ref, np.arange(n))
    assert (ref["periods"] > 0).sum() > 20
    live = np.arange(360)[None, :] < ref["iters"][:, None]
    assert np.array_equal(got["trace"][live], ref["trace"][live])


def test_overtime_equals_the_oracle_in_player_mode(engine, oracle, models_s2, oto):
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ctx = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    use = tuple(usage.resolve_team(tc, models_s2) for tc in ctx)
    n = 20_000
    spec = MatchupSpec("Kansas State", "Iowa State", ctx[0].sp, ctx[1].sp, n, 0, n, 0, usage=use)
    engine.set_matchups([spec])
    got = engine.simulate_host(1234, want_iters=True, want_players=True, overtime=RULES, want_ot_periods=True,
                               want_ot_hist=True)
    ref = _oracle(oto, oracle.make_config(models_s2, spec.sp_a, spec.sp_b), n, seed=1234, usage=oracle.make_usage(use),
                  n_slots=engine.n_slots)
    _check_against_oracle(got, ref, np.arange(n))
    _box_equal_philox(got["players"].dense(), ref["players"])


# ---- 2. the scripted streams -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("memo", ["on", "off"])
def test_scripted_streams(memo_engines, memo):
    e = memo_engines[memo]
    names = sorted(osc.SCENARIOS)
    for max_periods in sorted({osc.SCENARIOS[k][1] for k in names}):
        group = [k for k in names if osc.SCENARIOS[k][1] == max_periods]
        start = GameState(offense=0, seconds=0, score=osc.START_SCORE)
        specs = [MatchupSpec("A", "B", KSU, ISU, 2, 0, 2, 2 * i, start=start) for i in range(len(group))]
        e.set_matchups(specs)
        stream = np.concatenate([np.stack([osc.stream_for(osc.SCENARIOS[k][0])[0]] * 2) for k in group])
        got = e.simulate_host(0, stream=stream, want_iters=True, want_trace=True,
                              overtime=OvertimeRules(max_periods, 120), want_ot_periods=True)
        for i, k in enumerate(group):
            for g in (0, 1):
                sc, iters, periods = osc.expected(k, g)
                row = 2 * i + g
                assert (tuple(got["scores"][row]), got["iters"][row], got["ot_periods"][row]) == (sc, iters, periods), (k, g)
                assert (got["trace"][row, :iters, 2] == 120).all()


# ---- 3. overtime on against off at the same seed ---------------------------------------------------------------------
def test_on_against_off_at_one_million_games(memo_engines):
    e = memo_engines["on"]
    n = 1_000_000
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    off = e.simulate_host(7, want_iters=True)
    on = e.simulate_host(7, want_iters=True, overtime=RULES, want_ot_periods=True, want_ot_hist=True)
    level = off["scores"][:, 0] == off["scores"][:, 1]
    assert 0.01 < level.mean() < 0.06
    d = ~level
    assert np.array_equal(on["scores"][d], off["scores"][d]) and np.array_equal(on["iters"][d], off["iters"][d])
    assert (on["ot_periods"][d] == 0).all() and (on["ot_periods"][level] >= 1).all()
    extra = int((on["iters"][level] - off["iters"][level]).sum())
    assert extra > 0
    assert on["counters"]["iters"] - off["counters"]["iters"] == extra
    assert on["counters"]["games"] == off["counters"]["games"] == n
    assert on["counters"]["ot_games"] == int(level.sum())
    assert on["counters"]["ot_periods"] == int(on["ot_periods"].sum())
    assert off["counters"]["ot_games"] == off["counters"]["ot_periods"] == 0
    # each overtime iteration is one snap: a play, or a fourth-down kick
    snaps = lambda c: c["plays"] + c["fga"] + c["punt"]
    assert snaps(on["counters"]) - snaps(off["counters"]) == extra
    assert np.array_equal(on["ot_hist"][0].astype(np.int64), hist_from_rows(on["scores"], on["ot_periods"].astype(np.int64),
                                                                            np.arange(n)))
    # the score histogram holds the final scores, overtime included
    h = outputs.histogram_from_scores(on["scores"])
    assert np.array_equal(on["hist"][0].astype(np.int64), h)


# ---- 4. live starts: 0:00 level and late in the fourth quarter -------------------------------------------------------
def _curve():
    """150 states of the last 5 minutes, ending at 0:00 with the score level."""
    st = []
    for i in range(149):
        sec = 300 - 2 * i
        st.append(GameState(offense=i & 1, seconds=sec, down=1 + i % 4, distance=float(1 + i % 10),
                            yards_to_goal=float(10 + (7 * i) % 80), score=(14 + (i % 3) * 3, 14 + (i % 2) * 3)))
    st.append(GameState(offense=0, seconds=0, score=(17, 17)))
    return st


@pytest.mark.parametrize("memo", ["on", "off"])
def test_live_curve_equals_the_oracle(memo_engines, oracle, models_s2, oto, memo):
    e = memo_engines[memo]
    states = _curve()
    k = 300
    specs = [MatchupSpec("A", "B", KSU, ISU, k, 0, k, i * k, start=s) for i, s in enumerate(states)]
    e.set_matchups(specs)
    got = e.simulate_host(5, want_iters=True, overtime=RULES, want_ot_periods=True, want_ot_hist=True)
    cfg = oracle.make_config(models_s2, KSU, ISU)
    for i, s in enumerate(states):
        ref = oto.simulate(cfg, k, start=s, matchup=i, seed=5)
        rows = slice(i * k, (i + 1) * k)
        assert np.array_equal(got["scores"][rows], ref["scores"]), i
        assert np.array_equal(got["iters"][rows], ref["iters"]), i
        assert np.array_equal(got["ot_periods"][rows].astype(np.int64), ref["periods"]), i
        assert np.array_equal(got["ot_hist"][i].astype(np.int64), hist_from_rows(ref["scores"], ref["periods"], np.arange(k)))
    last = slice(149 * k, 150 * k)
    assert (got["ot_periods"][last] >= 1).all()


# ---- 5. the API ------------------------------------------------------------------------------------------------------
def test_simulate_live_overtime(engine):
    ks, isu = "Kansas State", "Iowa State"
    entries = [(ks, isu, api.LiveState(ks, 0, 1, 10.0, 75.0, (14, 14))),
               (ks, isu, api.LiveState(isu, 30, 1, 10.0, 75.0, (21, 21))),
               (ks, isu, api.LiveState(ks, 0, 1, 10.0, 75.0, (17, 14)))]
    plain = api.simulate_live(entries, 20_000, seed=21, engine=engine)
    res = api.simulate_live(entries, 20_000, seed=21, engine=engine, overtime=True)
    assert plain[0]["p_tie"] == 1.0 and res[0]["p_tie"] < 0.01
    assert res[0]["overtime"]["p_ot"] == 1.0 and res[0]["overtime"]["regulation"]["level"]["p"] == 1.0
    assert res[0]["p_win"][ks] == pytest.approx(res[0]["overtime"]["ot_win"][ks])
    assert 0.5 < res[1]["overtime"]["p_ot"] < 1.0
    assert res[2]["overtime"]["p_ot"] == 0.0 and np.array_equal(res[2]["hist"], plain[2]["hist"])
    for r in res:
        odds = outputs.live_odds_from_hist(r["hist"], ks, isu)
        assert r["p_win"] == odds["p_win"] and r["p_tie"] == odds["p_tie"]


def test_simulate_slate_and_matchup_overtime(engine):
    pairs = [("Kansas State", "Iowa State"), ("UTSA", "Ohio State")]
    plain = api.simulate_slate(pairs, n=20_000, seed=3, engine=engine)
    res = api.simulate_slate(pairs, n=20_000, seed=3, engine=engine, overtime=True,
                             markets={pairs[0]: {"spread": -3.5, "total": 50.5}})
    assert res["_counters"]["ot_games"] > 0 and plain["_counters"]["ot_games"] == 0
    for p in pairs:
        r = res[p]
        o = r["overtime"]
        assert 0.005 < o["p_ot"] < 0.1
        assert o["games"] == r["games"] == plain[p]["games"]
        pt = r["moneyline"]["team"]["p_win"] + r["moneyline"]["opp"]["p_win"]
        assert pt > plain[p]["moneyline"]["team"]["p_win"] + plain[p]["moneyline"]["opp"]["p_win"]
    assert res[pairs[0]]["markets"]["spread"]["samples"] == res[pairs[0]]["games"] // 2
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    A = priors.build_team_context_from_sp_flex("Kansas State", 2025, 1, sp)
    B = priors.build_team_context_from_sp_flex("Iowa State", 2025, 1, sp)
    df, _ = api.simulate_matchup(A, B, n=20_000, seed=3, engine=engine, overtime=True, show_progress=False)
    assert df.attrs["overtime"]["games"] == 40_000 and df.attrs["overtime"]["p_ot"] > 0
    ties = (df["pts"] == df["opp_pts"]).mean()
    assert ties < 0.001
