"""Start states inside overtime on the B200 (fmc_set_start_states_overtime, the overtime instantiations of both simulation
kernels): the resume states of the harness's own level games in one launch, all twelve overtime instantiations against
the overtime start harness game by game (injected draws with traces, Philox with the memo off, on and persistent, player
mode with box lines, with and without forced choices), the draw identity of forced overtime choices, the independence of
regulation entries, the refusals and the API."""
import dataclasses
import os

import numpy as np
import pytest

from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import api, native, outputs, priors, usage
from fast_monte_carlo_b200.engine import GameState, MatchupSpec, OvertimeRules
from test_gpu_players import _box_equal_philox
from test_gpu_segments import memo_engines  # noqa: F401  (fixture)
from test_overtime_live import (FOURTH_DOWNS, ORACLE_COUNTERS, SCRIPTS, _ot, level_games, olive,  # noqa: F401
                                resume_stream, script_stream, table_states)

pytestmark = pytest.mark.gpu

CODE = {None: 0, "go": 1, "fg": 2, "punt": 3}
S_U_GO = 8

# (state, forced choice): every kind of overtime snap, and the fourth downs with each available choice
STARTS = [(_ot(0, (24, 24), 1, 1), None), (_ot(1, (24, 21), 1, 2, down=2, distance=6.0, ytg=19.0), None),
          (_ot(1, (30, 27), 2, 2), None), (_ot(0, (33, 27), 2, 1, True), None), (_ot(1, (35, 35), 3, 1, True), None),
          (_ot(0, (37, 39), 5, 2, True), None)]
FORCED = [(st, c) for st in FOURTH_DOWNS for c in (None, "go", "fg", "punt")
          if not (c == "fg" and st.yards_to_goal > 38) and not (c == "punt" and st.yards_to_goal < 16)]


def _spec(st, c, k, i, usage_=None, a=("A", KSU), b=("B", ISU), g0=0):
    return MatchupSpec(a[0], b[0], a[1], b[1], k, g0, g0 + k, i * k, usage=usage_,
                       start=dataclasses.replace(st, fourth_down=CODE[c]))


def _check(got, olive, cfg, entries, k, trace=False, stream=None, seed=0, use=None, n_slots=0):
    tot = {c: 0 for c in ORACLE_COUNTERS}
    for i, (st, c) in enumerate(entries):
        rows = slice(i * k, (i + 1) * k)
        kw = dict(stream=stream[rows]) if stream is not None else dict(seed=seed)
        ref = olive.simulate_start(cfg, k, start=st, choice=c, matchup=i, trace=trace, usage=use, n_slots=n_slots, **kw)
        assert np.array_equal(got["scores"][rows], ref["scores"]), (i, c)
        assert np.array_equal(got["iters"][rows], ref["iters"]), (i, c)
        assert np.array_equal(got["ot_periods"][rows].astype(np.int64), ref["periods"]), (i, c)
        if trace:
            live = np.arange(360)[None, :] < ref["iters"][:, None]
            assert np.array_equal(got["trace"][rows][live], ref["trace"][live]), (i, c)
        if use is not None:
            if stream is not None:
                assert np.array_equal(got["players"].dense()[rows], ref["players"]), (i, c)
            else:
                _box_equal_philox(got["players"].dense()[rows], ref["players"])
        for n in ORACLE_COUNTERS:
            tot[n] += ref["counters"][n]
    assert {n: got["counters"][n] for n in ORACLE_COUNTERS} == tot


def _run(e, entries, k, **kw):
    e.set_matchups([_spec(st, c, k, i, kw.pop("usage_", None)) for i, (st, c) in enumerate(entries)])
    return e.simulate_host(kw.pop("seed", 0), want_iters=True, overtime=OvertimeRules(), want_ot_periods=True, **kw)


# ---- 1. resume in one launch -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("memo", ["off", "on"])
def test_resume_states_in_one_launch(memo_engines, olive, level_games, memo):
    """Every resume state of the harness's level games as a one-game entry (its original game id), all in one launch:
    the rest of the original game, bit for bit, with traces."""
    cfg, stream, res, rows, states = level_games
    e = memo_engines[memo]
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, 1, i, i + 1, q, start=g) for q, (i, j, g) in enumerate(states)])
    st = np.stack([resume_stream(stream, i, j) for i, j, _ in states])
    got = e.simulate_host(0, stream=st, want_trace=True, want_iters=True, overtime=OvertimeRules(), want_ot_periods=True)
    tot = {c: 0 for c in ORACLE_COUNTERS}
    for q, (i, j, g) in enumerate(states):
        n = int(res["iters"][i]) - j
        assert tuple(got["scores"][q]) == tuple(res["scores"][i]), (i, j)
        assert got["iters"][q] == n and got["ot_periods"][q] == res["periods"][i], (i, j)
        assert np.array_equal(got["trace"][q, :n], res["trace"][i, j:j + n]), (i, j)
    ref = [olive.simulate_start(cfg, 1, start=g, stream=st[q:q + 1], game0=i)["counters"]
           for q, (i, j, g) in enumerate(states)]
    tot = {c: sum(r[c] for r in ref) for c in ORACLE_COUNTERS}
    assert {c: got["counters"][c] for c in ORACLE_COUNTERS} == tot
    assert got["counters"]["ot_games"] == len(states)


# ---- 2. the twelve overtime instantiations against the harness --------------------------------------------------------
@pytest.mark.parametrize("forced", [False, True])
@pytest.mark.parametrize("memo", ["off", "on"])
def test_injected_draws_with_traces(memo_engines, oracle, models_s2, olive, memo, forced):
    e, entries, k = memo_engines[memo], FORCED if forced else STARTS, 300
    stream = oracle.make_stream(k * len(entries), 29)
    got = _run(e, entries, k, stream=stream, want_trace=True)
    _check(got, olive, oracle.make_config(models_s2, KSU, ISU), entries, k, trace=True, stream=stream)


@pytest.mark.parametrize("forced", [False, True])
@pytest.mark.parametrize("memo", ["off", "on", "persistent"])
def test_philox_games(memo_engines, oracle, models_s2, olive, memo, forced):
    e, entries, k = memo_engines[memo], FORCED if forced else STARTS, 2000
    cfg = oracle.make_config(models_s2, KSU, ISU)
    for _ in range(2 if memo == "persistent" else 1):
        got = _run(e, entries, k, seed=20251023)
        _check(got, olive, cfg, entries, k, seed=20251023)
    if memo != "off":
        assert got["counters"]["memo_hits"] > 0


@pytest.fixture(scope="module")
def players_setup(models_s2):
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ctx = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    return ctx, tuple(usage.resolve_team(tc, models_s2) for tc in ctx)


@pytest.mark.parametrize("forced", [False, True])
@pytest.mark.parametrize("rng", ["stream", "philox"])
def test_player_mode(engine, oracle, models_s2, olive, players_setup, rng, forced):
    """The player instantiations with per-game box lines counted from the start state (a try credits none)."""
    ctx, use = players_setup
    entries, k = (FORCED if forced else STARTS), 400
    kw = dict(stream=oracle.make_stream(k * len(entries), 31)) if rng == "stream" else dict(seed=78)
    engine.set_matchups([_spec(st, c, k, i, use, ("Kansas State", ctx[0].sp), ("Iowa State", ctx[1].sp))
                         for i, (st, c) in enumerate(entries)])
    got = engine.simulate_host(kw.get("seed", 0), stream=kw.get("stream"), want_iters=True, want_players=True,
                               overtime=OvertimeRules(), want_ot_periods=True)
    _check(got, olive, oracle.make_config(models_s2, ctx[0].sp, ctx[1].sp), entries, k, stream=kw.get("stream"),
           seed=kw.get("seed", 0), use=oracle.make_usage(use), n_slots=engine.n_slots)


@pytest.mark.parametrize("name", sorted(SCRIPTS))
def test_scripts(memo_engines, name):
    """The hand-built streams from overtime states, as games 0 and 1 (either team the opening-kickoff receiver)."""
    start, plan, max_periods, final, periods = SCRIPTS[name]
    stream, n = script_stream(plan)
    for memo in ("off", "on"):
        e = memo_engines[memo]
        e.set_matchups([MatchupSpec("A", "B", KSU, ISU, 2, 0, 2, 0, start=start)])
        got = e.simulate_host(0, stream=np.stack([stream, stream]), want_iters=True, want_trace=True,
                              overtime=OvertimeRules(max_periods=max_periods), want_ot_periods=True, want_ot_hist=True)
        for g in (0, 1):
            assert tuple(got["scores"][g]) == final and got["iters"][g] == n and got["ot_periods"][g] == periods, (memo, g)
            assert got["trace"][g, 0, 0] == (1.0 if start.offense == g else 0.0)
        res = 0 if final[0] > final[1] else (1 if final[1] > final[0] else 2)
        assert got["ot_hist"][0, :, periods, res].tolist() == [1, 1]


# ---- 3. the draw identity ------------------------------------------------------------------------------------------------
def test_forced_to_its_own_branch_is_the_same_game(memo_engines):
    """Every game of a policy launch equals, game by game, the same game of the launch forced to the branch its own draw
    picks at the overtime snap (score, iterations, overtime periods), at 200,000 games per state."""
    import oracle_fourth_down as fd
    e, n, seed = memo_engines["on"], 200_000, 777

    def launch(st, c):
        e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0, start=dataclasses.replace(st, fourth_down=CODE[c]))])
        return e.simulate_host(seed, want_iters=True, want_hist=False, overtime=OvertimeRules(), want_ot_periods=True)

    for i, st in enumerate(FOURTH_DOWNS):
        base = launch(st, None)
        # the policy's draw at the snap, which is played at the snap clock
        b = fd.branches(fd.philox_u_many(seed, np.arange(n), 0, S_U_GO), dataclasses.replace(st, seconds=120, overtime=None))
        assert 0.02 < (b == "go").mean() < 0.98
        for c in set(b):
            forced = launch(st, c)
            sel = b == c
            for key in ("scores", "iters", "ot_periods"):
                assert np.array_equal(forced[key][sel], base[key][sel]), (i, c, key)
            assert not np.array_equal(forced["scores"][~sel], base["scores"][~sel]), (i, c)


# ---- 4. independence of the entries -------------------------------------------------------------------------------------
@pytest.mark.parametrize("memo", ["off", "on"])
def test_regulation_entries_are_unchanged_by_overtime_entries(memo_engines, memo):
    e, k = memo_engines[memo], 20_000
    reg = [GameState(), GameState(offense=1, seconds=0, down=1, distance=10.0, yards_to_goal=25.0, score=(14, 14)),
           GameState(offense=0, seconds=400, down=3, distance=4.0, yards_to_goal=30.0, score=(17, 20))]
    mixed = [reg[0], STARTS[0][0], reg[1], FORCED[1][0], reg[2], STARTS[4][0]]
    plain = [reg[0], reg[0], reg[1], reg[1], reg[2], reg[2]]
    out = []
    for sts in (mixed, plain):
        e.set_matchups([MatchupSpec("A", "B", KSU, ISU, k, 0, k, i * k, start=s) for i, s in enumerate(sts)])
        out.append(e.simulate_host(9, want_iters=True, overtime=OvertimeRules(), want_ot_periods=True))
    for i in (0, 2, 4):
        rows = slice(i * k, (i + 1) * k)
        for key in ("scores", "iters", "ot_periods"):
            assert np.array_equal(out[0][key][rows], out[1][key][rows]), (i, key)
        assert np.array_equal(out[0]["hist"][i], out[1]["hist"][i])


# ---- 5. refusals ---------------------------------------------------------------------------------------------------------
def _raw(kw):
    """A start state that bypasses GameState's own checks: the library checks again."""
    ot = kw.get("overtime")
    d = dict(kw, fourth_down=kw.get("fourth_down", 0),
             overtime=None if ot is None else type("RawOt", (), dict(period=ot.period, possession=ot.possession,
                                                                   two_point_try=ot.two_point_try))())
    return type("Raw", (), d)()


def test_abi_validation_of_the_margins(engine):
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, 10, 0, 10, 0)])
    for kw, ok in table_states():
        if ok:
            engine.ctx.set_start_states([_raw(kw)])
        else:
            with pytest.raises(native.FmcError, match="margin"):
                engine.ctx.set_start_states([_raw(kw)])


@pytest.mark.parametrize("kw, match", [
    (dict(seconds=5), "seconds 0"), (dict(offense=-1), "offense"), (dict(period=1, two_point_try=True), "period 1"),
    (dict(period=3, two_point_try=False), "period 3"), (dict(period=17), "period"), (dict(possession=3), "possession"),
    (dict(period=3, two_point_try=True, down=2), "down 1"), (dict(period=3, two_point_try=True, fourth_down=1, down=4), "fourth"),
])
def test_abi_refuses_other_fields(engine, kw, match):
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, 10, 0, 10, 0)])
    ot = {f: kw.pop(f) for f in ("period", "possession", "two_point_try") if f in kw}
    base = dict(offense=0, seconds=0, down=1, distance=10.0, yards_to_goal=25.0, score=(20, 20), fourth_down=0)
    if ot.get("two_point_try"):
        base.update(distance=3.0, yards_to_goal=3.0)
    base.update(kw)
    o = dict(period=1, possession=1, two_point_try=False)
    o.update(ot)
    st = type("Raw", (), dict(base, overtime=type("RawOt", (), o)()))()
    with pytest.raises(native.FmcError, match=match):
        engine.ctx.set_start_states([st])


def test_launch_refusals(engine):
    st = _ot(0, (30, 30), 4, 1, True)
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, 10, 0, 10, 0, start=st)])
    with pytest.raises(native.FmcError, match="overtime"):
        engine.simulate_host(1)
    with pytest.raises(native.FmcError, match="max_periods"):
        engine.simulate_host(1, overtime=OvertimeRules(max_periods=3))
    with pytest.raises(native.FmcError, match="overtime"):
        engine.simulate_host(1, want_segments=True)
    assert engine.simulate_host(1, overtime=OvertimeRules(max_periods=4))["hist"].sum() == 10
    # fmc_set_matchups and fmc_set_start_states return every entry to regulation
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, 10, 0, 10, 0)])
    assert engine.simulate_host(1)["hist"].sum() == 10
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, 10, 0, 10, 0, start=st)])
    engine.ctx.set_start_states([GameState()])
    assert engine.simulate_host(1)["hist"].sum() == 10


# ---- 6. the API ----------------------------------------------------------------------------------------------------------
def _count_launches(engine, monkeypatch):
    calls = []
    real = engine.ctx.simulate_device
    monkeypatch.setattr(engine.ctx, "simulate_device", lambda **kw: calls.append(1) or real(**kw))
    return calls


def test_simulate_live_curve_through_overtime(engine, level_games, monkeypatch):
    """Every snap of one overtime game as a curve, in one launch."""
    ks, isu = "Kansas State", "Iowa State"
    cfg, stream, res, rows, states = level_games
    i = max(rows, key=lambda r: sum(1 for ii, _, _ in states if ii == r))
    snaps = [g for ii, _, g in states if ii == i]
    assert len(snaps) >= 4
    names = (ks, isu)
    entries = [(ks, isu, api.LiveState(names[g.offense], 0, g.down, g.distance, g.yards_to_goal, g.score,
                                       overtime=g.overtime)) for g in snaps]
    calls = _count_launches(engine, monkeypatch)
    games = 20_000
    out = api.simulate_live(entries, games, seed=4, engine=engine, overtime=True)
    assert len(calls) == 1 and len(out) == len(snaps)
    for g, r in zip(snaps, out):
        ot = r["overtime"]
        assert r["games"] == games and ot["p_ot"] == pytest.approx(1.0)
        assert r["p_win"][ks] + r["p_win"][isu] + r["p_tie"] == pytest.approx(1.0)
        k = g.overtime.period
        assert all(p >= k for p, v in enumerate(ot["periods"]) if v > 0)
    # the same entries without the curve: the histograms do not depend on the other entries' presence
    one = api.simulate_live(entries[:1], games, seed=4, engine=engine, overtime=True)
    assert np.array_equal(one[0]["hist"], out[0]["hist"])


def test_fourth_down_decisions_in_overtime(engine, monkeypatch):
    """Iowa State has 4th & 3 at the 8 on the second possession of the first overtime, down 24-21: kick or go?"""
    ks, isu = "Kansas State", "Iowa State"
    states = [(ks, isu, api.LiveState(isu, 0, 4, 3.0, 8.0, (24, 21), overtime=api.OvertimeState(1, 2))),
              (ks, isu, api.LiveState(ks, 0, 4, 2.0, 30.0, (24, 24), overtime=api.OvertimeState(2, 1))),
              (ks, isu, api.LiveState(ks, 0, 4, 3.0, 45.0, (21, 21), overtime=api.OvertimeState(1, 1)))]
    calls = _count_launches(engine, monkeypatch)
    games = 40_000
    res = api.fourth_down_decisions(states, games, seed=12, engine=engine)
    assert len(calls) == 1 and len(res) == 3
    assert res[0]["choices"]["punt"] is None and res[2]["choices"]["fg"] is None
    for (a, b, st), r in zip(states, res):
        got = {k: v for k, v in r["choices"].items() if v is not None}
        dec = outputs.fourth_down_from_hists(dict({k: v["hist"] for k, v in got.items()}, policy=r["policy"]["hist"]),
                                             offense_is_a=st.offense == a)
        assert r["equity"] == dec["equity"] and r["best"] == dec["best"] and r["delta"] == dec["delta"]
        for c, v in got.items():
            assert v["games"] == games and v["overtime"]["p_ot"] == pytest.approx(1.0)
    with pytest.raises(ValueError, match="overtime"):
        api.fourth_down_decisions(states[:1], 100, engine=engine, overtime=False)


def test_simulate_live_refusals(engine):
    ks, isu = "Kansas State", "Iowa State"
    st = api.LiveState(isu, 0, 4, 3.0, 8.0, (24, 21), overtime=api.OvertimeState(1, 2))
    with pytest.raises(ValueError, match="overtime"):
        api.simulate_live([(ks, isu, st)], 100, engine=engine)
    with pytest.raises(ValueError, match="max_periods"):
        api.simulate_live([(ks, isu, dataclasses.replace(st, overtime=api.OvertimeState(2, 2)))], 100, engine=engine,
                          overtime=api.OvertimeRules(max_periods=1))
    with pytest.raises(ValueError, match="segments"):
        api.simulate_live([(ks, isu, st)], 100, engine=engine, overtime=True, segments=True)
    with pytest.raises(ValueError, match="margin"):
        api.simulate_live([(ks, isu, dataclasses.replace(st, score=(24, 20)))], 100, engine=engine, overtime=True)
