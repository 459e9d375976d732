"""Start states inside overtime (include/fmc.h fmc_overtime_state) on the CPU: the overtime harness started from every
overtime iteration of its own level games plays the rest of each game bit for bit; hand-built draw streams from
overtime states; forced fourth-down choices in overtime; the validation of the states the rules can reach."""
import dataclasses

import numpy as np
import pytest

import overtime_scripts as osc
from conftest import ISU, KSU
from fast_monte_carlo_b200 import api
from fast_monte_carlo_b200.engine import GameState, OvertimeState

ORACLE_COUNTERS = ("plays", "iters", "pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg", "punt", "go")


@pytest.fixture(scope="module")
def olive(models_s2):
    import oracle_overtime_live
    oracle_overtime_live.load_models(models_s2)
    return oracle_overtime_live


@pytest.fixture(scope="module")
def level_games(oracle, models_s2, olive):
    """20,000 harness games under a Philox-generated injected stream, with the overtime state of every iteration, and
    the resume states of their level games that did not end at the iteration cap."""
    cfg = oracle.make_config(models_s2, KSU, ISU)
    n = 20_000
    stream = oracle.make_stream(n, 5)
    res = olive.simulate_states(cfg, n, stream=stream, trace=True)
    rows = [int(i) for i in np.nonzero(res["periods"] > 0)[0] if res["iters"][i] < oracle.MAX_ITERS]
    return cfg, stream, res, rows, olive.resume_states(res, rows=rows)


def resume_stream(stream, i, j):
    """The draws of game i from iteration j on, as the stream of a game that starts there (the tail repeats the last
    record; a resumed game never reads it, since the original game ended before the cap)."""
    s = np.empty_like(stream[i])
    s[:stream.shape[1] - j] = stream[i, j:]
    s[stream.shape[1] - j:] = stream[i, -1]
    return s


# ---- 1. resume ---------------------------------------------------------------------------------------------------------
def test_the_states_of_the_overtime_harness_are_its_overtime_game(oracle, models_s2, level_games):
    """The state-recording copy of the overtime loop plays oracle_overtime.c's games."""
    import oracle_overtime
    cfg, stream, res, rows, _ = level_games
    oracle_overtime.load_models(models_s2)
    ref = oracle_overtime.simulate(cfg, len(res["iters"]), stream=stream, trace=True)
    for k in ("scores", "iters", "periods"):
        assert np.array_equal(res[k], ref[k]), k
    live = np.arange(oracle.MAX_ITERS)[None, :] < ref["iters"][:, None]
    assert np.array_equal(res["trace"][live], ref["trace"][live])
    assert res["counters"] == ref["counters"]
    assert 400 < len(rows) < 900      # about 3 % of the games are level after regulation


def test_resume_from_every_overtime_iteration(oracle, olive, level_games):
    cfg, stream, res, rows, states = level_games
    assert len(states) > 4000 and {g.overtime.two_point_try for _, _, g in states} == {False, True}
    assert {g.overtime.period for _, _, g in states} >= {1, 2, 3}
    firsts = {}
    for i, j, g in states:
        got = olive.simulate_start(cfg, 1, start=g, stream=resume_stream(stream, i, j)[None], game0=i, trace=True,
                                   states=True)
        n = int(got["iters"][0])
        assert tuple(got["scores"][0]) == tuple(res["scores"][i]), (i, j)
        assert n == res["iters"][i] - j, (i, j)
        assert got["periods"][0] == res["periods"][i], (i, j)
        assert np.array_equal(got["trace"][0, :n], res["trace"][i, j:j + n]), (i, j)
        assert np.array_equal(got["states"][0, :n], res["states"][i, j:j + n]), (i, j)
        if i not in firsts:
            firsts[i] = got["counters"]
    # counters: regulation of every game plus overtime resumed from its first snap = the original games
    reg = oracle.simulate(cfg, len(res["iters"]), stream=stream)["counters"]
    assert set(firsts) == set(rows)
    tot = {c: reg[c] + sum(f[c] for f in firsts.values()) for c in ORACLE_COUNTERS}
    assert tot == {c: res["counters"][c] for c in ORACLE_COUNTERS}


# ---- 2. hand-built streams from overtime states --------------------------------------------------------------------------
def _snaps(plan):
    """The snap records of a plan of possession kinds (overtime_scripts.KINDS) and single records."""
    return [r for k in plan for r in (osc.KINDS[k][0] if isinstance(k, str) else [k])]


def script_stream(plan):
    recs = _snaps(plan)
    s = np.tile(osc.INCOMPLETE, (osc.MAX_ITERS, 1))
    s[:len(recs)] = recs
    return s, len(recs)


def _ot(offense, score, period, possession=1, two_point_try=False, down=1, distance=10.0, ytg=25.0):
    if two_point_try:
        down, distance, ytg = 1, 3.0, 3.0
    return GameState(offense=offense, seconds=0, down=down, distance=distance, yards_to_goal=ytg, score=score,
                     overtime=OvertimeState(period, possession, two_point_try))


# name: (start, plan, max_periods, final score (A, B), last period played)
SCRIPTS = {
    # period 2, A scored the first touchdown (6): its try made, then B's touchdown does not win and its try fails
    "p2_first_try_made": (_ot(0, (27, 21), 2, 1, True), ["ok", "td", "fail"], 16, (29, 27), 2),
    # ... A's try failed, B's touchdown levels and its try wins
    "p2_first_try_failed": (_ot(0, (27, 21), 2, 1, True), ["fail", "td", "ok"], 16, (27, 29), 2),
    # B's try on the second possession of period 2 made: level, period 3 (B first) decides it
    "p2_second_try_made": (_ot(1, (29, 27), 2, 2, True), ["ok", "ok", "fail"], 16, (29, 31), 3),
    # ... failed: level after it, A wins period 3 on the second try
    "p2_second_try_failed": (_ot(1, (27, 27), 2, 2, True), ["fail", "fail", "ok"], 16, (29, 27), 3),
    # B, 3 down on the second possession of period 2, scores a touchdown that wins: no try
    "p2_td_wins_without_try": (_ot(1, (24, 21), 2, 2), ["td"], 16, (24, 27), 2),
    # the second try of period 3, then a shoot-out to period 6
    "p3_shoot_out": (_ot(1, (31, 29), 3, 2, True), ["ok", "fail", "fail", "ok", "ok", "ok", "fail"], 16, (33, 35), 6),
    # the first try of the last period allowed: level at the cap
    "cap_from_the_last_period": (_ot(0, (30, 30), 4, 1, True), ["fail", "fail"], 4, (30, 30), 4),
    # mid-possession: 3rd & 7 at the 10 on the second possession of period 1, 7 down; the touchdown levels
    "p1_mid_possession": (_ot(1, (28, 21), 1, 2, down=3, distance=7.0, ytg=10.0), [osc.SHORT_TD, "fg", "none"], 16,
                          (28, 31), 2),
}


@pytest.mark.parametrize("name", sorted(SCRIPTS))
@pytest.mark.parametrize("game", [0, 1])
def test_scripts_from_overtime_states(oracle, models_s2, olive, name, game):
    start, plan, max_periods, final, periods = SCRIPTS[name]
    stream, n = script_stream(plan)
    got = olive.simulate_start(oracle.make_config(models_s2, KSU, ISU), 1, start=start, stream=stream[None], game0=game,
                               max_periods=max_periods, trace=True, states=True)
    assert tuple(got["scores"][0]) == final
    assert got["iters"][0] == n and got["periods"][0] == periods
    assert tuple(got["states"][0, 0]) == (start.overtime.period, start.overtime.possession, int(start.overtime.two_point_try))
    first = game & 1
    assert got["trace"][0, 0, 0] == (1.0 if start.offense == first else 0.0)


# ---- 3. forced choices ---------------------------------------------------------------------------------------------------
FOURTH_DOWNS = [
    _ot(0, (24, 24), 1, 1, down=4, distance=2.0, ytg=30.0),      # level, inside the 38: go / kick to lead
    _ot(1, (27, 24), 2, 2, down=4, distance=5.0, ytg=20.0),      # 3 down: go / kick to level
    _ot(1, (21, 21), 2, 1, down=4, distance=3.0, ytg=45.0),      # level, outside the 38: go / punt (a team behind
                                                                 # at the snap clock of 120 s always goes)
]


def _available(st):
    return ["go"] + (["fg"] if st.yards_to_goal <= 38 else []) + (["punt"] if st.yards_to_goal >= 16 else [])


@pytest.mark.parametrize("i", range(len(FOURTH_DOWNS)))
def test_forced_choices_in_overtime(oracle, models_s2, olive, i):
    """A game whose own draw picks a branch is the same game forced to it; a forced choice plays its branch."""
    import oracle_fourth_down as fd
    st, n, seed = FOURTH_DOWNS[i], 20_000, 99
    cfg = oracle.make_config(models_s2, KSU, ISU)
    base = olive.simulate_start(cfg, n, start=st, seed=seed, matchup=i)
    # the policy's draw at the snap, which is played at the snap clock
    b = fd.branches(fd.philox_u_many(seed, np.arange(n), i, 8), dataclasses.replace(st, seconds=120, overtime=None))
    assert len(set(b)) == 2 and 0.02 < (b == "go").mean() < 0.98
    for c in _available(st):
        forced = olive.simulate_start(cfg, n, start=st, choice=c, seed=seed, matchup=i)
        sel = b == c       # (the policy never punts inside the 38 nor kicks outside it)
        for key in ("scores", "iters", "periods"):
            assert np.array_equal(forced[key][sel], base[key][sel]), (c, key)
        assert not np.array_equal(forced["scores"][~sel], base["scores"][~sel]), c
        assert forced["counters"][{"go": "go", "fg": "fga", "punt": "punt"}[c]] >= n


# ---- 4. validation -------------------------------------------------------------------------------------------------------
# (period, possession, try) -> the margins of the team with the ball the rules can reach
TABLE = [((1, 1, False), {0}), ((2, 1, False), {0}), ((1, 2, False), {0, -3, -7}), ((2, 2, False), {0, -3, -6, -8}),
         ((2, 1, True), {6}), ((2, 2, True), {0, -2})] + \
        [((k, 1, True), {0}) for k in (3, 4, 16)] + [((k, 2, True), {0, -2}) for k in (3, 4, 16)]


def table_states():
    """Every row of TABLE at its allowed margins and their neighbours: (GameState kwargs, allowed)."""
    out = []
    for (k, p, t), ok in TABLE:
        for d in sorted({x + e for x in ok for e in (-1, 0, 1)}):
            for off in (0, 1):
                sc = [20, 20]
                sc[off] += d
                kw = dict(offense=off, seconds=0, down=1, distance=3.0 if t else 10.0, yards_to_goal=3.0 if t else 25.0,
                          score=tuple(sc), overtime=OvertimeState(k, p, t))
                out.append((kw, d in ok))
    return out


def test_validation_of_the_margins():
    states = table_states()
    assert sum(ok for _, ok in states) == 2 * sum(len(ok) for _, ok in TABLE)
    for kw, ok in states:
        if ok:
            GameState(**kw)
        else:
            with pytest.raises(ValueError, match="margin"):
                GameState(**kw)


@pytest.mark.parametrize("kw, match", [
    (dict(overtime=OvertimeState(1, 1), seconds=5), "seconds 0"),
    (dict(overtime=OvertimeState(1, 1), offense=-1), "offense"),
    (dict(overtime=OvertimeState(3, 2, True), down=2), "down 1, distance 3"),
    (dict(overtime=OvertimeState(2, 1, True), yards_to_goal=25.0, distance=3.0, score=(26, 20)), "down 1, distance 3"),
    (dict(overtime=OvertimeState(2, 1, True), fourth_down=1, down=4, score=(26, 20)), "fourth"),
    (dict(overtime=(1, 1, False)), "OvertimeState"),
])
def test_validation_of_the_other_fields(kw, match):
    base = dict(offense=0, seconds=0, down=1, distance=3.0, yards_to_goal=3.0, score=(20, 20))
    if not kw["overtime"] or isinstance(kw["overtime"], tuple) or not kw["overtime"].two_point_try:
        base.update(distance=10.0, yards_to_goal=25.0)
    base.update(kw)
    with pytest.raises(ValueError, match=match):
        GameState(**base)


@pytest.mark.parametrize("args, match", [((1, 3), "possession"), ((0,), "period"), ((17,), "period"),
                                         ((1, 1, True), "period 1"), ((3, 1, False), "period 3")])
def test_overtime_state_refusals(args, match):
    with pytest.raises(ValueError, match=match):
        OvertimeState(*args)


def test_forced_choices_at_overtime_fourth_downs():
    for st in FOURTH_DOWNS:
        for c in (1, 2, 3):
            if (c == 2 and st.yards_to_goal > 38) or (c == 3 and st.yards_to_goal < 16):
                with pytest.raises(ValueError):
                    dataclasses.replace(st, fourth_down=c)
            else:
                dataclasses.replace(st, fourth_down=c)


def test_api_refusals_without_a_gpu():
    """simulate_live and fourth_down_decisions refuse overtime states before any launch."""
    ks, isu = "Kansas State", "Iowa State"
    st = api.LiveState(isu, 0, 4, 3.0, 8.0, (24, 21), overtime=api.OvertimeState(1, 2))
    assert api.live_game_state(ks, isu, st).overtime == OvertimeState(1, 2)
    as_dict = dict(offense=isu, seconds=0, down=4, distance=3.0, yards_to_goal=8.0, score=(24, 21),
                   overtime=dict(period=1, possession=2))
    assert api.live_game_state(ks, isu, as_dict) == api.live_game_state(ks, isu, st)
    with pytest.raises(ValueError, match="overtime"):
        api.simulate_live([(ks, isu, st)], 10, engine=object())
    with pytest.raises(ValueError, match="max_periods"):
        api.simulate_live([(ks, isu, api.LiveState(ks, 0, 1, 3.0, 3.0, (30, 30), overtime=api.OvertimeState(5, 1, True)))],
                          10, engine=object(), overtime=api.OvertimeRules(max_periods=4))
    try_state = api.LiveState(ks, 0, 1, 3.0, 3.0, (30, 30), overtime=api.OvertimeState(3, 1, True))
    with pytest.raises(ValueError, match="fourth down"):
        api.fourth_down_decisions([(ks, isu, try_state)], 10, engine=object())
    with pytest.raises(ValueError, match="margin"):
        api.live_game_state(ks, isu, dataclasses.replace(st, score=(24, 22)))
