"""Fourth-down decisions on the B200 (fmc_game_state.fourth_down, the decision instantiations of both simulation
kernels): the forced-choice oracle game by game for all twelve instantiations (injected draws with traces, Philox with the
memo off, on and persistent, player mode with box lines, overtime on and off), the draw identity at one million games,
policy entries in a decision launch, the refusals, and the API."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import api, native, outputs, priors, usage
from fast_monte_carlo_b200.engine import GameState, MatchupSpec, OvertimeRules
from test_gpu_players import _box_equal_philox
from test_gpu_segments import memo_engines  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

ORACLE_COUNTERS = ("plays", "iters", "pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg", "punt", "go")
CODE = {None: 0, "go": 1, "fg": 2, "punt": 3}
S_U_GO = 8

# (state, choices): late and early, both sides of the 38, a tie-making kick, a punt from deep
CASES = [
    (GameState(offense=0, seconds=1500, down=4, distance=2.0, yards_to_goal=34.0, score=(10, 14)), (None, "go", "fg", "punt")),
    (GameState(offense=1, seconds=240, down=4, distance=6.0, yards_to_goal=55.0, score=(21, 17)), ("go", "punt", None)),
    (GameState(offense=0, seconds=25, down=4, distance=3.0, yards_to_goal=20.0, score=(14, 17)), ("fg", "go")),
    (GameState(offense=1, seconds=3000, down=4, distance=9.0, yards_to_goal=72.0, score=(0, 3)), ("punt", "go")),
]


@pytest.fixture(scope="module")
def fd(models_s2):
    import oracle_fourth_down
    oracle_fourth_down.load_models(models_s2)
    return oracle_fourth_down


def _entries():
    return [(st, c) for st, cs in CASES for c in cs]


def _specs(entries, k, usage_=None, a=("A", KSU), b=("B", ISU)):
    return [MatchupSpec(a[0], b[0], a[1], b[1], k, 0, k, i * k, usage=usage_,
                        start=GameState(**{**st.__dict__, "fourth_down": CODE[c]})) for i, (st, c) in enumerate(entries)]


def _check(got, fd, cfg, entries, k, overtime, trace=False, stream=None, seed=0, use=None, n_slots=0):
    tot = {c: 0 for c in ORACLE_COUNTERS}
    for i, (st, c) in enumerate(entries):
        rows = slice(i * k, (i + 1) * k)
        kw = dict(stream=stream[rows]) if stream is not None else dict(seed=seed)
        ref = fd.simulate(cfg, k, start=st, choice=c, matchup=i, overtime=overtime, trace=trace, usage=use,
                          n_slots=n_slots, **kw)
        assert np.array_equal(got["scores"][rows], ref["scores"]), (i, c)
        assert np.array_equal(got["iters"][rows], ref["iters"]), (i, c)
        if overtime:
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


def _run(e, entries, k, overtime, **kw):
    e.set_matchups(_specs(entries, k, kw.pop("usage_", None)))
    rules = OvertimeRules() if overtime else None
    return e.simulate_host(kw.pop("seed", 0), want_iters=True, overtime=rules, want_ot_periods=overtime, **kw)


# ---- 1. the twelve instantiations against the harness ----------------------------------------------------------------
@pytest.mark.parametrize("overtime", [False, True])
@pytest.mark.parametrize("memo", ["off", "on"])
def test_injected_draws_with_traces(memo_engines, oracle, models_s2, fd, memo, overtime):
    """The TEST instantiations of sim_kernel (memo off) and sim_memo_kernel (memo on), bit for bit with traces."""
    e, entries, k = memo_engines[memo], _entries(), 400
    stream = oracle.make_stream(k * len(entries), 17)
    got = _run(e, entries, k, overtime, stream=stream, want_trace=True)
    _check(got, fd, oracle.make_config(models_s2, KSU, ISU), entries, k, overtime, trace=True, stream=stream)


@pytest.mark.parametrize("overtime", [False, True])
@pytest.mark.parametrize("memo", ["off", "on", "persistent"])
def test_philox_games(memo_engines, oracle, models_s2, fd, memo, overtime):
    """The production instantiations, game by game under Philox (persistent: twice, the second on the kept memo)."""
    e, entries, k = memo_engines[memo], _entries(), 2000
    cfg = oracle.make_config(models_s2, KSU, ISU)
    for _ in range(2 if memo == "persistent" else 1):
        got = _run(e, entries, k, overtime, seed=20251022)
        _check(got, fd, cfg, entries, k, overtime, seed=20251022)
    if memo != "off":
        assert got["counters"]["memo_hits"] > 0


@pytest.fixture(scope="module")
def players_setup(models_s2):
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ctx = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    return ctx, tuple(usage.resolve_team(tc, models_s2) for tc in ctx)


@pytest.mark.parametrize("overtime", [False, True])
@pytest.mark.parametrize("rng", ["stream", "philox"])
def test_player_mode(engine, oracle, models_s2, fd, players_setup, rng, overtime):
    """The player instantiations (TEST with injected draws, production with Philox) with per-game box lines."""
    ctx, use = players_setup
    entries, k = _entries(), 500
    kw = dict(stream=oracle.make_stream(k * len(entries), 23)) if rng == "stream" else dict(seed=77)
    engine.set_matchups([MatchupSpec("Kansas State", "Iowa State", ctx[0].sp, ctx[1].sp, k, 0, k, i * k, usage=use,
                                     start=GameState(**{**st.__dict__, "fourth_down": CODE[c]}))
                         for i, (st, c) in enumerate(entries)])
    rules = OvertimeRules() if overtime else None
    got = engine.simulate_host(kw.get("seed", 0), stream=kw.get("stream"), want_iters=True, want_players=True,
                               overtime=rules, want_ot_periods=overtime)
    _check(got, fd, oracle.make_config(models_s2, ctx[0].sp, ctx[1].sp), entries, k, overtime,
           stream=kw.get("stream"), seed=kw.get("seed", 0), use=oracle.make_usage(use), n_slots=engine.n_slots)


# ---- 2. the draw identity at one million games -----------------------------------------------------------------------
def test_forced_to_its_own_branch_is_the_same_game_at_one_million(memo_engines, fd):
    """Every game of an unforced launch equals, game by game, the same game of the launch forced to the branch its own
    draw picks (score, iterations, overtime periods): go / kick from the 30, go / punt from midfield."""
    e = memo_engines["on"]
    n, seed = 1_000_000, 4242
    sts = [GameState(offense=0, seconds=1300, down=4, distance=2.0, yards_to_goal=30.0, score=(10, 13)),
           GameState(offense=1, seconds=700, down=4, distance=2.0, yards_to_goal=52.0, score=(17, 17))]
    other = ("fg", "punt")

    def launch(codes):
        e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, i * n, start=GameState(**{**st.__dict__, "fourth_down": c}))
                        for i, (st, c) in enumerate(zip(sts, codes))])
        return e.simulate_host(seed, want_iters=True, want_hist=False, overtime=OvertimeRules(), want_ot_periods=True)

    base = launch((0, 0))
    go = launch((CODE["go"], CODE["go"]))
    kick = launch((CODE[other[0]], CODE[other[1]]))
    for i, st in enumerate(sts):
        rows = slice(i * n, (i + 1) * n)
        b = fd.branches(fd.philox_u_many(seed, np.arange(n), i, S_U_GO), st)
        assert set(b) == {"go", other[i]} and 0.05 < (b == "go").mean() < 0.95
        for forced, name in ((go, "go"), (kick, other[i])):
            sel = b == name
            for key in ("scores", "iters", "ot_periods"):
                assert np.array_equal(forced[key][rows][sel], base[key][rows][sel]), (i, name, key)
            # ... and the games forced to the other branch are different games
            assert not np.array_equal(forced["scores"][rows][~sel], base["scores"][rows][~sel])


# ---- 3. policy entries in a decision launch --------------------------------------------------------------------------
@pytest.mark.parametrize("memo", ["off", "on"])
def test_policy_entries_of_a_decision_launch_are_unchanged(memo_engines, memo):
    e, k = memo_engines[memo], 20_000
    # each forced choice differs from the policy in some games (the policy always goes from CASES[1], always punts from
    # CASES[3])
    mixed = [(CASES[0][0], None), (CASES[0][0], "go"), (CASES[1][0], None), (CASES[1][0], "punt"),
             (CASES[2][0], None), (CASES[2][0], "fg"), (CASES[3][0], None), (CASES[3][0], "go")]
    plain = [(st, None) for st, _ in mixed]
    for overtime in (False, True):
        got = _run(e, mixed, k, overtime, seed=5)
        ref = _run(e, plain, k, overtime, seed=5)
        for i, (_, c) in enumerate(mixed):
            rows = slice(i * k, (i + 1) * k)
            same = np.array_equal(got["scores"][rows], ref["scores"][rows]) and np.array_equal(got["iters"][rows],
                                                                                               ref["iters"][rows])
            assert same == (c is None), (i, c, overtime)
            if c is None:
                assert np.array_equal(got["hist"][i], ref["hist"][i])


# ---- 4. refusals -------------------------------------------------------------------------------------------------------
def _state(**kw):
    base = dict(offense=0, seconds=600, down=4, distance=3.0, yards_to_goal=30.0, score=(7, 3), fourth_down=0)
    base.update(kw)
    return type("Raw", (), base)()     # bypasses GameState's own checks: the library checks again


@pytest.mark.parametrize("kw", [dict(fourth_down=4), dict(fourth_down=-1), dict(down=3, fourth_down=1),
                                dict(seconds=0, fourth_down=1), dict(yards_to_goal=38.5, fourth_down=2),
                                dict(yards_to_goal=15.0, fourth_down=3)])
def test_abi_refuses_invalid_choices(engine, kw):
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, 10, 0, 10, 0)])
    with pytest.raises(native.FmcError, match="fourth|field goal|punt"):
        engine.ctx.set_start_states([_state(**kw)])
    engine.ctx.set_start_states([_state(yards_to_goal=38.0, fourth_down=2)])
    engine.ctx.set_start_states([_state(yards_to_goal=16.0, fourth_down=3)])


@pytest.mark.parametrize("want", [dict(want_segments=True), dict(want_sequence=True), dict(want_period_scores=True)])
def test_abi_refuses_choices_with_period_or_sequence_outputs(engine, want):
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, 10, 0, 10, 0, start=CASES[0][0]),
                         MatchupSpec("A", "B", KSU, ISU, 10, 0, 10, 10,
                                     start=GameState(**{**CASES[0][0].__dict__, "fourth_down": 1}))])
    with pytest.raises(native.FmcError, match="fourth-down"):
        engine.simulate_host(1, **want)
    assert engine.simulate_host(1)["hist"].sum() == 20


# ---- 5. the API ------------------------------------------------------------------------------------------------------
def test_fourth_down_decisions(engine, monkeypatch):
    ks, isu = "Kansas State", "Iowa State"
    states = [(ks, isu, api.LiveState(ks, 420, 4, 2.0, 34.0, (17, 20))),
              (ks, isu, api.LiveState(isu, 1500, 4, 7.0, 65.0, (3, 0))),
              (ks, isu, api.LiveState(ks, 30, 4, 1.0, 6.0, (21, 24)))]
    calls = []
    real = engine.ctx.simulate_device
    monkeypatch.setattr(engine.ctx, "simulate_device", lambda **kw: calls.append(1) or real(**kw))
    games = 40_000
    res = api.fourth_down_decisions(states, games, seed=11, engine=engine, markets={0: {"spread": 2.5}})
    assert len(calls) == 1 and len(res) == 3
    assert set(res[0]["choices"]) == {"go", "fg", "punt"} and all(res[0]["choices"].values())
    assert res[1]["choices"]["fg"] is None and "fg" in res[1]["unavailable"]
    assert res[2]["choices"]["punt"] is None and "punt" in res[2]["unavailable"]
    for (a, b, st), r in zip(states, res):
        got = {k: v for k, v in r["choices"].items() if v is not None}
        for v in list(got.values()) + [r["policy"]]:
            assert {"hist", "p_win", "p_tie", "mean_points", "markets", "overtime"} <= set(v) and v["games"] == games
        dec = outputs.fourth_down_from_hists(dict({k: v["hist"] for k, v in got.items()}, policy=r["policy"]["hist"]),
                                             offense_is_a=st.offense == a)
        assert r["equity"] == dec["equity"] and r["best"] == dec["best"] and r["delta"] == dec["delta"]
        for c, v in got.items():
            assert r["equity"][c]["equity"] == pytest.approx(v["p_win"][st.offense] + v["p_tie"] / 2)
    assert res[0]["policy"]["markets"] is not None and res[0]["choices"]["go"]["markets"] is not None
    # the shared launch path: simulate_live on the same entries at the same seed gives the same histograms
    launch, mk, plan, _ = api._fourth_down_plan(states, None)
    live = api.simulate_live(launch, games, seed=11, engine=engine, overtime=True)
    for r, rows in zip(res, plan):
        for key, j in rows:
            mine = r["policy"] if key == "policy" else r["choices"][key]
            assert np.array_equal(mine["hist"], live[j]["hist"]), key
    # overtime off on request
    off = api.fourth_down_decisions(states[:1], 1000, seed=1, engine=engine, overtime=False)
    assert "overtime" not in off[0]["policy"]


def test_simulate_live_with_a_forced_choice(engine):
    ks, isu = "Kansas State", "Iowa State"
    st = api.LiveState(ks, 600, 4, 3.0, 30.0, (10, 10))
    forced = api.simulate_live([(ks, isu, st), (ks, isu, api.LiveState(ks, 600, 4, 3.0, 30.0, (10, 10), fourth_down="fg"))],
                               20_000, seed=3, engine=engine)
    plain = api.simulate_live([(ks, isu, st), (ks, isu, st)], 20_000, seed=3, engine=engine)
    assert np.array_equal(forced[0]["hist"], plain[0]["hist"])
    assert not np.array_equal(forced[1]["hist"], plain[1]["hist"])
