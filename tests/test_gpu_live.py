"""Games from an in-game state on the B200 (fmc_set_start_states, shared specialisations, `simulate_live`): the GPU
against the kickoff launch, the reference's own games resumed mid-game, and the C oracle from chosen states."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import api, outputs, priors, usage
from fast_monte_carlo_b200.engine import Engine, GameState, MatchupSpec

pytestmark = pytest.mark.gpu

OSU, UTSA = (29.5, 39.6, 10.1), (0.0, 33.9, 33.9)
GAME_COUNTERS = ("games", "plays", "iters", "pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg", "punt", "go",
                 "hist_overflow")
ORACLE_COUNTERS = ("plays", "iters", "pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg", "punt", "go")


@pytest.fixture(scope="module")
def live(models_s2):
    """The C oracle with a start record per game (tests/oracle_live.py), every forest loaded."""
    import oracle_live
    oracle_live.load_models(models_s2)
    return oracle_live

# states a user asks about, each with what makes it interesting
STATES = {
    "goal_line_4th": GameState(offense=0, seconds=2000, down=4, distance=1.0, yards_to_goal=1.0, score=(10, 14)),
    "own_1": GameState(offense=1, seconds=3000, down=1, distance=10.0, yards_to_goal=99.0, score=(3, 0)),
    "crosses_half": GameState(offense=0, seconds=1801, down=2, distance=7.0, yards_to_goal=60.0, score=(14, 7)),
    "four_min_trailing": GameState(offense=1, seconds=240, down=1, distance=10.0, yards_to_goal=70.0, score=(21, 17)),
    "over": GameState(offense=1, seconds=0, down=3, distance=4.0, yards_to_goal=32.0, score=(24, 17)),
    "rout_130_0": GameState(offense=0, seconds=900, down=1, distance=10.0, yards_to_goal=75.0, score=(130, 0)),
}


@pytest.fixture(scope="module")
def memo_engines(models_s2, native_lib):
    engines = {m: Engine(models_s2, device=0, stage2="standin", memo=m) for m in ("on", "off", "persistent")}
    yield engines
    for e in engines.values():
        e.close()


def _trace_equal(a, b):
    return bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


def _game_counters(c):
    return {k: c[k] for k in GAME_COUNTERS}


@pytest.mark.parametrize("memo", ["on", "off", "persistent"])
def test_kickoff_state_equals_default_launch(memo_engines, memo):
    """200 k Philox games with an explicit kickoff start record (offense -1) are the default launch's games."""
    e = memo_engines[memo]
    n = 200_000
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    base = e.simulate_host(20251018, want_iters=True)
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0, start=GameState())])
    got = e.simulate_host(20251018, want_iters=True)
    assert np.array_equal(got["scores"], base["scores"])
    assert np.array_equal(got["iters"], base["iters"])
    assert np.array_equal(got["hist"], base["hist"])
    assert _game_counters(got["counters"]) == _game_counters(base["counters"])
    assert (got["counters"]["memo_probes"] > 0) == (memo != "off")


def _reference_resume_entries():
    """One-game entries for every iteration start of both reference fixtures whose state is a real game state (the
    reference's rules also reach downs past 4 and yard lines past 100, which fmc_set_start_states rejects; the CPU test
    resumes the oracle at those too): (specs, stream rows, expected (iters, trace rows, scores))."""
    from oracle import c_oracle as co
    from streams import adversarial_stream
    specs, rows, want = [], [], []
    for name, make in (("ref_trajectories.npz", co.make_stream), ("ref_trajectories_adversarial.npz", adversarial_stream)):
        t = np.load(os.path.join(GOLDEN, name))
        meta = json.loads(str(t["meta"]))
        stream = make(len(meta), int(t["stream_seed"]))
        for g, m in enumerate(meta):
            spA, spB = (m["sp_second"], m["sp_first"]) if g & 1 else (m["sp_first"], m["sp_second"])
            first, n = g & 1, int(t["iters"][g])
            for k in range(n):
                r = t["traces"][g, k]
                if r[1] > 4 or not (0.0 < r[6] < 100.0):
                    continue
                score = [0, 0]
                score[first], score[first ^ 1] = int(r[3]), int(r[4])
                st = GameState(offense=first if r[0] == 1.0 else first ^ 1, seconds=int(r[2]), down=int(r[1]),
                               distance=float(r[5]), yards_to_goal=float(r[6]), score=tuple(score))
                specs.append(MatchupSpec("A", "B", tuple(spA), tuple(spB), g + 1, g, g + 1, len(specs), start=st))
                row = np.zeros((co.MAX_ITERS, co.N_SLOTS))
                row[:co.MAX_ITERS - k] = stream[g, k:]
                rows.append(row)
                want.append((n - k, t["traces"][g, k:n], (t["scores"][g][0], t["scores"][g][1]) if first == 0
                             else (t["scores"][g][1], t["scores"][g][0])))
    return specs, np.stack(rows), want


@pytest.mark.parametrize("memo", ["on", "off"])
def test_reference_games_resumed_in_one_launch(memo_engines, memo):
    """Every iteration start of the reference's own games as a one-game entry with its own start state and draw row, all
    in ONE launch: each entry plays the rest of the reference's game bit for bit.  The entries share a handful of
    specialisations, so the memo stays on past 1,024 entries."""
    e = memo_engines[memo]
    specs, stream, want = _reference_resume_entries()
    assert len(specs) > 6000
    e.set_matchups(specs)
    got = e.simulate_host(0, stream=stream, want_trace=True, want_iters=True)
    for i, (n, rows, sc) in enumerate(want):
        assert got["iters"][i] == n, i
        assert np.array_equal(got["trace"][i, :n], rows), i
        assert tuple(got["scores"][i]) == tuple(sc), i
    assert (got["counters"]["memo_probes"] > 0) == (memo == "on")


@pytest.mark.parametrize("name", list(STATES))
def test_chosen_states_vs_oracle(engine, oracle, models_s2, name, live):
    """Game by game against the oracle from the same start state: injected draws (trajectories bit for bit) and Philox
    (scores, iterations, counters)."""
    st = STATES[name]
    cfg = oracle.make_config(models_s2, KSU, ISU)
    n = 4096
    stream = oracle.make_stream(n, 23)
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0, start=st)])
    got = engine.simulate_host(0, stream=stream, want_trace=True, want_iters=True)
    ref = live.simulate(cfg, n, stream=stream, trace=True, start=st)
    assert np.array_equal(got["scores"], ref["scores"])
    assert np.array_equal(got["iters"], ref["iters"])
    assert _trace_equal(got["trace"], ref["trace"])
    n = 50_000
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0, start=st)])
    got = engine.simulate_host(77, want_iters=True)
    ref = live.simulate(cfg, n, seed=77, start=st)
    assert np.array_equal(got["scores"], ref["scores"])
    assert np.array_equal(got["iters"], ref["iters"])
    for k in ORACLE_COUNTERS:
        assert got["counters"][k] == ref["counters"][k], k
    assert got["counters"]["games"] == n
    h = got["hist"][0]
    assert int(h.sum()) == n
    if name == "over":
        assert (got["iters"] == 0).all() and (got["scores"] == [24, 17]).all()
    if name == "rout_130_0":
        assert got["counters"]["hist_overflow"] == n and int(h[:, 127, :].sum()) == n
    else:
        assert got["counters"]["hist_overflow"] == 0


def _random_states(rng, k):
    out = []
    for _ in range(k):
        ytg = float(rng.integers(1, 100))
        out.append(GameState(offense=int(rng.integers(-1, 2)), seconds=int(rng.integers(0, 3601)), down=int(rng.integers(1, 5)),
                             distance=float(min(ytg, rng.integers(1, 16))), yards_to_goal=ytg,
                             score=(int(rng.integers(0, 50)), int(rng.integers(0, 50)))))
    return out


def test_one_pair_many_states_shares_tables_and_memo(oracle, models_s2, live):
    """1,500 entries of one pair: one table set, one memo id, the memo engaged (a memo per entry would be switched off
    past 1,024 entries), and every entry equals the oracle's games of that entry index."""
    e = Engine(models_s2, device=0, stage2="standin", memo="on")
    try:
        states = _random_states(np.random.default_rng(3), 1500)
        per = 32
        specs = [MatchupSpec("A", "B", KSU, ISU, per, 0, per, m * per, start=s) for m, s in enumerate(states)]
        e.set_matchups(specs)
        got = e.simulate_host(4242, want_iters=True)
        assert got["counters"]["memo_probes"] > 0 and got["counters"]["memo_hits"] > 0
        assert np.array_equal(e.ctx.packed_slots(1499), e.ctx.packed_slots(0))
        cfg = oracle.make_config(models_s2, KSU, ISU)
        for m, s in enumerate(states):
            ref = live.simulate(cfg, per, matchup=m, seed=4242, start=s, threads=1)
            assert np.array_equal(got["scores"][m * per:(m + 1) * per], ref["scores"]), m
            assert np.array_equal(got["iters"][m * per:(m + 1) * per], ref["iters"]), m
    finally:
        e.close()


def test_mixed_slate_of_pairs_and_states(engine, oracle, models_s2, live):
    """Three pairs, several states each, interleaved: entry by entry equal to the oracle."""
    pairs = [(KSU, ISU), (OSU, UTSA), (ISU, KSU)]
    states = _random_states(np.random.default_rng(9), 12)
    per = 3000
    specs = [MatchupSpec("A", "B", *pairs[m % 3], per, 0, per, m * per, start=s) for m, s in enumerate(states)]
    engine.set_matchups(specs)
    got = engine.simulate_host(31337, want_iters=True)
    for m, s in enumerate(states):
        cfg = oracle.make_config(models_s2, *pairs[m % 3])
        ref = live.simulate(cfg, per, matchup=m, seed=31337, start=s)
        assert np.array_equal(got["scores"][m * per:(m + 1) * per], ref["scores"]), m
        assert np.array_equal(got["iters"][m * per:(m + 1) * per], ref["iters"]), m
        h = got["hist"][m]
        assert np.array_equal(h, outputs.histogram_from_scores(got["scores"][m * per:(m + 1) * per]))


def test_warm_memo_survives_a_state_change(models_s2):
    """memo="persistent": a new start state keeps the tables and the memo, so state s2 after s1 hits more than s2 on a
    fresh engine -- with the same games."""
    s1 = GameState(offense=0, seconds=2700, down=1, distance=10.0, yards_to_goal=75.0, score=(7, 3))
    s2 = GameState(offense=1, seconds=2650, down=2, distance=6.0, yards_to_goal=68.0, score=(7, 3))
    n = 200_000
    warm = Engine(models_s2, device=0, stage2="standin", memo="persistent")
    cold = Engine(models_s2, device=0, stage2="standin", memo="persistent")
    try:
        warm.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0, start=s1)])
        warm.simulate_host(1)
        warm.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0, start=s2)])
        a = warm.simulate_host(2)
        cold.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0, start=s2)])
        b = cold.simulate_host(2)
        assert np.array_equal(a["scores"], b["scores"])
        assert a["counters"]["memo_hits"] > b["counters"]["memo_hits"] > 0
    finally:
        warm.close()
        cold.close()


def test_player_mode_from_a_start_state(engine, oracle, models_s2, live):
    """The player instantiation from a start state against fo_simulate_players: scores and boxes bit for bit under
    injected draws."""
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ctx = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    use = tuple(usage.resolve_team(tc, models_s2) for tc in ctx)
    st = GameState(offense=1, seconds=1361, down=3, distance=4.0, yards_to_goal=32.0, score=(24, 17))
    n = 4096
    stream = oracle.make_stream(n, 41)
    spec = MatchupSpec("Kansas State", "Iowa State", ctx[0].sp, ctx[1].sp, n, 0, n, 0, usage=use, start=st)
    engine.set_matchups([spec])
    assert engine.ctx.has_usage and engine.n_slots > 0
    got = engine.simulate_host(0, stream=stream, want_trace=True, want_iters=True, want_players=True)
    cfg = oracle.make_config(models_s2, spec.sp_a, spec.sp_b)
    ref = live.simulate(cfg, n, stream=stream, trace=True, usage=oracle.make_usage(use), n_slots=engine.n_slots, start=st)
    assert np.array_equal(got["scores"], ref["scores"])
    assert np.array_equal(got["iters"], ref["iters"])
    assert _trace_equal(got["trace"], ref["trace"])
    assert np.array_equal(got["players"].dense(), ref["players"])
    assert got["players"].dense()[..., 1].sum() > 0


def test_split_game_range_adds_up(engine):
    st = STATES["four_min_trailing"]
    n = 60_000
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0, start=st)])
    whole = engine.simulate_host(5)["hist"]
    parts = 0
    for g0, g1 in (api.shard_range(n, r, 3) for r in range(3)):
        engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, g0, g1, 0, start=st)])
        parts = parts + engine.simulate_host(5)["hist"].astype(np.int64)
    assert np.array_equal(parts, whole)


def test_simulate_live_api(engine):
    ks, isu = "Kansas State", "Iowa State"
    entries = [
        (ks, isu, api.LiveState(isu, 900 + 461, 3, 4.0, 32.0, (24, 17))),
        (ks, isu, api.LiveState(isu, 10, 1, 10.0, 75.0, (50, 0))),            # a 50-point lead with 10 s left
        (isu, ks, dict(offense=isu, seconds=3000, down=1, distance=10.0, yards_to_goal=75.0, score=(0, 7))),
    ]
    out = api.simulate_live(entries, 20_000, seed=11, engine=engine, markets={0: {"spread": -3.5, "total": 55.5}})
    assert [r["state"] for r in out] == [e[2] for e in entries]
    for r, (a, b, _) in zip(out, entries):
        assert r["games"] == 20_000 and int(r["hist"].sum()) == 20_000 and r["hist"].shape == (128, 128)
        assert r["p_win"][a] + r["p_win"][b] + r["p_tie"] == pytest.approx(1.0, abs=1e-12)
        assert r["hist_overflow"] == 0
    assert out[1]["p_win"][ks] == 1.0 and out[1]["mean_points"][ks] >= 50
    assert out[0]["mean_points"][ks] >= 24 and out[0]["mean_points"][isu] >= 17
    assert set(out[0]["markets"]) == {"spread", "total"} and out[1]["markets"] is None
    with pytest.raises(ValueError):
        api.simulate_live([(ks, isu, api.LiveState("Kansas", 100, 1, 10.0, 75.0))], 10, engine=engine)
