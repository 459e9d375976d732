"""Next-score, drive-result and race-to-N markets on the B200 (fmc_simulate_markets, the sequence hooks of both simulation
kernels): the reference's games under their injected draws, the sequence harness game by game from the kickoff and from
live starts, the histograms against the per-game rows, nothing else moving, and the API."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import api, outputs, priors, usage
from fast_monte_carlo_b200.engine import GameState, MatchupSpec
from fast_monte_carlo_b200.native import SEQ_NONE, seq_bin_next
from test_gpu_segments import GAME_COUNTERS, _reference_entries, memo_engines  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

NB = outputs.SEQ_BINS


@pytest.fixture(scope="module")
def seqo(models_s2):
    import oracle_sequence
    oracle_sequence.load_models(models_s2)
    return oracle_sequence


def hist_from_rows(seq, race, games):
    """[2][SEQ_BINS] of per-game sequence words and race results (harness layout), game ids `games`."""
    h = np.zeros((2, NB), dtype=np.int64)
    race = np.asarray(race, dtype=np.int64)
    o = np.asarray(games) & 1
    w0, w1 = seq[:, 0].astype(np.int64), seq[:, 1].astype(np.int64)
    none = w0 == SEQ_NONE
    nb = np.where(none, outputs.SEQ_BIN_NONE, seq_bin_next(w0 & 1, (w0 >> 1) & 1, np.maximum(w0 >> 2, 1)))
    np.add.at(h, (o, nb), 1)
    np.add.at(h, (o, outputs.SEQ_BIN_DRIVE0 + (w1 & 0xFF)), 1)
    for k in range(len(outputs.RACE_TARGETS)):
        ok = race[:, k] >= 0
        np.add.at(h, (o[ok], outputs.SEQ_BIN_RACE0 + 3 * k + race[ok, k]), 1)
    return h


def _harness(seqo, cfg, n, seed, start, matchup=0, chunk=5000, **kw):
    parts = [seqo.simulate(cfg, min(chunk, n - lo), game0=lo, matchup=matchup, seed=seed, start=start, **kw)
             for lo in range(0, n, chunk)]
    return {k: np.concatenate([p[k] for p in parts]) for k in ("scores", "sequence", "race")}


def _check_sums(h, n_games_by_orientation, settled):
    for o in range(2):
        n = n_games_by_orientation[o]
        assert int(h[o, :outputs.SEQ_BIN_DRIVE0].sum()) == n
        assert int(h[o, outputs.SEQ_BIN_DRIVE0:outputs.SEQ_BIN_RACE0].sum()) == n
        for k in range(len(outputs.RACE_TARGETS)):
            assert int(h[o, outputs.SEQ_BIN_RACE0 + 3 * k:outputs.SEQ_BIN_RACE0 + 3 * k + 3].sum()) == (0 if settled[k] else n)


# ---- 1. the reference's games under their injected draws --------------------------------------------------------------
@pytest.mark.parametrize("memo", ["on", "off"])
def test_reference_games_sequence(memo_engines, oracle, models_s2, seqo, memo):
    e = memo_engines[memo]
    specs, stream, _ = _reference_entries()
    e.set_matchups(specs)
    got = e.simulate_host(0, stream=stream, want_trace=True, want_sequence=True, want_sequence_hist=True)
    kick = GameState()
    for i, s in enumerate(specs):
        ref = seqo.simulate(oracle.make_config(models_s2, s.sp_a, s.sp_b), 1, game0=s.game_begin, stream=stream[i:i + 1],
                            start=kick)
        assert tuple(got["scores"][i]) == tuple(ref["scores"][0]), i
        assert np.array_equal(got["sequence"][i], ref["sequence"][0]), i
        assert np.array_equal(got["sequence_hist"][i].astype(np.int64), hist_from_rows(ref["sequence"], ref["race"],
                                                                                       [s.game_begin])), i


# ---- 2. Philox games from the kickoff, game by game ------------------------------------------------------------------
@pytest.mark.parametrize("memo", ["on", "off", "persistent"])
def test_sequence_equals_the_harness(memo_engines, oracle, models_s2, seqo, memo):
    e = memo_engines[memo]
    n = 20_000
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    got = e.simulate_host(8675309, want_sequence=True, want_sequence_hist=True)
    ref = _harness(seqo, oracle.make_config(models_s2, KSU, ISU), n, 8675309, GameState())
    assert np.array_equal(got["scores"][:, 0], ref["scores"][:, 0]) and np.array_equal(got["scores"][:, 1], ref["scores"][:, 1])
    assert np.array_equal(got["sequence"], ref["sequence"])
    assert np.array_equal(got["sequence_hist"][0].astype(np.int64), hist_from_rows(ref["sequence"], ref["race"], np.arange(n)))


def test_sequence_equals_the_harness_in_player_mode(engine, oracle, models_s2, seqo):
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ctx = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    use = tuple(usage.resolve_team(tc, models_s2) for tc in ctx)
    n = 20_000
    spec = MatchupSpec("Kansas State", "Iowa State", ctx[0].sp, ctx[1].sp, n, 0, n, 0, usage=use)
    engine.set_matchups([spec])
    got = engine.simulate_host(1234, want_sequence=True, want_sequence_hist=True, want_players=True)
    ref = _harness(seqo, oracle.make_config(models_s2, spec.sp_a, spec.sp_b), n, 1234, GameState(),
                   usage=oracle.make_usage(use))
    assert np.array_equal(got["sequence"], ref["sequence"])
    assert np.array_equal(got["sequence_hist"][0].astype(np.int64), hist_from_rows(ref["sequence"], ref["race"], np.arange(n)))


# ---- 3. live starts, game by game --------------------------------------------------------------------------------------
def _live_states():
    st = [GameState(offense=0, seconds=1500, down=4, distance=2.0, yards_to_goal=30.0, score=(7, 3)),     # 4th down: FG range
          GameState(offense=1, seconds=2400, down=4, distance=8.0, yards_to_goal=70.0),                   # 4th down: punt
          GameState(offense=0, seconds=0, down=1, distance=10.0, yards_to_goal=75.0, score=(21, 14)),     # clock 0
          GameState(offense=1, seconds=1200, down=1, distance=10.0, yards_to_goal=75.0, score=(10, 15)),  # at targets
          GameState(offense=0, seconds=600, down=2, distance=5.0, yards_to_goal=45.0, score=(30, 24))]    # past targets
    # one snap before each quarter boundary
    st += [GameState(offense=b % 2, seconds=b + 5, down=2, distance=7.0, yards_to_goal=52.0, score=(3, 7)) for b in (2700, 1800, 900)]
    st += [GameState(offense=0, seconds=5, down=3, distance=3.0, yards_to_goal=20.0, score=(17, 17))]
    return st


def _curve_states(k=150):
    rng = np.random.default_rng(7)
    out = []
    for i in range(k):
        sec = int(3600 - i * 24)
        out.append(GameState(offense=i % 2, seconds=sec, down=int(rng.integers(1, 5)), distance=float(rng.integers(1, 15)),
                             yards_to_goal=float(rng.integers(15, 95)), score=(int(rng.integers(0, 5)) * 7,
                                                                                 int(rng.integers(0, 4)) * 3)))
    return out


def _check_entries(e, oracle, models_s2, seqo, states, per, seed, check_games):
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, per, 0, per, m * per, start=s) for m, s in enumerate(states)])
    got = e.simulate_host(seed, want_sequence=True, want_sequence_hist=True)
    cfg = oracle.make_config(models_s2, KSU, ISU)
    for m, s in enumerate(states):
        rows = got["sequence"][m * per:(m + 1) * per]
        ref = _harness(seqo, cfg, check_games, seed, s, matchup=m)
        assert np.array_equal(rows[:check_games], ref["sequence"]), m
        settled = [max(s.score) >= t for t in outputs.RACE_TARGETS]
        h = got["sequence_hist"][m].astype(np.int64)
        _check_sums(h, ((per + 1) // 2, per // 2), settled)
        if check_games == per:
            assert np.array_equal(h, hist_from_rows(ref["sequence"], ref["race"], np.arange(per))), m
        if s.seconds == 0:
            assert (rows[:, 0] == SEQ_NONE).all() and (rows[:, 1] == outputs.DRIVE_RESULTS.index("end_of_game")).all()
    return got


@pytest.mark.parametrize("memo", ["on", "off"])
def test_live_starts_equal_the_harness(memo_engines, oracle, models_s2, seqo, memo):
    _check_entries(memo_engines[memo], oracle, models_s2, seqo, _live_states(), 10_000, 4711, 10_000)


def test_curve_of_150_states_equals_the_harness(memo_engines, oracle, models_s2, seqo):
    _check_entries(memo_engines["on"], oracle, models_s2, seqo, _curve_states(), 2000, 99, 2000)


# ---- 4. the histograms are the per-game rows ---------------------------------------------------------------------------
def test_sequence_hist_equals_the_per_game_rows(engine, oracle, models_s2, seqo):
    n = 1_000_000
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    got = engine.simulate_host(99, want_sequence=True, want_sequence_hist=True)
    h = got["sequence_hist"][0].astype(np.int64)
    _check_sums(h, (n // 2, n // 2), [False] * len(outputs.RACE_TARGETS))
    # next-score and drive bins from the rows (the race is not in them: its bins against the final scores)
    rows = got["sequence"]
    no_race = np.full((n, len(outputs.RACE_TARGETS)), -1, dtype=np.int64)
    want = hist_from_rows(rows, no_race, np.arange(n))
    assert np.array_equal(h[:, :outputs.SEQ_BIN_RACE0], want[:, :outputs.SEQ_BIN_RACE0])
    assert ((rows[:, 0] == SEQ_NONE) == (got["scores"] == 0).all(axis=1)).all()
    sc, o = got["scores"].astype(np.int64), np.arange(n) & 1
    for k, t in enumerate(outputs.RACE_TARGETS):
        for side in range(2):
            sel = o == side
            r = h[side, outputs.SEQ_BIN_RACE0 + 3 * k:outputs.SEQ_BIN_RACE0 + 3 * k + 3]
            assert r[2] == int(((sc[sel, 0] < t) & (sc[sel, 1] < t)).sum())
            assert r[0] <= int((sc[sel, 0] >= t).sum()) and r[1] <= int((sc[sel, 1] >= t).sum())


# ---- 5. nothing else moves ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("memo", ["on", "off"])
def test_outputs_unchanged_by_the_sequence_hooks(memo_engines, memo):
    e = memo_engines[memo]
    n = 300_000
    st = GameState(offense=0, seconds=2000, down=3, distance=4.0, yards_to_goal=48.0, score=(7, 10))
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0), MatchupSpec("A", "B", ISU, KSU, n, 0, n, n, start=st)])
    base = e.simulate_host(2024, want_iters=True, want_period_scores=True, want_segments=True)
    seq = e.simulate_host(2024, want_iters=True, want_sequence=True, want_sequence_hist=True)
    both = e.simulate_host(2024, want_iters=True, want_period_scores=True, want_segments=True, want_sequence=True,
                           want_sequence_hist=True)
    for k in ("scores", "hist", "iters"):
        assert np.array_equal(seq[k], base[k]) and np.array_equal(both[k], base[k]), k
    for k in ("period_scores", "segment_hist"):
        assert np.array_equal(both[k], base[k]), k
    for k in ("sequence", "sequence_hist"):
        assert np.array_equal(both[k], seq[k]), k
    want = {k: base["counters"][k] for k in GAME_COUNTERS}
    assert {k: seq["counters"][k] for k in GAME_COUNTERS} == want and {k: both["counters"][k] for k in GAME_COUNTERS} == want


def test_injected_draws_unchanged_by_the_sequence_hooks(engine, oracle):
    """The TEST instantiations with both hooks: trajectories, scores and iterations are those without hooks."""
    n = 2048
    stream = oracle.make_stream(n, 5)
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    a = engine.simulate_host(0, stream=stream, want_trace=True, want_iters=True)
    b = engine.simulate_host(0, stream=stream, want_trace=True, want_iters=True, want_period_scores=True,
                             want_sequence=True, want_sequence_hist=True)
    same = (a["trace"] == b["trace"]) | (np.isnan(a["trace"]) & np.isnan(b["trace"]))
    assert same.all()
    for k in ("scores", "iters", "hist"):
        assert np.array_equal(a[k], b[k]), k
    _check_sums(b["sequence_hist"][0].astype(np.int64), (n // 2, n // 2), [False] * 5)


# ---- 6. the API ----------------------------------------------------------------------------------------------------
def test_simulate_slate_sequence(engine):
    pairs = [("Kansas State", "Iowa State"), ("UTSA", "Ohio State")]
    plain = api.simulate_slate(pairs, n=5000, seed=3, engine=engine)
    res = api.simulate_slate(pairs, n=5000, seed=3, engine=engine, sequence=True)
    for p in pairs:
        r = res[p]
        assert np.array_equal(r["hist"], plain[p]["hist"])
        h = r["sequence_hist"]
        assert h.shape == (2, NB)
        odds = outputs.sequence_odds_from_hist(h, *p)
        assert r["first_score"] == odds["next_score"] and r["race"] == odds["race"]
        for o, t in enumerate(p):
            assert r["opening_drive"][t] == outputs.sequence_odds_from_hist(h[o], *p)["drive"]
    # the pregame first score is that of an entry started from the kickoff as a live state (the first pair is matchup 0)
    sp_df = priors.load_sp_flex(priors.packaged_priors_path())
    a, b = pairs[0]
    engine.set_matchups([MatchupSpec(a, b, priors.lookup_sp_flex(a, sp_df), priors.lookup_sp_flex(b, sp_df), 10_000, 0,
                                     10_000, 0, start=GameState())])
    live = engine.simulate_host(3, want_sequence_hist=True)
    assert np.array_equal(live["sequence_hist"][0], res[pairs[0]]["sequence_hist"])
    assert outputs.sequence_odds_from_hist(live["sequence_hist"][0], a, b)["next_score"] == res[pairs[0]]["first_score"]


def test_simulate_live_sequence(engine):
    ks, isu = "Kansas State", "Iowa State"
    entries = [
        (ks, isu, api.LiveState(ks, 3600, 1, 10.0, 75.0)),
        (ks, isu, api.LiveState(isu, 1805, 4, 12.0, 70.0, (10, 7))),
        (ks, isu, api.LiveState(ks, 400, 1, 10.0, 75.0, (24, 21))),
        (ks, isu, api.LiveState(ks, 0, 1, 10.0, 75.0, (14, 14))),
    ]
    plain = api.simulate_live(entries, 20_000, seed=21, engine=engine)
    res = api.simulate_live(entries, 20_000, seed=21, engine=engine, sequence=True)
    for i, (r, q) in enumerate(zip(res, plain)):
        assert np.array_equal(r["hist"], q["hist"])
        st = entries[i][2]
        odds = outputs.sequence_odds_from_hist(r["sequence_hist"], ks, isu, start_score=st.score)
        assert (r["next_score"], r["drive"], r["race"]) == (odds["next_score"], odds["drive"], odds["race"])
    assert res[1]["drive"]["p"]["punt"] > 0.5 and res[1]["race"][10] == {"settled": True, "winner": ks}
    assert res[2]["race"][25]["settled"] is False and res[2]["race"][20] == {"settled": True, "winner": None}
    assert res[3]["next_score"]["none"] == 1.0 and res[3]["drive"]["p"]["end_of_game"] == 1.0
    assert res[3]["race"][10] == {"settled": True, "winner": None} and res[3]["race"][15]["p"]["neither"] == 1.0
