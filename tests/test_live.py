"""Games from an in-game state (start states, `simulate_live`) on the CPU: the oracle resumed at the reference's own
states, the kickoff as an explicit state, the live odds and the host-side validation."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import outputs
from fast_monte_carlo_b200.engine import GameState

FIXTURES = ("ref_trajectories.npz", "ref_trajectories_adversarial.npz")


@pytest.fixture(scope="module")
def live(models_s2):
    """The C oracle with a start record per game (tests/oracle_live.py), every forest loaded."""
    import oracle_live
    oracle_live.load_models(models_s2)
    return oracle_live


def fixture_stream(name, n, seed):
    if name == "ref_trajectories.npz":
        from oracle import c_oracle as co
        return co.make_stream(n, seed)
    from streams import adversarial_stream
    return adversarial_stream(n, seed)


def resume_points(name):
    """(meta, traces, iters, scores, stream) of a reference fixture."""
    t = np.load(os.path.join(GOLDEN, name))
    meta = json.loads(str(t["meta"]))
    return meta, t["traces"], t["iters"], t["scores"], fixture_stream(name, len(meta), int(t["stream_seed"]))


class _Raw:
    """A start record outside GameState's ranges: the reference's rules reach downs past 4 (an incomplete pass on
    fourth down is not a turnover) and yard lines past 100 (sacks), which no real game has."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def raw_state_at(trace_row, first):
    r = trace_row
    score = [0, 0]
    score[first], score[first ^ 1] = int(r[3]), int(r[4])
    return _Raw(offense=first if r[0] == 1.0 else first ^ 1, seconds=int(r[2]), down=int(r[1]), distance=float(r[5]),
                yards_to_goal=float(r[6]), score=score)


@pytest.mark.parametrize("name", FIXTURES)
def test_resume_at_every_reference_state(models, oracle, name, live):
    """For every game g and every iteration k of the reference's own games: the oracle started at the state of iteration k
    with draws stream[g, k:], as game g, plays the rest of the reference's game bit for bit (trace rows k.., iterations
    minus k, final score).  Game i of one oracle call has id g + i, so the states of game g go to the even i (the
    parity of g: the trace is relative to the kickoff receiver g & 1) and the odd i start with the clock at 0."""
    meta, traces, iters, scores, stream = resume_points(name)
    done = 0
    for g, m in enumerate(meta):
        spA, spB = (m["sp_second"], m["sp_first"]) if g & 1 else (m["sp_first"], m["sp_second"])
        cfg = oracle.make_config(models, spA, spB)
        first, n = g & 1, int(iters[g])
        over = _Raw(offense=0, seconds=0, down=1, distance=10.0, yards_to_goal=75.0, score=(0, 0))
        starts, draws = [], np.zeros((2 * n, oracle.MAX_ITERS, oracle.N_SLOTS))
        for k in range(n):
            starts += [raw_state_at(traces[g, k], first), over]
            draws[2 * k, :oracle.MAX_ITERS - k] = stream[g, k:]
        r = live.simulate(cfg, 2 * n, game0=g, stream=draws, trace=True, start=starts)
        for k in range(n):
            i = 2 * k
            assert r["iters"][i] == n - k, (g, k)
            assert np.array_equal(r["trace"][i, :n - k], traces[g, k:n]), (g, k)
            assert (r["scores"][i, first], r["scores"][i, first ^ 1]) == tuple(scores[g]), (g, k)
            assert r["iters"][i + 1] == 0
        done += n
    assert done == int(iters.sum())


@pytest.mark.parametrize("rng", ["philox", "stream"])
def test_kickoff_state_is_the_kickoff(models_s2, oracle, rng, live):
    """An explicit kickoff start record (offense -1: the receiver by game parity) plays exactly today's games."""
    cfg = oracle.make_config(models_s2, KSU, ISU, stage2="booster")
    n = 512
    kw = dict(stream=oracle.make_stream(n, 11)) if rng == "stream" else dict(seed=20251018)
    base = oracle.simulate(cfg, n, game0=3, trace=True, **kw)
    got = live.simulate(cfg, n, game0=3, trace=True, start=GameState(), **kw)
    assert np.array_equal(got["scores"], base["scores"])
    assert np.array_equal(got["iters"], base["iters"])
    assert np.array_equal(got["trace"], base["trace"], equal_nan=True)
    assert got["counters"] == base["counters"]


def test_kickoff_state_is_the_kickoff_in_player_mode(models_s2, oracle, live):
    """The same in player mode (usage tables, per-game box), against fo_simulate_players."""
    from fast_monte_carlo_b200 import priors, usage
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    tcs = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    use = oracle.make_usage(tuple(usage.resolve_team(tc, models_s2) for tc in tcs))
    cfg = oracle.make_config(models_s2, tcs[0].sp, tcs[1].sp)
    n, slots = 256, 12
    stream = oracle.make_stream(n, 13)
    base = oracle.simulate(cfg, n, stream=stream, usage=use, n_slots=slots)
    got = live.simulate(cfg, n, stream=stream, usage=use, n_slots=slots, start=GameState())
    assert np.array_equal(got["scores"], base["scores"]) and np.array_equal(got["iters"], base["iters"])
    assert np.array_equal(got["players"], base["players"]) and got["players"][..., 1].sum() > 0


def test_start_state_semantics(models, oracle, live):
    """A game that starts with the clock at 0 ends at once with the start score; the first trace row of a game is its
    start state; per-game start records apply game by game."""
    cfg = oracle.make_config(models, KSU, ISU)
    over = GameState(offense=1, seconds=0, down=3, distance=4.0, yards_to_goal=32.0, score=(24, 17))
    r = live.simulate(cfg, 8, seed=1, start=over)
    assert (r["iters"] == 0).all() and (r["scores"] == [24, 17]).all() and r["counters"]["plays"] == 0
    third_q = GameState(offense=1, seconds=1361, down=3, distance=4.0, yards_to_goal=32.0, score=(24, 17))
    r = live.simulate(cfg, 4, game0=6, seed=2, trace=True, start=third_q)
    for i in range(4):
        first = (6 + i) & 1
        assert list(r["trace"][i, 0]) == [float(first == 1), 3.0, 1361.0, float(third_q.score[first]),
                                          float(third_q.score[first ^ 1]), 4.0, 32.0, 0.0]
        assert (r["scores"][i] >= [24, 17]).all()
    mixed = [over, GameState(), third_q]
    r = live.simulate(cfg, 3, seed=3, start=mixed)
    assert r["iters"][0] == 0 and r["iters"][1] > 0 and r["iters"][2] > 0


def test_live_odds_brute_force():
    """live_odds_from_hist against a direct count over a random score table, ties and clamped bins included."""
    rng = np.random.default_rng(5)
    n = 20_000
    a = rng.integers(0, 60, n)
    b = rng.integers(0, 60, n)
    a[:300] = b[:300]                                  # ties
    a[300:350] = 127 + rng.integers(0, 40, 50)         # past the last bin on both sides
    b[340:380] = 130
    parity = rng.integers(0, 2, n)
    h = np.zeros((2, outputs.HIST_BINS, outputs.HIST_BINS), dtype=np.int64)
    ca, cb = np.minimum(a, 127), np.minimum(b, 127)
    np.add.at(h, (parity, ca, cb), 1)
    got = outputs.live_odds_from_hist(h, "A", "B", spread=-3.5, total=61.0)
    assert got["games"] == n
    assert got["p_win"]["A"] == pytest.approx(np.mean(ca > cb), abs=1e-15)
    assert got["p_win"]["B"] == pytest.approx(np.mean(cb > ca), abs=1e-15)
    assert got["p_tie"] == pytest.approx(np.mean(ca == cb), abs=1e-15)
    assert got["p_win"]["A"] + got["p_win"]["B"] + got["p_tie"] == pytest.approx(1.0, abs=1e-12)
    assert got["mean_points"]["A"] == pytest.approx(ca.mean(), rel=1e-12)
    assert got["mean_points"]["B"] == pytest.approx(cb.mean(), rel=1e-12)
    sp, to = got["markets"]["spread"], got["markets"]["total"]
    assert sp["p_cover"] == round(float(np.mean(ca - cb > 3.5)), 6)
    assert sp["p_notcover"] == round(float(np.mean(ca - cb < 3.5)), 6)
    assert sp["mean_margin"] == pytest.approx((ca - cb).mean(), rel=1e-12)
    assert sp["median_margin"] == float(np.median(ca - cb))
    assert to["p_over"] == round(float(np.mean(ca + cb > 61)), 6)
    assert to["push_rate"] == round(float(np.mean(ca + cb == 61)), 6)
    assert to["median_total"] == float(np.median(ca + cb))
    # the same games in a [128, 128] table (orientations already summed) give the same odds
    assert outputs.live_odds_from_hist(h.sum(axis=0), "A", "B")["p_win"] == got["p_win"]
    assert outputs.live_odds_from_hist(h, "A", "B")["markets"] is None
    with pytest.raises(ValueError):
        outputs.live_odds_from_hist(np.zeros_like(h), "A", "B")


@pytest.mark.parametrize("bad", [
    dict(offense=2), dict(offense=-2), dict(seconds=-1), dict(seconds=3601), dict(seconds=12.5), dict(down=0),
    dict(down=5), dict(score=(251, 0)), dict(score=(0, -1)), dict(score=(1, 2, 3)), dict(distance=0.0),
    dict(distance=-1.0), dict(distance=float("nan")), dict(distance=float("inf")), dict(distance=100.5),
    dict(yards_to_goal=0.0), dict(yards_to_goal=100.0), dict(yards_to_goal=float("nan")),
])
def test_game_state_validation(bad):
    with pytest.raises(ValueError):
        GameState(**bad)


def test_game_state_edges_accepted():
    GameState(offense=1, seconds=0, down=4, distance=100.0, yards_to_goal=99.0, score=(250, 0))
    GameState(offense=0, seconds=3600, down=1, distance=0.5, yards_to_goal=0.5)


def test_live_state_team_resolution():
    from fast_monte_carlo_b200 import api
    st = api.LiveState("Iowa State", 7 * 60 + 41 + 900, 3, 4.0, 32.0, (24, 17))
    gs = api.live_game_state("Kansas State", "Iowa State", st)
    assert gs == GameState(offense=1, seconds=1361, down=3, distance=4.0, yards_to_goal=32.0, score=(24, 17))
    assert api.live_game_state("Kansas State", "Iowa State", dict(st.__dict__)) == gs
    with pytest.raises(ValueError, match="neither"):
        api.live_game_state("Kansas State", "Iowa State", api.LiveState("Kansas", 100, 1, 10.0, 75.0))
    with pytest.raises(ValueError):
        api.live_game_state("Kansas State", "Iowa State", api.LiveState("Iowa State", 100, 7, 10.0, 75.0))


def test_simulate_live_rejects_unknown_teams_before_the_gpu():
    from fast_monte_carlo_b200 import api
    st = api.LiveState("Nowhere U", 100, 1, 10.0, 75.0)
    with pytest.raises(ValueError, match="not found"):
        api.simulate_live([("Nowhere U", "Iowa State", st)], 10, engine=object())
