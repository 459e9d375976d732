"""Fourth-down decisions on the CPU: the forced-choice oracle (tests/oracle_fourth_down.py) pinned on the reference's own
games and on the policy's games (the draw identity), the edges of the choices' ranges, `fourth_down_from_hists` against
a brute-force count, the validation, and the single all-reduce of a multi-state call over two gloo ranks."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ISU, KSU, ROOT
from fast_monte_carlo_b200 import api, native, outputs
from fast_monte_carlo_b200.engine import FOURTH_DOWN_FG, FOURTH_DOWN_GO, FOURTH_DOWN_PUNT, GameState
from test_live import FIXTURES, raw_state_at, resume_points

S_U_GO, S_U_FG = 8, 9


@pytest.fixture(scope="module")
def fd(models_s2):
    import oracle_fourth_down
    oracle_fourth_down.load_models(models_s2)
    return oracle_fourth_down


@pytest.fixture(scope="module")
def live(models_s2):
    import oracle_live
    oracle_live.load_models(models_s2)
    return oracle_live


@pytest.fixture(scope="module")
def ot(models_s2):
    import oracle_overtime
    oracle_overtime.load_models(models_s2)
    return oracle_overtime


def _same(a, b):
    return bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


# ---- pinned on the reference ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", FIXTURES)
def test_forced_to_the_reference_branch_plays_the_reference_game(models, oracle, fd, name):
    """Every fourth down (with time left) at an iteration start of the reference's own games: resumed there with the
    draws from that iteration on and forced to the branch the reference took (its S_U_GO draw against the oracle's
    go_for_it_prob), the harness plays the rest of the reference's game bit for bit."""
    meta, traces, iters, scores, stream = resume_points(name)
    seen = {"go": 0, "fg": 0, "punt": 0}
    for g, m in enumerate(meta):
        spA, spB = (m["sp_second"], m["sp_first"]) if g & 1 else (m["sp_first"], m["sp_second"])
        cfg = oracle.make_config(models, spA, spB)
        first, n = g & 1, int(iters[g])
        ks = [k for k in range(n) if traces[g, k, 1] == 4.0 and traces[g, k, 2] > 0]
        if not ks:
            continue
        starts, choices = [], []
        draws = np.zeros((len(ks), oracle.MAX_ITERS, oracle.N_SLOTS))
        for j, k in enumerate(ks):
            st = raw_state_at(traces[g, k], first)
            starts.append(st)
            choices.append(fd.branch_of(stream[g, k, S_U_GO], st))
            draws[j, :oracle.MAX_ITERS - k] = stream[g, k:]
        # every game of the call is game g (game0 = g, one game per call keeps the kickoff receiver's parity)
        for j, k in enumerate(ks):
            r = fd.simulate(cfg, 1, game0=g, stream=draws[j:j + 1], trace=True, start=starts[j], choice=choices[j])
            assert r["iters"][0] == n - k, (g, k)
            assert np.array_equal(r["trace"][0, :n - k], traces[g, k:n]), (g, k)
            assert (r["scores"][0, first], r["scores"][0, first ^ 1]) == tuple(scores[g]), (g, k)
            seen[choices[j]] += 1
    assert sum(seen.values()) > 0
    if name == "ref_trajectories.npz":
        assert min(seen.values()) > 0, seen           # the reference's games take every branch


# ---- the draw identity in the harness -------------------------------------------------------------------------------
STATES = [
    GameState(offense=0, seconds=1500, down=4, distance=2.0, yards_to_goal=34.0, score=(10, 14)),
    GameState(offense=1, seconds=240, down=4, distance=6.0, yards_to_goal=55.0, score=(21, 17)),
    GameState(offense=0, seconds=95, down=4, distance=1.0, yards_to_goal=8.0, score=(17, 20)),
    GameState(offense=1, seconds=3000, down=4, distance=9.0, yards_to_goal=72.0, score=(0, 3)),
    GameState(offense=0, seconds=20, down=4, distance=4.0, yards_to_goal=21.0, score=(24, 27)),
]


@pytest.mark.parametrize("overtime", [False, True])
def test_forced_to_its_own_branch_every_game_is_the_same_game(oracle, models_s2, fd, live, ot, overtime):
    """20,000 Philox games from five fourth-down states: every game forced to the branch its own draws pick is the game
    fo_live_simulate / fo_overtime_simulate plays (score, iterations, trace, overtime periods, event counters)."""
    cfg = oracle.make_config(models_s2, KSU, ISU)
    n, seed = 4000, 31
    picked = set()
    for m, st in enumerate(STATES):
        kw = dict(game0=5, matchup=m, seed=seed, trace=True)
        ref = (ot.simulate(cfg, n, start=st, **kw) if overtime else live.simulate(cfg, n, start=st, **kw))
        choice = list(fd.branches(fd.philox_u_many(seed, 5 + np.arange(n), m, S_U_GO), st))
        got = fd.simulate(cfg, n, start=[st] * n, choice=choice, overtime=overtime, **kw)
        assert np.array_equal(got["scores"], ref["scores"]), m
        assert np.array_equal(got["iters"], ref["iters"]), m
        assert _same(got["trace"], ref["trace"]), m
        assert got["counters"] == ref["counters"], m
        if overtime:
            assert np.array_equal(got["periods"], ref["periods"]), m
        picked |= set(choice)
        # the policy (choice None) is fo_live_simulate / fo_overtime_simulate itself
        pol = fd.simulate(cfg, n, start=st, overtime=overtime, **kw)
        assert np.array_equal(pol["scores"], ref["scores"]) and pol["counters"] == ref["counters"]
    assert picked == {"go", "fg", "punt"}


def test_vectorised_philox_draws_are_the_oracles(oracle, fd):
    games = np.array([0, 1, 7, 4095, (1 << 33) + 5])
    for seed, m, slot, it in ((31, 0, S_U_GO, 0), (0xFEDCBA9876543210, 4, S_U_FG, 3)):
        want = [fd.philox_u(seed, int(g), m, slot, it) for g in games]
        assert np.array_equal(fd.philox_u_many(seed, games, m, slot, it), want)


# ---- the edges of the ranges ----------------------------------------------------------------------------------------
def _stream(n, seed, **iter0):
    from oracle import c_oracle as co
    s = co.make_stream(n, seed)
    for slot, v in iter0.items():
        s[:, 0, {"go": S_U_GO, "fg": S_U_FG}[slot]] = v
    return s


def test_forced_field_goal_from_the_38(oracle, models_s2, fd, live):
    """A 55-yard try (p = 0.50): made with u_fg 0.3 (3 points, the opponent at its 25, 12 s), missed with 0.7 (the
    opponent at the spot of the kick); either is the policy's game when its go draw declines (u_go ~ 1)."""
    cfg = oracle.make_config(models_s2, KSU, ISU)
    st = GameState(offense=0, seconds=1200, down=4, distance=5.0, yards_to_goal=38.0, score=(7, 7))
    for u_fg, pts, ytg in ((0.3, 3, 75.0), (0.7, 0, 62.0)):
        forced = fd.simulate(cfg, 16, start=st, choice="fg", trace=True, stream=_stream(16, 5, go=0.0, fg=u_fg))
        row = forced["trace"][:, 1]
        assert (row[:, 0] == (np.arange(16) % 2 == 1)).all()      # team B has the ball: 1 iff B received first
        assert (row[:, 2] == 1188).all() and (row[:, 6] == ytg).all() and (row[:, 1] == 1).all()
        a_first = np.arange(16) % 2 == 0          # the trace is relative to team (g & 1)
        assert (row[a_first, 3] == 7 + pts).all() and (row[~a_first, 4] == 7 + pts).all()
        pol = live.simulate(cfg, 16, start=st, trace=True, stream=_stream(16, 5, go=1 - 1e-12, fg=u_fg))
        assert np.array_equal(forced["scores"], pol["scores"]) and _same(forced["trace"], pol["trace"])


def test_forced_punt_from_the_16(oracle, models_s2, fd):
    """From the 16 the net distance is clipped to exactly 15: the receiving team takes over at its own 1 (yards to goal
    99) after 16 s -- a punt the reference itself never makes there (it kicks)."""
    cfg = oracle.make_config(models_s2, KSU, ISU)
    st = GameState(offense=1, seconds=700, down=4, distance=3.0, yards_to_goal=16.0, score=(3, 0))
    r = fd.simulate(cfg, 64, start=st, choice="punt", trace=True, seed=9)
    row = r["trace"][:, 1]
    first = np.arange(64) % 2
    assert (row[:, 0] == (first == 0)).all()      # team A (0) has the ball: the offense column is 1 iff A received first
    assert (row[:, 1] == 1).all() and (row[:, 2] == 684).all() and (row[:, 5] == 10.0).all() and (row[:, 6] == 99.0).all()
    assert r["counters"]["punt"] >= 64


@pytest.mark.parametrize("bad", [dict(choice="go", start=GameState(down=3)),
                                 dict(choice="punt", start=GameState(down=4, seconds=0))])
def test_harness_refuses_a_forced_choice_off_a_fourth_down(oracle, models_s2, fd, bad):
    cfg = oracle.make_config(models_s2, KSU, ISU)
    st = bad["start"]
    raw = type("S", (), dict(offense=st.offense, seconds=st.seconds, down=st.down, distance=st.distance,
                             yards_to_goal=st.yards_to_goal, score=st.score))()
    with pytest.raises(ValueError):
        fd.simulate(cfg, 4, start=raw, choice=bad["choice"], seed=1)


# ---- the decision arithmetic ----------------------------------------------------------------------------------------
def test_fourth_down_from_hists_brute_force():
    rng = np.random.default_rng(3)
    per = {}
    hists = {}
    for k, (n, mu) in {"policy": (3000, 20), "go": (2500, 24), "fg": (2700, 21), "punt": (2900, 18)}.items():
        a = rng.poisson(mu, n)
        b = rng.poisson(21, n)
        b[:60] = a[:60]                              # some level games
        h = np.zeros((2, outputs.HIST_BINS, outputs.HIST_BINS), dtype=np.int64)
        np.add.at(h, (np.arange(n) % 2, a, b), 1)
        hists[k] = h.sum(axis=0)
        per[k] = (a, b)
    for off_a in (True, False):
        got = outputs.fourth_down_from_hists(hists, offense_is_a=off_a)
        val = {}
        for k, (a, b) in per.items():
            mine, theirs = (a, b) if off_a else (b, a)
            x = np.where(mine > theirs, 1.0, np.where(mine == theirs, 0.5, 0.0))
            val[k] = (x.mean(), x.std(ddof=1) / np.sqrt(len(x)))
            assert got["equity"][k]["equity"] == pytest.approx(val[k][0], abs=1e-12)
            assert got["equity"][k]["se"] == pytest.approx(val[k][1], rel=1e-9)
            assert got["equity"][k]["games"] == len(x)
        best = max(outputs.FOURTH_DOWN_CHOICES, key=lambda c: val[c][0])
        assert got["best"] == best and set(got["delta"]) == set(outputs.FOURTH_DOWN_CHOICES) - {best}
        for c, d in got["delta"].items():
            assert d["equity"] == pytest.approx(val[best][0] - val[c][0], abs=1e-12)
            assert d["se"] == pytest.approx(np.hypot(val[best][1], val[c][1]), rel=1e-9)
    # a choice left out is left out of best and delta
    part = outputs.fourth_down_from_hists(dict(hists, fg=None), offense_is_a=True)
    assert "fg" not in part["equity"] and "fg" not in part["delta"] and part["best"] != "fg"
    with pytest.raises(ValueError):
        outputs.fourth_down_from_hists({"policy": hists["policy"]}, offense_is_a=True)


# ---- validation ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw", [
    dict(down=4, seconds=600, yards_to_goal=40.0, fourth_down=4),
    dict(down=4, seconds=600, yards_to_goal=40.0, fourth_down=-1),
    dict(down=4, seconds=600, yards_to_goal=40.0, fourth_down=1.0),
    dict(down=3, seconds=600, yards_to_goal=40.0, fourth_down=FOURTH_DOWN_GO),
    dict(down=4, seconds=0, yards_to_goal=40.0, fourth_down=FOURTH_DOWN_GO),
    dict(down=4, seconds=600, yards_to_goal=38.5, fourth_down=FOURTH_DOWN_FG),
    dict(down=4, seconds=600, yards_to_goal=15.5, fourth_down=FOURTH_DOWN_PUNT),
])
def test_game_state_refuses_bad_choices(kw):
    with pytest.raises(ValueError):
        GameState(**kw)


def test_game_state_accepts_the_edges():
    GameState(down=4, seconds=1, yards_to_goal=38.0, fourth_down=FOURTH_DOWN_FG)
    GameState(down=4, seconds=1, yards_to_goal=16.0, fourth_down=FOURTH_DOWN_PUNT)
    GameState(down=4, seconds=1, yards_to_goal=99.0, fourth_down=FOURTH_DOWN_GO)
    assert GameState().fourth_down == 0


def test_abi_layout_and_codes():
    """fmc_game_state keeps its layout (the field replaces `reserved`) and the codes match include/fmc.h."""
    assert C.sizeof(native.GameStateC) == 40 and native.GameStateC.fourth_down.offset == 20
    with open(os.path.join(ROOT, "include", "fmc.h")) as fh:
        h = fh.read()
    assert "enum { FMC_4TH_POLICY = 0, FMC_4TH_GO, FMC_4TH_FG, FMC_4TH_PUNT };" in h
    assert outputs.FOURTH_DOWN_CHOICES == ("go", "fg", "punt")
    assert (FOURTH_DOWN_GO, FOURTH_DOWN_FG, FOURTH_DOWN_PUNT) == (1, 2, 3)


def _live_state(**kw):
    base = dict(offense="Kansas State", seconds=600, down=4, distance=3.0, yards_to_goal=30.0, score=(14, 17))
    base.update(kw)
    return api.LiveState(**base)


def test_live_state_maps_to_the_codes():
    for name, code in (("go", 1), ("fg", 2), ("punt", 3), (None, 0)):
        gs = api.live_game_state("Kansas State", "Iowa State", _live_state(fourth_down=name))
        assert gs.fourth_down == code
    with pytest.raises(ValueError):
        api.live_game_state("Kansas State", "Iowa State", _live_state(fourth_down="kick"))
    with pytest.raises(ValueError):
        api.live_game_state("Kansas State", "Iowa State", _live_state(yards_to_goal=45.0, fourth_down="fg"))


@pytest.mark.parametrize("extra", [dict(segments=True), dict(sequence=True)])
def test_forced_choice_with_period_or_sequence_outputs_is_refused_before_the_gpu(extra):
    with pytest.raises(ValueError, match="fourth-down"):
        api.simulate_live([("Kansas State", "Iowa State", _live_state(fourth_down="go"))], 10, **extra)


@pytest.mark.parametrize("state", [_live_state(down=3), _live_state(seconds=0), _live_state(fourth_down="go")])
def test_fourth_down_decisions_refuses_other_states(state):
    with pytest.raises(ValueError):
        api.fourth_down_decisions([("Kansas State", "Iowa State", state)], 10)


def test_fourth_down_plan():
    """Each state becomes its policy entry plus one entry per available choice; the markets of a state go to all of them;
    the reasons of the choices left out are kept."""
    deep = _live_state(offense="Iowa State", yards_to_goal=70.0)
    near = _live_state(yards_to_goal=10.0)
    launch, mk, plan, why = api._fourth_down_plan(
        [("Kansas State", "Iowa State", _live_state()), ("Kansas State", "Iowa State", deep),
         ("Kansas State", "Iowa State", near)], {1: {"spread": 3.5}})
    assert [k for k, _ in plan[0]] == ["policy", "go", "fg", "punt"]
    assert [k for k, _ in plan[1]] == ["policy", "go", "punt"] and set(why[1]) == {"fg"}
    assert [k for k, _ in plan[2]] == ["policy", "go", "fg"] and set(why[2]) == {"punt"}
    assert [j for rows in plan for _, j in rows] == list(range(len(launch))) == list(range(10))
    assert [launch[j][2].fourth_down for _, j in plan[0]] == [None, "go", "fg", "punt"]
    assert set(mk) == {4, 5, 6} and all(v == {"spread": 3.5} for v in mk.values())


# ---- one all-reduce over two ranks ----------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


ENTRIES = [("Kansas State", "Iowa State", _live_state()),
           ("Kansas State", "Iowa State", _live_state(offense="Iowa State", yards_to_goal=70.0))]


def _parts(rank, n_entries):
    g = torch.Generator().manual_seed(300 + rank)
    hist = torch.randint(0, 5, (n_entries, 2, outputs.HIST_BINS, outputs.HIST_BINS), generator=g, dtype=torch.int32)
    oth = torch.randint(0, 50, (n_entries, 2, outputs.OT_MAX_PERIODS + 1, 3), generator=g, dtype=torch.int32)
    return hist, oth


def _decisions(hist, oth):
    launch, mk, plan, why = api._fourth_down_plan(ENTRIES, None)
    starts = [api.live_game_state(a, b, s) for a, b, s in launch]
    res = api._live_results(launch, starts, mk, hist, None, None, oth)
    return api._fourth_down_group(ENTRIES, plan, why, res)


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    calls = []
    real = dist.all_reduce

    def counting(t, *a, **kw):
        calls.append(t.numel())
        return real(t, *a, **kw)

    dist.all_reduce = counting
    try:
        n = len(api._fourth_down_plan(ENTRIES, None)[0])
        out = _decisions(*_parts(rank, n))
    finally:
        dist.all_reduce = real
    if rank == 0:
        q.put(([(d["best"], d["equity"], d["policy"]["hist"], d["choices"]["punt"]["overtime"]["p_ot"]) for d in out],
               calls))
    dist.barrier()
    dist.destroy_process_group()


def test_multi_state_histograms_merge_in_one_all_reduce():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got, calls = q.get(timeout=300)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    n = len(api._fourth_down_plan(ENTRIES, None)[0])
    parts = [_parts(r, n) for r in range(2)]
    want = _decisions(*[sum(p[i].to(torch.int64) for p in parts) for i in range(2)])
    assert len(calls) == 1
    for (best, eq, hpol, p_ot), w in zip(got, want):
        assert best == w["best"] and eq == w["equity"] and p_ot == w["choices"]["punt"]["overtime"]["p_ot"]
        assert np.array_equal(hpol, w["policy"]["hist"])
