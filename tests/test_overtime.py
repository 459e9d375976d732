"""Overtime on the CPU: the overtime oracle (tests/oracle_overtime.py) against the regulation oracle and against the rules
re-derived here from its trace rows, hand-built draw streams that force each rule, `overtime_odds_from_hist` against a
brute-force count, the validation, and the single all-reduce over two gloo ranks."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import overtime_scripts as osc
from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import api, outputs
from fast_monte_carlo_b200.engine import GameState, OvertimeRules

SNAP = 120


@pytest.fixture(scope="module")
def ot(models_s2):
    import oracle_overtime
    oracle_overtime.load_models(models_s2)
    return oracle_overtime


@pytest.fixture(scope="module")
def live(models_s2):
    import oracle_live
    oracle_live.load_models(models_s2)
    return oracle_live


@pytest.fixture(scope="module")
def philox_runs(oracle, models_s2, ot, live):
    """8,000 Philox games of Kansas State - Iowa State from the kickoff, regulation only and with overtime."""
    cfg = oracle.make_config(models_s2, KSU, ISU)
    n = 8000
    kick = GameState()
    reg = live.simulate(cfg, n, start=kick, seed=7, trace=True)
    over = ot.simulate(cfg, n, start=kick, seed=7, trace=True)
    return reg, over


def _same(a, b):
    return bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


def test_games_not_level_are_unchanged_and_level_ones_share_regulation(philox_runs):
    reg, over = philox_runs
    level = reg["scores"][:, 0] == reg["scores"][:, 1]
    assert 0.01 < level.mean() < 0.08                      # about 3 % of games are level after regulation
    d = ~level
    assert np.array_equal(over["scores"][d], reg["scores"][d])
    assert np.array_equal(over["iters"][d], reg["iters"][d])
    assert _same(over["trace"][d], reg["trace"][d])
    assert (over["periods"][d] == 0).all() and (over["periods"][level] >= 1).all()
    for g in np.flatnonzero(level):
        r = reg["iters"][g]
        assert over["iters"][g] > r
        assert _same(over["trace"][g, :r], reg["trace"][g, :r])
    # nearly every level game gets a result
    assert (over["scores"][level, 0] != over["scores"][level, 1]).mean() > 0.99


def _check_rules(rows, final, level_score, max_periods=16):
    """The overtime of one game re-derived from its overtime trace rows (offense is the first team, down, seconds, points
    of the first team, of the other, distance, yards to goal, going) and final score (first team, other): possession
    order, start spots, points (TD 7 in period 1, 6 and a try in period 2, tries from period 3), end conditions.
    Returns the periods played."""
    n = len(rows)
    cur = [float(level_score), float(level_score)]
    assert tuple(rows[0][3:5]) == tuple(cur)
    assert (rows[:, 2] == SNAP).all()
    after = lambda j: tuple(rows[j + 1][3:5]) if j + 1 < n else tuple(float(x) for x in final)
    j, k = 0, 1

    def play_try(team):
        nonlocal j
        assert (rows[j][0] == (team == 0)) and tuple(rows[j][[1, 5, 6, 7]]) == (1, 3, 3, 0)
        gain = np.subtract(after(j), cur)
        assert gain[team ^ 1] == 0 and gain[team] in (0, 2)
        cur[team] += gain[team]
        j += 1

    while True:
        for second in (0, 1):
            team = ((k - 1) & 1) ^ second                      # 0: the team with the first possession of period 1
            if k >= 3:
                play_try(team)
                continue
            assert (rows[j][0] == (team == 0)) and tuple(rows[j][[1, 5, 6, 7]]) == (1, 10, 25, 0)
            while True:                                        # to the snap that ends the possession
                nxt = after(j)
                if nxt != tuple(cur) or j + 1 == n or (rows[j + 1][0] == 1.0) != (team == 0):
                    break
                # the period's second possession, ended without a score: the next period starts with the same team,
                # and its first row is the only way to see the change (no snap reaches exactly 1st & 10 at the 25)
                if second and tuple(rows[j + 1][[1, 5, 6, 7]]) == (1, 10, 25, 0):
                    break
                j += 1
            gain = np.subtract(after(j), cur)
            j += 1
            assert gain[team ^ 1] == 0
            pts = gain[team]
            if k == 1:
                assert pts in (0, 3, 7)
                cur[team] += pts
            else:
                assert pts in (0, 3, 6)
                cur[team] += pts
                if pts == 6:
                    if second and cur[team] > cur[team ^ 1]:
                        assert j == n and tuple(cur) == tuple(final)
                        return k
                    play_try(team)
        if cur[0] != cur[1] or k == max_periods:
            assert j == n and tuple(cur) == tuple(float(x) for x in final)
            return k
        k += 1


def test_rules_rederived_from_the_trace_rows(philox_runs):
    reg, over = philox_runs
    level = np.flatnonzero(reg["scores"][:, 0] == reg["scores"][:, 1])
    assert len(level) > 100
    seen = set()
    for g in level:
        first = g & 1
        r, it = reg["iters"][g], over["iters"][g]
        assert it < 360
        final = (over["scores"][g, first], over["scores"][g, first ^ 1])
        k = _check_rules(over["trace"][g, r:it], final, reg["scores"][g, 0])
        assert k == over["periods"][g]
        seen.add(k)
    assert {1, 2} <= seen


@pytest.mark.parametrize("name", sorted(osc.SCENARIOS))
def test_scripted_streams(oracle, models_s2, ot, name):
    plan, max_periods, *_ = osc.SCENARIOS[name]
    cfg = oracle.make_config(models_s2, KSU, ISU)
    s, _ = osc.stream_for(plan)
    start = GameState(offense=0, seconds=0, down=1, distance=10.0, yards_to_goal=75.0, score=osc.START_SCORE)
    for game0 in (0, 1):
        r = ot.simulate(cfg, 1, start=start, game0=game0, stream=s[None], max_periods=max_periods, trace=True)
        sc, iters, periods = osc.expected(name, game0)
        assert tuple(r["scores"][0]) == sc and r["iters"][0] == iters and r["periods"][0] == periods, (game0, r)
        assert (r["trace"][0, :iters, 2] == SNAP).all()


def test_start_at_zero_level_and_not_level(oracle, models_s2, ot, live):
    cfg = oracle.make_config(models_s2, KSU, ISU)
    lvl = GameState(offense=1, seconds=0, score=(10, 10))
    r = ot.simulate(cfg, 400, start=lvl, seed=3)
    assert (r["periods"] >= 1).all() and (r["iters"] > 0).all()
    assert (r["scores"] >= 10).all() and (r["scores"][:, 0] != r["scores"][:, 1]).mean() > 0.99
    up = GameState(offense=1, seconds=0, score=(10, 3))
    r = ot.simulate(cfg, 50, start=up, seed=3)
    assert (r["periods"] == 0).all() and (r["iters"] == 0).all() and (r["scores"] == (10, 3)).all()


def test_player_mode_tries_credit_nothing(oracle, models_s2, ot, live):
    """A try adds nothing to the box: a game that reaches period 3 (a made and a failed try) has the box of the same game
    capped after period 2, while its event counters count the two try snaps."""
    from fast_monte_carlo_b200 import priors, usage
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    tcs = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    cu = oracle.make_usage(tuple(usage.resolve_team(tc, models_s2) for tc in tcs))
    cfg = oracle.make_config(models_s2, tcs[0].sp, tcs[1].sp)
    slots = 12
    plan = ["none"] * 4 + ["ok", "fail"]
    s, _ = osc.stream_for(plan)
    start = GameState(offense=0, seconds=0, score=osc.START_SCORE)
    full = ot.simulate(cfg, 1, start=start, stream=s[None], max_periods=3, usage=cu, n_slots=slots)
    s2, _ = osc.stream_for(["none"] * 4)
    part = ot.simulate(cfg, 1, start=start, stream=s2[None], max_periods=2, usage=cu, n_slots=slots)
    assert full["periods"][0] == 3 and part["periods"][0] == 2
    assert np.array_equal(full["players"], part["players"]) and full["players"][..., 1].sum() > 0
    assert full["counters"]["pass"] == part["counters"]["pass"] + 2


def test_overtime_odds_brute_force():
    rng = np.random.default_rng(5)
    n = 20000
    per = np.where(rng.random(n) < 0.9, 0, rng.integers(1, 17, n))
    res = rng.integers(0, 3, n)
    res[(per == 0) & (res == 2)] = rng.integers(0, 2, int(((per == 0) & (res == 2)).sum()))
    res[(per > 0) & (per < 16) & (res == 2)] = 0
    orient = rng.integers(0, 2, n)
    h = np.zeros((2, outputs.OT_MAX_PERIODS + 1, 3), dtype=np.int64)
    np.add.at(h, (orient, per, res), 1)
    o = outputs.overtime_odds_from_hist(h, "A", "B")
    assert o["games"] == n
    assert o["p_ot"] == pytest.approx((per > 0).mean())
    assert o["regulation"]["A"]["p"] == pytest.approx(((per == 0) & (res == 0)).mean())
    assert o["regulation"]["B"]["p"] == pytest.approx(((per == 0) & (res == 1)).mean())
    assert o["regulation"]["level"]["p"] == pytest.approx((per > 0).mean())
    assert o["regulation"]["A"]["american"] == outputs.prob_to_american(((per == 0) & (res == 0)).mean())
    assert o["ot_win"]["A"] == pytest.approx(((per > 0) & (res == 0)).mean())
    assert o["ot_win"]["B"] == pytest.approx(((per > 0) & (res == 1)).mean())
    assert o["periods"] == pytest.approx([(per == k).mean() for k in range(17)])
    assert o["p_level"] == pytest.approx(((per > 0) & (res == 2)).mean())
    assert outputs.overtime_odds_from_hist(h[0], "A", "B")["games"] == int(h[0].sum())
    with pytest.raises(ValueError):
        outputs.overtime_odds_from_hist(np.zeros_like(h), "A", "B")


@pytest.mark.parametrize("kw", [dict(max_periods=0), dict(max_periods=17), dict(snap_clock=0), dict(snap_clock=901),
                                dict(max_periods=2.0)])
def test_overtime_rules_validation(kw):
    with pytest.raises(ValueError):
        OvertimeRules(**kw)


def test_overtime_argument():
    from fast_monte_carlo_b200.engine import overtime_rules
    assert overtime_rules(False) is None and overtime_rules(None) is None
    assert overtime_rules(True) == OvertimeRules(16, 120)
    r = OvertimeRules(4, 60)
    assert overtime_rules(r) is r
    with pytest.raises(ValueError):
        overtime_rules("yes")


@pytest.mark.parametrize("extra", [dict(segments=True), dict(sequence=True)])
def test_overtime_with_period_or_sequence_outputs_is_refused_before_the_gpu(extra):
    state = api.LiveState(offense="Kansas State", seconds=0, down=1, distance=10.0, yards_to_goal=75.0, score=(7, 7))
    with pytest.raises(ValueError, match="overtime"):
        api.simulate_live([("Kansas State", "Iowa State", state)], 10, overtime=True, **extra)
    with pytest.raises(ValueError, match="overtime"):
        api.simulate_slate([("Kansas State", "Iowa State")], 10, overtime=True, **extra)


# ---- one all-reduce over two ranks -----------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _parts(rank):
    g = torch.Generator().manual_seed(200 + rank)
    hist = torch.randint(0, 50, (3, 2, outputs.HIST_BINS, outputs.HIST_BINS), generator=g, dtype=torch.int32)
    oth = torch.randint(0, 50, (3, 2, outputs.OT_MAX_PERIODS + 1, 3), generator=g, dtype=torch.int32)
    return hist, oth


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
        hist, oth = _parts(rank)
        h64, s64, q64, o64 = api._merge_all(None, hist, None, None, oth)
    finally:
        dist.all_reduce = real
    if rank == 0:
        q.put((h64.numpy(), s64, q64, o64.numpy(), calls))
    dist.barrier()
    dist.destroy_process_group()


def test_score_and_overtime_histograms_merge_in_one_all_reduce():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    h, s, sq, o, calls = q.get(timeout=300)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    parts = [_parts(r) for r in range(2)]
    want = [sum(p[i].to(torch.int64) for p in parts).numpy() for i in range(2)]
    assert np.array_equal(h, want[0]) and np.array_equal(o, want[1]) and s is None and sq is None
    assert len(calls) == 1
