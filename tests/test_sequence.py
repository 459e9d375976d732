"""Next-score, drive-result and race-to-N markets on the CPU: the sequence harness (tests/oracle_sequence.py) against the
reference's own games and resumed mid-game states, the drive definition at the half, `sequence_odds_from_hist` against a
brute-force count, and the single all-reduce over two gloo ranks."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from fast_monte_carlo_b200 import api, outputs
from fast_monte_carlo_b200.native import SEQ_NONE, seq_bin_next
from test_live import FIXTURES, _Raw, raw_state_at, resume_points

DR = {r: i for i, r in enumerate(outputs.DRIVE_RESULTS)}
KICKOFF = _Raw(offense=-1, seconds=3600, down=1, distance=10.0, yards_to_goal=75.0, score=(0, 0))


@pytest.fixture(scope="module")
def seqo(models):
    import oracle_sequence
    oracle_sequence.load_models(models)
    return oracle_sequence


def sequence_from_trace(trace, n, final, first):
    """Next score and race results of one game from its trace rows (columns 2 = seconds, 3 / 4 = scores of the first /
    second team) and final score (first, second): (team, kind, clock) or None, and {target: 0 / 1 / 2 / -1} with teams
    A / B = first ^ 0 / first ^ 1 turned into the matchup's indices (0 = A)."""
    rows = [(int(trace[k, 2]), int(trace[k, 3]), int(trace[k, 4])) for k in range(n)]
    after = [(r[1], r[2]) for r in rows[1:]] + [tuple(int(x) for x in final)]
    s0 = (rows[0][1], rows[0][2])
    nxt = None
    race = {t: (-1 if max(s0) >= t else None) for t in outputs.RACE_TARGETS}
    prev = s0
    for (clock, _, _), cur in zip(rows, after):
        if cur != prev:
            side = 0 if cur[0] != prev[0] else 1
            pts = cur[side] - prev[side]
            assert pts in (3, 7) and cur[side ^ 1] == prev[side ^ 1]
            team = first if side == 0 else first ^ 1
            if nxt is None:
                nxt = (team, 0 if pts == 7 else 1, clock)
            for t in outputs.RACE_TARGETS:
                if race[t] is None and prev[side] < t <= cur[side] and cur[side ^ 1] < t:
                    race[t] = team
        prev = cur
    return nxt, {t: (2 if v is None else v) for t, v in race.items()}


def unpack_next(w):
    w = int(w)
    return None if w == SEQ_NONE else (w & 1, (w >> 1) & 1, w >> 2)


def check_game(r, i, trace, n, final_fs, first, start_offense):
    nxt, race = sequence_from_trace(trace, n, final_fs, first)
    got = unpack_next(r["sequence"][i, 0])
    assert got == nxt, (got, nxt)
    assert {t: int(r["race"][i, k]) for k, t in enumerate(outputs.RACE_TARGETS)} == race
    code, clock = int(r["sequence"][i, 1]) & 0xFF, int(r["sequence"][i, 1]) >> 8
    if code in (DR["td"], DR["fg"]):            # a scoring drive is the next score: same team, same snap
        assert got == (start_offense, 0 if code == DR["td"] else 1, clock)
    if code == DR["end_of_game"]:
        assert clock == 0 and got is None        # every score ends the drive: a drive still on has seen none
    return code


@pytest.mark.parametrize("name", FIXTURES)
def test_harness_on_the_reference_games(models, oracle, seqo, name):
    """The reference's 40 games under their own draws, from the kickoff and resumed at mid-game states: the harness's
    next score and races are those read off the reference's traces."""
    meta, traces, iters, scores, stream = resume_points(name)
    codes = set()
    for g, m in enumerate(meta):
        spA, spB = (m["sp_second"], m["sp_first"]) if g & 1 else (m["sp_first"], m["sp_second"])
        cfg = oracle.make_config(models, spA, spB)
        first, n = g & 1, int(iters[g])
        half = int(np.argmax(traces[g, :n, 2] <= 1800))
        ks = sorted({0, n // 3, half - 1, half, (2 * n) // 3, n - 1})
        starts = [KICKOFF] + [raw_state_at(traces[g, k], first) for k in ks]
        draws = np.zeros((len(starts), oracle.MAX_ITERS, oracle.N_SLOTS))
        draws[0] = stream[g]
        for j, k in enumerate(ks):
            draws[1 + j, :oracle.MAX_ITERS - k] = stream[g, k:]
        # game ids g, g + 2, ...: every start keeps the kickoff receiver g & 1 its trace is relative to
        r = {key: [] for key in ("scores", "sequence", "race")}
        for j, st in enumerate(starts):
            one = seqo.simulate(cfg, 1, game0=g, stream=draws[j:j + 1], start=st)
            for key in r:
                r[key].append(one[key][0])
        r = {key: np.stack(v) for key, v in r.items()}
        fin = tuple(int(x) for x in scores[g])
        assert (r["scores"][0, first], r["scores"][0, first ^ 1]) == fin
        codes.add(check_game(r, 0, traces[g], n, fin, first, first))
        for j, k in enumerate(ks):
            st = starts[1 + j]
            codes.add(check_game(r, 1 + j, traces[g, k:], n - k, fin, first, st.offense))
    assert {DR["td"], DR["punt"]} <= codes


def test_play_result_comes_before_the_end_of_the_half(models, oracle, seqo):
    """A play whose tick crosses 1800 ends the drive with its own result: a forced punt (4th and 20 at the own 30,
    5 s before the half) is a punt snapped at 1805, never the end of the half; a touchdown from the 1 at 1810 is a
    touchdown; the end of the half is reported only for a play that changes nothing else."""
    cfg = oracle.make_config(models, (15.6, 35.7, 20.0), (11.0, 31.5, 20.6))
    punt = seqo.simulate(cfg, 2000, seed=5, start=_Raw(offense=0, seconds=1805, down=4, distance=20.0, yards_to_goal=70.0,
                                                         score=(3, 0)))
    assert (punt["sequence"][:, 1] == (DR["punt"] | 1805 << 8)).all()
    goal = seqo.simulate(cfg, 2000, seed=6, start=_Raw(offense=1, seconds=1810, down=1, distance=1.0, yards_to_goal=1.0,
                                                         score=(0, 0)))
    code, clock = goal["sequence"][:, 1] & 0xFF, goal["sequence"][:, 1] >> 8
    td = code == DR["td"]
    assert td.sum() > 1000 and (clock[td] == 1810).all()
    assert (goal["sequence"][td, 0] == (1 | 0 << 1 | 1810 << 2)).all()
    half = code == DR["end_of_half"]
    assert half.any() and (clock[half] == 1810).all()
    assert set(np.unique(code)) <= {DR["td"], DR["end_of_half"], DR["interception"]}


def test_harness_edge_starts(models, oracle, seqo):
    """Clock 0: no next score, drive "end of game", races settled or "neither"; start scores at and past the targets."""
    cfg = oracle.make_config(models, (15.6, 35.7, 20.0), (11.0, 31.5, 20.6))
    over = seqo.simulate(cfg, 4, seed=1, start=_Raw(offense=0, seconds=0, down=1, distance=10.0, yards_to_goal=75.0,
                                                     score=(14, 3)))
    assert (over["sequence"][:, 0] == SEQ_NONE).all() and (over["sequence"][:, 1] == DR["end_of_game"]).all()
    assert (over["race"] == [-1, 2, 2, 2, 2]).all()
    late = seqo.simulate(cfg, 3000, seed=2, start=_Raw(offense=1, seconds=900, down=1, distance=10.0, yards_to_goal=75.0,
                                                        score=(20, 10)))
    assert (late["race"][:, :3] == -1).all()
    for k, t in enumerate(outputs.RACE_TARGETS[3:], start=3):
        s = late["scores"]
        a_first = late["race"][:, k] == 0
        assert (s[a_first, 0] >= t).all()
        assert ((late["race"][:, k] == 2) == ((s[:, 0] < t) & (s[:, 1] < t))).all()


# ---- odds from the histogram -----------------------------------------------------------------------------------------
def _random_rows(rng, n, start_score):
    """Per-game next score (team, kind, clock or None), drive code and race results consistent with `start_score`."""
    nxt = [None if rng.random() < 0.1 else (int(rng.integers(2)), int(rng.integers(2)), int(rng.integers(1, 3601)))
           for _ in range(n)]
    drive = rng.integers(0, len(outputs.DRIVE_RESULTS), n)
    race = rng.integers(0, 3, (n, len(outputs.RACE_TARGETS)))
    for k, t in enumerate(outputs.RACE_TARGETS):
        if max(start_score) >= t:
            race[:, k] = -1
    return nxt, drive, race


def _hist(nxt, drive, race):
    h = np.zeros(outputs.SEQ_BINS, dtype=np.int64)
    for x in nxt:
        h[outputs.SEQ_BIN_NONE if x is None else int(seq_bin_next(*x))] += 1
    for d in drive:
        h[outputs.SEQ_BIN_DRIVE0 + d] += 1
    for k in range(len(outputs.RACE_TARGETS)):
        for r in race[:, k]:
            if r >= 0:
                h[outputs.SEQ_BIN_RACE0 + 3 * k + r] += 1
    return h


@pytest.mark.parametrize("start_score", [(0, 0), (10, 3), (24, 31)])
def test_sequence_odds_equal_a_brute_force_count(start_score):
    rng = np.random.default_rng(sum(start_score))
    n = 5000
    nxt, drive, race = _random_rows(rng, n, start_score)
    o = outputs.sequence_odds_from_hist(_hist(nxt, drive, race), "A", "B", start_score=start_score,
                                        before=(0, 900, 1800, 3540, 3600))
    assert o["games"] == n
    for t, name in enumerate(("A", "B")):
        for k, kind in enumerate(("td", "fg")):
            assert o["next_score"]["p"][name][kind] == pytest.approx(sum(x is not None and x[:2] == (t, k) for x in nxt) / n)
        assert o["next_score"]["p"][name]["any"] == pytest.approx(sum(x is not None and x[0] == t for x in nxt) / n)
        for c in (0, 900, 1800, 3540, 3600):
            want = sum(x is not None and x[0] == t and x[2] > c for x in nxt) / n
            assert o["next_score"]["before"][c][name] == pytest.approx(want)
        assert o["next_score"]["american"][name]["td"] == outputs.prob_to_american(o["next_score"]["p"][name]["td"])
    assert o["next_score"]["none"] == pytest.approx(sum(x is None for x in nxt) / n)
    for i, r in enumerate(outputs.DRIVE_RESULTS):
        assert o["drive"]["p"][r] == pytest.approx((drive == i).mean())
    assert o["drive"]["p_scores"] == pytest.approx(((drive == DR["td"]) | (drive == DR["fg"])).mean())
    for k, t in enumerate(outputs.RACE_TARGETS):
        rt = o["race"][t]
        if max(start_score) >= t:
            a, b = start_score[0] >= t, start_score[1] >= t
            assert rt == {"settled": True, "winner": None if a and b else ("A" if a else "B")}
            continue
        assert not rt["settled"]
        assert rt["p"]["A"] == pytest.approx((race[:, k] == 0).mean())
        assert rt["p"]["B"] == pytest.approx((race[:, k] == 1).mean())
        assert rt["p"]["neither"] == pytest.approx((race[:, k] == 2).mean())
    # both orientations at once: the leading axis is summed
    h = _hist(nxt, drive, race)
    two = outputs.sequence_odds_from_hist(np.stack([h, h]), "A", "B", start_score=start_score)
    assert two["games"] == 2 * n and two["drive"]["p"] == o["drive"]["p"]


def test_sequence_odds_reject_malformed_input():
    rng = np.random.default_rng(0)
    h = _hist(*_random_rows(rng, 100, (0, 0)))
    bad = [
        (np.zeros(outputs.SEQ_BINS - 1, dtype=np.int64), {}),
        (np.zeros(outputs.SEQ_BINS, dtype=np.int64), {}),
        (h.astype(np.float64), {}),
        (-h, {}),
        (h, {"start_score": (1, 2, 3)}),
        (h, {"start_score": (-1, 0)}),
        (h, {"start_score": (10, 0)}),           # settled target with games in its bins
        (h, {"before": (61,)}),
        (h, {"before": (3660,)}),
    ]
    drive_short = h.copy()
    drive_short[outputs.SEQ_BIN_DRIVE0] -= 1
    race_short = h.copy()
    race_short[outputs.SEQ_BIN_RACE0] += 1
    bad += [(drive_short, {}), (race_short, {})]
    for arr, kw in bad:
        with pytest.raises(ValueError):
            outputs.sequence_odds_from_hist(arr, "A", "B", **kw)


# ---- one all-reduce over two ranks -----------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _parts(rank):
    g = torch.Generator().manual_seed(100 + rank)
    hist = torch.randint(0, 50, (3, 2, outputs.HIST_BINS, outputs.HIST_BINS), generator=g, dtype=torch.int32)
    seg = torch.randint(0, 50, (3, 2, len(outputs.SEGMENTS), outputs.HIST_BINS, outputs.HIST_BINS), generator=g,
                        dtype=torch.int32)
    seq = torch.randint(0, 50, (3, 2, outputs.SEQ_BINS), generator=g, dtype=torch.int32)
    return hist, seg, seq


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
        hist, seg, seq = _parts(rank)
        h64, s64, q64 = api._merge_segments(hist, seg, None, seq)
        h2, s2, q2 = api._merge_segments(hist, None, None, seq)
    finally:
        dist.all_reduce = real
    if rank == 0:
        q.put((h64.numpy(), s64.numpy(), q64.numpy(), h2.numpy(), s2, q2.numpy(), calls))
    dist.barrier()
    dist.destroy_process_group()


def test_score_period_and_sequence_histograms_merge_in_one_all_reduce():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    h, s, sq, h2, s2, sq2, calls = q.get(timeout=300)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    parts = [_parts(r) for r in range(2)]
    want = [sum(p[i].to(torch.int64) for p in parts).numpy() for i in range(3)]
    assert np.array_equal(h, want[0]) and np.array_equal(s, want[1]) and np.array_equal(sq, want[2])
    assert np.array_equal(h2, want[0]) and s2 is None and np.array_equal(sq2, want[2])
    assert len(calls) == 2        # one collective per merge
