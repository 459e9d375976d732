"""Quarter and half markets on the CPU: the period definition on the reference's own games, `segment_odds_from_hist`
against a brute-force count, and the live period inputs (`LiveState.quarter_start_score` / `half_start_score`)."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from fast_monte_carlo_b200 import api, outputs

BOUNDARIES = (2700, 1800, 900)           # end of Q1, Q2, Q3 (include/fmc.h FMC_N_SEGMENTS)
SEG_START = {"Q1": 3600, "Q2": 2700, "Q3": 1800, "Q4": 900, "H1": 3600, "H2": 1800}
SEG_END = {"Q1": 2700, "Q2": 1800, "Q3": 900, "Q4": 0, "H1": 1800, "H2": 0}


def periods_from_trace(trace, n_iters, final, start_sec=None, start_score=None):
    """The period outputs of one game from its per-iteration trace (rows [iteration][FMC_TRACE_COLS]: column 2 = seconds
    left, columns 3 / 4 = the scores of the first / second team) and its final score, all in the trace's orientation.
    The start state is the first row (or `start_sec` / `start_score` for a game without iterations).  Returns (ends,
    segments): ends[q] = score at the end of quarter q + 1 (the score at the first iteration start at or below the
    boundary, else the final score), None for a boundary at or before the start; segments[name] = points scored in the
    period, None for one that ended at or before the start."""
    n = int(n_iters)
    sec0 = int(trace[0, 2]) if n else int(start_sec)
    s0 = (int(trace[0, 3]), int(trace[0, 4])) if n else tuple(int(x) for x in start_score)
    final = (int(final[0]), int(final[1]))
    ends = []
    for B in BOUNDARIES:
        if sec0 <= B:
            ends.append(None)
            continue
        k = next((i for i in range(n) if trace[i, 2] <= B), None)
        ends.append(final if k is None else (int(trace[k, 3]), int(trace[k, 4])))
    at = {3600: s0, 2700: ends[0], 1800: ends[1], 900: ends[2], 0: final}

    def base(b):                       # score at boundary b, or the start if b is not after it
        return s0 if sec0 <= b or b == 3600 else at[b]

    segs = {}
    for name in outputs.SEGMENTS:
        b0, b1 = SEG_START[name], SEG_END[name]
        if b1 > 0 and sec0 <= b1:
            segs[name] = None
            continue
        e, s = at[b1], base(b0)
        segs[name] = (e[0] - s[0], e[1] - s[1])
    return ends, segs


def _reference_games():
    for name in ("ref_trajectories.npz", "ref_trajectories_adversarial.npz"):
        t = np.load(os.path.join(GOLDEN, name))
        for g in range(len(json.loads(str(t["meta"])))):
            yield t["traces"][g], int(t["iters"][g]), (int(t["scores"][g][0]), int(t["scores"][g][1]))


def test_period_definition_on_the_reference_games():
    games = list(_reference_games())
    assert len(games) == 40
    for trace, n, final in games:
        ends, seg = periods_from_trace(trace, n, final)
        assert all(e is not None for e in ends)
        add = lambda x, y: (x[0] + y[0], x[1] + y[1])
        assert add(seg["Q1"], seg["Q2"]) == seg["H1"]
        assert add(seg["Q3"], seg["Q4"]) == seg["H2"]
        assert add(seg["H1"], seg["H2"]) == final
        assert all(p >= 0 for v in seg.values() for p in v)
        assert ends[0][0] <= ends[1][0] <= ends[2][0] <= final[0] and ends[0][1] <= ends[1][1] <= ends[2][1] <= final[1]
    # the quarters are not all alike: some game scores in every one, and some quarter is scoreless for a team
    assert any(all(sum(s) > 0 for k, s in periods_from_trace(*g)[1].items()) for g in games)


def test_period_definition_from_a_mid_game_row():
    """Resuming a reference game at a row counts only what follows it, and still adds up to final - start."""
    trace, n, final = next(_reference_games())
    for k in (0, 40, int(np.argmax(trace[:n, 2] <= 1800)), n - 1):
        ends, seg = periods_from_trace(trace[k:], n - k, final)
        sec0, s0 = int(trace[k, 2]), (int(trace[k, 3]), int(trace[k, 4]))
        for q, B in enumerate(BOUNDARIES):
            assert (ends[q] is None) == (sec0 <= B)
        h1 = seg["H1"] or (0, 0)
        assert (h1[0] + seg["H2"][0], h1[1] + seg["H2"][1]) == (final[0] - s0[0], final[1] - s0[1])
    _, seg = periods_from_trace(trace[:0], 0, (24, 17), start_sec=0, start_score=(24, 17))
    assert seg == {"Q1": None, "Q2": None, "Q3": None, "Q4": (0, 0), "H1": None, "H2": (0, 0)}


def _hist(a, b):
    h = np.zeros((outputs.HIST_BINS, outputs.HIST_BINS), dtype=np.int64)
    np.add.at(h, (np.minimum(a, outputs.HIST_BINS - 1), np.minimum(b, outputs.HIST_BINS - 1)), 1)
    return h


@pytest.mark.parametrize("offset", [(0, 0), (7, 3), (0, 14)])
def test_segment_odds_against_brute_force(offset):
    rng = np.random.default_rng(17 + offset[0])
    n = 5000
    a = rng.choice([0, 3, 6, 7, 10, 13, 14, 17, 21], size=n)
    b = rng.choice([0, 3, 7, 10, 14, 17], size=n)
    a[:3] = 140                                    # past the last bin: counted as 127 + offset
    pa, pb = np.minimum(a, 127) + offset[0], np.minimum(b, 127) + offset[1]
    spread, total = -3.0, 17.0                     # integer lines: pushes happen
    got = outputs.segment_odds_from_hist(_hist(a, b), "A", "B", offset=offset, spread=spread, total=total)
    assert got["games"] == n
    assert got["p_win"]["A"] == pytest.approx(np.mean(pa > pb), abs=1e-12)
    assert got["p_win"]["B"] == pytest.approx(np.mean(pb > pa), abs=1e-12)
    assert got["p_tie"] == pytest.approx(np.mean(pa == pb), abs=1e-12)
    assert got["p_tie"] > 0
    assert got["mean_points"]["A"] == pytest.approx(pa.mean(), abs=1e-9)
    assert got["mean_points"]["B"] == pytest.approx(pb.mean(), abs=1e-9)
    sp, tt = got["markets"]["spread"], got["markets"]["total"]
    margin, tot = pa - pb, pa + pb
    assert sp["spread"] == spread and tt["total"] == total and sp["team"] == "A" and sp["samples"] == n
    assert sp["p_cover"] == round(np.mean(margin > -spread), 6)
    assert sp["p_notcover"] == round(np.mean(margin < -spread), 6)
    assert sp["push_rate"] == round(np.mean(margin == -spread), 6) and sp["push_rate"] > 0
    assert sp["mean_margin"] == pytest.approx(margin.mean(), abs=1e-9)
    assert sp["median_margin"] == float(np.median(margin))
    assert tt["p_over"] == round(np.mean(tot > total), 6)
    assert tt["p_under"] == round(np.mean(tot < total), 6)
    assert tt["push_rate"] == round(np.mean(tot == total), 6) and tt["push_rate"] > 0
    assert tt["mean_total"] == pytest.approx(tot.mean(), abs=1e-9)
    assert tt["median_total"] == float(np.median(tot))
    assert sp["american_cover"] == outputs.prob_to_american(sp["p_cover"])


def test_segment_odds_equal_live_odds_on_a_final_histogram():
    rng = np.random.default_rng(5)
    h = _hist(rng.integers(0, 60, 20000), rng.integers(0, 60, 20000))
    for kw in ({}, {"spread": -6.5}, {"total": 51.0}, {"spread": 3.0, "total": 44.5}):
        assert outputs.segment_odds_from_hist(h, "A", "B", **kw) == outputs.live_odds_from_hist(h, "A", "B", **kw)
    with pytest.raises(ValueError):
        outputs.segment_odds_from_hist(np.zeros_like(h), "A", "B")


def _state(seconds, score=(0, 0), **kw):
    return api.LiveState("A", seconds, 1, 10.0, 75.0, score, **kw)


@pytest.mark.parametrize("state", [
    _state(3000, (7, 3), quarter_start_score=(0, 3)),                       # non-zero in Q1
    _state(3000, (7, 3), half_start_score=(7, 0)),                          # the half began at 0-0
    _state(2000, (14, 10), half_start_score=(3, 0)),                        # ... in Q2 too
    _state(1500, (21, 10), quarter_start_score=(14, 10), half_start_score=(14, 7)),   # Q3: they must agree
    _state(2000, (14, 10), quarter_start_score=(17, 3)),                    # quarter start above the score
    _state(600, (28, 17), quarter_start_score=(21, 10), half_start_score=(24, 7)),    # half start above quarter start
    _state(600, (28, 17), half_start_score=(30, 7)),                        # half start above the score
    _state(600, (28, 17), quarter_start_score=(21,)),
    _state(900, (21, 10), quarter_start_score=(14, 10)),                    # a boundary state: the quarter began now
    _state(1800, (21, 10), half_start_score=(14, 10)),
])
def test_contradictory_period_starts_raise(state):
    with pytest.raises(ValueError):
        api.period_starts(state)


def test_implied_period_starts():
    assert api.period_starts(_state(3000, (7, 3))) == ((0, 0), (0, 0))
    assert api.period_starts(_state(2000, (14, 10))) == (None, (0, 0))
    assert api.period_starts(_state(1500, (21, 10), half_start_score=(14, 10))) == ((14, 10), (14, 10))
    assert api.period_starts(_state(1500, (21, 10), quarter_start_score=(14, 10))) == ((14, 10), (14, 10))
    assert api.period_starts(_state(600, (28, 17))) == (None, None)
    # exactly on a boundary the quarter (and at 1800 the half) began at the score
    assert api.period_starts(_state(2700, (7, 3))) == ((7, 3), (0, 0))
    assert api.period_starts(_state(1800, (14, 10))) == ((14, 10), (14, 10))
    assert api.period_starts(_state(900, (21, 10), half_start_score=(14, 10))) == ((21, 10), (14, 10))
    assert api.period_starts(_state(900, (21, 10), quarter_start_score=(21, 10))) == ((21, 10), None)
    assert api.period_starts(dict(offense="A", seconds=0, down=1, distance=10.0, yards_to_goal=75.0, score=(3, 3),
                                  quarter_start_score=(3, 0))) == ((3, 0), None)


def _seg_hist(rng):
    h = np.zeros((len(outputs.SEGMENTS), outputs.HIST_BINS, outputs.HIST_BINS), dtype=np.int64)
    for k in range(len(outputs.SEGMENTS)):
        h[k] = _hist(rng.integers(0, 20, 1000), rng.integers(0, 20, 1000))
    return h


def test_live_segments_status_offsets_and_none_odds():
    sg = _seg_hist(np.random.default_rng(2))
    sg[0] = 0                                            # Q1 ended before a Q2 state: the kernel counted nothing there
    st = _state(2000, (14, 10))                          # Q2, quarter start unknown
    out = api.live_segments(st, sg, "A", "B", {"Q2": {"spread": 1.5}, "H1": {"total": 30.5}})
    assert [out[k]["status"] for k in outputs.SEGMENTS] == ["ended", "in_progress", "future", "future", "in_progress",
                                                            "future"]
    assert out["Q1"]["odds"] is None and not out["Q1"]["hist"].any()
    assert out["Q2"]["odds"] is None and out["Q2"]["offset"] is None and out["Q2"]["hist"].sum() == 1000
    assert out["H1"]["offset"] == (14, 10)
    assert out["H1"]["odds"] == outputs.segment_odds_from_hist(sg[4], "A", "B", offset=(14, 10), total=30.5)
    assert out["Q3"]["odds"] == outputs.segment_odds_from_hist(sg[2], "A", "B")
    known = api.live_segments(_state(2000, (14, 10), quarter_start_score=(7, 3)), sg, "A", "B", {"Q2": {"spread": 1.5}})
    assert known["Q2"]["offset"] == (7, 7)
    assert known["Q2"]["odds"] == outputs.segment_odds_from_hist(sg[1], "A", "B", offset=(7, 7), spread=1.5)
    # a Q4 state without start scores: Q4 and H2 in progress with unknown starts, everything else ended
    late = api.live_segments(_state(300, (28, 17)), sg, "A", "B")
    assert [late[k]["status"] for k in outputs.SEGMENTS] == ["ended", "ended", "ended", "in_progress", "ended",
                                                             "in_progress"]
    assert all(late[k]["odds"] is None for k in outputs.SEGMENTS)
    # the clock at 0: Q4 and H2 are in progress and end at once
    over = api.live_segments(_state(0, (28, 17), quarter_start_score=(21, 17), half_start_score=(14, 10)), sg, "A", "B")
    assert over["Q4"]["offset"] == (7, 0) and over["H2"]["offset"] == (14, 7)


@pytest.mark.parametrize("lines", [{"H1": 3.5}, {"Q2": {}}, {"Q3": {"spread": 1.0, "moneyline": -110}}])
def test_bad_period_lines_raise(lines):
    with pytest.raises(ValueError):
        api.live_segments(_state(3000), _seg_hist(np.random.default_rng(0)), "A", "B", lines)
