"""Hand-built injected-draw streams that force overtime possessions, for the CPU and GPU overtime tests.

Every possession kind below takes a fixed number of snaps whatever the two teams' strengths, so a plan (a list of
possession kinds in overtime order) gives the game's whole stream and its result can be worked out by hand.  The games
start at 0:00 with the score level (a live entry), so overtime starts at iteration 0.  Draw slots are the kernel's
(fmc_sim.cuh S_U_CALL ...): a u slot holds the uniform, a z slot the normal deviate itself."""
from __future__ import annotations

import numpy as np

MAX_ITERS, N_SLOTS = 360, 16
U_CALL, U_COMP, Z_YARDS, U_EX, U_BOOST, U_FIN, U_S2, Z_INT, U_GO, U_FG, Z_GROSS, Z_RET, U_TB, U_P1, U_WR, U_YQ = range(16)


def _rec(**kw):
    r = np.full(N_SLOTS, 0.5)
    r[[Z_YARDS, Z_INT, Z_GROSS, Z_RET]] = 0.0
    for k, v in kw.items():
        r[globals()[k]] = v
    return r


# one snap each
INCOMPLETE = _rec(U_CALL=0.999, U_COMP=0.9999, U_S2=0.0)                 # pass, not complete, stage 2 -> incomplete
SACK = _rec(U_CALL=0.999, U_COMP=0.9999, U_S2=0.9999, Z_YARDS=-1000.0)    # stage 2 -> sack, the 20-yard maximum loss
LONG_TD = _rec(U_CALL=0.999, U_COMP=0.0, Z_YARDS=1000.0, U_EX=0.0, U_BOOST=0.999, U_FIN=0.999)   # explosive, to the goal
SHORT_TD = _rec(U_CALL=0.999, U_COMP=0.0, U_EX=0.999, U_FIN=0.0)         # red-zone finish (inside the 12, down <= 3)
FG_GOOD = _rec(U_GO=0.999, U_FG=0.0)                                       # fourth down: no go, field goal made
FG_MISSED = _rec(U_GO=0.999, U_FG=0.9999)
PUNT = _rec(U_GO=0.999, U_TB=0.999)

# possession kinds (from the opponent's 25, or a try) -> their snaps, and the points they add
KINDS = {
    "td": ([SACK, LONG_TD], 7),                                      # 7 in period 1; 6 (+ try) in period 2
    "fg": ([INCOMPLETE] * 3 + [FG_GOOD], 3),
    "none": ([INCOMPLETE] * 3 + [FG_MISSED], 0),
    "punt": ([SACK] * 3 + [PUNT], 0),                                # sacked back to the 15, fourth and 70: punt
    "ok": ([SHORT_TD], 2),                                           # two-point try made
    "fail": ([INCOMPLETE], 0),                                       # two-point try failed
}


def stream_for(plan) -> tuple:
    """(stream [MAX_ITERS][N_SLOTS], iterations) of a plan; the draws after the plan are incomplete passes."""
    recs = [r for k in plan for r in KINDS[k][0]]
    s = np.tile(INCOMPLETE, (MAX_ITERS, 1))
    s[:len(recs)] = recs
    return s, len(recs)


# (plan, max_periods, points of the team with the first possession of period 1, of the other, overtime periods)
SCENARIOS = {
    "td_td_in_period_1": (["td", "td", "fg", "none"], 16, 7, 10, 2),
    "period_2_td_wins_without_try": (["none", "none", "none", "td"], 16, 6, 0, 2),
    "failed_and_made_tries": (["td", "td", "td", "ok", "td", "fail"], 16, 13, 15, 2),
    "shoot_out_from_period_3": (["fg", "fg", "td", "fail", "td", "fail", "ok", "ok", "ok", "fail"], 16, 11, 13, 4),
    "max_periods_cap": (["none"] * 4 + ["fail", "fail"], 3, 0, 0, 3),
    "punt_after_sacks": (["punt", "fg"], 16, 0, 3, 1),
}
START_SCORE = (7, 7)


def expected(name, game: int):
    """(scores (A, B), iterations, periods) of scenario `name` as game `game` (team game & 1 has the first possession)."""
    plan, _, first_pts, other_pts, periods = SCENARIOS[name]
    first = game & 1
    sc = [START_SCORE[0], START_SCORE[1]]
    sc[first] += first_pts
    sc[first ^ 1] += other_pts
    return tuple(sc), stream_for(plan)[1], periods
