"""What fourth-down decisions inside overtime cost on the GPU: python scripts/overtime_live_bench.py [--games 20000]
[--reps 5] [--out FILE]

Workload: an overtime fourth-down chart of one pair (Kansas State with the ball against Iowa State) in one launch.
Scenarios: periods 1 and 2; on the first possession level at 24-24, and on the second possession trailing by 3 and by
7 in period 1, by 3 and by 8 in period 2 (a touchdown and a made try; 7 behind is not a margin the rules reach there).
In each, 4th & 1..10 (distance at most the yards to goal) at yards to goal 1, 6, 11, 16 and 21.  Each state carries
its policy entry and one entry per available choice (go; field goal, every state being inside the 38; punt from the 16
out), `--games` games each -- the launch `api.fourth_down_decisions` makes for the chart.  Two arms on the same entries
and seed: "decision" with the forced choices and "policy" with every code 0 (the overtime instantiations without the
decision rule).  The arms do not play the same games, so the counters report the plays of each arm next to the times.
The arms run alternately, `--reps` times each after one warm-up call of each, timed with CUDA events around the launch
(output buffers are zeroed before the window).  Prints the card's name, power limit and max SM clock beside the numbers,
as one JSON object (and writes it to --out)."""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from fast_monte_carlo_b200 import artifacts as art  # noqa: E402
from fast_monte_carlo_b200.engine import (FOURTH_DOWN_FG, FOURTH_DOWN_GO, FOURTH_DOWN_PUNT, Engine, GameState,  # noqa: E402
                                          MatchupSpec, OvertimeState)
from fourth_down_bench import timed  # noqa: E402
from live_bench import ISU, KSU, card  # noqa: E402

# (period, possession, points of Kansas State with the ball, of Iowa State)
SCENARIOS = [(1, 1, 24, 24), (1, 2, 21, 24), (1, 2, 17, 24), (2, 1, 24, 24), (2, 2, 21, 24), (2, 2, 16, 24)]


def chart():
    """(state, code) of every entry of the chart."""
    out = []
    for k, p, a, b in SCENARIOS:
        for ytg in range(1, 26, 5):
            for dist in range(1, 11):
                if dist > ytg:
                    continue
                st = dict(offense=0, seconds=0, down=4, distance=float(dist), yards_to_goal=float(ytg), score=(a, b),
                          overtime=OvertimeState(k, p))
                codes = [0, FOURTH_DOWN_GO, FOURTH_DOWN_FG] + ([FOURTH_DOWN_PUNT] if ytg >= 16 else [])
                out += [(st, c) for c in codes]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=20_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=20251023)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("overtime_live_bench.py measures the GPU: no CUDA device")
    entries = chart()
    g = args.games
    eng = Engine(art.load_default_models(), device=0, memo="on")

    def arm(decision):
        eng.set_matchups([MatchupSpec("Kansas State", "Iowa State", KSU, ISU, g, 0, g, m * g,
                                      start=GameState(**st, fourth_down=c if decision else 0))
                          for m, (st, c) in enumerate(entries)])

    for d in (True, False):                       # warm-up: tables, memo layout
        arm(d)
        timed(eng, len(entries), args.seed)
    ms = {True: [], False: []}
    cs = {}
    for r in range(args.reps):
        for d in ((True, False) if r % 2 == 0 else (False, True)):
            arm(d)                                # same pairs: only the start words change
            t, cs[d] = timed(eng, len(entries), args.seed)
            ms[d].append(t)
    eng.close()
    dec, pol = statistics.median(ms[True]), statistics.median(ms[False])
    res = {"card": card(), "how": "median of --reps CUDA-event times per arm, arms alternated, same entries and seed",
           "states": len({(s["overtime"], s["score"], s["distance"], s["yards_to_goal"]) for s, _ in entries}),
           "entries": len(entries), "games_per_entry": g, "games": cs[True]["games"],
           "ms_decision": round(dec, 3), "ms_policy": round(pol, 3),
           "ms_decision_all": [round(x, 3) for x in ms[True]], "ms_policy_all": [round(x, 3) for x in ms[False]],
           "time_overhead_pct": round(100.0 * (dec - pol) / pol, 2),
           "plays_decision": cs[True]["plays"], "plays_policy": cs[False]["plays"],
           "ns_per_play_decision": round(1e6 * dec / cs[True]["plays"], 3),
           "ns_per_play_policy": round(1e6 * pol / cs[False]["plays"], 3),
           "ot_periods_decision": cs[True]["ot_periods"], "ot_periods_policy": cs[False]["ot_periods"]}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
