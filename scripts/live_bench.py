"""Live pricing on the GPU: python scripts/live_bench.py [--games 100000] [--calls 50] [--call-games 1000000] [--out FILE]

(a) a win-probability curve: the iteration-start states of one Philox game of Kansas State - Iowa State (about 150),
    every state x `--games` games, all in ONE launch (one entry per state; the entries share one specialisation);
(b) re-pricing after every snap: `--calls` successive calls of `--call-games` games, each from the next state of that
    game, with the memo kept between calls (memo="persistent");
(c) the card and its power limit.
Shipped models (stage 2 stand-in, heuristic play call).  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from fast_monte_carlo_b200 import artifacts as art  # noqa: E402
from fast_monte_carlo_b200.engine import Engine, GameState, MatchupSpec  # noqa: E402

KSU, ISU = (15.6, 35.7, 20.0), (11.0, 31.5, 20.6)


def curve_states(eng, seed):
    """The iteration-start states of Philox game 0 (Kansas State receives), from the engine's own trace."""
    eng.set_matchups([MatchupSpec("Kansas State", "Iowa State", KSU, ISU, 1, 0, 1, 0)])
    r = eng.simulate_host(seed, want_trace=True, want_iters=True)
    out = []
    for row in r["trace"][0, :int(r["iters"][0])]:
        off = 0 if row[0] == 1.0 else 1                       # trace column 0 is relative to the receiver, team 0 here
        if row[1] > 4 or not (0.0 < row[6] < 100.0):
            continue                                          # downs past 4 / yard lines past 100: not a real game state
        out.append(GameState(offense=off, seconds=int(row[2]), down=int(row[1]), distance=float(row[5]),
                             yards_to_goal=float(row[6]), score=(int(row[3]), int(row[4]))))
    return out


def hit_rate(c):
    return c["memo_hits"] / c["memo_probes"] if c["memo_probes"] else 0.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True, check=False)
    return q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=100_000)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--call-games", type=int, default=1_000_000)
    ap.add_argument("--seed", type=int, default=20251018)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ms = art.load_default_models()
    res = {"card": card()}

    # (a) the curve in one launch
    eng = Engine(ms, device=0, memo="on")
    states = curve_states(eng, args.seed)
    n = args.games
    specs = [MatchupSpec("Kansas State", "Iowa State", KSU, ISU, n, 0, n, m * n, start=s) for m, s in enumerate(states)]
    distinct = len({(s.sp_a, s.sp_b, eng.coach_col(s.team_a), eng.coach_col(s.team_b)) for s in specs})
    eng.set_matchups(specs)
    t0 = time.perf_counter()
    eng.simulate_host(args.seed + 1, want_scores=False)       # specialises and uploads the tables; warms the kernel
    first = time.perf_counter() - t0
    walls = []
    for rep in range(3):
        t0 = time.perf_counter()
        r = eng.simulate_host(args.seed + 2 + rep, want_scores=False)
        walls.append(time.perf_counter() - t0)
    c = r["counters"]
    wall = min(walls)
    res["curve"] = {"states": len(states), "games_per_state": n, "games": c["games"], "specialisations": distinct,
                    "packed_slots_equal": bool((eng.ctx.packed_slots(0) == eng.ctx.packed_slots(len(specs) - 1)).all()),
                    "first_call_s": round(first, 4), "wall_s": round(wall, 4), "wall_s_all": [round(w, 4) for w in walls],
                    "plays_per_s": c["plays"] / wall, "memo_hit_rate": round(hit_rate(c), 4),
                    "how": "fmc_simulate_host of all states in one launch (per-entry histograms copied back, no per-game "
                           "scores), host clock around the synchronous call, best of 3 after one warm-up call"}
    eng.close()

    # (b) re-pricing after every snap, memo kept between calls
    eng = Engine(ms, device=0, memo="persistent")
    g = args.call_games
    calls = []
    t_all = time.perf_counter()
    for i in range(args.calls):
        s = states[i % len(states)]
        t0 = time.perf_counter()
        eng.set_matchups([MatchupSpec("Kansas State", "Iowa State", KSU, ISU, g, 0, g, 0, start=s)])
        r = eng.simulate_host(args.seed + 100 + i, want_scores=False)
        calls.append({"s": round(time.perf_counter() - t0, 4), "hit_rate": round(hit_rate(r["counters"]), 4),
                      "plays": r["counters"]["plays"]})
    total = time.perf_counter() - t_all
    steady = calls[1:] if len(calls) > 1 else calls
    res["reprice"] = {"calls": len(calls), "games_per_call": g, "total_s": round(total, 3),
                      "calls_per_s": len(calls) / total,
                      "calls_per_s_after_first": len(steady) / sum(x["s"] for x in steady),
                      "per_call": calls,
                      "how": "set_matchups (same pair: the tables stay, only the start state changes) + fmc_simulate_host "
                             "per call, host clock; the first call specialises the tables and starts with an empty memo"}
    eng.close()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
