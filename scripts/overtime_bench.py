"""What overtime costs on the GPU: python scripts/overtime_bench.py [--games 10000000] [--curve-games 100000] [--reps 5]
[--out FILE]

(a) BASELINE configs[1]: `--games` games of Kansas State - Iowa State from the kickoff, memo on, with overtime off and on
    (fmc_simulate vs fmc_simulate_overtime with the overtime histogram).  About 3 % of games are level after regulation
    and play about 15 more snaps, so the expected extra work is under 0.5 % of the plays;
(b) a live curve of 150 entries that ends at 0:00 with the score level: the iteration-start states of one Philox game
    (the first 149) and the level state, x `--curve-games` games, in one launch, overtime off and on.  There the last
    entry plays nothing but overtime.
The two arms of each workload run alternately, `--reps` times each after one warm-up call of each, with the same seed,
and are timed with CUDA events around the launch (output buffers are zeroed before the window).  The counters report
the plays of each arm, so the extra work is measured next to the extra time.  Prints the card's name, power limit and
max SM clock beside the numbers, as one JSON object (and writes it to --out)."""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from fast_monte_carlo_b200 import artifacts as art, outputs  # noqa: E402
from fast_monte_carlo_b200.engine import Engine, GameState, MatchupSpec, OvertimeRules  # noqa: E402
from fast_monte_carlo_b200.native import COUNTER_NAMES  # noqa: E402
from live_bench import ISU, KSU, card, curve_states  # noqa: E402


def timed(eng, n_entries, seed, overtime):
    """(kernel ms by CUDA events, counters) of one launch on the current matchup list."""
    dev = torch.device("cuda", eng.ctx.device)
    hist = torch.zeros((n_entries, 2, outputs.HIST_BINS, outputs.HIST_BINS), dtype=torch.int32, device=dev)
    cnt = torch.zeros(32, dtype=torch.int64, device=dev)
    oth = torch.zeros((n_entries, 2, outputs.OT_MAX_PERIODS + 1, 3), dtype=torch.int32, device=dev) if overtime else None
    st = torch.cuda.current_stream(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    t0.record(st)
    eng.ctx.simulate_device(seed=seed, hist=hist.data_ptr(), counters=cnt.data_ptr(), cuda_stream=st.cuda_stream,
                            overtime=OvertimeRules() if overtime else None, ot_hist=oth.data_ptr() if oth is not None else 0)
    t1.record(st)
    t1.synchronize()
    c = dict(zip(COUNTER_NAMES, cnt.cpu().tolist()))
    if oth is not None:
        assert int(oth.sum()) == c["games"]
    return t0.elapsed_time(t1), c


def compare(eng, n_entries, seed, reps):
    timed(eng, n_entries, seed, False)                 # warm-up: tables, memo layout
    timed(eng, n_entries, seed, True)
    ms = {False: [], True: []}
    cs = {}
    for r in range(reps):
        for arm in ((False, True) if r % 2 == 0 else (True, False)):
            t, cs[arm] = timed(eng, n_entries, seed, arm)
            ms[arm].append(t)
    off, on = statistics.median(ms[False]), statistics.median(ms[True])
    return {"games": cs[False]["games"], "ms_off": round(off, 3), "ms_on": round(on, 3),
            "ms_off_all": [round(x, 3) for x in ms[False]], "ms_on_all": [round(x, 3) for x in ms[True]],
            "time_overhead_pct": round(100.0 * (on - off) / off, 2),
            "plays_off": cs[False]["plays"], "plays_on": cs[True]["plays"],
            "plays_overhead_pct": round(100.0 * (cs[True]["plays"] - cs[False]["plays"]) / cs[False]["plays"], 3),
            "ot_games": cs[True]["ot_games"], "ot_periods": cs[True]["ot_periods"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=10_000_000)
    ap.add_argument("--curve-games", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=20251018)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("overtime_bench.py measures the GPU: no CUDA device")
    ms = art.load_default_models()
    res = {"card": card(), "how": "median of --reps CUDA-event times per arm, arms alternated, same seed"}
    eng = Engine(ms, device=0, memo="on")
    n = args.games
    eng.set_matchups([MatchupSpec("Kansas State", "Iowa State", KSU, ISU, n, 0, n, 0)])
    res["configs1"] = compare(eng, 1, args.seed, args.reps)
    states = curve_states(eng, args.seed)[:149] + [GameState(offense=0, seconds=0, score=(21, 21))]
    g = args.curve_games
    eng.set_matchups([MatchupSpec("Kansas State", "Iowa State", KSU, ISU, g, 0, g, m * g, start=s)
                      for m, s in enumerate(states)])
    res["curve"] = dict(states=len(states), games_per_state=g, **compare(eng, len(states), args.seed + 1, args.reps))
    eng.close()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
