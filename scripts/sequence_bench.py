"""What the next-score / drive / race histograms cost on the GPU: python scripts/sequence_bench.py [--games 10000000]
[--curve-games 100000] [--reps 5] [--out FILE]

(a) BASELINE configs[1]: `--games` games of Kansas State - Iowa State from the kickoff, memo on, with and without
    sequence_hist (fmc_simulate vs fmc_simulate_markets, the per-game rows in library scratch);
(b) a live curve: the iteration-start states of one Philox game (about 150 entries of one pair) x `--curve-games`
    games, in one launch, with and without sequence_hist.
The two arms of each workload run alternately, `--reps` times each after one warm-up call of each, with the same seed,
and are timed with CUDA events around the launch (output buffers are zeroed before the window).  The score histograms
of the two arms are compared.  Prints the card's name, power limit and max SM clock beside the numbers, as one JSON
object (and writes it to --out)."""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from fast_monte_carlo_b200 import artifacts as art, outputs  # noqa: E402
from fast_monte_carlo_b200.engine import Engine, MatchupSpec  # noqa: E402
from live_bench import ISU, KSU, card, curve_states  # noqa: E402


def timed(eng, n_entries, seed, sequence):
    """(kernel ms by CUDA events, score histogram, games) of one launch on the current matchup list."""
    dev = torch.device("cuda", eng.ctx.device)
    hist = torch.zeros((n_entries, 2, outputs.HIST_BINS, outputs.HIST_BINS), dtype=torch.int32, device=dev)
    cnt = torch.zeros(32, dtype=torch.int64, device=dev)
    sq = torch.zeros((n_entries, 2, outputs.SEQ_BINS), dtype=torch.int32, device=dev) if sequence else None
    st = torch.cuda.current_stream(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    t0.record(st)
    eng.ctx.simulate_device(seed=seed, hist=hist.data_ptr(), counters=cnt.data_ptr(), cuda_stream=st.cuda_stream,
                            sequence_hist=sq.data_ptr() if sq is not None else 0)
    t1.record(st)
    t1.synchronize()
    if sq is not None:
        assert int(sq[:, :, outputs.SEQ_BIN_DRIVE0:outputs.SEQ_BIN_RACE0].sum()) == int(cnt[0])
    return t0.elapsed_time(t1), hist.cpu(), int(cnt[0])


def compare(eng, n_entries, seed, reps):
    timed(eng, n_entries, seed, False)                 # warm-up: tables, memo layout, the device scratch of the rows
    timed(eng, n_entries, seed, True)
    ms = {False: [], True: []}
    hists = {}
    games = 0
    for r in range(reps):
        for arm in ((False, True) if r % 2 == 0 else (True, False)):
            t, h, games = timed(eng, n_entries, seed, arm)
            ms[arm].append(t)
            hists[arm] = h
    plain, withseq = statistics.median(ms[False]), statistics.median(ms[True])
    return {"games": games, "ms_without": round(plain, 3), "ms_with_sequence_hist": round(withseq, 3),
            "ms_without_all": [round(x, 3) for x in ms[False]], "ms_with_all": [round(x, 3) for x in ms[True]],
            "overhead_pct": round(100.0 * (withseq - plain) / plain, 2),
            "score_hist_equal": bool(torch.equal(hists[False], hists[True]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=10_000_000)
    ap.add_argument("--curve-games", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=20251018)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sequence_bench.py measures the GPU: no CUDA device")
    ms = art.load_default_models()
    res = {"card": card(), "how": "median of --reps CUDA-event times per arm, arms alternated, same seed"}
    eng = Engine(ms, device=0, memo="on")
    n = args.games
    eng.set_matchups([MatchupSpec("Kansas State", "Iowa State", KSU, ISU, n, 0, n, 0)])
    res["configs1"] = compare(eng, 1, args.seed, args.reps)
    states = curve_states(eng, args.seed)
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
