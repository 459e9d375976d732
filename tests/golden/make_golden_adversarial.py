"""Golden trajectories of the UNMODIFIED reference simulate_game under ADVERSARIAL injected draws
(tests/streams.py: all-zero / all-one uniforms, +-4 sigma normals, mixtures) -- pins the oracle on the rare
branches (touchback punts, missed field goals, sacks past the 100, down >= 5 chains, late-game go-for-it).
Needs the original project (FMC_REFERENCE_DIR=<its directory>):   python tests/golden/make_golden_adversarial.py
"""
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ref_harness as rh     # noqa: E402
from streams import adversarial_stream   # noqa: E402


def main():
    t0 = time.time()
    mod = rh.load_reference(cache_off=True)
    pairs = [("Kansas State", "Iowa State"), ("UTSA", "Ohio State")]
    n_games = int(os.environ.get("FMC_GOLDEN_GAMES", "24"))
    stream = adversarial_stream(n_games, 2025)
    traces = np.full((n_games, rh.MAX_ITERS, 8), np.nan)
    scores = np.zeros((n_games, 2), dtype=np.int32)
    iters = np.zeros(n_games, dtype=np.int32)
    plays = np.zeros(n_games, dtype=np.int32)
    meta = []
    for g in range(n_games):
        a, b = pairs[(g // 2) % len(pairs)]
        if g & 1:
            a, b = b, a
        ca, cb = rh.team_context(mod, a), rh.team_context(mod, b)
        res, trc, used = rh.run_game_injected(mod, ca, cb, stream[g])
        traces[g, :trc.shape[0]] = trc
        scores[g] = (res["off_score"], res["def_score"])
        iters[g] = trc.shape[0]
        plays[g] = res["box"][a]["plays"] + res["box"][b]["plays"]
        meta.append(dict(first=a, second=b, sp_first=[ca.sp_rating, ca.sp_offense, ca.sp_defense],
                         sp_second=[cb.sp_rating, cb.sp_offense, cb.sp_defense], pattern=g % 6))
        print(f"game {g} pattern {g % 6}: {a} {scores[g,0]} - {b} {scores[g,1]}  iters {iters[g]} plays {plays[g]} ({time.time()-t0:.0f}s)", flush=True)
    np.savez_compressed(os.path.join(HERE, "ref_trajectories_adversarial.npz"), stream_seed=2025, traces=traces,
                        scores=scores, iters=iters, plays=plays, meta=json.dumps(meta))


if __name__ == "__main__":
    main()
