"""Golden fixtures for the binary play-call model path (SURVEY 8a row a4 / 8f row 3), from the UNMODIFIED reference.

Needs the original project (FMC_REFERENCE_DIR=<its directory>):   python tests/golden/make_golden_play_json.py

`play_model.json` and `calibration.json` are not in the reference snapshot, so the reference falls back to
`pass_prob_v1` (FMC:326-328).  This script gives the reference module a SYNTHETIC `play_model.json` of the trained
shape (fast_monte_carlo_b200.synth.synthetic_play_model_json: multi:softprob over [pass, run], 16 features of the
shipped features.pkl, categorical `head_coach`) plus a `calibration.json`, lets its own `_load_play_policy`
(FMC:319-337) load them (xgboost = oracle/fake_xgboost.py), and records

  play_json.npz   the synthetic model (JSON text), the temperature, P(pass) of the reference's own
                  `play_call_pass_prob_binary` (FMC:407-427) on 400 random states for two offense teams, and 8
                  injected-stream trajectories of its `simulate_game` with the model policy on.
"""
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from fast_monte_carlo_b200 import synth                # noqa: E402
from oracle import ref_harness as rh                   # noqa: E402
from oracle.c_oracle import make_stream                # noqa: E402

TEMPERATURE = 1.3
PAIRS = [("Kansas State", "Iowa State"), ("UTSA", "Ohio State")]


def main():
    t0 = time.time()
    mod = rh.load_reference()
    model = synth.synthetic_play_model_json()
    text = json.dumps(model)
    scratch = mod._scratch_dir
    with open(os.path.join(scratch, "play_model.json"), "w") as f:
        f.write(text)
    with open(os.path.join(scratch, "calibration.json"), "w") as f:
        json.dump({"temperature": TEMPERATURE}, f)
    old = os.getcwd()
    os.chdir(scratch)
    try:
        mod._load_play_policy()                          # FMC:319-337: booster, features.pkl, label_encoder.pkl, T
    finally:
        os.chdir(old)
    assert mod._PLAY_BOOSTER is not None and mod._PLAY_TEMP == TEMPERATURE
    assert mod._PLAY_CLASSES == ["pass", "run"] and len(mod._PLAY_FEATURES) == 16

    # ---- the wrapper on random states -----------------------------------------------------------------
    rng = np.random.default_rng(12)
    n = 400
    states = np.zeros((n, 7))
    states[:, 0] = rng.choice([1, 2, 3, 4, 5], size=n)
    states[:, 1] = np.where(rng.random(n) < 0.5, np.round(rng.uniform(0.5, 20, n), 1), rng.uniform(0.1, 25, n))
    states[:, 2] = np.where(rng.random(n) < 0.5, rng.integers(1, 100, n), rng.uniform(0.5, 99.5, n))
    states[:, 3] = np.round(rng.normal(0, 12, n))
    states[rng.random(n) < 0.25, 3] = 0
    states[:, 4] = rng.integers(1, 3601, n)
    states[:, 5] = rng.integers(0, 2, n)             # which team of the pair is on offense
    states[:, 6] = rng.integers(0, len(PAIRS), n)
    p_pass = np.zeros(n)
    ctxs = {t: rh.team_context(mod, t) for p in PAIRS for t in p}
    for i in range(n):
        a, b = PAIRS[int(states[i, 6])]
        off, de = (ctxs[a], ctxs[b]) if states[i, 5] == 0 else (ctxs[b], ctxs[a])
        row = mod.build_state_row(off, de, int(states[i, 0]), float(states[i, 1]), float(states[i, 2]), int(states[i, 4]), 3, 3)
        mod._fill_row(row, off, de, int(states[i, 0]), float(states[i, 1]), float(states[i, 2]), int(states[i, 4]), 3, 3,
                      passer_name="Unknown", target_name="Unknown", score_diff=int(states[i, 3]))
        p_pass[i] = mod.play_call_pass_prob_binary(row, offense_team_name=off.name)

    # ---- trajectories with the model policy on -----------------------------------------------------------
    n_games = int(os.environ.get("FMC_GOLDEN_GAMES", "8"))
    stream = make_stream(n_games, 13)
    traces = np.full((n_games, rh.MAX_ITERS, 8), np.nan)
    scores = np.zeros((n_games, 2), dtype=np.int32)
    iters = np.zeros(n_games, dtype=np.int32)
    meta = []
    for g in range(n_games):
        a, b = PAIRS[(g // 2) % len(PAIRS)]
        first, second = (b, a) if (g & 1) else (a, b)
        ca, cb = rh.team_context(mod, first), rh.team_context(mod, second)
        res, trc, used = rh.run_game_injected(mod, ca, cb, stream[g])
        traces[g, :trc.shape[0]] = trc
        scores[g] = (res["off_score"], res["def_score"])
        iters[g] = trc.shape[0]
        meta.append(dict(team_a=a, team_b=b, sp_a=[ctxs[a].sp_rating, ctxs[a].sp_offense, ctxs[a].sp_defense],
                         sp_b=[ctxs[b].sp_rating, ctxs[b].sp_offense, ctxs[b].sp_defense]))
        print(f"game {g}: {first} {scores[g,0]} - {second} {scores[g,1]}  iters {iters[g]}  ({time.time()-t0:.0f}s)", flush=True)
    np.savez_compressed(os.path.join(HERE, "play_json.npz"), model_json=np.frombuffer(text.encode(), dtype=np.uint8),
                        temperature=TEMPERATURE, states=states, p_pass=p_pass, stream_seed=13, traces=traces,
                        scores=scores, iters=iters, meta=json.dumps(meta),
                        features=json.dumps([str(c) for c in mod._PLAY_FEATURES]),      # features.pkl
                        classes=json.dumps(list(mod._PLAY_CLASSES)),                    # label_encoder.pkl
                        pairs=json.dumps(PAIRS))
    print("done in %.0fs" % (time.time() - t0))


if __name__ == "__main__":
    main()
