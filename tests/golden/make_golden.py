"""Regenerates every fixture under tests/golden/ from the REAL reference objects.

Needs the original project (FMC_REFERENCE_DIR=<its directory>):   python tests/golden/make_golden.py

  sklearn_quantiles.npz   live `Pipeline.predict` of the nine quantile pipelines (FMC:658-668) on random
                          rows, incl. exact-zero features, down >= 5 and real player names
  transformers.npz        live `ColumnTransformer.transform` column layout (FMC:651-654) and
                          `scaler.pkl.transform`
  priors.json             load_sp_flex / lookup_sp_flex / _norm_team / csv_base_from of the reference
                          module itself on PregameSPPlus2025_1.csv (FMC:1573-1644, 1717-1722)
  ref_scalars.json        pass_prob_v1, go_for_it_prob, field_goal_prob, explosive_prob, rz_finish_prob_*,
                          matchup_bias, yardage_multiplier evaluated by the reference module
  ref_trajectories.npz    per-iteration states of the reference's own simulate_game under an injected
                          draw stream (oracle/ref_harness.py); xgboost replaced by oracle/fake_xgboost.py
  xgb_provisional.json    SURVEY Appendix G vectors for the XGBoost boosters (xgboost is not installed:
                          these are provisional, "two independent implementations agree" anchors)
"""
import json
import os
import sys
import time

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from fast_monte_carlo_b200 import artifacts as art   # noqa: E402
from oracle import ref_harness as rh                  # noqa: E402

REF = rh.REFERENCE_DIR

NUM = art.NUM_FEATURES


def random_rows(rng, n, teams_sp):
    down = rng.choice([1, 2, 3, 4, 5, 6], size=n, p=[.36, .30, .20, .10, .03, .01])
    dist = np.clip(np.round(rng.normal(8, 4, n), 1), 0.5, 30)
    ytg = rng.integers(1, 100, n).astype(float)
    frac = rng.random(n) < 0.5
    ytg = np.where(frac, ytg + rng.random(n), ytg)
    dist = np.where(frac, dist + rng.random(n) * 0.1, dist)
    sd = np.round(rng.normal(0, 14, n)).astype(int)
    sd[rng.random(n) < 0.2] = 0
    sec = rng.integers(1, 3601, n)
    pair = np.stack([rng.permutation(len(teams_sp))[:2] for _ in range(n)])
    off = teams_sp[pair[:, 0]]
    de = teams_sp[pair[:, 1]]
    num = np.zeros((n, 17))
    num[:, 0] = down; num[:, 1] = dist; num[:, 2] = ytg; num[:, 3] = ytg <= 20; num[:, 4] = sd; num[:, 5] = sec
    num[:, 6] = 3; num[:, 7] = 3
    num[:, 8] = off[:, 0]; num[:, 9] = off[:, 1]; num[:, 10] = de[:, 2]; num[:, 11] = de[:, 0]
    num[:, 12] = dist >= (ytg - 0.5); num[:, 13] = (down == 4) & (dist <= 2.0); num[:, 14] = ytg <= 33
    num[:, 15] = np.where(sec > 1800, 1, 2); num[:, 16] = (sec % 1800) <= 120
    return num


def frame(num, **names):
    df = pd.DataFrame(num, columns=NUM)
    for c in ("down", "is_red_zone", "score_diff", "seconds_remaining", "offenseTimeouts", "defenseTimeouts",
              "goal_to_go", "fourth_and_short", "fg_range", "half", "two_minute"):
        df[c] = df[c].astype("int64")
    for k, v in names.items():
        df[k] = v
    return df


def main():
    t0 = time.time()
    mod = rh.load_reference()
    sp = mod.load_sp_flex(os.path.join(REF, "PregameSPPlus2025_1.csv"))
    teams_sp = sp[["RATING", "OFFENSE", "DEFENSE"]].to_numpy(dtype=float)

    # ---- priors ---------------------------------------------------------------------------------
    queries = ["Kansas State", "Iowa State", "kansas state", "App State", "Appalachian State", "UMass",
               "Massachusetts", "UTSA", "UT San Antonio", "Miami (OH)", "miami oh", "Hawai'i", "Ole Miss",
               "Texas A&M", "texas a&m", "San José State", "Sam Houston", "UL Monroe", "Louisiana Monroe",
               "Southern Miss", "UConn", "Connecticut", "Alabam", "State"]
    lookups = {}
    for q in queries:
        try:
            lookups[q] = list(mod.lookup_sp_flex(q, sp))
        except ValueError as e:
            lookups[q] = {"error": str(e)}
    priors = dict(
        table=[dict(team=r.team, RATING=float(r.RATING), OFFENSE=float(r.OFFENSE), DEFENSE=float(r.DEFENSE),
                    norm_team=r.norm_team) for r in sp.itertuples()],
        lookups=lookups,
        csv_base={f"{a}|{b}|{w}": mod.csv_base_from(a, b, w) for a, b, w in
                  [("Kansas State", "Iowa State", 1), ("Miami (OH)", "Texas A&M", 12), ("Hawai'i", "UL Monroe", 3)]},
    )
    json.dump(priors, open(os.path.join(HERE, "priors.json"), "w"), indent=0)

    # ---- scalar helper functions of the reference ------------------------------------------------
    rng = np.random.default_rng(11)
    A = rh.team_context(mod, "Kansas State"); B = rh.team_context(mod, "Iowa State")
    U = rh.team_context(mod, "UTSA"); O = rh.team_context(mod, "Ohio State")
    sc = dict(pass_prob_v1=[], go_for_it_prob=[], field_goal_prob=[], modifiers=[])
    for _ in range(400):
        down = int(rng.integers(1, 8)); dist = float(np.round(rng.uniform(0.2, 25), 2)); ytg = float(np.round(rng.uniform(-3, 104), 2))
        sec = int(rng.integers(1, 3601)); sd = int(rng.integers(-21, 22))
        sc["pass_prob_v1"].append([down, dist, ytg, sec, sd, mod.pass_prob_v1(down, dist, ytg, sec, sd)])
        d4 = float(rng.choice([0.5, 1, 1.0001, 2, 2.5, 3, 4, 4.2, 7]))
        sc["go_for_it_prob"].append([ytg, d4, sd, sec, mod.go_for_it_prob(ytg, d4, sd, sec)])
        sc["field_goal_prob"].append([ytg, mod.field_goal_prob(ytg + 17)])
    for off, de in ((A, B), (B, A), (U, O), (O, U)):
        for ytg in (1.0, 3.5, 7.0, 9.0, 12.0, 25.0, 40.0, 40.5, 60.0, 61.0, 99.0):
            for down in (1, 2, 3, 4, 5):
                sc["modifiers"].append(dict(
                    off=[off.sp_rating, off.sp_offense, off.sp_defense], de=[de.sp_rating, de.sp_offense, de.sp_defense],
                    ytg=ytg, down=down, matchup_bias=mod.matchup_bias(off, de),
                    yardage_multiplier=mod.yardage_multiplier(off, de), mismatch_z=mod.mismatch_z(off, de),
                    explosive_prob=mod.explosive_prob(off, de, ytg),
                    rz_finish_prob_pass=mod.rz_finish_prob_pass(ytg, off, de, down),
                    rz_finish_prob_run=mod.rz_finish_prob_run(ytg, off, de, down)))
    json.dump(sc, open(os.path.join(HERE, "ref_scalars.json"), "w"))

    # ---- live sklearn pipelines -------------------------------------------------------------------
    n = 4000
    num = random_rows(np.random.default_rng(5), n, teams_sp)
    ms = art.compile_reference_dir(REF)
    out = dict(num=num)
    r2 = np.random.default_rng(6)
    fams = dict(pass_yards=("PY10", "PY50", "PY90"), run_yards=("RY10", "RY50", "RY90"), sack_yards=("SY10", "SY50", "SY90"))
    for fam, objs in fams.items():
        f = ms[fam]
        names = {}
        active = np.full((n, 2), -1, dtype=np.int32)
        for gi, g in enumerate(f.groups):
            pick = r2.integers(0, len(g.categories), n)
            vals = np.array(g.categories, dtype=object)[pick]
            unk = r2.random(n) < 0.5
            vals[unk] = "Unknown"
            nope = r2.random(n) < 0.1
            vals[nope] = "Nobody Atall"
            names[g.name] = vals
            active[:, gi] = [g.column_of(v) for v in vals]
        df = frame(num, passer_name="Unknown", target_name="Unknown", rusher_name="Unknown")
        for k, v in names.items():
            df[k] = v
        preds = np.stack([getattr(mod, o).predict(df) for o in objs], axis=1)
        out[f"{fam}/active"] = active
        out[f"{fam}/pred"] = preds
    np.savez_compressed(os.path.join(HERE, "sklearn_quantiles.npz"), **out)

    # ---- transformers -------------------------------------------------------------------------------
    tr = {}
    k = 64
    numk = num[:k]
    for nm, obj, cols in (("pass_stage1", mod.PASS1_META, mod.ST1_FEATURES), ("pass_stage2", mod.PASS2_PRE, mod.ST2_FEATURES)):
        f = ms.forests.get(nm)
        groups = f.groups if f is not None else art.preprocessor_groups(os.path.join(REF, "pass_stage2_preprocessor.joblib"))
        names = {}
        for g in groups:
            pick = r2.integers(0, len(g.categories), k)
            vals = np.array(g.categories, dtype=object)[pick]
            vals[::3] = "Unknown"; vals[1::7] = "Nobody Atall"
            names[g.name] = vals
        df = frame(numk, passer_name="Unknown", target_name="Unknown")
        for kk, v in names.items():
            df[kk] = v
        X = obj.transform(df[cols]).tocsr()
        tr[f"{nm}/indptr"] = X.indptr; tr[f"{nm}/indices"] = X.indices; tr[f"{nm}/data"] = X.data
        tr[f"{nm}/shape"] = np.asarray(X.shape)
        for g in groups:
            tr[f"{nm}/name/{g.name}"] = np.asarray([str(v) for v in names[g.name]])
            tr[f"{nm}/groupbase/{g.name}"] = np.asarray([g.base, len(g.categories)])
    tr["num"] = numk
    import joblib
    scaler = art.load_sklearn_object(os.path.join(REF, "scaler.pkl"))
    cols11 = [c for c in art.PLAY_FEATURES if c != "is_red_zone"]
    raw11 = pd.DataFrame(numk[:, [NUM.index(c) for c in cols11]], columns=cols11)
    tr["scaler/in"] = raw11.to_numpy()
    tr["scaler/out"] = scaler.transform(raw11)
    np.savez_compressed(os.path.join(HERE, "transformers.npz"), **tr)

    # ---- reference trajectories under injected draws ---------------------------------------------------
    pairs = [("Kansas State", "Iowa State"), ("UTSA", "Ohio State")]
    n_games = int(os.environ.get("FMC_GOLDEN_GAMES", "16"))
    from oracle.c_oracle import make_stream
    stream = make_stream(n_games, 7)
    traces = np.full((n_games, rh.MAX_ITERS, 8), np.nan)
    scores = np.zeros((n_games, 2), dtype=np.int32)     # [first team, second team]
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
                         sp_second=[cb.sp_rating, cb.sp_offense, cb.sp_defense]))
        print(f"game {g}: {a} {scores[g,0]} - {b} {scores[g,1]}  iters {iters[g]}  ({time.time()-t0:.0f}s)", flush=True)
    np.savez_compressed(os.path.join(HERE, "ref_trajectories.npz"), stream_seed=7, traces=traces, scores=scores,
                        iters=iters, plays=plays, meta=json.dumps(meta))

    # ---- provisional XGBoost vectors (SURVEY Appendix G) ----------------------------------------------------
    r0 = dict(down=3, distance=7, yardsToGoal=35, is_red_zone=0, score_diff=-3, seconds_remaining=742,
              offenseTimeouts=2, defenseTimeouts=2, sp_rating_off=12.0, sp_offense_rating_off=18.0,
              sp_defense_rating_def=10.0, sp_rating_def=7.0, goal_to_go=0, fourth_and_short=0, fg_range=0, half=2,
              two_minute=0)
    prov = dict(
        source="SURVEY.md Appendix G (survey-time probe; xgboost itself is unavailable)",
        r0=[r0[c] for c in NUM],
        stage1=[
            dict(passer="Caleb Williams", score_diff=-3, trees=188, margin=-0.1976059, p=0.4507587),
            dict(passer="Caleb Williams", score_diff=-3, trees=68, margin=-0.1526048, p=0.4619227),
            dict(passer="Unknown", score_diff=0, trees=188, margin=-0.2032859, p=0.4493528),
        ],
        play_model=[
            dict(off="Kansas State", de="Iowa State", down=1, distance=10, ytg=75, sd=0, sec=3500,
                 margins=[-9.346, 1.652, -8.433, 1.991, -4.913]),
        ],
        sklearn_r0_unknown=dict(pass_yards=[4.39653395, 14.01793596, 38.62077971],
                                run_yards=[-0.38032156, 2.99471273, 11.03926082],
                                sack_yards=[-11.2073078, -7.04441875, -2.0]),
    )
    json.dump(prov, open(os.path.join(HERE, "xgb_provisional.json"), "w"), indent=1)
    print("done in %.0fs" % (time.time() - t0))


if __name__ == "__main__":
    main()
