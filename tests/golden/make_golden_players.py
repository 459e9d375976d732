"""Golden fixtures for the per-player path (SURVEY 8a row a16 / 8f row 1), from the UNMODIFIED reference.

Needs the original project (FMC_REFERENCE_DIR=<its directory>):   python tests/golden/make_golden_players.py

The shipped reference has no usage data (every name is "Unknown", nothing is tracked, FMC:246-249), so
the fixture gives the reference module a synthetic focus sheet (`players_focus.csv`, the format of
`2025_week1_players.csv`, FMC:511-602) whose names exercise every case: names that the models split
on, names outside every OneHotEncoder category list, percentage usages, duplicate rows, a NaN usage,
a remainder that becomes `__Other__`, a total above 1 that is renormalised, and a team without any
focus rows.  Then it drives the reference's own `simulate_game` with injected draw streams
(oracle/ref_harness.py) and stores

  players_focus.csv        the synthetic sheet
  usage_*_share.csv        synthetic fallback usage files (committed; written once by hand)
  ref_players.npz          per team the reference's share tables + track sets
                           (`_build_focus_usage_tables` / `_usage_from_focus_or_fallback`), per game the
                           per-iteration states, final scores and `flatten_player_box_rows` (FMC:1266-1299)
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

from oracle import ref_harness as rh                  # noqa: E402
from streams import adversarial_stream                # noqa: E402
from oracle.c_oracle import make_stream               # noqa: E402

SHEET = """team,player,pos,usage,stat,yards
Kansas State,Taylen Green,QB,70,pass_yards,245.5
Kansas State,Zach Gibson,QB,20,pass_yards,40.5
Kansas State,Blake Watson,RB,0.45,rush_yards,71.5
Kansas State,Anthony Grant,RB,0.30,rush_yards,44.5
Kansas State,Taylen Green,QB,0.05,rush_yards,18.5
Kansas State,Benjamin Brahmer,TE,0.3,rec_yards,51.5
Kansas State,Braelon Allen,WR,0.2,rec_yards,38.5
Kansas State,Nobody Known,WR,0.1,rec_yards,20.5
Iowa State,Levi Williams,QB,1.0,pass_yards,212.5
Iowa State,Bo Nix,RB,0.5,rush_yards,60.5
Iowa State,Bo Nix,RB,0.2,rush_yards,60.5
Iowa State,Brady Cook,RB,0.5,rush_yards,33.5
Iowa State,Carson Hansen,WR,0.4,rec_yards,55.5
Iowa State,Cam Barfield,WR,0.35,rec_yards,47.5
Iowa State,Avery Morrow,WR,,rec_yards,12.5
Iowa State,Zed Unknown,WR,0.25,rec_yards,30.5
"""

# Ohio State has no focus rows: its usage comes from the fallback files usage_{qb,rush,target}_share.csv in this
# directory (FMC:243-245, 487-505): 21 rushers (one with a negative share), 12 targets, nothing tracked
PAIRS = [("Kansas State", "Iowa State"), ("UTSA", "Iowa State"), ("Ohio State", "Kansas State")]
PLAYER_COLS = ["sim", "start", "team", "opp", "player", "role", "pass_att", "pass_comp", "pass_yds", "pass_td", "INT",
               "sacks", "rush_att", "rush_yds", "rush_td", "rec", "tgt", "rec_yds", "rec_td"]


def main():
    t0 = time.time()
    mod = rh.load_reference()
    sheet_path = os.path.join(HERE, "players_focus.csv")
    with open(sheet_path, "w") as f:
        f.write(SHEET)
    mod._FOCUS_USAGE = mod._build_focus_usage_tables(sheet_path)      # FMC:605 does this at import from the cwd
    assert mod.OTHER_SENTINEL == "__Other__"

    os.chdir(HERE)      # `_load_usage_table` reads the fallback files relative to the working directory
    teams = {}
    for name in sorted({t for p in PAIRS for t in p}):
        tc = rh.team_context(mod, name)
        teams[name] = dict(
            qb=[list(map(str, tc.qb_share["passer_name"])), [float(x) for x in tc.qb_share["share"].values]],
            ru=[list(map(str, tc.rush_share["rusher_name"])), [float(x) for x in tc.rush_share["share"].values]],
            tg=[list(map(str, tc.target_share["receiver_name"])), [float(x) for x in tc.target_share["share"].values]],
            track_pass=sorted(tc.track_pass or []), track_rush=sorted(tc.track_rush or []),
            track_rec=sorted(tc.track_rec or []),
            sp=[tc.sp_rating, tc.sp_offense, tc.sp_defense])

    n_games = int(os.environ.get("FMC_GOLDEN_GAMES", "12"))
    stream = make_stream(n_games, 11)
    traces = np.full((n_games, rh.MAX_ITERS, 8), np.nan)
    scores = np.zeros((n_games, 2), dtype=np.int32)
    iters = np.zeros(n_games, dtype=np.int32)
    meta, rows = [], []
    for g in range(n_games):
        a, b = PAIRS[(g // 2) % len(PAIRS)]
        first, second = (b, a) if (g & 1) else (a, b)
        ca, cb = rh.team_context(mod, first), rh.team_context(mod, second)
        res, trc, used = rh.run_game_injected(mod, ca, cb, stream[g])
        traces[g, :trc.shape[0]] = trc
        scores[g] = (res["off_score"], res["def_score"])
        iters[g] = trc.shape[0]
        meta.append(dict(team_a=a, team_b=b, first=first, second=second))
        for r in mod.flatten_player_box_rows(res, sim_id=g, start_flag="B" if (g & 1) else "A"):
            rows.append([r[c] for c in PLAYER_COLS])
        print(f"game {g}: {first} {scores[g,0]} - {second} {scores[g,1]}  iters {iters[g]}  "
              f"player rows so far {len(rows)}  ({time.time()-t0:.0f}s)", flush=True)
    # ---- the same under ADVERSARIAL draws (tests/streams.py): u = 0 picks the first entry with a positive share
    # (zero-share entries are skipped by searchsorted(..., 'right')), u just below 1 the last one, and so on
    n_adv = int(os.environ.get("FMC_GOLDEN_ADV_GAMES", "12"))
    adv = adversarial_stream(n_adv, 77)
    a_traces = np.full((n_adv, rh.MAX_ITERS, 8), np.nan)
    a_scores = np.zeros((n_adv, 2), dtype=np.int32)
    a_iters = np.zeros(n_adv, dtype=np.int32)
    a_meta, a_rows = [], []
    for g in range(n_adv):
        a, b = PAIRS[(g // 2) % len(PAIRS)]
        first, second = (b, a) if (g & 1) else (a, b)
        ca, cb = rh.team_context(mod, first), rh.team_context(mod, second)
        res, trc, used = rh.run_game_injected(mod, ca, cb, adv[g])
        a_traces[g, :trc.shape[0]] = trc
        a_scores[g] = (res["off_score"], res["def_score"])
        a_iters[g] = trc.shape[0]
        a_meta.append(dict(team_a=a, team_b=b, first=first, second=second, pattern=g % 6))
        for r in mod.flatten_player_box_rows(res, sim_id=g, start_flag="B" if (g & 1) else "A"):
            a_rows.append([r[c] for c in PLAYER_COLS])
        print(f"adversarial game {g} pattern {g % 6}: {first} {a_scores[g,0]} - {second} {a_scores[g,1]}  iters {a_iters[g]}  "
              f"player rows so far {len(a_rows)}  ({time.time()-t0:.0f}s)", flush=True)
    np.savez_compressed(os.path.join(HERE, "ref_players.npz"), stream_seed=11, traces=traces, scores=scores, iters=iters,
                        meta=json.dumps(meta), teams=json.dumps(teams), player_cols=json.dumps(PLAYER_COLS),
                        player_rows=json.dumps(rows), adv_stream_seed=77, adv_traces=a_traces, adv_scores=a_scores,
                        adv_iters=a_iters, adv_meta=json.dumps(a_meta), adv_player_rows=json.dumps(a_rows))
    print("done in %.0fs" % (time.time() - t0))


if __name__ == "__main__":
    main()
