"""Drop-in Python entry points of the reference (fast_monte_carlo_cfb.py:1467-1521, 1661-1722),
executed by the B200 engine.

    simulate_upcoming_matchup(teamA, teamB, *, year, week, sp_path, n, show_progress,
                              collect_players, save_csv, processes)
        -> (sims_df, players_df, summary, A, B, meta)
    simulate_matchup(teamA_ctx, teamB_ctx, n, seed, show_progress, collect_players, players_csv,
                     processes) -> (sims_df, players_df | None)

Same argument meaning, return shapes, file names (`scores_<save_csv>`, `players_<save_csv>`) and
error behaviour (ValueError for an unknown team / schema).  `n` counts PAIRS of games (A receives,
then B receives); `processes` and `show_progress` are accepted and ignored (the GPU replaces the
process pool).  Differences, all documented in DESIGN.md: a given `seed` makes the run
reproducible game by game (counter-based Philox keyed by (seed, game id)) instead of re-seeding
NumPy before every game (SURVEY Appendix E.8).

Players (SURVEY 8f row 1): when a team has usage data -- the focus sheet `2025_week1_players.csv`
(FMC:508-605) or `usage_*_share.csv` (FMC:487-505), looked up in the working directory exactly like
the reference, or passed with `focus_csv=` / `usage_dir=` -- passer, target and rusher are sampled
per play on the GPU, feed the models' one-hot columns, and the focus names get per-game box lines:
`players_df` has the reference's PLAYER_COLS rows (`flatten_player_box_rows`, FMC:1266-1299).  Without
usage data every name is "Unknown" and `players_df` is empty, as in the shipped reference.
"""
from __future__ import annotations

import os
import threading
import time
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import pandas as pd

from . import outputs
from . import usage as _usage
from .engine import Engine, GameState, MatchupSpec, OvertimeRules, overtime_rules  # noqa: F401
from .priors import (TeamContext, build_team_context_from_sp_flex, csv_base_from, load_sp_flex,
                     lookup_sp_flex, packaged_priors_path)

# FMC:1259-1264
PLAYER_COLS = [
    "sim", "start", "team", "opp", "player", "role",
    "pass_att", "pass_comp", "pass_yds", "pass_td", "INT", "sacks",
    "rush_att", "rush_yds", "rush_td",
    "rec", "tgt", "rec_yds", "rec_td",
]

_ENGINES: Dict[tuple, Engine] = {}
# The engine of a device is shared process-wide (like the reference's module-level models) and holds the matchup list
# of the call in progress: calls from several threads are serialised.
_ENGINE_LOCK = threading.RLock()
# joint score histogram [2, 128, 128] + event counters of the most recent simulate_matchup call
LAST_RUN: Dict[str, object] = {}


def get_engine(device: Optional[int] = None, **kw) -> Engine:
    """Process-wide engine per (device, options) -- the analogue of the reference's module-level
    model objects.  Raises when the CUDA library or a GPU is missing: there is no CPU path."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    key = (device,) + tuple(sorted(kw.items()))
    if key not in _ENGINES:
        _ENGINES[key] = Engine(device=device, **kw)
    return _ENGINES[key]


class _Attached:
    """A value riding in DataFrame.attrs: compared by identity, so that pandas' own attrs comparisons (concat, astype)
    never evaluate an array for truth."""
    __slots__ = ("value",)

    def __init__(self, value):
        self.value = value

    def __eq__(self, other):
        return self is other

    def __hash__(self):
        return id(self)


def _fresh_seed() -> int:
    return int.from_bytes(os.urandom(8), "little")


def simulate_matchup(teamA: TeamContext, teamB: TeamContext, n: int = 100, seed: Optional[int] = None,
                     show_progress: bool = True, collect_players: bool = False,
                     players_csv: Optional[str] = None, processes: Optional[int] = None,
                     *, engine: Optional[Engine] = None,
                     game_range: Optional[Tuple[int, int]] = None,
                     overtime=False) -> Tuple[pd.DataFrame, Optional[pd.DataFrame]]:
    """`game_range=(g0, g1)` (ours, for one process per GPU): simulate only games [g0, g1) of the 2n -- `shard_range`
    gives a rank its slice; the rows returned are those games, and the histograms of the ranks add up to the run's
    (`merge_histograms`).  A given seed gives the same games whatever the split.
    `overtime` (False, True or an engine.OvertimeRules): play games level after regulation to a result under college
    overtime rules.  The scores are then final scores, overtime included, and sims_df.attrs["overtime"] holds
    `outputs.overtime_odds_from_hist` of the games.  The default is the reference's end of the game at 0:00."""
    rules = overtime_rules(overtime)
    eng = engine if engine is not None else get_engine()
    games = 2 * int(n)
    g0, g1 = (0, games) if game_range is None else (int(game_range[0]), int(game_range[1]))
    if not (0 <= g0 <= g1 <= max(games, 0)):
        raise ValueError("game_range must lie inside [0, 2n]")
    box = None
    use = (_usage.resolve_team(teamA, eng.models), _usage.resolve_team(teamB, eng.models))
    if g1 - g0 <= 0:
        sims_df = pd.DataFrame(columns=["team", "opp", "pts", "opp_pts"])
    else:
        # the name columns of the result depend on the names and the game parity only: built while the GPU plays
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=1) as side:
            names_f = side.submit(outputs.name_columns, teamA.name, teamB.name, g1 - g0, g0)
            with _ENGINE_LOCK:
                # the sampled names feed the models whether or not the box is collected (FMC:1058-1081, 1203-1216)
                eng.set_matchups([MatchupSpec(teamA.name, teamB.name, teamA.sp, teamB.sp, games, g0, g1, 0, usage=use)])
                want_box = bool(collect_players) and eng.n_slots > 0
                ot_kw = dict(overtime=rules, want_ot_hist=True) if rules is not None else {}
                res = eng.simulate_host(_fresh_seed() if seed is None else int(seed), want_scores=True, want_hist=True,
                                        want_players=want_box, **ot_kw)
            names = names_f.result()
        box = res.get("players")
        sims_df = outputs.sims_frame(teamA.name, teamB.name, res["scores"], first_game=g0, names=names)
        sims_df.attrs["counters"] = dict(res["counters"])
        sims_df.attrs["hist"] = _Attached(res["hist"][0])
        if rules is not None:
            sims_df.attrs["overtime"] = outputs.overtime_odds_from_hist(res["ot_hist"][0], teamA.name, teamB.name)
        LAST_RUN.clear()
        LAST_RUN.update(hist=res["hist"][0], counters=dict(res["counters"]), teams=(teamA.name, teamB.name),
                        scores=res["scores"], player_box=box, usage=use, game_range=(g0, g1))
    players_df = None
    if collect_players:
        players_df = (_usage.player_rows(box, 0, (teamA.name, teamB.name), use) if box is not None
                      else pd.DataFrame(columns=PLAYER_COLS))
        if players_csv:
            if players_csv.lower().endswith(".parquet"):
                players_df.to_parquet(players_csv, index=False)
            else:
                players_df.to_csv(players_csv, index=False)
    return sims_df, players_df


def simulate_upcoming_matchup(teamA: str, teamB: str, *, year: int = 2025, week: int = 1,
                              sp_path: str = "Pregame_SPPlus2025_1.csv", n: int = 1000,
                              show_progress: bool = True, collect_players: bool = True,
                              save_csv: Optional[str] = None, processes: Optional[int] = None,
                              seed: Optional[int] = None, engine: Optional[Engine] = None,
                              focus_csv: Optional[str] = None, usage_dir: str = ".", overtime=False):
    """`overtime` as in `simulate_matchup`; with it, meta["overtime"] holds `outputs.overtime_odds_from_hist`."""
    overtime_rules(overtime)
    sp_df = load_sp_flex(sp_path)
    # FMC:605 builds the focus tables at import from `2025_week1_players.csv` in the working directory
    focus = _usage.build_focus_usage_tables(focus_csv if focus_csv is not None else _usage.FOCUS_PLAYERS_CSV)
    A = build_team_context_from_sp_flex(teamA, year, week, sp_df, focus=focus, usage_dir=usage_dir)
    B = build_team_context_from_sp_flex(teamB, year, week, sp_df, focus=focus, usage_dir=usage_dir)

    t0 = time.perf_counter()
    sims_df, players_df = simulate_matchup(A, B, n=n, seed=seed, show_progress=show_progress,
                                           collect_players=collect_players, processes=processes, engine=engine,
                                           overtime=overtime)
    t1 = time.perf_counter()
    # FMC:1681-1687.  The group-by over the 2n rows and the joint score histogram the kernel accumulated hold the same
    # information; the histogram gives the five statistics in microseconds (tests check the two agree)
    c = sims_df.attrs.get("counters")
    h = sims_df.attrs.get("hist")
    h = h.value if isinstance(h, _Attached) else None
    if h is not None and c and c.get("hist_overflow", 1) == 0 and min(int(h[0].sum()), int(h[1].sum())) > 1:
        summary = outputs.summary_from_hist(h, A.name, B.name)
    else:
        summary = outputs.summary_frame(sims_df)

    write_time = 0.0
    if save_csv:
        tw = time.perf_counter()
        try:
            if save_csv.lower().endswith(".parquet"):
                raw = sims_df.attrs.get("scores_raw")
                if raw is None:
                    raw = LAST_RUN.get("scores") if LAST_RUN.get("teams") == (A.name, B.name) else None
                if raw is not None and len(raw) == len(sims_df):   # chunked, dictionary-encoded writer straight from the score array
                    outputs.write_scores_table(f"scores_{save_csv}", A.name, B.name, raw)
                else:
                    sims_df.to_parquet(f"scores_{save_csv}", index=False)
                if players_df is not None:
                    players_df.to_parquet(f"players_{save_csv}", index=False)
            else:
                sims_df.to_csv(f"scores_{save_csv}", index=False)
                if players_df is not None:
                    players_df.to_csv(f"players_{save_csv}", index=False)
        except Exception:
            sims_df.to_csv(f"scores_{save_csv}.csv", index=False)
            if players_df is not None:
                players_df.to_csv(f"players_{save_csv}.csv", index=False)
        write_time = time.perf_counter() - tw

    sim_time = t1 - t0
    meta = {"sim_time_sec": sim_time, "io_time_sec": write_time, "total_time_sec": sim_time + write_time, "sims": n}
    c = sims_df.attrs.get("counters")
    if c:
        meta["plays"] = c["plays"]
        meta["games"] = c["games"]
    if "overtime" in sims_df.attrs:
        meta["overtime"] = sims_df.attrs["overtime"]
    return sims_df, players_df, summary, A, B, meta


# ---------------------------------------------------------------------------------------------
# slates (BASELINE configs 4 and 5): many matchups, games sharded over ranks, one histogram merge
# ---------------------------------------------------------------------------------------------
def shard_range(total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous slice of [0, total) owned by `rank`; slices tile the range exactly."""
    return (total * rank) // world, (total * (rank + 1)) // world


def slate_specs(pairs: Sequence[Tuple[str, str]], games_per_matchup: int, sp_df: pd.DataFrame,
                rank: int = 0, world: int = 1, shard: str = "games") -> List[MatchupSpec]:
    """The matchup list of one rank.  Results do not depend on `world` or `shard`: the Philox key is (seed, matchup,
    game id) and the ranks' integer histograms add up (`merge_histograms`).
      shard="games":    every rank simulates its contiguous game-id slice of every matchup (FMC:1321-1328 treats a pair
                        of games as the unit of work);
      shard="matchups": rank r simulates all games of matchups r, r + world, ... and none of the others (their ranges are
                        empty) -- a matchup's node tables and its memo entries then live on one GPU only, which keeps the
                        memo's hit rate at that of an unsharded matchup."""
    if shard not in ("games", "matchups"):
        raise ValueError("shard must be 'games' or 'matchups'")
    specs = []
    off = 0
    for i, (a, b) in enumerate(pairs):
        spa, spb = lookup_sp_flex(a, sp_df), lookup_sp_flex(b, sp_df)
        if shard == "games":
            g0, g1 = shard_range(int(games_per_matchup), rank, world)
        else:
            g0, g1 = (0, int(games_per_matchup)) if i % world == rank else (0, 0)
        specs.append(MatchupSpec(a, b, spa, spb, int(games_per_matchup), g0, g1, off))
        off += g1 - g0
    return specs


def merge_histograms(hist, counters=None):
    """The single exchange step of the multi-GPU path: all-reduce(sum) of the integer histograms
    (+ counters) over the default torch.distributed group (NCCL over NVLink on GPUs, gloo on CPU).
    `hist` / `counters` are int64 torch tensors and are reduced in place.  No-op without a group."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(hist, op=dist.ReduceOp.SUM)
        if counters is not None:
            dist.all_reduce(counters, op=dist.ReduceOp.SUM)
    return hist, counters


def _segment_buffer(n_entries: int, dev):
    """The kernels' per-period histograms [n_entries][2][N_SEGMENTS][BINS][BINS] (768 KB an entry), zeroed."""
    import torch
    return torch.zeros((n_entries, 2, len(outputs.SEGMENTS), outputs.HIST_BINS, outputs.HIST_BINS), dtype=torch.int32,
                       device=dev)


def _merge_all(counters, *hists):
    """int64 copies of the integer histograms `hists` (each may be None), merged over ranks by ONE `merge_histograms`
    all-reduce of them laid end to end.  Returns them in order, None where None was given."""
    import torch
    parts = [t for t in hists if t is not None]
    flat = torch.cat([t.reshape(-1) for t in parts]).to(torch.int64)
    merge_histograms(flat, counters)
    out, at = [], 0
    for t in hists:
        if t is None:
            out.append(None)
            continue
        out.append(flat[at:at + t.numel()].reshape(t.shape))
        at += t.numel()
    return tuple(out)


def _merge_segments(hist, seg, counters=None, seq=None):
    """int64 copies of the score histograms, the period histograms `seg` and the scoring-sequence histograms `seq` (each
    may be None), merged over ranks by ONE `merge_histograms` all-reduce of them laid end to end.  Returns (hist, seg,
    seq), None where None was given."""
    return _merge_all(counters, hist, seg, seq)


def _overtime_buffer(n_entries: int, dev):
    """The kernels' overtime histograms [n_entries][2][OT_MAX_PERIODS + 1][3] (408 B an entry), zeroed."""
    import torch
    return torch.zeros((n_entries, 2, outputs.OT_MAX_PERIODS + 1, 3), dtype=torch.int32, device=dev)


def _overtime_args(overtime, segments: bool, sequence: bool):
    """The OvertimeRules of an API call; ValueError when combined with period or sequence outputs (their definitions
    are for regulation)."""
    rules = overtime_rules(overtime)
    if rules is not None and (segments or sequence):
        raise ValueError("overtime cannot be combined with segments=True or sequence=True")
    return rules


def _sequence_buffer(n_entries: int, dev):
    """The kernels' scoring-sequence histograms [n_entries][2][SEQ_BINS] (2 KB an entry), zeroed."""
    import torch
    return torch.zeros((n_entries, 2, outputs.SEQ_BINS), dtype=torch.int32, device=dev)


def _segment_lines(mk) -> None:
    """ValueError unless every period line of a market entry ({..., "H1": {"spread": s, "total": t}}) is a mapping with
    a spread and / or a total and nothing else."""
    for name in outputs.SEGMENTS:
        if name not in (mk or {}):
            continue
        line = mk[name]
        if not isinstance(line, dict) or not line or not set(line) <= {"spread", "total"}:
            raise ValueError(f"the {name} line must be a mapping with 'spread' and / or 'total', got {line!r}")


def gather_player_box(local_rec, total_games: int):
    """The exchange step of the player path across ranks: every rank holds the per-game box of its contiguous
    game-id slice (`shard_range`), fmc_player_rec[games_local][2][n_slots]; one all-gather over the default
    torch.distributed group (NCCL for a CUDA tensor, gloo for a CPU tensor / NumPy array) returns the whole run's
    box in game order on every rank.  `local_rec` may be a NumPy structured array (native.PLAYER_REC), a
    native.PlayerBox or an int64 torch tensor [games_local, 2, n_slots, 2].  No-op without a process group.
    Memory: 32 bytes x n_slots x total_games on every rank -- meant for one matchup, not for a slate."""
    import torch
    import torch.distributed as dist
    from .native import PLAYER_REC, PlayerBox
    if isinstance(local_rec, PlayerBox):
        local_rec = local_rec.rec
    as_numpy = isinstance(local_rec, np.ndarray)
    t = torch.from_numpy(np.ascontiguousarray(local_rec).view(np.int64).reshape(local_rec.shape + (2,))) if as_numpy else local_rec
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return PlayerBox(local_rec) if as_numpy else t
    rank, world = dist.get_rank(), dist.get_world_size()
    sizes = [shard_range(int(total_games), r, world) for r in range(world)]
    assert t.shape[0] == sizes[rank][1] - sizes[rank][0], "local box does not match this rank's game slice"
    longest = max(b - a for a, b in sizes)
    pad = torch.zeros((longest,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[:t.shape[0]] = t
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad)
    whole = torch.cat([parts[r][:sizes[r][1] - sizes[r][0]] for r in range(world)], dim=0)
    if as_numpy:
        return PlayerBox(whole.cpu().numpy().view(PLAYER_REC).reshape(whole.shape[:-1]))
    return whole


def simulate_slate(pairs: Sequence[Tuple[str, str]], n: int = 1000, *, sp_path: Optional[str] = None,
                   year: int = 2025, week: int = 1, seed: Optional[int] = None,
                   engine: Optional[Engine] = None, markets: Optional[Dict[Tuple[str, str], Dict[str, float]]] = None,
                   focus_csv: Optional[str] = None, usage_dir: str = ".", segments: bool = False,
                   sequence: bool = False, overtime=False):
    """A whole slate in one launch (BASELINE configs 3-4): every (teamA, teamB) of `pairs` is simulated for
    `n` PAIRS of games (2n games, A receives / B receives alternately, exactly like `simulate_matchup`).

    Under torch.distributed (one process per GPU) every rank plays its contiguous game-id slice of every
    matchup and the integer histograms are merged with ONE all-reduce; the result does not depend on the
    number of ranks.  No per-game table is materialised: everything `edge_finder.py` derives from
    `scores_*` -- `summary` (FMC:1681-1687), moneyline (edge_finder.py:249-281) and, for pairs listed in
    `markets` ({(A, B): {"spread": s, "total": t}}), spread / total odds (edge_finder.py:283-336) -- comes
    from the joint score histogram.  Returns {(A, B): {"hist", "summary", "moneyline", "markets", "games"}},
    plus the key "_counters" with the event counters of the whole slate.

    Players: when a team of the slate has usage data (`focus_csv`, default `2025_week1_players.csv` in the working
    directory, or `usage_*_share.csv` under `usage_dir`; FMC:228-249) the slate runs in player mode and every
    matchup also returns "player_hist" ([2][n_slots][PH_BINS], merged over ranks with the same all-reduce),
    "usage" and "props": `edge_finder.scan_props_for_matchup` (edge_finder.py:340-390) for the sheet's lines,
    computed from the histograms (`usage.player_prop_odds_from_hist`).

    Periods: with `segments=True` every pair also returns "segments" = {name: {"hist", "odds"}} for each name of
    `outputs.SEGMENTS` (quarters Q1..Q4, halves H1, H2; include/fmc.h defines them): "hist" = [2][BINS][BINS] of the
    (A, B) points scored in the period per orientation (A receives first / B receives first), "odds" =
    `outputs.segment_odds_from_hist` over BOTH orientations (the opening-kickoff coin toss is part of the pregame
    uncertainty).  Period lines come through `markets` under the period's name:
    {(A, B): {"spread": s, "H1": {"spread": s1, "total": t1}, "Q1": {...}}}.  The period histograms are merged over
    ranks in the same all-reduce as the score histograms.

    Scoring sequence: with `sequence=True` every pair also returns "sequence_hist" ([2][SEQ_BINS] per orientation, A
    receives first / B receives first; include/fmc.h defines the bins), "first_score" and "race" (the next-score and
    race-to-N parts of `outputs.sequence_odds_from_hist` over BOTH orientations) and "opening_drive" = {receiving team:
    the drive part of `outputs.sequence_odds_from_hist` of the orientation in which that team receives the kickoff}.
    These histograms ride in the same all-reduce too.

    Overtime: `overtime` (False, True or an engine.OvertimeRules) plays games level after regulation to a result under
    college overtime rules; "hist", "summary", "moneyline" and "markets" then come from the final scores, overtime
    included, and every pair also returns "overtime" = `outputs.overtime_odds_from_hist` over both orientations (its
    histogram rides in the same all-reduce).  ValueError with `segments=True` or `sequence=True`.
    """
    import torch
    import torch.distributed as dist
    rules = _overtime_args(overtime, segments, sequence)
    eng = engine if engine is not None else get_engine()
    sp_df = load_sp_flex(sp_path if sp_path is not None else packaged_priors_path())
    sheet = focus_csv if focus_csv is not None else _usage.FOCUS_PLAYERS_CSV
    focus = _usage.build_focus_usage_tables(sheet)
    uses = []
    for a, b in pairs:                                    # same errors as the reference for unknown teams
        ta = build_team_context_from_sp_flex(a, year, week, sp_df, focus=focus, usage_dir=usage_dir)
        tb = build_team_context_from_sp_flex(b, year, week, sp_df, focus=focus, usage_dir=usage_dir)
        uses.append((_usage.resolve_team(ta, eng.models), _usage.resolve_team(tb, eng.models)))
    rank, world = 0, 1
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(), dist.get_world_size()
    specs = slate_specs(pairs, 2 * int(n), sp_df, rank, world)
    for sp_, u in zip(specs, uses):
        sp_.usage = u
    eng.set_matchups(specs)
    with_players = eng.ctx.has_usage and eng.n_slots > 0
    dev = torch.device("cuda", eng.ctx.device)
    if segments:
        for mk in (markets or {}).values():
            _segment_lines(mk)
    hist = torch.zeros((len(specs), 2, outputs.HIST_BINS, outputs.HIST_BINS), dtype=torch.int32, device=dev)
    counters = torch.zeros(len(native_counter_names()), dtype=torch.int64, device=dev)
    padded = torch.zeros(32, dtype=torch.int64, device=dev)
    st = torch.cuda.current_stream(dev)
    phist = (torch.zeros((len(specs), 2, eng.n_slots, _usage.PH_BINS), dtype=torch.int32, device=dev)
             if with_players else None)
    seg = _segment_buffer(len(specs), dev) if segments else None
    sq = _sequence_buffer(len(specs), dev) if sequence else None
    ot = _overtime_buffer(len(specs), dev) if rules is not None else None
    eng.ctx.simulate_device(seed=_fresh_seed() if seed is None else int(seed), hist=hist.data_ptr(),
                            counters=padded.data_ptr(), cuda_stream=st.cuda_stream,
                            player_hist=phist.data_ptr() if phist is not None else 0,
                            segment_hist=seg.data_ptr() if seg is not None else 0,
                            sequence_hist=sq.data_ptr() if sq is not None else 0,
                            overtime=rules, ot_hist=ot.data_ptr() if ot is not None else 0)
    counters.copy_(padded[:counters.numel()])
    hist64, seg64, sq64, ot64 = _merge_all(counters, hist, seg, sq, ot)
    oth = ot64.cpu().numpy() if ot64 is not None else None           # [pairs][2][OT_MAX_PERIODS + 1][3]
    ph = None
    if phist is not None:
        ph64 = phist.to(torch.int64)
        merge_histograms(ph64)
        ph = ph64.cpu().numpy()
    h = hist64.cpu().numpy()
    sgs = seg64.cpu().numpy() if seg64 is not None else None       # [pairs][2][N_SEGMENTS][BINS][BINS]
    sqs = sq64.cpu().numpy() if sq64 is not None else None          # [pairs][2][SEQ_BINS]
    c = counters.cpu().numpy()
    out: Dict[object, object] = {"_counters": {k: int(c[i]) for i, k in enumerate(native_counter_names())}}
    for m, (a, b) in enumerate(pairs):
        entry = {"hist": h[m], "games": int(h[m].sum()), "summary": outputs.summary_from_hist(h[m], a, b),
                 "moneyline": outputs.moneyline_from_hist(h[m], a, b), "markets": None}
        mk = (markets or {}).get((a, b))
        # with segments, a pair whose lines are all period lines has no final-score market
        if mk and not (segments and set(mk) <= set(outputs.SEGMENTS)):
            entry["markets"] = outputs.game_market_odds_from_hist(h[m], a, b, spread=mk.get("spread"), total=mk.get("total"))
        if sgs is not None:
            sg = sgs[m]
            entry["segments"] = {}
            for k, name in enumerate(outputs.SEGMENTS):
                both = sg[:, k].sum(axis=0)
                line = (mk or {}).get(name) or {}
                odds = (outputs.segment_odds_from_hist(both, a, b, spread=line.get("spread"), total=line.get("total"))
                        if both.sum() > 0 else None)
                entry["segments"][name] = {"hist": sg[:, k], "odds": odds}
        if sqs is not None:
            entry["sequence_hist"] = sqs[m]
            if entry["games"] > 0:
                both = outputs.sequence_odds_from_hist(sqs[m], a, b)
                entry["first_score"], entry["race"] = both["next_score"], both["race"]
                entry["opening_drive"] = {t: outputs.sequence_odds_from_hist(sqs[m][o], a, b)["drive"]
                                          for o, t in enumerate((a, b))}
            else:
                entry["first_score"] = entry["race"] = entry["opening_drive"] = None
        if oth is not None:
            entry["overtime"] = outputs.overtime_odds_from_hist(oth[m], a, b) if entry["games"] > 0 else None
        if ph is not None:
            entry["player_hist"] = ph[m]
            entry["usage"] = uses[m]
            entry["props"] = _usage.scan_props_from_hist(ph[m], (a, b), uses[m], sheet)
        out[(a, b)] = entry
    return out


# ---------------------------------------------------------------------------------------------
# live games: the rest of a game in progress, from any in-game state
# ---------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class LiveState:
    """A game in progress as `simulate_live` takes it: `offense` = the NAME of the team with the ball, `score` = (points
    of teamA, points of teamB) of the entry, `seconds` remaining in regulation, down, distance and yards to goal.
    `quarter_start_score` / `half_start_score` (optional, (A, B) like `score`): the score when the current quarter and the
    current half began; they let the odds of a period in progress cover the whole period.  A first-quarter state needs
    neither (both are 0-0), a third-quarter state only one of them (the half and the quarter began together)."""
    offense: str
    seconds: int
    down: int
    distance: float
    yards_to_goal: float
    score: Tuple[int, int] = (0, 0)
    quarter_start_score: Optional[Tuple[int, int]] = None
    half_start_score: Optional[Tuple[int, int]] = None


# (start, end) clock boundaries of every period of outputs.SEGMENTS; Q4 and H2 end with the game
SEGMENT_BOUNDS = {"Q1": (3600, 2700), "Q2": (2700, 1800), "Q3": (1800, 900), "Q4": (900, None), "H1": (3600, 1800),
                  "H2": (1800, None)}


def quarter_of(seconds: int) -> int:
    """The quarter of a clock reading, as the engine derives it: 4 - (seconds - 1) // 900, and 4 at 0."""
    return 4 - (int(seconds) - 1) // 900 if seconds > 0 else 4


def period_starts(state) -> Tuple[Optional[Tuple[int, int]], Optional[Tuple[int, int]]]:
    """(score when the current quarter began, score when the current half began) of a LiveState (or a mapping with its
    fields), each None when it is neither given nor implied (the clock implies 0-0 in the first quarter and half, and
    the current score exactly on a quarter boundary).  ValueError for contradictory values: a start score that is not
    componentwise half start <= quarter start <= score, a non-zero half start in the first half or a non-zero quarter
    start in the first quarter, quarter and half start scores that differ in the third quarter, a start score of the
    period that begins on a boundary state other than the score."""
    get = (lambda k: state.get(k)) if isinstance(state, dict) else (lambda k: getattr(state, k, None))
    sec = int(get("seconds"))
    score = tuple(int(x) for x in get("score"))
    qs, hs = get("quarter_start_score"), get("half_start_score")
    qs = None if qs is None else tuple(int(x) for x in qs)
    hs = None if hs is None else tuple(int(x) for x in hs)
    for name, v in (("quarter_start_score", qs), ("half_start_score", hs)):
        if v is not None and len(v) != 2:
            raise ValueError(f"{name} must be (points A, points B)")
    q = quarter_of(sec)
    if q <= 2:
        if hs is not None and hs != (0, 0):
            raise ValueError(f"half_start_score {hs} in the first half: the half began at 0-0")
        hs = (0, 0)
    if q == 1:
        if qs is not None and qs != (0, 0):
            raise ValueError(f"quarter_start_score {qs} in the first quarter: the quarter began at 0-0")
        qs = (0, 0)
    if q == 3:
        if qs is not None and hs is not None and qs != hs:
            raise ValueError(f"quarter_start_score {qs} and half_start_score {hs} differ in the third quarter")
        qs = hs = qs if qs is not None else hs
    if sec in (2700, 1800, 900):
        # on a boundary the quarter (and at 1800 the half) has just begun: the play that crossed it belongs to the
        # previous quarter, so the current one began at the current score
        for name, v in (("quarter_start_score", qs), ("half_start_score", hs if sec == 1800 else None)):
            if v is not None and v != score:
                raise ValueError(f"{name} {v} at {sec} s: the period began at the score {score}")
        qs = score
        if sec == 1800:
            hs = score
    le = lambda x, y: x[0] <= y[0] and x[1] <= y[1]
    if qs is not None and not le(qs, score):
        raise ValueError(f"quarter_start_score {qs} exceeds the score {score}")
    if hs is not None and not le(hs, score):
        raise ValueError(f"half_start_score {hs} exceeds the score {score}")
    if qs is not None and hs is not None and not le(hs, qs):
        raise ValueError(f"half_start_score {hs} exceeds quarter_start_score {qs}")
    return qs, hs


def live_segments(state, seg_hist: np.ndarray, team_a: str, team_b: str, lines=None) -> Dict[str, Dict[str, object]]:
    """The periods of a live entry from its [N_SEGMENTS][BINS][BINS] histograms (both orientations summed): for every name
    of outputs.SEGMENTS {"status", "offset", "hist", "odds"}.  status "ended": the period ended at or before the state;
    its histogram is empty and its odds None.  "in_progress": the histogram counts from the state; `offset` = the points
    already scored in the period (from `period_starts`), and the odds cover the whole period, or are None when the
    period's start score is unknown (offset None).  "future": the period starts after the state.  `lines`: a market entry
    with the period lines under the periods' names ({"H1": {"spread": s, "total": t}, ...})."""
    get = (lambda k: state.get(k)) if isinstance(state, dict) else (lambda k: getattr(state, k, None))
    sec = int(get("seconds"))
    score = tuple(int(x) for x in get("score"))
    qs, hs = period_starts(state)
    _segment_lines(lines)
    out: Dict[str, Dict[str, object]] = {}
    for k, name in enumerate(outputs.SEGMENTS):
        begin, end = SEGMENT_BOUNDS[name]
        h = np.asarray(seg_hist[k])
        if end is not None and sec <= end:
            out[name] = {"status": "ended", "offset": None, "hist": np.zeros_like(h), "odds": None}
            continue
        if sec > begin:
            status, offset = "future", (0, 0)
        else:
            base = (0, 0) if begin == 3600 else (hs if name in ("Q3", "H2") else qs)
            status, offset = "in_progress", None if base is None else (score[0] - base[0], score[1] - base[1])
        line = (lines or {}).get(name) or {}
        odds = (outputs.segment_odds_from_hist(h, team_a, team_b, offset=offset, spread=line.get("spread"),
                                               total=line.get("total")) if offset is not None and h.sum() > 0 else None)
        out[name] = {"status": status, "offset": offset, "hist": h, "odds": odds}
    return out


def live_game_state(team_a: str, team_b: str, state) -> GameState:
    """The engine's GameState of `state` (a LiveState, or a mapping with its fields) for the pair (team_a, team_b).
    ValueError when the team with the ball is neither team, or a field is out of range."""
    get = (lambda k: state[k]) if isinstance(state, dict) else (lambda k: getattr(state, k))
    off = get("offense")
    if off == team_a:
        o = 0
    elif off == team_b:
        o = 1
    else:
        raise ValueError(f"Team '{off}' with the ball is neither '{team_a}' nor '{team_b}'.")
    sc = tuple(get("score"))
    return GameState(offense=o, seconds=int(get("seconds")), down=int(get("down")), distance=float(get("distance")),
                     yards_to_goal=float(get("yards_to_goal")), score=(int(sc[0]), int(sc[1])))


def simulate_live(entries: Sequence[Tuple[str, str, object]], games: int = 100_000, *, sp_path: Optional[str] = None,
                  year: int = 2025, week: int = 1, seed: Optional[int] = None, engine: Optional[Engine] = None,
                  markets: Optional[Dict[int, Dict[str, float]]] = None, segments: bool = False,
                  sequence: bool = False, overtime=False) -> List[Dict[str, object]]:
    """Who wins from here?  Every entry (teamA, teamB, state) -- `state` a LiveState (or a mapping with its fields) --
    plays `games` GAMES (not pairs) from its state, all entries in one launch: a win-probability curve (one pair, a state
    per snap) and a live slate (many pairs) alike.  Entries of the same pair share one specialised table set and one memo,
    so a curve costs little more than one entry with as many games.

    Under torch.distributed every rank plays its `shard_range` slice of every entry's games and the integer histograms
    are merged with ONE all-reduce (as in `simulate_slate`); the result does not depend on the number of ranks.
    Returns a list in entry order of dicts: "state", "games", "hist" (the [128, 128] histogram of final (A, B) points,
    both orientations summed), "p_win" ({teamA: p, teamB: p}), "p_tie" (without overtime the games level at 0:00, as in
    the reference; with it only those level at the cap of periods),
    "mean_points" ({teamA: x, teamB: y}), "hist_overflow" (games in the last bin: a team with 127 or more points, which
    the odds count as 127), and "markets": for entries whose index is in `markets` ({i: {"spread": s, "total": t}},
    spread from teamA's side) the spread / total odds of `outputs.game_market_odds_from_hist`, else None.
    Teams are rated from the SP+ table at `sp_path` (default: the packaged week-1 2025 table); `year` / `week` are
    accepted as `simulate_slate` accepts them and change nothing here, since no usage data is read (every name is
    "Unknown": player props are not returned).

    Periods: with `segments=True` every entry also returns "segments" = `live_segments(...)`: per period of
    `outputs.SEGMENTS` its status (ended / in_progress / future), the histogram of the points scored in it from the
    state on (both orientations summed) and its odds, with the period lines of `markets` under the period's name
    ({i: {"spread": s, "H2": {"spread": s2, "total": t2}}}).  A period in progress is priced as a whole when its start
    score is known (LiveState.quarter_start_score / half_start_score, or implied by the clock).

    Scoring sequence: with `sequence=True` every entry also returns "sequence_hist" ([SEQ_BINS], both orientations
    summed) and, from `outputs.sequence_odds_from_hist` with the state's score as the start score, "next_score" (which
    team scores next and how, or no further score), "drive" (how the drive in progress ends) and "race" (first to
    10 / 15 / 20 / 25 / 30, targets already reached reported as settled).

    Overtime: `overtime` (False, True or an engine.OvertimeRules) plays games level after regulation to a result under
    college overtime rules, also from a state at 0:00 with the score level; "hist", "p_win", "p_tie", "mean_points" and
    "markets" then come from the final scores, and every entry also returns "overtime" =
    `outputs.overtime_odds_from_hist` (P(overtime), the 3-way result at the end of regulation, P(win in overtime) per
    team, the distribution of overtime periods).  ValueError with `segments=True` or `sequence=True`."""
    import torch
    import torch.distributed as dist
    rules = _overtime_args(overtime, segments, sequence)
    eng = engine if engine is not None else get_engine()
    sp_df = load_sp_flex(sp_path if sp_path is not None else packaged_priors_path())
    entries = list(entries)
    if not entries:
        raise ValueError("simulate_live needs at least one entry")
    if int(games) < 1:
        raise ValueError("games must be at least 1")
    starts = []
    sps = []
    for m, (a, b, st) in enumerate(entries):  # same errors as the reference for unknown teams
        sps.append((lookup_sp_flex(a, sp_df), lookup_sp_flex(b, sp_df)))
        starts.append(live_game_state(a, b, st))
        period_starts(st)
        if segments:
            _segment_lines((markets or {}).get(m))
    rank, world = 0, 1
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(), dist.get_world_size()
    g0, g1 = shard_range(int(games), rank, world)
    specs = [MatchupSpec(a, b, spa, spb, int(games), g0, g1, i * (g1 - g0), start=gs)
             for i, ((a, b, _), (spa, spb), gs) in enumerate(zip(entries, sps, starts))]
    dev = torch.device("cuda", eng.ctx.device)
    hist = torch.zeros((len(specs), 2, outputs.HIST_BINS, outputs.HIST_BINS), dtype=torch.int32, device=dev)
    seg = _segment_buffer(len(specs), dev) if segments else None
    sq = _sequence_buffer(len(specs), dev) if sequence else None
    ot = _overtime_buffer(len(specs), dev) if rules is not None else None
    with _ENGINE_LOCK:
        eng.set_matchups(specs)
        if g1 > g0:
            st = torch.cuda.current_stream(dev)
            eng.ctx.simulate_device(seed=_fresh_seed() if seed is None else int(seed), hist=hist.data_ptr(),
                                    cuda_stream=st.cuda_stream, segment_hist=seg.data_ptr() if seg is not None else 0,
                                    sequence_hist=sq.data_ptr() if sq is not None else 0,
                                    overtime=rules, ot_hist=ot.data_ptr() if ot is not None else 0)
    hist64, seg64, sq64, ot64 = _merge_all(None, hist, seg, sq, ot)
    oth = ot64.cpu().numpy() if ot64 is not None else None
    h = hist64.cpu().numpy()
    sg = seg64.sum(dim=1).cpu().numpy() if seg64 is not None else None      # [entries][N_SEGMENTS][BINS][BINS]
    sqh = sq64.sum(dim=1).cpu().numpy() if sq64 is not None else None       # [entries][SEQ_BINS]
    out = []
    for m, (a, b, st) in enumerate(entries):
        h2 = h[m].sum(axis=0)
        mk = (markets or {}).get(m) or {}
        odds = outputs.live_odds_from_hist(h2, a, b, spread=mk.get("spread"), total=mk.get("total"))
        last = outputs.HIST_BINS - 1
        out.append({"state": st, "games": odds["games"], "hist": h2, "p_win": odds["p_win"], "p_tie": odds["p_tie"],
                    "mean_points": odds["mean_points"],
                    "hist_overflow": int(h2[last, :].sum() + h2[:last, last].sum()), "markets": odds["markets"]})
        if sg is not None:
            out[-1]["segments"] = live_segments(st, sg[m], a, b, mk)
        if sqh is not None:
            seq = outputs.sequence_odds_from_hist(sqh[m], a, b, start_score=tuple(starts[m].score))
            out[-1].update(sequence_hist=sqh[m], next_score=seq["next_score"], drive=seq["drive"], race=seq["race"])
        if oth is not None:
            out[-1]["overtime"] = outputs.overtime_odds_from_hist(oth[m], a, b)
    return out


def native_counter_names():
    from .native import COUNTER_NAMES
    return COUNTER_NAMES
