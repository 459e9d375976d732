"""Outputs the consumer (`edge_finder.py`) reads, computed either from the per-game score table or
directly from the joint (points A, points B) histogram the kernels accumulate.

`edge_finder.game_market_odds` / `moneyline_from_sims` (edge_finder.py:235-336) only use the joint
distribution of (pts, opp_pts) per orientation, so every statistic they print is a function of the
histogram; `scores_*.csv` can still be materialised for a literal drop-in.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import pandas as pd

HIST_BINS = 128


def _chunks(n: int, workers: int):
    """Even-aligned row ranges for the worker threads (numpy copies release the GIL)."""
    step = max(2, ((n + workers - 1) // workers + 1) & ~1)
    return [(lo, min(n, lo + step)) for lo in range(0, n, step)]


def _pool(n: int):
    import os
    from concurrent.futures import ThreadPoolExecutor
    try:
        cpus = len(os.sched_getaffinity(0))
    except AttributeError:          # pragma: no cover
        cpus = os.cpu_count() or 1
    w = max(1, min(16, cpus, n // 500_000))
    return (ThreadPoolExecutor(max_workers=w) if w > 1 else None), w


def _alternating_names(first: str, second: str, n: int, pool=None, workers: int = 1):
    """Arrow large_string array `first, second, first, ...` of length n, assembled from its buffers (no Python string
    objects: a 10 M-row column takes tens of milliseconds instead of seconds)."""
    import pyarrow as pa
    fb, sb = first.encode("utf-8"), second.encode("utf-8")
    la, lb = len(fb), len(sb)
    offsets = np.empty(n + 1, dtype=np.int64)
    total = (n // 2) * (la + lb) + (n & 1) * la
    data = np.empty(total, dtype=np.uint8)
    pair = np.frombuffer(fb + sb, dtype=np.uint8)

    def fill(lo, hi):          # lo is even
        m = hi - lo
        base = (lo // 2) * (la + lb)
        k = np.arange(0, (m + 1) // 2 + 1, dtype=np.int64) * (la + lb) + base
        offsets[lo:hi + 1:2] = k[: (m + 2) // 2]
        offsets[lo + 1:hi + 1:2] = k[: (m + 1) // 2] + la
        nb = int(offsets[hi]) - base
        full = nb // (la + lb)
        if full:
            data[base:base + full * (la + lb)].reshape(full, la + lb)[:] = pair
        if nb - full * (la + lb):
            data[base + full * (la + lb):base + nb] = pair[: nb - full * (la + lb)]

    parts = _chunks(n, workers) if n else []
    if pool is not None and len(parts) > 1:
        list(pool.map(lambda r: fill(*r), parts))
    else:
        for r in parts:
            fill(*r)
    if n == 0:
        offsets[0] = 0
    return pa.LargeStringArray.from_buffers(n, pa.py_buffer(offsets), pa.py_buffer(data))


def name_columns(team_a: str, team_b: str, n: int, first_game: int = 0):
    """The `team` / `opp` columns of `sims_frame` for games [first_game, first_game + n): they depend on the names and
    the game parity only, so `api.simulate_matchup` builds them on a worker thread WHILE the kernel runs."""
    n = int(n)
    p = int(first_game) & 1
    names = (team_a, team_b) if p == 0 else (team_b, team_a)
    dt = pd.Series(["x"]).dtype        # what `pd.DataFrame(rows)` of the reference gives its name columns
    if dt == object:
        nm = np.array(names, dtype=object)
        idx = np.arange(n) & 1
        return nm[idx], nm[1 - idx]
    pool, workers = _pool(n)
    try:
        team = pd.array(_alternating_names(names[0], names[1], n, pool, workers), dtype=dt)
        other = pd.array(_alternating_names(names[1], names[0], n, pool, workers), dtype=dt)
    finally:
        if pool is not None:
            pool.shutdown()
    return team, other


def sims_frame(team_a: str, team_b: str, scores: np.ndarray, first_game: int = 0, names=None) -> pd.DataFrame:
    """Per-game table with the reference's columns and row order (FMC:1501-1509): game g has the
    opening-kickoff receiver as `team`; even games are A-first, odd games B-first.  The two name columns have
    the dtype pandas infers for the reference's own lists of names; they are assembled from Arrow buffers and the
    point columns by strided copies, on a few threads (10 M rows: ~0.1 s instead of 2.5 s through 20 M Python
    string objects).  `names` = a `name_columns(...)` result computed ahead of time."""
    n = int(scores.shape[0])
    p = int(first_game) & 1
    pts = np.empty(n, dtype=np.int64)
    opp = np.empty(n, dtype=np.int64)
    pool, workers = _pool(n)

    def points(lo, hi):        # rows lo, lo + 2, ... (lo even) have parity p: A first when p == 0
        pts[lo:hi:2] = scores[lo:hi:2, p]; opp[lo:hi:2] = scores[lo:hi:2, 1 - p]
        pts[lo + 1:hi:2] = scores[lo + 1:hi:2, 1 - p]; opp[lo + 1:hi:2] = scores[lo + 1:hi:2, p]

    try:
        parts = _chunks(n, workers) if n else []
        if pool is not None and len(parts) > 1:
            list(pool.map(lambda r: points(*r), parts))
        else:
            for r in parts:
                points(*r)
    finally:
        if pool is not None:
            pool.shutdown()
    team, other = names if names is not None else name_columns(team_a, team_b, n, first_game)
    return pd.DataFrame({"team": team, "opp": other, "pts": pts, "opp_pts": opp}, copy=False)


def summary_frame(sims_df: pd.DataFrame) -> pd.DataFrame:
    """groupby(team) mean/sd/win_rate exactly as FMC:1681-1687 (sample std, ties are not wins).  The scores are final
    scores: without overtime a game level at 0:00 is a tie; with it (engine.OvertimeRules) only a game still level at the
    cap of periods is."""
    win = (sims_df["pts"].to_numpy() > sims_df["opp_pts"].to_numpy())
    tmp = sims_df.assign(_win=win)
    out = tmp.groupby("team").agg(
        mean_pts=("pts", "mean"), sd_pts=("pts", "std"),
        mean_opp=("opp_pts", "mean"), sd_opp=("opp_pts", "std"),
        win_rate=("_win", "mean"))
    return out


def histogram_from_scores(scores: np.ndarray, first_game: int = 0) -> np.ndarray:
    """[2, BINS, BINS] joint histogram (orientation = game parity) from a per-game (A, B) table."""
    h = np.zeros((2, HIST_BINS, HIST_BINS), dtype=np.int64)
    g = np.arange(first_game, first_game + scores.shape[0]) & 1
    a = np.minimum(scores[:, 0], HIST_BINS - 1)
    b = np.minimum(scores[:, 1], HIST_BINS - 1)
    np.add.at(h, (g, a, b), 1)
    return h


def _oriented(hist2: np.ndarray, team_is_a: bool):
    """(pts, opp_pts, weight) grids of the orientation in which `team` received the kickoff --
    the only rows edge_finder.game_market_odds keeps (edge_finder.py:301-302)."""
    o = 0 if team_is_a else 1
    w = hist2[o].astype(np.float64)
    a = np.arange(HIST_BINS)[:, None] + np.zeros((1, HIST_BINS), dtype=np.int64)
    b = np.arange(HIST_BINS)[None, :] + np.zeros((HIST_BINS, 1), dtype=np.int64)
    return (a, b, w) if team_is_a else (b, a, w)


def _weighted_median(values: np.ndarray, weights: np.ndarray) -> float:
    """np.median of the multiset (even counts average the two middle values)."""
    order = np.argsort(values, kind="stable")
    v = values[order]
    w = weights[order]
    keep = w > 0
    v, w = v[keep], w[keep]
    c = np.cumsum(w)
    n = c[-1]
    lo = v[np.searchsorted(c, (n + 1) // 2, side="left")]
    hi = v[np.searchsorted(c, n // 2 + 1, side="left")]
    return float(lo + hi) / 2.0 if n % 2 == 0 else float(lo)


def prob_to_american(p: float) -> int:
    """edge_finder._prob_to_american (edge_finder.py:70-75)."""
    p = float(np.clip(p, 1e-6, 1 - 1e-6))
    return int(round(-100 * p / (1 - p))) if p >= 0.5 else int(round(100 * (1 - p) / p))


def moneyline_from_hist(hist2: np.ndarray, team: str, opp: str) -> Dict[str, Dict]:
    """edge_finder.moneyline_from_sims (edge_finder.py:249-281) with `team` = A: p_team from the
    A-first orientation, p_opp from the B-first one (they need not sum to 1).  Ties are not wins: without overtime the
    games level at 0:00, with it only those level at the cap of periods."""
    a, b, w = _oriented(hist2, True)
    p_team = float((w * (a > b)).sum() / w.sum())
    b2, a2, w2 = _oriented(hist2, False)
    p_opp = float((w2 * (b2 > a2)).sum() / w2.sum())
    return {"team": {"name": team, "p_win": round(p_team, 6), "ml_fair": prob_to_american(p_team)},
            "opp": {"name": opp, "p_win": round(p_opp, 6), "ml_fair": prob_to_american(p_opp)}}


def game_market_odds_from_hist(hist2: np.ndarray, team: str, opp: str, *, team_is_a: bool = True,
                               spread: Optional[float] = None, total: Optional[float] = None) -> Dict[str, Dict]:
    """edge_finder.game_market_odds (edge_finder.py:283-336) from the histogram."""
    pts, opp_pts, w = _oriented(hist2, team_is_a)
    n = w.sum()
    if n <= 0:
        raise ValueError("No rows from the TEAM perspective found in scores file.")
    out: Dict[str, Dict] = {}
    if spread is not None:
        margin = (pts - opp_pts).astype(np.float64)
        tgt = -float(spread)
        p_cover = float((w * (margin > tgt)).sum() / n)
        p_not = float((w * (margin < tgt)).sum() / n)
        p_push = float((w * np.isclose(margin, tgt, atol=1e-9)).sum() / n)
        out["spread"] = {
            "team": team, "opp": opp, "spread": float(spread), "samples": int(n),
            "p_cover": round(p_cover, 6), "p_notcover": round(p_not, 6), "push_rate": round(p_push, 6),
            "american_cover": prob_to_american(p_cover), "american_notcover": prob_to_american(p_not),
            "mean_margin": float((w * margin).sum() / n),
            "median_margin": _weighted_median(margin.ravel(), w.ravel()),
        }
    if total is not None:
        totals = (pts + opp_pts).astype(np.float64)
        T = float(total)
        p_over = float((w * (totals > T)).sum() / n)
        p_under = float((w * (totals < T)).sum() / n)
        p_push = float((w * np.isclose(totals, T, atol=1e-9)).sum() / n)
        out["total"] = {
            "team": team, "opp": opp, "total": float(total), "samples": int(n),
            "p_over": round(p_over, 6), "p_under": round(p_under, 6), "push_rate": round(p_push, 6),
            "american_over": prob_to_american(p_over), "american_under": prob_to_american(p_under),
            "mean_total": float((w * totals).sum() / n),
            "median_total": _weighted_median(totals.ravel(), w.ravel()),
        }
    if not out:
        raise ValueError("Provide at least one of spread= or total=.")
    return out


def live_odds_from_hist(hist2: np.ndarray, team_a: str, team_b: str, *, spread: Optional[float] = None,
                        total: Optional[float] = None) -> Dict[str, object]:
    """Odds of games played from a live state (api.simulate_live), over BOTH orientations: unlike a game from the
    kickoff, the start state fixes who has the ball, so the game-id parity carries no meaning.  Returns games, p_win per
    team, p_tie (without overtime the games level at 0:00, as in the reference; with it, engine.OvertimeRules, only the
    games still level at the cap of periods), mean final points per team, and for `spread` (team A's line: A covers
    when its margin beats -spread) / `total` the fields of `game_market_odds_from_hist` with team A as the team.
    Scores past the last bin count as HIST_BINS - 1 points, as the histogram holds them."""
    h = np.asarray(hist2).reshape(-1, HIST_BINS, HIST_BINS).sum(axis=0).astype(np.float64)
    n = h.sum()
    if n <= 0:
        raise ValueError("the histogram holds no games")
    a = np.arange(HIST_BINS, dtype=np.float64)[:, None]
    b = np.arange(HIST_BINS, dtype=np.float64)[None, :]
    p_a = float((h * (a > b)).sum() / n)
    p_b = float((h * (b > a)).sum() / n)
    out: Dict[str, object] = {
        "games": int(n),
        "p_win": {team_a: p_a, team_b: p_b},
        "p_tie": float((h * (a == b)).sum() / n),
        "mean_points": {team_a: float((h * a).sum() / n), team_b: float((h * b).sum() / n)},
        "markets": None,
    }
    if spread is not None or total is not None:
        out["markets"] = game_market_odds_from_hist(np.stack([h, np.zeros_like(h)]), team_a, team_b, spread=spread, total=total)
    return out


OT_MAX_PERIODS = 16        # include/fmc.h FMC_OT_MAX_PERIODS


def overtime_odds_from_hist(ot_hist2: np.ndarray, team_a: str, team_b: str) -> Dict[str, object]:
    """Overtime markets of one entry from its overtime histogram ([2][OT_MAX_PERIODS + 1][3] or [OT_MAX_PERIODS + 1][3]:
    games by overtime periods played and final result A won / B won / level; both orientations are summed).  Returns
    games; p_ot, the probability of overtime; "regulation", the 3-way result at the end of regulation (A, B, level =
    p_ot) with fair American odds; "ot_win", the probability per team of winning in overtime (unconditional: the two sum
    to p_ot - p_level); "periods", P(the game ends after exactly k overtime periods) for k = 0..OT_MAX_PERIODS; and
    p_level, the probability that a game is still level when the cap of periods ends it."""
    h = np.asarray(ot_hist2, dtype=np.float64).reshape(-1, OT_MAX_PERIODS + 1, 3).sum(axis=0)
    n = h.sum()
    if n <= 0:
        raise ValueError("the overtime histogram holds no games")
    p = h / n
    p_ot = float(p[1:].sum())
    reg = {team_a: float(p[0, 0]), team_b: float(p[0, 1]), "level": float(p[0, 2]) + p_ot}
    return {
        "games": int(n),
        "p_ot": p_ot,
        "regulation": {k: {"p": v, "american": prob_to_american(v)} for k, v in reg.items()},
        "ot_win": {team_a: float(p[1:, 0].sum()), team_b: float(p[1:, 1].sum())},
        "periods": [float(x) for x in p.sum(axis=1)],
        "p_level": float(p[1:, 2].sum()),
    }


# periods of a game (include/fmc.h FMC_N_SEGMENTS), in the order of the kernels' segment histograms
SEGMENTS = ("Q1", "Q2", "Q3", "Q4", "H1", "H2")


def segment_odds_from_hist(h2: np.ndarray, team_a: str, team_b: str, *, offset=(0, 0), spread: Optional[float] = None,
                           total: Optional[float] = None) -> Dict[str, object]:
    """Odds of one period (quarter or half) from a [BINS, BINS] histogram of the (A, B) points scored in it: games,
    p_win per team, p_tie (a period can end level), mean points per team, and for `spread` (team A's line) / `total`
    the fields of `game_market_odds_from_hist` with team A as the team.  `offset` = (A, B) points already scored in the
    period (a live period in progress whose histogram counts from the live state) and is added to every bin, without
    clamping.  Points past the last bin count as HIST_BINS - 1, as the histogram holds them.  With offset (0, 0) on a
    final-score histogram this is `live_odds_from_hist`."""
    h = np.asarray(h2).reshape(HIST_BINS, HIST_BINS).astype(np.float64)
    n = h.sum()
    if n <= 0:
        raise ValueError("the histogram holds no games")
    oa, ob = int(offset[0]), int(offset[1])
    a = np.arange(HIST_BINS, dtype=np.float64)[:, None] + oa
    b = np.arange(HIST_BINS, dtype=np.float64)[None, :] + ob
    out: Dict[str, object] = {
        "games": int(n),
        "p_win": {team_a: float((h * (a > b)).sum() / n), team_b: float((h * (b > a)).sum() / n)},
        "p_tie": float((h * (a == b)).sum() / n),
        "mean_points": {team_a: float((h * a).sum() / n), team_b: float((h * b).sum() / n)},
        "markets": None,
    }
    if spread is not None or total is not None:
        # the offset moves every margin by oa - ob and every total by oa + ob: price the lines moved the other way on the
        # histogram as it is, then put the line and the margin / total statistics back where the period has them
        d, s = oa - ob, oa + ob
        mk = game_market_odds_from_hist(np.stack([h, np.zeros_like(h)]), team_a, team_b,
                                        spread=None if spread is None else float(spread) + d,
                                        total=None if total is None else float(total) - s)
        if "spread" in mk:
            mk["spread"].update(spread=float(spread), mean_margin=mk["spread"]["mean_margin"] + d,
                                median_margin=mk["spread"]["median_margin"] + d)
        if "total" in mk:
            mk["total"].update(total=float(total), mean_total=mk["total"]["mean_total"] + s,
                               median_total=mk["total"]["median_total"] + s)
        out["markets"] = mk
    return out


# scoring sequence (include/fmc.h FMC_SEQ_NONE): layout of one orientation's sequence histogram
DRIVE_RESULTS = ("td", "fg", "missed_fg", "punt", "interception", "downs", "end_of_half", "end_of_game")
RACE_TARGETS = (10, 15, 20, 25, 30)
SEQ_MINUTES = 60
SEQ_BIN_NONE = 4 * SEQ_MINUTES
SEQ_BIN_DRIVE0 = SEQ_BIN_NONE + 1
SEQ_BIN_RACE0 = SEQ_BIN_DRIVE0 + len(DRIVE_RESULTS)
SEQ_BINS = SEQ_BIN_RACE0 + 3 * len(RACE_TARGETS)
SCORE_KINDS = ("td", "fg")


def sequence_odds_from_hist(h, team_a: str, team_b: str, *, start_score=(0, 0), before=()) -> Dict[str, object]:
    """Next-score, drive-result and race-to-N odds from a scoring-sequence histogram: [SEQ_BINS] of one orientation or
    [..., SEQ_BINS] (summed over the leading axes, e.g. both orientations).  `start_score` = (A, B) points at the start
    state the histogram was played from: a race target either team had reached there is settled.  `before` = clocks C
    (multiples of 60 in 0..3600) for P(the next score is by a team and snapped with more than C seconds left).
    Returns {"games",
             "next_score": {"p": {team: {"td", "fg", "any"}}, "none", "american": {team: {...}}, "before": {C: {team: p}}},
             "drive": {"p": {result: p}, "p_scores", "american": {result: odds}},
             "race": {N: {"settled": False, "p": {team_a, team_b, "neither"}, "american": {...}} or
                         {"settled": True, "winner": team or None (both teams had reached N)}}}.
    ValueError for a histogram of another shape, negative or empty counts, drive or race bins that do not hold every
    game, or a malformed start score or clock."""
    a = np.asarray(h)
    if a.ndim < 1 or a.shape[-1] != SEQ_BINS:
        raise ValueError(f"a sequence histogram has {SEQ_BINS} bins in its last axis, got shape {a.shape}")
    if not np.issubdtype(a.dtype, np.integer) or (a < 0).any():
        raise ValueError("a sequence histogram holds non-negative integer counts")
    a = a.reshape(-1, SEQ_BINS).astype(np.int64).sum(axis=0)
    sc = tuple(start_score)
    if len(sc) != 2 or any(int(x) != x or x < 0 for x in sc):
        raise ValueError(f"start_score must be (points A, points B) >= 0, got {start_score!r}")
    nxt = a[:SEQ_BIN_NONE].reshape(2, 2, SEQ_MINUTES)              # [team][kind][minute]
    n = int(nxt.sum() + a[SEQ_BIN_NONE])
    if n <= 0:
        raise ValueError("the histogram holds no games")
    drive = a[SEQ_BIN_DRIVE0:SEQ_BIN_RACE0]
    if int(drive.sum()) != n:
        raise ValueError(f"the drive bins hold {int(drive.sum())} games, the next-score bins {n}")
    teams = (team_a, team_b)
    p_next = {teams[t]: {SCORE_KINDS[k]: float(nxt[t, k].sum() / n) for k in range(2)} for t in range(2)}
    for t in teams:
        p_next[t]["any"] = p_next[t]["td"] + p_next[t]["fg"]
    p_none = float(a[SEQ_BIN_NONE] / n)
    out_before = {}
    for c in before:
        if int(c) != c or c < 0 or c > 3600 or int(c) % 60:
            raise ValueError(f"a clock of `before` must be a multiple of 60 in 0..3600, got {c!r}")
        # snap clock > C  <=>  minute bin (clock - 1) // 60 >= C // 60
        out_before[int(c)] = {teams[t]: float(nxt[t, :, int(c) // 60:].sum() / n) for t in range(2)}
    p_drive = {r: float(drive[i] / n) for i, r in enumerate(DRIVE_RESULTS)}
    race = {}
    for i, target in enumerate(RACE_TARGETS):
        bins = a[SEQ_BIN_RACE0 + 3 * i:SEQ_BIN_RACE0 + 3 * i + 3]
        if sc[0] >= target or sc[1] >= target:
            if bins.sum():
                raise ValueError(f"race to {target} was settled at the start score {sc} but its bins hold games")
            race[target] = {"settled": True,
                            "winner": None if (sc[0] >= target and sc[1] >= target) else teams[0 if sc[0] >= target else 1]}
            continue
        if int(bins.sum()) != n:
            raise ValueError(f"the race-to-{target} bins hold {int(bins.sum())} games, the next-score bins {n}")
        p = {team_a: float(bins[0] / n), team_b: float(bins[1] / n), "neither": float(bins[2] / n)}
        race[target] = {"settled": False, "p": p, "american": {k: prob_to_american(v) for k, v in p.items()}}
    return {
        "games": n,
        "next_score": {"p": p_next, "none": p_none,
                       "american": {t: {k: prob_to_american(v) for k, v in p_next[t].items()} for t in teams},
                       "before": out_before},
        "drive": {"p": p_drive, "p_scores": p_drive["td"] + p_drive["fg"],
                  "american": {k: prob_to_american(v) for k, v in p_drive.items()}},
        "race": race,
    }


def summary_from_hist(hist2: np.ndarray, team_a: str, team_b: str) -> pd.DataFrame:
    """The `summary` frame of simulate_upcoming_matchup (FMC:1681-1687) from the histogram: each
    team's row covers the orientation in which it received the opening kickoff."""
    rows = {}
    for name, is_a in ((team_a, True), (team_b, False)):
        pts, opp_pts, w = _oriented(hist2, is_a)
        n = w.sum()
        def mean_sd(x):
            m = (w * x).sum() / n
            var = (w * (x - m) ** 2).sum() / (n - 1) if n > 1 else np.nan
            return float(m), float(np.sqrt(var))
        mp, sp_ = mean_sd(pts.astype(np.float64))
        mo, so = mean_sd(opp_pts.astype(np.float64))
        rows[name] = dict(mean_pts=mp, sd_pts=sp_, mean_opp=mo, sd_opp=so,
                          win_rate=float((w * (pts > opp_pts)).sum() / n))
    df = pd.DataFrame.from_dict(rows, orient="index")
    df.index.name = "team"
    return df.sort_index()


# ---------------------------------------------------------------------------------------------
# literal score tables at scale (SURVEY 8f row 2): the file edge_finder.py opens
# ---------------------------------------------------------------------------------------------
def write_scores_table(path: str, team_a: str, team_b: str, scores: np.ndarray, first_game: int = 0,
                       chunk_rows: int = 4_000_000) -> int:
    """Writes `scores_<base>.parquet|csv` (columns team, opp, pts, opp_pts; rows alternate A-first /
    B-first exactly like FMC:1501-1509) straight from the per-game (A, B) score array, in row-group
    chunks, with the two team-name columns dictionary-encoded -- a 10 M-game table is ~25 MB of parquet
    and never exists as a pandas object frame.  Returns the number of rows written."""
    import pyarrow as pa
    import pyarrow.parquet as pq
    n = int(scores.shape[0])
    names = pa.array([team_a, team_b], type=pa.string())
    schema = pa.schema([("team", pa.dictionary(pa.int8(), pa.string())), ("opp", pa.dictionary(pa.int8(), pa.string())),
                        ("pts", pa.int64()), ("opp_pts", pa.int64())])
    is_parquet = path.lower().endswith(".parquet")
    writer = pq.ParquetWriter(path, schema, compression="zstd") if is_parquet else None
    try:
        for lo in range(0, max(n, 1), chunk_rows):
            sc = scores[lo:lo + chunk_rows]
            g = np.arange(first_game + lo, first_game + lo + sc.shape[0])
            b_first = (g & 1).astype(np.int8)
            pts = np.where(b_first == 0, sc[:, 0], sc[:, 1]).astype(np.int64)
            opp = np.where(b_first == 0, sc[:, 1], sc[:, 0]).astype(np.int64)
            tbl = pa.table({
                "team": pa.DictionaryArray.from_arrays(pa.array(b_first), names),
                "opp": pa.DictionaryArray.from_arrays(pa.array((1 - b_first).astype(np.int8)), names),
                "pts": pa.array(pts), "opp_pts": pa.array(opp)}, schema=schema)
            if is_parquet:
                writer.write_table(tbl)
            else:
                import pyarrow.csv as pacsv
                cols = {c: (tbl[c].cast(pa.string()) if c in ("team", "opp") else tbl[c]) for c in tbl.column_names}
                plain = pa.table(cols)
                with open(path, "ab" if lo else "wb") as fh:
                    pacsv.write_csv(plain, fh, write_options=pacsv.WriteOptions(include_header=(lo == 0)))
    finally:
        if writer is not None:
            writer.close()
    return n
