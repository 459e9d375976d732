"""Every simulation-kernel instantiation, every memo schedule and any split of the game range on the B200.

`launch_sim` picks one of 30 kernels: sim_kernel<TEST, PLAYERS, HOOKS, OT> (plain and player mode) and
sim_memo_kernel<TEST, HOOKS, OT>, each with TEST on or off and with no optional outputs, period outputs, sequence
outputs, both, or overtime.  This file runs all of them against the oracles game by game (1), shows that no memo
schedule changes a result (2), that launches over a split game range (odd bounds, out_offsets out of entry order, empty
slices) add up to the launch over the whole range (3), and checks the edges of the overtime rules (4).  Every engine is
built here with an explicit memo mode, so nothing depends on FMC_MEMO."""
import hashlib
import itertools
import os
from dataclasses import dataclass
from typing import Optional

import numpy as np
import pytest

from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import outputs, priors, usage
from fast_monte_carlo_b200.engine import Engine, GameState, MatchupSpec, OvertimeRules
from fast_monte_carlo_b200.native import FmcError
from test_gpu_overtime import hist_from_rows as ot_hist_from_rows
from test_gpu_players import _box_equal_philox
from test_gpu_segments import GAME_COUNTERS, host_segment_hist, oracle_period_words, segments_from_rows
from test_gpu_sequence import hist_from_rows as seq_hist_from_rows

pytestmark = pytest.mark.gpu

SEED = 20261022
N_TEST = 1024                    # games per entry under injected draws (46 KB of stream a game)
N_PHILOX = 10_000                # games per entry under Philox draws
ORACLE_COUNTERS = ("plays", "iters", "pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg", "punt", "go")
ALL_GAME_COUNTERS = GAME_COUNTERS + ("ot_games", "ot_periods")
RULES = OvertimeRules()
LAST = outputs.HIST_BINS - 1

# One launch carries three entries of one pair: the kickoff, 3rd & 4 in the third quarter, and level at 0:20, so that
# quarter and half boundaries, the end of the game and overtime all happen.
ENTRIES = (GameState(),
           GameState(offense=0, seconds=1361, down=3, distance=4.0, yards_to_goal=48.0, score=(10, 14)),
           GameState(offense=1, seconds=20, down=1, distance=10.0, yards_to_goal=65.0, score=(17, 17)))

KERNELS = ("plain", "memo", "players")
OUTPUTS = {
    "none": {},
    "periods": dict(want_period_scores=True, want_segments=True),
    "sequence": dict(want_sequence=True, want_sequence_hist=True),
    "both": dict(want_period_scores=True, want_segments=True, want_sequence=True, want_sequence_hist=True),
    "overtime": dict(overtime=RULES, want_ot_periods=True, want_ot_hist=True),
}
HAS_PERIODS = ("periods", "both")
HAS_SEQUENCE = ("sequence", "both")
CASES = list(itertools.product(KERNELS, (False, True), OUTPUTS))


def _case_id(kernel, test, outs):
    return f"{kernel}-{'test' if test else 'philox'}-{outs}"


@dataclass(frozen=True)
class Pair:
    team_a: str
    team_b: str
    sp_a: tuple
    sp_b: tuple
    usage: Optional[tuple] = None

    @property
    def n_slots(self) -> int:
        return 0 if self.usage is None else max(len(tu.slots) for tu in self.usage)

    def spec(self, start, games, g0, g1, out_offset):
        return MatchupSpec(self.team_a, self.team_b, self.sp_a, self.sp_b, games, g0, g1, out_offset, usage=self.usage,
                           start=start)


def _entries(pair, n, starts=ENTRIES):
    """One entry per start state, games [0, n) each, out_offsets in reverse entry order."""
    k = len(starts)
    return [pair.spec(s, n, 0, n, (k - 1 - i) * n) for i, s in enumerate(starts)]


def _rows(i, n, k=len(ENTRIES)):
    """The rows of entry i of _entries."""
    return slice((k - 1 - i) * n, (k - i) * n)


def _nan_equal(a, b):
    return bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


def _digest(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


# ---- fixtures ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def live(models_s2):
    import oracle_live
    oracle_live.load_models(models_s2)
    return oracle_live


@pytest.fixture(scope="module")
def seqo(models_s2):
    import oracle_sequence
    oracle_sequence.load_models(models_s2)
    return oracle_sequence


@pytest.fixture(scope="module")
def oto(models_s2):
    import oracle_overtime
    oracle_overtime.load_models(models_s2)
    return oracle_overtime


@pytest.fixture(scope="module")
def pairs(models_s2):
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ctx = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    use = tuple(usage.resolve_team(tc, models_s2) for tc in ctx)
    assert use[0].slots and use[1].slots
    plain = Pair("A", "B", KSU, ISU)
    return {"plain": plain, "memo": plain, "players": Pair("Kansas State", "Iowa State", ctx[0].sp, ctx[1].sp, use)}


@pytest.fixture(scope="module")
def engines(models_s2, native_lib):
    es = {"plain": Engine(models_s2, device=0, stage2="standin", memo="off"),
          "memo": Engine(models_s2, device=0, stage2="standin", memo="on"),
          "players": Engine(models_s2, device=0, stage2="standin", memo="on")}
    yield es
    for e in es.values():
        e.close()


@pytest.fixture(scope="module")
def stream(oracle):
    return oracle.make_stream(len(ENTRIES) * N_TEST, 77)


def _entry_stream(stream, i, n=N_TEST):
    return stream[_rows(i, n)]


def _entry_oracle(oracle, models_s2, mods, pair, start, m, n, stream=None, rules=None):
    """The oracle's games [0, n) of entry m from `start`: scores, iters, counters, the player box; without overtime the
    period words (from the oracle's traces) and the sequence rows and races; with it the overtime periods.  Traces are
    kept under injected draws only; Philox games are run in chunks so that their traces are never all in memory."""
    live, seqo, oto = mods
    cfg = oracle.make_config(models_s2, pair.sp_a, pair.sp_b)
    use = {} if pair.usage is None else dict(usage=oracle.make_usage(pair.usage), n_slots=pair.n_slots)
    chunk = n if stream is not None else 2500
    parts = []
    for lo in range(0, n, chunk):
        k = min(chunk, n - lo)
        kw = dict(start=start, game0=lo, matchup=m, seed=SEED, **use)
        if stream is not None:
            kw["stream"] = stream[lo:lo + k]
        if rules is not None:
            r = oto.simulate(cfg, k, max_periods=rules.max_periods, snap_clock=rules.snap_clock, trace=stream is not None,
                             **kw)
        else:
            r = live.simulate(cfg, k, trace=True, **kw)
            r["words"] = oracle_period_words(r["trace"], r["iters"], r["scores"], np.arange(lo, lo + k), start.seconds)
            kw.pop("n_slots", None)
            s = seqo.simulate(cfg, k, **kw)
            assert np.array_equal(s["scores"], r["scores"])
            r["sequence"], r["race"] = s["sequence"], s["race"]
            if stream is None:
                r["trace"] = None
        parts.append(r)
    out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0] if k != "counters" and parts[0][k] is not None}
    out["counters"] = {k: sum(p["counters"][k] for p in parts) for k in ORACLE_COUNTERS}
    return out


@pytest.fixture(scope="module")
def refs(oracle, models_s2, live, seqo, oto, pairs, stream):
    """The oracle's games of the three entries, once per (players, draws, rules): they do not depend on the kernel."""
    cache = {}

    def get(kernel, test, ot):
        pair = pairs[kernel]
        key = (pair.usage is not None, test, ot)
        if key not in cache:
            n = N_TEST if test else N_PHILOX
            cache[key] = [_entry_oracle(oracle, models_s2, (live, seqo, oto), pair, s, i, n,
                                        _entry_stream(stream, i) if test else None, RULES if ot else None)
                          for i, s in enumerate(ENTRIES)]
        return cache[key]
    return get


def _launch(e, pair, test, outs, stream):
    """The entries of the matrix on engine `e` with one output set, under injected draws (and traces) when `test`."""
    e.set_matchups(_entries(pair, N_TEST if test else N_PHILOX))
    kw = dict(OUTPUTS[outs], want_iters=True)
    if test:
        kw.update(stream=stream, want_trace=True)
    if pair.usage is not None:
        kw.update(want_players=True, want_player_hist=True)
    return e.simulate_host(SEED, **kw)


def _kept(got):
    """What a later test compares a launch with: everything, the traces as a digest of their bits."""
    out = {k: v for k, v in got.items() if k not in ("trace", "players")}
    if "trace" in got:
        out["trace"] = _digest(got["trace"])
    if "players" in got:
        out["players"] = _digest(got["players"].rec)
    return out


@pytest.fixture(scope="module")
def runs(engines, pairs, stream):
    """Launches shared between tests: (kernel, test, outputs) -> _kept of the launch on the matrix engines."""
    cache = {}

    def get(kernel, test, outs):
        key = (kernel, test, outs)
        if key not in cache:
            cache[key] = _kept(_launch(engines[kernel], pairs[kernel], test, outs, stream))
        return cache[key]
    return get


def _assert_same(got, want):
    """Every output of two launches equal bit for bit (`want` as _kept keeps it), and every game counter."""
    got = _kept(got)
    assert set(got) == set(want)
    for k, v in want.items():
        if k == "counters":
            assert {c: got[k][c] for c in ALL_GAME_COUNTERS} == {c: v[c] for c in ALL_GAME_COUNTERS}
        elif isinstance(v, str):
            assert got[k] == v, k
        else:
            assert got[k].dtype == v.dtype and np.array_equal(got[k], v), k


# ---- 1. the instantiation matrix against the oracles ------------------------------------------------------------------
@pytest.mark.parametrize("kernel,test,outs", CASES, ids=[_case_id(*c) for c in CASES])
def test_instantiation_against_the_oracles(engines, pairs, refs, runs, stream, kernel, test, outs):
    e, pair = engines[kernel], pairs[kernel]
    ot = outs == "overtime"
    ref = refs(kernel, test, ot)
    n = N_TEST if test else N_PHILOX
    got = _launch(e, pair, test, outs, stream)
    c = got["counters"]
    # which kernel ran: only sim_memo_kernel counts trips; a box only in player mode; traces only under TEST
    assert (c["trips"] > 0) == (kernel == "memo")
    assert e.ctx.has_usage == (kernel == "players")
    if kernel == "players":
        assert got["players"].dense()[..., 1].sum() > 0
    if test:
        assert (got["iters"] > 0).all() and not np.isnan(got["trace"][:, 0, 2]).any()
    else:
        assert "trace" not in got
    games = np.arange(n)
    for i, (s, r) in enumerate(zip(ENTRIES, ref)):
        rows = _rows(i, n)
        assert np.array_equal(got["scores"][rows], r["scores"]), i
        assert np.array_equal(got["iters"][rows], r["iters"]), i
        assert np.array_equal(got["hist"][i].astype(np.int64), outputs.histogram_from_scores(r["scores"])), i
        if test:
            assert _nan_equal(got["trace"][rows], r["trace"]), i
        if outs in HAS_PERIODS:
            assert np.array_equal(got["period_scores"][rows], r["words"]), i
            pts, counted = segments_from_rows(r["words"], r["scores"], s.seconds, s.score)
            assert np.array_equal(got["segment_hist"][i].astype(np.int64), host_segment_hist(pts, counted, games)), i
        if outs in HAS_SEQUENCE:
            assert np.array_equal(got["sequence"][rows], r["sequence"]), i
            assert np.array_equal(got["sequence_hist"][i].astype(np.int64),
                                  seq_hist_from_rows(r["sequence"], r["race"], games)), i
        if ot:
            assert np.array_equal(got["ot_periods"][rows].astype(np.int64), r["periods"]), i
            assert np.array_equal(got["ot_hist"][i].astype(np.int64), ot_hist_from_rows(r["scores"], r["periods"], games)), i
        if kernel == "players":
            box = got["players"].dense()[rows]
            if test:
                assert np.array_equal(box, r["players"]), i          # float64 yards bit for bit
            else:
                _box_equal_philox(box, r["players"])
            assert np.array_equal(got["player_hist"][i], usage.player_hist_from_box(box, pair.usage)), i
    assert {k: c[k] for k in ORACLE_COUNTERS} == {k: sum(r["counters"][k] for r in ref) for k in ORACLE_COUNTERS}
    assert c["games"] == len(ENTRIES) * n
    assert c["hist_overflow"] == sum(int((r["scores"] > LAST).any(axis=1).sum()) for r in ref)
    if ot:
        assert c["ot_games"] == sum(int((r["periods"] > 0).sum()) for r in ref) > 0
        assert c["ot_periods"] == sum(int(r["periods"].sum()) for r in ref)
        assert (got["ot_periods"][_rows(2, n)] > 0).sum() > n // 10        # the level entry plays overtime
    else:
        assert c["ot_games"] == c["ot_periods"] == 0
    # the optional outputs move nothing else: the launch without them, same kernel and draws
    if outs != "none":
        base = runs(kernel, test, "none")
        if ot:
            d = base["scores"][:, 0] != base["scores"][:, 1]
            assert np.array_equal(got["scores"][d], base["scores"][d]) and np.array_equal(got["iters"][d], base["iters"][d])
            assert (got["ot_periods"][~d] > 0).all() and (got["ot_periods"][d] == 0).all()
        else:
            for k in ("scores", "hist", "iters"):
                assert np.array_equal(got[k], base[k]), k


# ---- 2. results do not depend on the memo schedule --------------------------------------------------------------------
# name -> (max_trips, break_parked, FMC_MEMO_BREAK_WAITING or None = the library's default, memo_bytes); 0 = default
SCHEDULES = {
    "trips1-parked1": (1, 1, None, 0),
    "trips1-parked32-waiting1": (1, 32, 1, 0),
    "trips2-parked32-waiting1e6": (2, 32, 10 ** 6, 0),
    "trips4096-parked32-waiting1e6": (4096, 32, 10 ** 6, 0),
    "trips4096-parked1-waiting1": (4096, 1, 1, 0),
    "table1MiB": (0, 0, None, 1 << 20),
}


def _memo_engine(models_s2, max_trips=0, break_parked=0, waiting=None, memo_bytes=0, mode="on"):
    """A fresh engine with the memo schedule set explicitly.  The library reads FMC_MEMO_BREAK_WAITING when the schedule is
    set and keeps it in the context: the variable is set only while the engine is made, and the engine is never given
    another schedule."""
    with pytest.MonkeyPatch.context() as mp:
        if waiting is None:
            mp.delenv("FMC_MEMO_BREAK_WAITING", raising=False)
        else:
            mp.setenv("FMC_MEMO_BREAK_WAITING", str(waiting))
        e = Engine(models_s2, device=0, stage2="standin", memo=mode, memo_bytes=memo_bytes)
        e.ctx.set_memo(mode, max_bytes=memo_bytes, max_trips=max_trips, break_parked=break_parked)
    return e


@pytest.fixture(scope="module", params=list(SCHEDULES))
def schedule(request, models_s2, native_lib):
    e = _memo_engine(models_s2, *SCHEDULES[request.param])
    yield request.param, e
    e.close()


@pytest.fixture(scope="module")
def default_schedule(models_s2, native_lib, pairs, stream):
    """Counters of the memo kernel under the default schedule, per (test, outputs)."""
    e = _memo_engine(models_s2)
    cache = {}

    def get(test, outs):
        if (test, outs) not in cache:
            cache[(test, outs)] = _launch(e, pairs["memo"], test, outs, stream)["counters"]
        return cache[(test, outs)]
    yield get
    e.close()


@pytest.mark.parametrize("outs", list(OUTPUTS))
@pytest.mark.parametrize("test", [False, True], ids=["philox", "test"])
def test_results_do_not_depend_on_the_memo_schedule(schedule, default_schedule, runs, pairs, stream, test, outs):
    name, e = schedule
    got = _launch(e, pairs["memo"], test, outs, stream)
    _assert_same(got, runs("plain", test, outs))
    c, d = got["counters"], default_schedule(test, outs)
    assert c["trips"] > 0 and d["trips"] > 0
    # the schedule did change: otherwise the case proves nothing
    assert (c["rounds"], c["trips"]) != (d["rounds"], d["trips"])
    if SCHEDULES[name][3]:
        assert c["memo_hits"] < d["memo_hits"]


def test_persistent_memo_across_instantiations(models_s2, native_lib, engines, pairs, stream):
    """One warm table through launches of different instantiations on the same entries: each equals memo off, and from
    the second launch on it hits more than a cold table.  A memo key that is not complete for a state only one
    instantiation reaches (the overtime snap clock, a two-point try) would hand another launch a wrong result."""
    warm = _memo_engine(models_s2, mode="persistent")
    try:
        pair = pairs["memo"]
        launches = [(False, {}), (False, dict(overtime=RULES, want_ot_periods=True, want_ot_hist=True)),
                    (False, OUTPUTS["both"]),
                    (False, dict(overtime=OvertimeRules(snap_clock=1), want_ot_periods=True, want_ot_hist=True)),
                    (True, dict(overtime=RULES, want_ot_periods=True, want_ot_hist=True))]
        for e in (warm, engines["memo"], engines["plain"]):
            e.set_matchups(_entries(pair, N_TEST))
        for j, (test, kw) in enumerate(launches):
            if test:
                kw = dict(kw, stream=stream, want_trace=True)
            w, cold, off = (e.simulate_host(SEED, want_iters=True, **kw) for e in (warm, engines["memo"], engines["plain"]))
            _assert_same(w, _kept(off))
            _assert_same(cold, _kept(off))
            assert cold["counters"]["memo_hits"] > 0, j
            if j:
                assert w["counters"]["memo_hits"] > cold["counters"]["memo_hits"], j
    finally:
        warm.close()


@pytest.mark.parametrize("knob", [dict(max_trips=4097), dict(max_trips=-1), dict(break_parked=33), dict(break_parked=-1)],
                         ids=["max_trips=4097", "max_trips=-1", "break_parked=33", "break_parked=-1"])
def test_set_memo_rejects_bad_schedules(engines, knob):
    with pytest.raises(FmcError, match="scheduling knob"):
        engines["memo"].ctx.set_memo("on", **knob)


# ---- 3. splits of the game range ----------------------------------------------------------------------------------------
N_SPLIT = 30_001
BOUNDS = (0, 7_777, 19_001, N_SPLIT)
ROW_KEYS = ("scores", "iters", "period_scores", "sequence", "ot_periods")
HIST_KEYS = ("hist", "segment_hist", "sequence_hist", "ot_hist", "player_hist")


def _split_specs(pair, k):
    """Launch k of three over [BOUNDS[k], BOUNDS[k + 1]) of entries 0 and 2.  Entry 1 is owned whole by launch 1 and
    has an empty range in the others.  out_offsets in reverse entry order."""
    lo, hi = BOUNDS[k], BOUNDS[k + 1]
    ranges = [(lo, hi), (0, N_SPLIT) if k == 1 else (lo, lo), (lo, hi)]
    specs, off = [None] * 3, 0
    for i in (2, 1, 0):
        specs[i] = pair.spec(ENTRIES[i], N_SPLIT, ranges[i][0], ranges[i][1], off)
        off += ranges[i][1] - ranges[i][0]
    return specs


def _sum(launches, key):
    return sum(g[key].astype(np.int64) for g in launches)


@pytest.mark.parametrize("outs", ["both", "overtime"])
@pytest.mark.parametrize("kernel", KERNELS)
def test_split_launches_add_up_to_the_whole(engines, pairs, kernel, outs):
    e, pair = engines[kernel], pairs[kernel]
    kw = dict(OUTPUTS[outs], want_iters=True)
    hist_only = {k: v for k, v in OUTPUTS[outs].items() if k not in ("want_period_scores", "want_sequence", "want_ot_periods")}
    if pair.usage is not None:
        kw.update(want_players=True, want_player_hist=True)
        hist_only.update(want_player_hist=True)
    whole_specs = _entries(pair, N_SPLIT)
    # the histograms alone: the per-game rows that are the hooks' state live in the library's grow-only scratch, which
    # the larger whole launch leaves behind for the three smaller ones (each rank of api.simulate_slate does this)
    e.set_matchups(whole_specs)
    whole_h = e.simulate_host(SEED, want_scores=False, **hist_only)
    split_h = []
    for k in range(3):
        e.set_matchups(_split_specs(pair, k))
        split_h.append(e.simulate_host(SEED, want_scores=False, **hist_only))
    e.set_matchups(whole_specs)
    whole = e.simulate_host(SEED, **kw)
    split = []
    for k in range(3):
        e.set_matchups(_split_specs(pair, k))
        split.append(e.simulate_host(SEED, **kw))
    assert (whole["counters"]["trips"] > 0) == (kernel == "memo")
    hists = [h for h in HIST_KEYS if h in whole]
    assert len(hists) == (3 if outs == "both" else 2) + (pair.usage is not None)
    if outs == "overtime":
        assert whole["counters"]["ot_games"] > N_SPLIT // 10
    for h in hists:
        assert np.array_equal(_sum(split, h), whole[h].astype(np.int64)), h
        assert np.array_equal(_sum(split_h, h), whole[h].astype(np.int64)), h
        assert np.array_equal(whole_h[h], whole[h]), h
    for c in ALL_GAME_COUNTERS:
        assert sum(g["counters"][c] for g in split) == whole["counters"][c], c
        assert sum(g["counters"][c] for g in split_h) == whole["counters"][c], c
    # per-game rows, put back by out_offset
    for k, got in enumerate(split):
        for i, (ws, s) in enumerate(zip(whole_specs, _split_specs(pair, k))):
            a = slice(s.out_offset, s.out_offset + s.game_end - s.game_begin)
            b = slice(ws.out_offset + s.game_begin, ws.out_offset + s.game_end)
            for r in ROW_KEYS:
                if r in whole:
                    assert np.array_equal(got[r][a], whole[r][b]), (k, i, r)
            if pair.usage is not None:
                x, y = got["players"].rec[a], whole["players"].rec[b]
                assert np.array_equal(x["counts"], y["counts"]) and np.array_equal(x["yds"].view(np.uint64),
                                                                                  y["yds"].view(np.uint64)), (k, i)


# ---- 4. edges of the overtime rules against the oracle ------------------------------------------------------------------
N_EDGE = 5000
LEVEL_126 = GameState(offense=0, seconds=0, score=(126, 126))
EDGES = {
    "max_periods=1": (OvertimeRules(max_periods=1), ENTRIES),
    "snap_clock=1": (OvertimeRules(snap_clock=1), ENTRIES),
    "snap_clock=900": (OvertimeRules(snap_clock=900), ENTRIES),
    "level_126_at_0:00": (RULES, (ENTRIES[0], LEVEL_126)),
}


@pytest.fixture(scope="module")
def edge_refs(oracle, models_s2, live, seqo, oto, pairs):
    cache = {}

    def get(name):
        if name not in cache:
            rules, starts = EDGES[name]
            cache[name] = [_entry_oracle(oracle, models_s2, (live, seqo, oto), pairs["plain"], s, i, N_EDGE, rules=rules)
                           for i, s in enumerate(starts)]
        return cache[name]
    return get


@pytest.mark.parametrize("memo", ["on", "off"])
@pytest.mark.parametrize("name", list(EDGES))
def test_overtime_edges_against_the_oracle(engines, pairs, edge_refs, name, memo):
    e = engines["memo" if memo == "on" else "plain"]
    rules, starts = EDGES[name]
    k = len(starts)
    e.set_matchups(_entries(pairs["plain"], N_EDGE, starts))
    got = e.simulate_host(SEED, want_iters=True, overtime=rules, want_ot_periods=True, want_ot_hist=True)
    ref = edge_refs(name)
    c = got["counters"]
    assert (c["trips"] > 0) == (memo == "on")
    games = np.arange(N_EDGE)
    for i, r in enumerate(ref):
        rows = _rows(i, N_EDGE, k)
        assert np.array_equal(got["scores"][rows], r["scores"]), i
        assert np.array_equal(got["iters"][rows], r["iters"]), i
        assert np.array_equal(got["ot_periods"][rows].astype(np.int64), r["periods"]), i
        assert np.array_equal(got["ot_hist"][i].astype(np.int64), ot_hist_from_rows(r["scores"], r["periods"], games)), i
        assert np.array_equal(got["hist"][i].astype(np.int64), outputs.histogram_from_scores(r["scores"])), i
        assert r["periods"].max() <= rules.max_periods
    assert {k_: c[k_] for k_ in ORACLE_COUNTERS} == {k_: sum(r["counters"][k_] for r in ref) for k_ in ORACLE_COUNTERS}
    over = sum(int((r["scores"] > LAST).any(axis=1).sum()) for r in ref)
    assert c["hist_overflow"] == over
    assert c["ot_games"] == sum(int((r["periods"] > 0).sum()) for r in ref) > 0
    assert c["ot_periods"] == sum(int(r["periods"].sum()) for r in ref)
    if name == "max_periods=1":
        assert any((r["periods"] == 1).any() and (r["scores"][:, 0] == r["scores"][:, 1]).any() for r in ref)
    if starts[-1] is LEVEL_126:
        # every game of that entry plays overtime, and those that score pass the last bin
        rows = _rows(k - 1, N_EDGE, k)
        assert (got["ot_periods"][rows] > 0).all()
        assert over > N_EDGE // 2
        assert int(got["hist"][k - 1][:, LAST, :].sum() + got["hist"][k - 1][:, :, LAST].sum()) >= over
