"""Quarter and half markets on the B200 (fmc_simulate_segments, the period hooks of both simulation kernels): the
reference's own games, the C oracle game by game, the histograms against the per-game rows, live starts on every
boundary, nothing else moving, and the API."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, ISU, KSU
from fast_monte_carlo_b200 import api, outputs, priors, usage
from fast_monte_carlo_b200.engine import Engine, GameState, MatchupSpec
from fast_monte_carlo_b200.native import PERIOD_NONE
from test_segments import BOUNDARIES, periods_from_trace

pytestmark = pytest.mark.gpu

GAME_COUNTERS = ("games", "plays", "iters", "pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg", "punt", "go",
                 "hist_overflow")
BINS = outputs.HIST_BINS
LAST = BINS - 1


@pytest.fixture(scope="module")
def live(models_s2):
    import oracle_live
    oracle_live.load_models(models_s2)
    return oracle_live


@pytest.fixture(scope="module")
def memo_engines(models_s2, native_lib):
    engines = {m: Engine(models_s2, device=0, stage2="standin", memo=m) for m in ("on", "off", "persistent")}
    yield engines
    for e in engines.values():
        e.close()


def _word(a, b):
    return (np.asarray(a).astype(np.uint32) | (np.asarray(b).astype(np.uint32) << 16)).astype(np.uint32)


def _unword(w):
    w = np.asarray(w, dtype=np.uint32)
    return (w & 0xFFFF).astype(np.int64), (w >> 16).astype(np.int64)


def oracle_period_words(trace, iters, scores, games, start_sec):
    """period_scores [n][3] of games from the oracle's traces (first-receiver orientation, NaN past the last iteration),
    their final (A, B) scores and their game ids: the definition of periods_from_trace, vectorised."""
    n = len(iters)
    first = np.asarray(games) & 1
    out = np.full((n, 3), PERIOD_NONE, dtype=np.uint32)
    sec = np.nan_to_num(trace[:, :, 2], nan=1e9)
    rows = np.arange(n)
    for q, B in enumerate(BOUNDARIES):
        if start_sec <= B:
            continue
        hit = sec <= B
        has, k = hit.any(axis=1), hit.argmax(axis=1)
        f, s = trace[rows, k, 3], trace[rows, k, 4]
        a = np.where(has, np.where(first == 0, f, s), scores[:, 0])
        b = np.where(has, np.where(first == 0, s, f), scores[:, 1])
        out[:, q] = _word(a, b)
    return out


def segments_from_rows(period, scores, start_sec, start_score):
    """Per-game points in each period (int64 [n][6][2]) and whether the period is counted, from period_scores rows, final
    scores and the entry's start state (include/fmc.h FMC_N_SEGMENTS)."""
    n = scores.shape[0]
    s0 = (np.full(n, start_score[0]), np.full(n, start_score[1]))
    at = {3600: s0, 0: (scores[:, 0].astype(np.int64), scores[:, 1].astype(np.int64))}
    for q, B in enumerate(BOUNDARIES):
        at[B] = _unword(period[:, q]) if start_sec > B else None
    base = lambda b: at[b] if (b == 3600 or start_sec > b) else s0
    spans = {"Q1": (3600, 2700), "Q2": (2700, 1800), "Q3": (1800, 900), "Q4": (900, 0), "H1": (3600, 1800), "H2": (1800, 0)}
    pts = np.zeros((n, 6, 2), dtype=np.int64)
    counted = []
    for k, name in enumerate(outputs.SEGMENTS):
        b0, b1 = spans[name]
        ok = b1 == 0 or start_sec > b1
        counted.append(ok)
        if ok:
            e, s = at[b1], base(b0)
            pts[:, k, 0], pts[:, k, 1] = e[0] - s[0], e[1] - s[1]
    return pts, counted


def host_segment_hist(pts, counted, games):
    """[2][6][BINS][BINS] from per-game period points, clamped into the last bin like the final histogram."""
    h = np.zeros((2, 6, BINS, BINS), dtype=np.int64)
    o = np.asarray(games) & 1
    for k in range(6):
        if counted[k]:
            np.add.at(h, (o, k, np.minimum(pts[:, k, 0], LAST), np.minimum(pts[:, k, 1], LAST)), 1)
    return h


# ---- 1. the reference's own games ---------------------------------------------------------------------------------
def _reference_entries():
    from oracle import c_oracle as co
    from streams import adversarial_stream
    specs, rows, want = [], [], []
    for name, make in (("ref_trajectories.npz", co.make_stream), ("ref_trajectories_adversarial.npz", adversarial_stream)):
        t = np.load(os.path.join(GOLDEN, name))
        meta = json.loads(str(t["meta"]))
        stream = make(len(meta), int(t["stream_seed"]))
        for g, m in enumerate(meta):
            spA, spB = (m["sp_second"], m["sp_first"]) if g & 1 else (m["sp_first"], m["sp_second"])
            n = int(t["iters"][g])
            fin = (int(t["scores"][g][0]), int(t["scores"][g][1]))
            ends, _ = periods_from_trace(t["traces"][g], n, fin)
            ab = [(e[0], e[1]) if g & 1 == 0 else (e[1], e[0]) for e in ends]
            specs.append(MatchupSpec("A", "B", tuple(spA), tuple(spB), g + 1, g, g + 1, len(specs)))
            rows.append(stream[g])
            want.append((n, t["traces"][g, :n], fin if g & 1 == 0 else fin[::-1], [int(_word(*x)) for x in ab]))
    return specs, np.stack(rows), want


@pytest.mark.parametrize("memo", ["on", "off"])
def test_reference_games_period_scores(memo_engines, memo):
    """The 40 reference games under their injected draws: period_scores are the reference's own quarter-end scores,
    integer for integer, and the games themselves are unchanged with the hooks in."""
    e = memo_engines[memo]
    specs, stream, want = _reference_entries()
    assert len(specs) == 40
    e.set_matchups(specs)
    got = e.simulate_host(0, stream=stream, want_trace=True, want_iters=True, want_period_scores=True, want_segments=True)
    for i, (n, rows, fin, words) in enumerate(want):
        assert got["iters"][i] == n, i
        assert np.array_equal(got["trace"][i, :n], rows), i
        assert tuple(got["scores"][i]) == tuple(fin), i
        assert list(got["period_scores"][i]) == words, i
        # the histogram path of the hooked TEST instantiations: the entry's one game in its periods' bins
        pts, counted = segments_from_rows(got["period_scores"][i:i + 1], got["scores"][i:i + 1], 3600, (0, 0))
        g = specs[i].game_begin
        assert all(counted)
        assert np.array_equal(got["segment_hist"][i].astype(np.int64), host_segment_hist(pts, counted, [g])), i
        ref = periods_from_trace(rows, n, fin if g & 1 == 0 else fin[::-1])[1]
        for k, name in enumerate(outputs.SEGMENTS):
            want = ref[name] if g & 1 == 0 else ref[name][::-1]
            assert tuple(pts[0, k]) == tuple(want), (i, name)
    assert (got["counters"]["memo_probes"] > 0) == (memo == "on")


# ---- 2. the oracle, game by game ----------------------------------------------------------------------------------
def _oracle_words(live, cfg, n, seed, start, chunk=5000, **kw):
    words, scores = [], []
    for lo in range(0, n, chunk):
        k = min(chunk, n - lo)
        ref = live.simulate(cfg, k, game0=lo, seed=seed, start=start, trace=True, **kw)
        words.append(oracle_period_words(ref["trace"], ref["iters"], ref["scores"], np.arange(lo, lo + k), start.seconds))
        scores.append(ref["scores"])
    return np.concatenate(words), np.concatenate(scores)


@pytest.mark.parametrize("memo", ["on", "off", "persistent"])
def test_period_scores_equal_the_oracle(memo_engines, oracle, models_s2, live, memo):
    e = memo_engines[memo]
    n = 20_000
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    got = e.simulate_host(8675309, want_period_scores=True)
    words, scores = _oracle_words(live, oracle.make_config(models_s2, KSU, ISU), n, 8675309, GameState())
    assert np.array_equal(got["scores"], scores)
    assert np.array_equal(got["period_scores"], words)
    assert (got["period_scores"] != PERIOD_NONE).all()


def test_period_scores_equal_the_oracle_in_player_mode(engine, oracle, models_s2, live):
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ctx = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    use = tuple(usage.resolve_team(tc, models_s2) for tc in ctx)
    n = 20_000
    spec = MatchupSpec("Kansas State", "Iowa State", ctx[0].sp, ctx[1].sp, n, 0, n, 0, usage=use)
    engine.set_matchups([spec])
    assert engine.ctx.has_usage and engine.n_slots > 0
    got = engine.simulate_host(1234, want_period_scores=True, want_players=True)
    cfg = oracle.make_config(models_s2, spec.sp_a, spec.sp_b)
    words, scores = _oracle_words(live, cfg, n, 1234, GameState(), usage=oracle.make_usage(use), n_slots=engine.n_slots)
    assert np.array_equal(got["scores"], scores)
    assert np.array_equal(got["period_scores"], words)


# ---- 3. the histograms are the per-game rows ----------------------------------------------------------------------
def test_segment_hist_equals_the_per_game_rows(engine):
    n = 1_000_000
    engine.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0)])
    got = engine.simulate_host(99, want_period_scores=True, want_segments=True)
    pts, counted = segments_from_rows(got["period_scores"], got["scores"], 3600, (0, 0))
    assert all(counted)
    want = host_segment_hist(pts, counted, np.arange(n))
    assert np.array_equal(got["segment_hist"][0].astype(np.int64), want)
    assert int(got["segment_hist"][0].sum()) == 6 * n
    # Q1 + Q2 = H1, Q3 + Q4 = H2, H1 + H2 = final, game by game
    assert np.array_equal(pts[:, 0] + pts[:, 1], pts[:, 4]) and np.array_equal(pts[:, 2] + pts[:, 3], pts[:, 5])
    assert np.array_equal(pts[:, 4] + pts[:, 5], got["scores"])


# ---- 4. live starts on every boundary --------------------------------------------------------------------------------
LIVE_SECONDS = (3600, 2701, 2700, 1801, 1800, 901, 900, 1, 0)


def _live_states():
    st = [GameState(offense=s % 2, seconds=s, down=1, distance=10.0, yards_to_goal=75.0) for s in LIVE_SECONDS]
    st += [GameState(offense=1, seconds=s, down=2, distance=6.0, yards_to_goal=40.0, score=(17, 10)) for s in (2000, 901, 0)]
    return st


@pytest.mark.parametrize("memo", ["on", "off"])
def test_live_starts_on_the_boundaries(memo_engines, oracle, models_s2, live, memo):
    e = memo_engines[memo]
    states = _live_states()
    per = 20_000
    e.set_matchups([MatchupSpec("A", "B", KSU, ISU, per, 0, per, m * per, start=s) for m, s in enumerate(states)])
    got = e.simulate_host(4711, want_period_scores=True, want_segments=True)
    cfg = oracle.make_config(models_s2, KSU, ISU)
    for m, s in enumerate(states):
        sl = slice(m * per, (m + 1) * per)
        ps, sc = got["period_scores"][sl], got["scores"][sl]
        for q, B in enumerate(BOUNDARIES):
            assert ((ps[:, q] == PERIOD_NONE).all() if s.seconds <= B else (ps[:, q] != PERIOD_NONE).all()), (m, q)
        pts, counted = segments_from_rows(ps, sc, s.seconds, s.score)
        sh = got["segment_hist"][m].astype(np.int64)
        assert np.array_equal(sh, host_segment_hist(pts, counted, np.arange(per))), m
        for k in range(6):
            assert int(sh[:, k].sum()) == (per if counted[k] else 0), (m, k)
        d = sc - np.array(s.score)
        h1 = pts[:, 4] if counted[4] else 0
        if counted[0]:
            assert np.array_equal(pts[:, 0] + pts[:, 1], pts[:, 4])
        if counted[2]:
            assert np.array_equal(pts[:, 2] + pts[:, 3], pts[:, 5])
        assert np.array_equal(h1 + pts[:, 5], d), m
        assert (pts >= 0).all()
        if s.seconds == 0:
            assert (pts[:, 3] == 0).all() and (pts[:, 5] == 0).all() and (sc == np.array(s.score)).all()
        # the oracle from the same start, for the first games of the entry
        k = 3000
        ref = live.simulate(cfg, k, matchup=m, seed=4711, start=s, trace=True)
        assert np.array_equal(sc[:k], ref["scores"]), m
        assert np.array_equal(ps[:k], oracle_period_words(ref["trace"], ref["iters"], ref["scores"], np.arange(k), s.seconds)), m


# ---- 5. nothing else moves -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("memo", ["on", "off"])
def test_outputs_unchanged_by_the_hooks(memo_engines, memo):
    e = memo_engines[memo]
    n = 300_000
    st = GameState(offense=0, seconds=2000, down=3, distance=4.0, yards_to_goal=48.0, score=(7, 10))
    specs = [MatchupSpec("A", "B", KSU, ISU, n, 0, n, 0), MatchupSpec("A", "B", ISU, KSU, n, 0, n, n, start=st)]
    e.set_matchups(specs)
    base = e.simulate_host(2024, want_iters=True)
    seg = e.simulate_host(2024, want_iters=True, want_segments=True)
    for k in ("scores", "hist", "iters"):
        assert np.array_equal(seg[k], base[k]), k
    assert {k: seg["counters"][k] for k in GAME_COUNTERS} == {k: base["counters"][k] for k in GAME_COUNTERS}
    # two game ranges launched separately add up to the one launch
    parts = 0
    for g0, g1 in (api.shard_range(n, r, 2) for r in range(2)):
        e.set_matchups([MatchupSpec("A", "B", KSU, ISU, n, g0, g1, 0), MatchupSpec("A", "B", ISU, KSU, n, g0, g1, g1 - g0, start=st)])
        parts = parts + e.simulate_host(2024, want_segments=True)["segment_hist"].astype(np.int64)
    assert np.array_equal(parts, seg["segment_hist"].astype(np.int64))


def test_injected_draws_unchanged_by_the_hooks_in_player_mode(engine, oracle, models_s2):
    """The player instantiation under injected draws (the TEST x PLAYERS x hooks kernel): trajectories, scores and boxes
    are those of the launch without period outputs."""
    focus = usage.build_focus_usage_tables(os.path.join(GOLDEN, "players_focus.csv"))
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    ctx = [priors.build_team_context_from_sp_flex(t, 2025, 1, sp, focus=focus, usage_dir=GOLDEN)
           for t in ("Kansas State", "Iowa State")]
    use = tuple(usage.resolve_team(tc, models_s2) for tc in ctx)
    n = 2048
    stream = oracle.make_stream(n, 5)
    engine.set_matchups([MatchupSpec("Kansas State", "Iowa State", ctx[0].sp, ctx[1].sp, n, 0, n, 0, usage=use)])
    a = engine.simulate_host(0, stream=stream, want_trace=True, want_iters=True, want_players=True)
    b = engine.simulate_host(0, stream=stream, want_trace=True, want_iters=True, want_players=True, want_period_scores=True,
                             want_segments=True)
    same = (a["trace"] == b["trace"]) | (np.isnan(a["trace"]) & np.isnan(b["trace"]))
    assert same.all()
    for k in ("scores", "iters", "hist"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["players"].dense(), b["players"].dense())
    pts, counted = segments_from_rows(b["period_scores"], b["scores"], 3600, (0, 0))
    assert np.array_equal(b["segment_hist"][0].astype(np.int64), host_segment_hist(pts, counted, np.arange(n)))


# ---- 6. the API ----------------------------------------------------------------------------------------------------
def test_simulate_slate_segments(engine):
    pairs = [("Kansas State", "Iowa State"), ("UTSA", "Ohio State"), ("Texas", "Michigan")]
    markets = {pairs[0]: {"spread": -3.5, "H1": {"spread": -1.5, "total": 24.5}, "Q1": {"total": 10.0}},
               pairs[1]: {"H2": {"spread": 7.0}}}
    plain = api.simulate_slate(pairs, n=5000, seed=3, engine=engine, markets={pairs[0]: {"spread": -3.5}})
    res = api.simulate_slate(pairs, n=5000, seed=3, engine=engine, markets=markets, segments=True)
    for p in pairs:
        r, q = res[p], plain[p]
        assert np.array_equal(r["hist"], q["hist"]) and r["games"] == q["games"] == 10_000
        assert r["moneyline"] == q["moneyline"] and r["summary"].equals(q["summary"]) and r["markets"] == q["markets"]
        assert set(r["segments"]) == set(outputs.SEGMENTS)
        for name, s in r["segments"].items():
            assert s["hist"].shape == (2, BINS, BINS) and int(s["hist"].sum()) == 10_000
            line = markets.get(p, {}).get(name, {})
            assert s["odds"] == outputs.segment_odds_from_hist(s["hist"].sum(axis=0), p[0], p[1], **line)
        assert r["segments"]["H1"]["odds"]["mean_points"][p[0]] + r["segments"]["H2"]["odds"]["mean_points"][p[0]] == \
            pytest.approx(r["summary"].loc[p[0], "mean_pts"] / 2 + r["summary"].loc[p[1], "mean_opp"] / 2, abs=1e-9)
    assert set(res[pairs[0]]["segments"]["H1"]["odds"]["markets"]) == {"spread", "total"}
    assert res[pairs[1]]["markets"] is None and res[pairs[2]]["segments"]["Q1"]["odds"]["markets"] is None
    assert res["_counters"]["games"] == plain["_counters"]["games"]


def test_simulate_live_segments(engine):
    ks, isu = "Kansas State", "Iowa State"
    entries = [
        (ks, isu, api.LiveState(ks, 3600, 1, 10.0, 75.0)),
        (ks, isu, api.LiveState(isu, 2400, 2, 7.0, 55.0, (10, 7), quarter_start_score=(7, 0))),
        (ks, isu, api.LiveState(isu, 2400, 2, 7.0, 55.0, (10, 7))),
        (ks, isu, api.LiveState(ks, 1200, 3, 3.0, 30.0, (17, 14), half_start_score=(14, 14))),
        (ks, isu, api.LiveState(ks, 400, 1, 10.0, 75.0, (24, 21))),
    ]
    markets = {1: {"spread": -2.5, "Q2": {"spread": 0.5}, "H1": {"total": 24.5}}, 3: {"H2": {"spread": -3.0}}}
    plain = api.simulate_live(entries, 20_000, seed=21, engine=engine, markets={1: {"spread": -2.5}})
    res = api.simulate_live(entries, 20_000, seed=21, engine=engine, markets=markets, segments=True)
    for i, (r, q) in enumerate(zip(res, plain)):
        assert np.array_equal(r["hist"], q["hist"])
        for k in ("games", "p_win", "p_tie", "mean_points", "hist_overflow", "markets"):
            assert r[k] == q[k], (i, k)
        for name, s in r["segments"].items():
            line = markets.get(i, {}).get(name, {})
            if s["status"] == "ended":
                assert s["odds"] is None and not s["hist"].any()
            elif s["offset"] is None:
                assert s["odds"] is None and int(s["hist"].sum()) == 20_000
            else:
                assert s["odds"] == outputs.segment_odds_from_hist(s["hist"], ks, isu, offset=s["offset"], **line)
    assert res[1]["segments"]["Q2"]["offset"] == (3, 7) and res[2]["segments"]["Q2"]["odds"] is None
    assert res[3]["segments"]["Q3"]["offset"] == (3, 0) and res[3]["segments"]["H2"]["offset"] == (3, 0)
    assert res[4]["segments"]["Q4"]["odds"] is None and res[4]["segments"]["Q3"]["status"] == "ended"
    assert res[0]["segments"]["H1"]["odds"]["p_win"] == pytest.approx(
        api.live_segments(entries[0][2], np.stack([res[0]["segments"][k]["hist"] for k in outputs.SEGMENTS]), ks,
                          isu)["H1"]["odds"]["p_win"])
