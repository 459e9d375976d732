#!/usr/bin/env python
"""Headline benchmark: simulated plays/s (and games/s) of the play-by-play Monte Carlo engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--games G] [--memo on|off]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): Kansas State vs Iowa State from the 2025 week-1 SP+ priors,
10,000,000 simulated games per GPU per step (weak scaling: rank r plays game ids
[r*G, (r+1)*G) of the same matchup; the integer histograms are merged with ONE all-reduce per
step).  Shipped model artifacts; the stage-2 booster the reference snapshot lacks is replaced by a
synthetic booster of the trained shape (fast_monte_carlo_b200/synth.py) so that the stage-2 tree
work is NOT skipped.  One step = one launch of the persistent simulation kernel over the batch.

Prints ONE JSON line (rank 0):
  value         plays/s with everything resident in HBM (CUDA events on the launch stream), the engine as shipped:
                exact memo in front of the tree walk ON (`memo`: hit rate, requests still walked);
  e2e           the same metric through the reference's Python entry point api.simulate_matchup (FMC:1467-1521) with
                HOST buffers: kernel, per-game score words + histogram copied back, the 2n-row sims_df; host clock;
  roofline      the tree walk, measured in the same run with the memo OFF (no tree work hidden): fraction of the L1
                data-pipe peak (the bound of a gather over cache-resident node tables), with the SURVEY 8(d)
                algorithmic-bytes figure, the gathered bytes against a warp-coherent gather probe, and DRAM traffic;
  tree_eval     BASELINE configs[2]: predict_kernel on 2^26 synthetic states, same accounting;
  cpu_baseline  the C oracle (a port of the reference's algorithm) on all host cores of this box, at every N.
`--impl reference` times that CPU port as its own arm.  `--workload slate | season` = configs[3] / configs[4].
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

KSU = ("Kansas State", (15.6, 35.7, 20.0))
ISU = ("Iowa State", (11.0, 31.5, 20.6))
SEED = 20251018
METRIC = "simulated_plays_per_sec"
UNIT = "plays/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--games", type=int, default=10_000_000, help="games per GPU per step (matchup workload)")
    ap.add_argument("--workload", default="matchup", choices=["matchup", "slate", "season"],
                    help="matchup = BASELINE configs[1] (default, the headline); slate = configs[3]: 60 matchups x "
                         "--slate-games games each, sharded over the GPUs by contiguous game-id ranges (strong scaling); "
                         "season = configs[4]: 12 weekly slates of 60 matchups from seeded shuffles of the 136 teams")
    ap.add_argument("--slate-games", type=int, default=1_000_000, help="games per matchup of the slate workload")
    ap.add_argument("--shard", default="matchups", choices=["games", "matchups"],
                    help="slate / season under several GPUs: whole matchups per rank (default; keeps a matchup's memo on one "
                         "GPU) or a game-id slice of every matchup per rank")
    ap.add_argument("--stage2", default="synthetic", choices=["synthetic", "standin"])
    ap.add_argument("--players", action="store_true",
                    help="matchup workload in player mode: usage tables from the synthetic focus sheet "
                         "(fast_monte_carlo_b200/data/players_focus_synthetic.csv), per-game player box written")
    ap.add_argument("--cpu-games", type=int, default=0, help="games of the bounded CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--memo", default=None, choices=["on", "off", "persistent"],
                    help="exact rank-keyed memo in front of the tree walk (default: on; FMC_MEMO overrides the default)")
    ap.add_argument("--roofline-steps", type=int, default=2, help="timed memo-off launches behind the roofline record")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-tree-eval", action="store_true")
    ap.add_argument("--tree-states", type=int, default=1 << 26, help="states of the configs[2] tree-eval sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, rank 0 writes what the last timed step computed as DIR/<name>.npy: "
                         "scores float32[games, 2] (points of team A, team B) and, with --players, players "
                         "float64[games, 2, slots, 6] of rank 0's games; hist float64[matchups, 2, 128, 128] and "
                         "counters float64[15] (games, plays, iters, pass, comp, inc, int, sack, run, td, fga, fg, punt, "
                         "go, hist_overflow) summed over all ranks, as every rank receives them. Larger outputs are "
                         "sampled with a fixed seed: scores of 2^20 games, the boxes of the first of those that fit "
                         "in 24 MiB, histograms of 64 matchups")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def slate_pairs():
    """SURVEY 8(d) config 4: the first 120 teams of the priors CSV paired (2i, 2i+1)."""
    from fast_monte_carlo_b200 import priors
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    teams = list(sp["team"])[:120]
    return [(teams[2 * i], teams[2 * i + 1]) for i in range(60)], sp


def season_pairs():
    """SURVEY 8(d) config 5: 12 weeks x 60 matchups, week w = default_rng(2025 + w) shuffle of the 136 teams,
    paired (2i, 2i+1)."""
    import numpy as np
    from fast_monte_carlo_b200 import priors
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    teams = list(sp.drop_duplicates(subset=["RATING", "OFFENSE", "DEFENSE"])["team"])
    pairs = []
    for week in range(1, 13):
        order = np.random.default_rng(2025 + week).permutation(len(teams))
        pairs += [(teams[order[2 * i]], teams[order[2 * i + 1]]) for i in range(60)]
    return pairs, sp


def workload(args, n_gpus):
    if args.workload == "season":
        return {
            "workload": "configs[4]: season slate, 12 weeks x 60 matchups (seeded shuffles of the 136 teams of "
                        f"PregameSPPlus2025_1) x {args.slate_games:,} simulated games each, sharded over {n_gpus} GPU(s) by "
                        f"{args.shard}, Philox seed {SEED}",
            "total_games_per_step": 720 * args.slate_games,
            "play_call": "pass_prob_v1 heuristic (reference behaviour when play_model.json is absent)",
            "stage2": ("synthetic booster of the trained shape (1086 trees, depth<=7)" if args.stage2 == "synthetic"
                       else "fixed stand-in probabilities"),
            "players": "Unknown (no usage tables shipped)",
            "parallelism": f"every matchup's games sharded over {n_gpus} GPU(s); one NCCL all-reduce of the "
                           "[720][2][128][128] histograms per step",
            "l2": "flushed between timed steps (256 MiB write); node tables: 720 matchups x ~0.6 MB",
        }
    if args.workload == "slate":
        return {
            "workload": "configs[3]: full-slate run, 60 matchups (first 120 teams of PregameSPPlus2025_1 paired) x "
                        f"{args.slate_games:,} simulated games each, sharded over {n_gpus} GPU(s) by {args.shard}, "
                        f"Philox seed {SEED}",
            "total_games_per_step": 60 * args.slate_games,
            "play_call": "pass_prob_v1 heuristic (reference behaviour when play_model.json is absent)",
            "stage2": ("synthetic booster of the trained shape (1086 trees, depth<=7)" if args.stage2 == "synthetic"
                       else "fixed stand-in probabilities"),
            "players": "Unknown (no usage tables shipped)",
            "parallelism": f"every matchup's games sharded over {n_gpus} GPU(s); one NCCL all-reduce of the "
                           "[60][2][128][128] histograms per step",
            "l2": "flushed between timed steps (256 MiB write); node tables (60 matchups x ~0.6 MB) are L2-resident",
        }
    return {
        "workload": "configs[1]: Kansas State vs Iowa State (PregameSPPlus2025_1 priors), "
                    f"{args.games:,} simulated games per GPU per step, Philox seed {SEED}",
        "games_per_gpu_per_step": args.games,
        "total_games_per_step": args.games * n_gpus,
        "play_call": "pass_prob_v1 heuristic (reference behaviour when play_model.json is absent)",
        "stage2": ("synthetic booster of the trained shape (1086 trees, depth<=7)" if args.stage2 == "synthetic"
                   else "fixed stand-in probabilities"),
        "players": ("synthetic focus sheet: 3 passers / 4 rushers / 4 targets per team sampled per play, one-hot "
                    "columns fed from the sampled names, 8 box lines per team per game written"
                    if getattr(args, "players", False) else "Unknown (no usage tables shipped)"),
        "parallelism": f"games sharded over {n_gpus} GPU(s); one NCCL all-reduce of the histograms per step",
        "l2": "flushed between timed steps (256 MiB write); node tables are meant to be cache-resident",
        "memo": "exact rank-keyed memo of model outputs in front of the tree walk, cleared at every step (--memo off: every "
                "request is walked; the roofline record is measured that way)",
    }


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------------------------
# algorithmic bytes (SURVEY 8d): 8 B per internal-node visit + one leaf fetch (4 B xgb / 8 B sklearn)
# per tree, visits = cover-weighted expected path length on the ORIGINAL (unpruned) forests
# ----------------------------------------------------------------------------------------------
def algorithmic_bytes_per_row(forest) -> float:
    import numpy as np
    leaf = forest.left < 0
    cover = forest.cover if forest.cover is not None else np.ones(forest.n_nodes)
    visits = 0.0
    bounds = np.append(forest.tree_root, forest.n_nodes)
    root_cover = cover[forest.tree_root]
    # expected internal-node visits of a tree = sum over internal nodes of cover(node)/cover(root)
    tree_of = np.repeat(np.arange(forest.n_trees), np.diff(bounds))
    w = cover / np.maximum(root_cover[tree_of], 1e-30)
    visits = float(w[~leaf].sum())
    leaf_bytes = 8 if forest.kind == 1 else 4
    return 8.0 * visits + leaf_bytes * forest.n_trees


def step_algorithmic_bytes(models, counters, stage2_booster: bool) -> float:
    b = {k: algorithmic_bytes_per_row(models[k]) for k in ("pass_stage1", "pass_yards", "run_yards", "sack_yards")}
    total = counters["pass"] * b["pass_stage1"] + counters["comp"] * b["pass_yards"] + \
        counters["run"] * b["run_yards"] + counters["sack"] * b["sack_yards"]
    if stage2_booster:
        total += (counters["pass"] - counters["comp"]) * algorithmic_bytes_per_row(models["pass_stage2"])
    return float(total)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(games_per_launch: int):
    """DRAM bytes per launch of sim_kernel, from the committed `ncu --set full` capture
    (profiles/sim_kernel_ncu_latest.json: dram__bytes_read.sum + dram__bytes_write.sum of one launch of
    `games_in_profiled_launch` games) scaled to this run's games per launch -- the kernel's DRAM traffic is
    the per-game score word + histogram atomics, i.e. proportional to the games."""
    p = os.path.join(ROOT, "profiles", "sim_kernel_ncu_latest.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["dram_bytes_per_launch"]) / float(d["games_in_profiled_launch"]) * games_per_launch
        except Exception:
            return None
    return None


# ----------------------------------------------------------------------------------------------
# CPU arm: the C oracle (port of the reference algorithm) on the host cores
# ----------------------------------------------------------------------------------------------
def load_models(stage2: str):
    from fast_monte_carlo_b200 import artifacts as art, synth
    ms = art.load_default_models()
    if stage2 == "synthetic":
        ms = synth.with_synthetic_stage2(ms)
    return ms


def synthetic_usage(ms):
    """Usage tables of the --players workload (both teams of the matchup)."""
    from fast_monte_carlo_b200 import priors, usage
    sheet = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fast_monte_carlo_b200", "data",
                         "players_focus_synthetic.csv")
    focus = usage.build_focus_usage_tables(sheet)
    sp_df = priors.load_sp_flex(priors.packaged_priors_path())
    return tuple(usage.resolve_team(priors.build_team_context_from_sp_flex(t, 2025, 1, sp_df, focus=focus,
                                                                           usage_dir=os.path.dirname(sheet)), ms)
                 for t in (KSU[0], ISU[0]))


def host_threads() -> int:
    """Host cores this process may use (the CPU arm always uses all of them, whatever OMP_NUM_THREADS says)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:      # pragma: no cover
        return max(1, os.cpu_count() or 1)


def cpu_run(ms, games: int, stage2: str, game0: int = 0, players: bool = False):
    from oracle import c_oracle as co
    co.load_models(ms)
    cfg = co.make_config(ms, KSU[1], ISU[1], stage2="booster" if stage2 == "synthetic" else "standin")
    threads = host_threads()      # explicit: torchrun exports OMP_NUM_THREADS=1, which must not shrink the CPU arm
    kw = {}
    if players:
        use = synthetic_usage(ms)
        kw = dict(usage=co.make_usage(use), n_slots=max(len(u.slots) for u in use))
    t = time.perf_counter()
    r = co.simulate(cfg, games, game0=game0, seed=SEED, threads=threads, **kw)
    dt = time.perf_counter() - t
    return r, dt, threads


def cpu_baseline(ms, args):
    games = args.cpu_games
    if games <= 0:
        _, dt, _ = cpu_run(ms, 2000, args.stage2, players=args.players)
        games = int(max(4000, min(400_000, 15.0 / (dt / 2000))))     # ~15 s of CPU work
    r, dt, threads = cpu_run(ms, games, args.stage2, players=args.players)
    return {"value": r["counters"]["plays"] / dt, "unit": UNIT, "games_per_sec": games / dt, "cores": threads,
            "host_cpus": os.cpu_count(), "kind": "port",
            "sample": f"{games} games of the same matchup/seed through oracle/fmc_oracle.c (OpenMP, {threads} threads), {dt:.1f} s"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ms = load_models(args.stage2)
    if args.cpu_games > 0:
        per_step = args.cpu_games
    else:
        _, dt0, threads = cpu_run(ms, 2000, args.stage2, players=args.players)
        per_step = int(max(4000, min(400_000, 20.0 / (dt0 / 2000))))       # ~20 s per step
    for w in range(args.warmup):
        cpu_run(ms, max(2000, per_step // 10), args.stage2, players=args.players)
    plays = 0
    t_tot = 0.0
    for s in range(args.steps):
        r, dt, threads = cpu_run(ms, per_step, args.stage2, game0=s * per_step, players=args.players)
        plays += r["counters"]["plays"]
        t_tot += dt
    value = plays / t_tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload(args, args.gpus),
        "games_per_sec": args.steps * per_step / t_tot,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "host_cpus": os.cpu_count(), "kind": "port",
                         "sample": f"{per_step} games per step (bounded sample of the {args.games:,}-game workload) "
                                   f"through oracle/fmc_oracle.c, the CPU port of the reference algorithm; the "
                                   f"reference itself cannot run (xgboost absent, stage-2 blob missing)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# roofline pieces
# ----------------------------------------------------------------------------------------------
def ncu_summary(name="sim_kernel_ncu_latest.json"):
    p = os.path.join(ROOT, "profiles", name)
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def l1_pipe_roofline(warp_steps, lane_visits, kernel_s, n_sms, sm_mhz, ncu, algo_bytes, traffic, kernel):
    """The bound of the tree walk is the L1 data pipe (one wavefront per clock per SM): every tree level of a warp
    costs one feature LDS wavefront plus the wavefronts of its 8-byte node gather.  `warp_steps` is counted by the
    kernel itself (FMC_C_WARP_STEPS / fmc_predict_stats); wavefronts per step come from the committed ncu capture
    of the same kernel (profiles/: l1tex__data_pipe_lsu_wavefronts over the step counter of the profiled launch,
    else 1 + lgds wavefronts per global load request)."""
    d = (ncu or {}).get("derived", {})
    per_step = d.get("l1_wavefronts_per_warp_step") or (1.0 + d.get("lgds_wavefronts_per_global_ld_request", 2.37))
    wavefronts = warp_steps * per_step
    peak = n_sms * sm_mhz * 1e6              # wavefronts / s
    achieved = wavefronts / kernel_s
    hbm, hbm_src = measured_peaks()
    return {
        "bound": "l1-data-pipe", "achieved": achieved / 1e9, "peak": peak / 1e9, "unit": "Gwavefront/s",
        "frac": achieved / peak, "traffic": traffic, "kernel": kernel, "kernel_ms_per_launch": kernel_s * 1e3,
        "warp_level_node_gathers_per_launch": warp_steps, "l1_wavefronts_per_gather_level": per_step,
        "peak_source": f"{n_sms} SMs x {sm_mhz:.0f} MHz (median SM clock sampled during the timed launches) x 1 wavefront/clk/SM",
        "ncu_crosscheck": {"l1_data_pipe_wavefronts_per_sm_cycle": d.get("l1_data_pipe_wavefronts_per_sm_cycle"),
                           "source": (ncu or {}).get("report")},
        "gathered": {"node_slots_per_launch": lane_visits, "gbs": lane_visits * 8.0 / kernel_s / 1e9},
        "algorithmic": {"bytes_per_launch": algo_bytes, "gbs": algo_bytes / kernel_s / 1e9,
                        "note": "SURVEY 8(d): 8 B per internal-node visit + leaf fetch per tree on the UNPRUNED forests x requests"},
        "hbm": {"peak_gbs": hbm, "peak_source": hbm_src, "traffic_bytes_per_launch": traffic,
                "frac": (traffic / kernel_s / 1e9 / hbm) if traffic else None,
                "note": "the node tables are cache-resident by design: DRAM carries score words, histogram atomics and spills"},
    }


def tree_states(n, seed=3):
    """SURVEY 8(d) config 3 states (see scripts/bench_trees.py)."""
    import numpy as np
    from fast_monte_carlo_b200 import priors
    sp = priors.load_sp_flex(priors.packaged_priors_path()).drop_duplicates(subset=["RATING", "OFFENSE", "DEFENSE"])
    teams = sp[["RATING", "OFFENSE", "DEFENSE"]].to_numpy(dtype=float)
    rng = np.random.default_rng(seed)
    x = np.zeros((n, 17))
    x[:, 0] = rng.choice([1, 2, 3, 4], size=n, p=[.38, .31, .21, .10])
    x[:, 1] = np.clip(np.round(rng.normal(8, 4, n), 1), 0.5, 30)
    x[:, 2] = rng.integers(1, 100, n)
    x[:, 3] = x[:, 2] <= 20
    x[:, 4] = np.round(rng.normal(0, 14, n))
    x[:, 5] = rng.integers(1, 3601, n)
    x[:, 6] = x[:, 7] = 3
    o = rng.integers(0, len(teams), n); d = (o + rng.integers(1, len(teams), n)) % len(teams)
    x[:, 8] = teams[o, 0]; x[:, 9] = teams[o, 1]; x[:, 10] = teams[d, 2]; x[:, 11] = teams[d, 0]
    x[:, 12] = x[:, 1] >= x[:, 2] - 0.5
    x[:, 13] = (x[:, 0] == 4) & (x[:, 1] <= 2)
    x[:, 14] = x[:, 2] <= 33
    x[:, 15] = np.where(x[:, 5] > 1800, 1, 2)
    x[:, 16] = (x[:, 5] % 1800) <= 120
    return x


def tree_eval_record(eng, ms, local, n_total=1 << 26, batch=1 << 22):
    """BASELINE configs[2]: play_model.xgb + the nine quantile models on 2^26 synthetic states through fmc_tree_predict
    (device buffers), with the same L1-data-pipe accounting as the simulation kernel."""
    import torch
    from fast_monte_carlo_b200 import artifacts as art
    names = ("play_model", "pass_yards", "run_yards", "sack_yards")
    rows = torch.from_numpy(tree_states(batch)).cuda(local)
    outs = {nm: torch.empty((batch, ms[nm].n_outputs), dtype=torch.float64, device=rows.device) for nm in names}
    st = torch.cuda.current_stream()

    def run_batch():
        for nm in names:
            eng.ctx.tree_predict_device(art.MODEL_IDS[nm], rows.data_ptr(), batch, outs[nm].data_ptr(), cuda_stream=st.cuda_stream)

    run_batch(); torch.cuda.synchronize()
    eng.ctx.predict_stats(reset=True)
    n_batches = max(1, n_total // batch)
    sampler = ClockSampler(local); sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_batches):
        run_batch()
    e1.record(); torch.cuda.synchronize()
    clocks = sampler.stop()
    sec = e0.elapsed_time(e1) / 1e3
    stats = eng.ctx.predict_stats(reset=True)
    n_done = n_batches * batch
    algo = sum(algorithmic_bytes_per_row(ms[nm]) for nm in names) * n_done
    mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
    rf = l1_pipe_roofline(stats["warp_steps"], stats["visits"], sec, eng.ctx.sm_count, mhz,
                          ncu_summary("predict_kernel_ncu_latest.json"), algo, None, "predict_kernel")
    return {"workload": f"configs[2]: {n_done:,} synthetic states x (play_model.xgb + pass/run/sack q10/q50/q90 = "
                        f"{sum(ms[nm].n_trees for nm in names)} trees), fmc_tree_predict on resident rows, batches of {batch:,}",
            "states_per_sec": n_done / sec, "ms": sec * 1e3, "gpu_launches": n_batches * len(names), "clocks": clocks,
            "roofline": rf}


# ----------------------------------------------------------------------------------------------
# outputs of the timed path (--dump-outputs): the same arguments give the same inputs, so that two builds
# can be compared output for output
# ----------------------------------------------------------------------------------------------
DUMP_GAMES = 1 << 20          # per-game scores: seeded sample of at most this many games (8 MiB)
DUMP_BOX_BYTES = 24 << 20     # per-game player boxes: the first games of that sample that fit in 24 MiB
DUMP_MATCHUPS = 64            # histograms: seeded sample of at most this many matchups (16 MiB)
DUMP_BYTES = 64 << 20
DUMP_COUNTERS = 15            # games .. hist_overflow: what the games did, not how the kernel scheduled them


def sample_ids(n: int, k: int):
    """Sorted, seeded sample of k of range(n); all of range(n) when n <= k."""
    import numpy as np
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(SEED).choice(n, size=k, replace=False))


def dump_outputs(path, scores, hist, counters, box):
    """Writes the device buffers of the last timed step as float32 / float64 .npy files under `path`."""
    import numpy as np
    import torch
    from fast_monte_carlo_b200 import native
    games = torch.from_numpy(sample_ids(scores.shape[0], DUMP_GAMES)).to(scores.device)
    words = scores[games].cpu().numpy().view(np.uint32)                  # points A | points B << 16
    out = {"scores": np.stack([words & 0xFFFF, words >> 16], axis=1).astype(np.float32),
           "hist": hist[torch.from_numpy(sample_ids(hist.shape[0], DUMP_MATCHUPS)).to(hist.device)].cpu().numpy()
           .astype(np.float64),
           "counters": counters[:DUMP_COUNTERS].cpu().numpy().astype(np.float64)}
    if box is not None:                                                  # int64 pairs = fmc_player_rec
        per_game = 2 * box.shape[2] * 6 * 8                              # float64 [2, slots, 6]
        rec = np.ascontiguousarray(box[games[:DUMP_BOX_BYTES // per_game]].cpu().numpy()).view(native.PLAYER_REC)[..., 0]
        out["players"] = native.unpack_player_box(rec)
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_BYTES, total
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_gpus = world

    from fast_monte_carlo_b200 import api, native, priors
    from fast_monte_carlo_b200.engine import Engine, MatchupSpec
    ms = load_models(args.stage2)
    eng = Engine(ms, device=local, stage2="booster" if args.stage2 == "synthetic" else "standin", memo=args.memo)
    if args.workload in ("slate", "season"):
        pairs, sp_df = slate_pairs() if args.workload == "slate" else season_pairs()
        spec = api.slate_specs(pairs, args.slate_games, sp_df, rank, world, shard=args.shard)
        G = sum(m.game_end - m.game_begin for m in spec)          # this rank's games per step
        total_games = len(pairs) * args.slate_games
    else:
        G = args.games
        g0, g1 = rank * G, (rank + 1) * G
        use = synthetic_usage(ms) if args.players else None
        spec = [MatchupSpec(KSU[0], ISU[0], KSU[1], ISU[1], G * world, g0, g1, 0, usage=use)]
        total_games = G * world
    n_m = len(spec)
    eng.set_matchups(spec)
    eng.ctx.packed_slots(0)          # forces the specialise + upload now, outside the timed region

    dev = torch.device("cuda", local)
    scores = torch.empty(G, dtype=torch.int32, device=dev)
    hist = torch.zeros((n_m, 2, native.HIST_BINS, native.HIST_BINS), dtype=torch.int32, device=dev)
    hist64 = torch.zeros((n_m, 2, native.HIST_BINS, native.HIST_BINS), dtype=torch.int64, device=dev)
    counters = torch.zeros(native.N_COUNTERS, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    box = None
    if args.workload == "matchup" and args.players and eng.n_slots:
        box = torch.zeros((G, 2, eng.n_slots, 2), dtype=torch.int64, device=dev)      # fmc_player_rec = 16 bytes

    def step():
        hist.zero_()
        counters.zero_()
        if box is not None:
            box.zero_()
        eng.ctx.simulate_device(seed=SEED, scores=scores.data_ptr(), hist=hist.data_ptr(), counters=counters.data_ptr(),
                                cuda_stream=stream.cuda_stream, players=box.data_ptr() if box is not None else 0)
        if world > 1:
            hist64.copy_(hist)
            dist.all_reduce(hist64)
            dist.all_reduce(counters)

    def timed(n_steps, n_warm):
        """n_warm untimed + n_steps timed steps, L2 flushed between steps; returns (total ms, per-step ms, counters of
        one step summed over ranks, clocks)."""
        for _ in range(n_warm):
            step()
            flush.zero_()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local)
        sampler.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_steps)]
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for i in range(n_steps):
            ev[i][0].record()
            step()
            ev[i][1].record()
            flush.zero_()
        k1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        clk = sampler.stop()
        tot = k0.elapsed_time(k1)
        per = [x.elapsed_time(y) for x, y in ev]
        c = counters.cpu().numpy()
        sc = {k: int(c[i]) for i, k in enumerate(native.COUNTER_NAMES)}
        t = torch.tensor([tot, sum(per)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), per, sc, clk

    # ---- headline: the engine as shipped (exact memo on unless --memo off) --------------------------------------
    total_ms, kernel_ms, step_ms, step_counters, clocks = timed(args.steps, max(args.warmup, 3))
    plays_step = step_counters["plays"]
    games_step = step_counters["games"]
    assert games_step == total_games, (games_step, total_games)
    value = plays_step * args.steps / (total_ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, scores, hist64 if world > 1 else hist, counters, box)

    # ---- end to end through the reference's Python entry point (FMC:1467-1521 simulate_matchup), host buffers ----
    # every sample: api.simulate_matchup -> fmc_simulate_host (tables specialised + uploaded when the pair changes,
    # kernel, per-game score words + histogram + counters copied back) -> the 2n-row sims_df the reference returns;
    # under torchrun every rank plays its slice of the 2n games (game_range) and the histograms are all-reduced
    e2e = None
    if args.workload == "matchup" and not args.players:
        sp_df = priors.load_sp_flex(priors.packaged_priors_path())
        A = priors.build_team_context_from_sp_flex(KSU[0], 2025, 1, sp_df)
        B = priors.build_team_context_from_sp_flex(ISU[0], 2025, 1, sp_df)
        samples, plays_e2e = [], 0
        sampler2 = ClockSampler(local)
        sampler2.start()
        for i in range(args.e2e_steps + 1):
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            df, _ = api.simulate_matchup(A, B, n=total_games // 2, seed=SEED, show_progress=False, engine=eng,
                                         game_range=(rank * G, (rank + 1) * G))
            h = torch.from_numpy(df.attrs["hist"].value.astype(np.int64))
            if world > 1:
                hd = h.to(dev)
                dist.all_reduce(hd)
                h = hd.cpu()
            dt = time.perf_counter() - t0
            assert len(df) == G and int(h.sum()) == total_games
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            pp = torch.tensor([df.attrs["counters"]["plays"]], dtype=torch.int64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dist.all_reduce(pp)
            if i == 0:
                first = float(tt[0])
                continue                                          # warm-up (also: first specialisation of the pair)
            samples.append(float(tt[0]))
            plays_e2e += int(pp[0])
            del df
        table_bytes = int(eng.ctx.packed_slots(0).sum()) * 8
        e2e = {"value": plays_e2e / sum(samples), "unit": UNIT,
               "h2d_bytes_per_step": 8 * n_m + 64, "d2h_bytes_per_step": G * 4 + 2 * native.HIST_BINS ** 2 * 4 + native.N_COUNTERS * 8,
               "step_seconds": samples, "first_call_seconds": first, "clocks": sampler2.stop(),
               "tables_h2d_bytes_first_call": table_bytes,
               "how": "api.simulate_matchup (the reference's Python entry point) -> fmc_simulate_host through ctypes: kernel, "
                      "per-game score words + histogram + counters copied to host, 2n-row sims_df built; host wall clock, "
                      "max over ranks.  The pair's tables are specialised + uploaded in the first (untimed) call and kept "
                      "while the pair stays the same (first_call_seconds includes it)"}
    else:
        # slates / player mode: the C-ABI host-buffer call (tables re-specialised + uploaded every sample)
        samples, plays_e2e = [], 0
        sampler2 = ClockSampler(local)
        sampler2.start()
        table_bytes = sum(int(eng.ctx.packed_slots(i).sum()) for i in range(n_m)) * 8
        for i in range(args.e2e_steps + 1):
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            eng.ctx.invalidate_tables()                            # every sample pays specialisation + upload again
            eng.set_matchups(spec)
            r = eng.simulate_host(SEED, want_scores=True, want_hist=True, want_players=box is not None)
            h = torch.from_numpy(r["hist"].astype(np.int64))
            if world > 1:
                hd = h.to(dev)
                dist.all_reduce(hd)
                h = hd.cpu()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            pp = torch.tensor([r["counters"]["plays"]], dtype=torch.int64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dist.all_reduce(pp)
            if i == 0:
                continue
            samples.append(float(tt[0]))
            plays_e2e += int(pp[0])
        e2e = {"value": plays_e2e / sum(samples) if samples else None, "unit": UNIT, "h2d_bytes_per_step": table_bytes + 200 + 8 * n_m,
               "d2h_bytes_per_step": G * 4 + int(np.prod(hist.shape)) * 4 + native.N_COUNTERS * 8 + (box.numel() * 8 if box is not None else 0),
               "step_seconds": samples, "clocks": sampler2.stop(), "tables_h2d_bytes_first_call": table_bytes,
               "how": "fmc_simulate_host through ctypes: kernel, per-game scores + histogram + counters (+ player box) copied "
                      "to host; host wall clock, max over ranks"}

    # ---- roofline of the tree walk: the same workload with the memo OFF, so that no tree work is hidden ----------
    roof = None
    memo_rec = {"mode": eng.memo, "probes_per_step": step_counters["memo_probes"], "hits_per_step": step_counters["memo_hits"],
                "hit_rate": step_counters["memo_hits"] / max(step_counters["memo_probes"], 1),
                "walked_requests_per_step": step_counters["requests"],
                "note": "exact rank-keyed memo (csrc/fmc_memo.hpp), cleared at the start of every step; results are "
                        "bit-identical with it off (tests/test_gpu_memo.py)"}
    if not args.no_roofline:
        eng.ctx.set_memo("off")
        r_total, r_kernel, r_steps, r_counters, r_clocks = timed(args.roofline_steps, 1)
        eng.ctx.set_memo(eng.memo)
        assert r_counters["plays"] == plays_step, "the memo must not change the games"
        if rank == 0:
            algo = step_algorithmic_bytes(ms, r_counters, args.stage2 == "synthetic") / world
            kern_s = (r_kernel / args.roofline_steps) / 1e3
            mhz = r_clocks.get("sm_mhz") or r_clocks.get("sm_max_mhz") or 1965.0
            roof = l1_pipe_roofline(r_counters["warp_steps"] / world, r_counters["visits"] / world, kern_s, eng.ctx.sm_count,
                                    mhz, ncu_summary(), algo, ncu_traffic(G), "fmc::sim_kernel (memo off)")
            roof["plays_per_sec_memo_off"] = r_counters["plays"] * args.roofline_steps / (r_total / 1e3)
            roof["step_ms"] = r_steps
            roof["clocks"] = r_clocks
            try:
                coh = eng.ctx.gather_probe_coherent(1 << 20, 256, 2000)
                coh2 = eng.ctx.gather_probe_coherent(1 << 20, 512, 2000)
                rnd_l1 = eng.ctx.gather_probe(64 << 10, 4000)
                rnd_l2 = eng.ctx.gather_probe(8 << 20, 1000)
                roof["gather_probe"] = {
                    "coherent_256B_gbs": coh["gbs"], "coherent_512B_gbs": coh2["gbs"], "random_l1_gbs": rnd_l1, "random_l2_gbs": rnd_l2,
                    "frac_of_coherent_probe": roof["gathered"]["gbs"] / coh["gbs"],
                    "note": "fmc_gather_probe_coherent: lanes of a warp gather 8-byte slots inside one 256 B / 512 B window "
                            "(1 MiB table, L2-resident, streamed through L1) like a tree level, nothing else per step; "
                            "the random-lane probes of round 1 are kept for reference (a walk's lanes are not random)"}
            except Exception as exc:                       # pragma: no cover
                print(f"gather probe failed: {exc}", file=sys.stderr)

    tree = None
    if rank == 0 and not args.no_tree_eval:
        try:
            tree = tree_eval_record(eng, load_models("standin") if args.stage2 != "standin" else ms, local,
                                    n_total=args.tree_states)
        except Exception as exc:                           # pragma: no cover
            print(f"tree_eval failed: {exc}", file=sys.stderr)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak" if args.workload == "matchup" else "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload(args, n_gpus),
            "games_per_sec": games_step * args.steps / (total_ms / 1e3),
            "plays_per_game": plays_step / games_step,
            "e2e": e2e,
            "gpu_launches": args.steps,
            "step_ms": step_ms,
            "clocks": clocks,
            "memo": memo_rec,
            "roofline": roof,
            "tree_eval": tree,
            "mix": {k: step_counters[k] for k in ("pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg", "punt", "go")},
            "device": eng.ctx.device_name,
        }
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(ms, args)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
