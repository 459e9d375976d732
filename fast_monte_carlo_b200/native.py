"""ctypes binding of libfmc_b200.so (include/fmc.h).

The shared library is built in-tree by `__graft_entry__.build()` (or `python -m
fast_monte_carlo_b200.build`).  There is no CPU fallback: if the library is missing, or no sm_100
GPU is present, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import sys
from typing import Optional

import numpy as np

from . import outputs as _out
from .outputs import DRIVE_RESULTS, RACE_TARGETS, SEQ_BINS  # noqa: F401  (scoring-sequence layout, include/fmc.h)

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FMC_LIB_PATH") or os.path.join(HERE, "libfmc_b200.so")

N_MODELS = 7
MODEL_INDEX = {"pass_stage1": 0, "pass_stage2": 1, "pass_yards": 2, "run_yards": 3, "sack_yards": 4,
               "play_model": 5, "run_fumble": 6}
HIST_BINS = 128
N_COUNTERS = 32
N_SLOTS = 16
MAX_ITERS = 360
TRACE_COLS = 8
COUNTER_NAMES = ("games", "plays", "iters", "pass", "comp", "inc", "int", "sack", "run", "td", "fga", "fg",
                 "punt", "go", "hist_overflow", "rounds", "requests", "visits", "ph_overflow", "warp_steps",
                 "memo_probes", "memo_hits", "trips", "_23", "memo_hits_s1", "memo_hits_s2", "memo_hits_pq", "memo_hits_rq",
                 "memo_hits_sq", "memo_hits_pm", "ot_games", "ot_periods")
PH_YDS_BINS, PH_YDS_OFFSET, PH_CNT_BINS = 8192, 1000, 128
PH_BINS = PH_YDS_BINS + 5 * PH_CNT_BINS
N_SEGMENTS = 6                     # FMC_N_SEGMENTS: Q1, Q2, Q3, Q4, H1, H2
PERIOD_NONE = 0xFFFFFFFF           # FMC_PERIOD_NONE: a quarter end at or before the start state
# scoring sequence (include/fmc.h FMC_SEQ_NONE): the per-game words; the histogram layout is outputs'
SEQ_NONE = 0xFFFFFFFF              # FMC_SEQ_NONE: no score after the start state
SEQ_TD, SEQ_FG = 0, 1              # kind of a scoring play
OT_MAX_PERIODS = 16                # FMC_OT_MAX_PERIODS; the overtime histogram is [n_matchups][2][OT_MAX_PERIODS + 1][3]
OT_A, OT_B, OT_LEVEL = 0, 1, 2      # its last index: the final result


def seq_bin_next(team, kind, clock):
    """FMC_SEQ_BIN_NEXT: bin of a next score by `team` of `kind` snapped with `clock` (1..3600) seconds left"""
    return (team * 2 + kind) * _out.SEQ_MINUTES + (np.asarray(clock) - 1) // 60


class FmcError(RuntimeError):
    pass


class ForestDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("n_outputs", C.c_int32), ("n_features", C.c_int32), ("num_base", C.c_int32),
        ("n_num", C.c_int32), ("zero_is_missing", C.c_int32),
        ("base", C.c_double * 8), ("scale", C.c_double),
        ("n_nodes", C.c_int32), ("n_trees", C.c_int32),
        ("feat", C.POINTER(C.c_int32)), ("thr", C.POINTER(C.c_float)), ("left", C.POINTER(C.c_int32)),
        ("right", C.POINTER(C.c_int32)), ("default_left", C.POINTER(C.c_uint8)), ("value", C.POINTER(C.c_double)),
        ("tree_root", C.POINTER(C.c_int32)), ("tree_out", C.POINTER(C.c_int32)),
    ]


class Params(C.Structure):
    _fields_ = [
        ("policy", C.c_int32), ("sampler", C.c_int32), ("stage2_mode", C.c_int32), ("pass_class", C.c_int32),
        ("play_temp", C.c_double), ("qy_noise", C.c_double), ("stage2_standin", C.c_double * 3),
    ]


class Matchup(C.Structure):
    _fields_ = [
        ("sp", (C.c_double * 3) * 2), ("coach_col", C.c_int32 * 2),
        ("game_begin", C.c_uint64), ("game_end", C.c_uint64), ("out_offset", C.c_uint64),
    ]


class GameStateC(C.Structure):
    """fmc_game_state"""
    _fields_ = [
        ("offense", C.c_int32), ("seconds", C.c_int32), ("down", C.c_int32), ("score", C.c_int32 * 2),
        ("reserved", C.c_int32), ("distance", C.c_double), ("yards_to_goal", C.c_double),
    ]


class SimArgs(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("n_matchups", C.c_int32), ("reserved", C.c_int32),
        ("scores_dev", C.c_void_p), ("hist_dev", C.c_void_p), ("counters_dev", C.c_void_p),
        ("stream_dev", C.c_void_p), ("trace_dev", C.c_void_p), ("iters_dev", C.c_void_p),
        ("stream", C.c_void_p), ("players_dev", C.c_void_p), ("player_hist_dev", C.c_void_p),
    ]


class SegmentArgs(C.Structure):
    """fmc_segment_args"""
    _fields_ = [("period_scores_dev", C.c_void_p), ("segment_hist_dev", C.c_void_p)]


class SequenceArgs(C.Structure):
    """fmc_sequence_args"""
    _fields_ = [("sequence_dev", C.c_void_p), ("sequence_hist_dev", C.c_void_p)]


class OvertimeArgs(C.Structure):
    """fmc_overtime_args"""
    _fields_ = [("max_periods", C.c_int32), ("snap_clock", C.c_int32), ("ot_periods_dev", C.c_void_p),
                ("ot_hist_dev", C.c_void_p)]


MAX_USAGE = 32
ROLE_INDEX = {"pass": 0, "rush": 1, "rec": 2}
PLAYER_REC = np.dtype([("yds", "<f8"), ("counts", "<u8")])     # fmc_player_rec


class Usage(C.Structure):
    _fields_ = [("n", C.c_int32), ("reserved", C.c_int32), ("share", C.c_double * MAX_USAGE),
                ("slot", C.c_int32 * MAX_USAGE), ("col", (C.c_int32 * MAX_USAGE) * N_MODELS)]


class TeamUsageC(C.Structure):
    _fields_ = [("role", Usage * 3)]


class PlayerBox:
    """The per-game player box as the kernel wrote it (fmc_player_rec[games][2][n_slots]), unpacked on demand:
    a 10 M-game run holds a gigabyte of records, and a prop question reads one slot of it."""

    def __init__(self, rec: np.ndarray):
        self.rec = rec
        self.shape = rec.shape + (6,)

    def slot(self, team: int, slot: int) -> np.ndarray:
        """float64[games, 6] = yds, att|tgt, comp|rec, td, INT, sacks of one box line."""
        return unpack_player_box(self.rec[:, team, slot])

    def dense(self) -> np.ndarray:
        """float64[games, 2, n_slots, 6] (tests; small runs)."""
        return unpack_player_box(self.rec)


def box_slot(box, team: int, slot: int) -> np.ndarray:
    """[games, 6] of one box line from a PlayerBox or from a dense float64[games, 2, n_slots, 6] array."""
    return box.slot(team, slot) if isinstance(box, PlayerBox) else np.asarray(box)[:, team, slot, :]


def unpack_player_box(rec: np.ndarray) -> np.ndarray:
    """fmc_player_rec[...] -> float64[..., 6] = yds, att|tgt, comp|rec, td, INT, sacks (10-bit count fields)."""
    out = np.zeros(rec.shape + (6,), dtype=np.float64)
    out[..., 0] = rec["yds"]
    c = rec["counts"]
    for k in range(5):
        out[..., 1 + k] = ((c >> np.uint64(10 * k)) & np.uint64(0x3FF)).astype(np.float64)
    return out


_lib = None


def library_path() -> str:
    return LIB_PATH


def load_library():
    """dlopen libfmc_b200.so; raises FmcError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FmcError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.fmc_last_error.restype = C.c_char_p
    L.fmc_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.fmc_destroy.argtypes = [C.c_void_p]
    L.fmc_destroy.restype = None
    L.fmc_device_info.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_char_p, C.c_int32]
    L.fmc_load_forest.argtypes = [C.c_void_p, C.c_int32, C.POINTER(ForestDesc)]
    L.fmc_set_scaler.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                 C.POINTER(C.c_double)]
    L.fmc_set_active_columns.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]
    L.fmc_set_params.argtypes = [C.c_void_p, C.POINTER(Params)]
    L.fmc_set_matchups.argtypes = [C.c_void_p, C.c_int32, C.POINTER(Matchup)]
    L.fmc_simulate.argtypes = [C.c_void_p, C.POINTER(SimArgs)]
    L.fmc_set_memo.argtypes = [C.c_void_p, C.c_int32, C.c_uint64, C.c_int32, C.c_int32]
    L.fmc_simulate_host.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    L.fmc_simulate_players_host.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.fmc_simulate_segments.argtypes = [C.c_void_p, C.POINTER(SimArgs), C.POINTER(SegmentArgs)]
    L.fmc_simulate_segments_host.argtypes = [C.c_void_p, C.c_uint64] + [C.c_void_p] * 10
    L.fmc_simulate_markets.argtypes = [C.c_void_p, C.POINTER(SimArgs), C.POINTER(SegmentArgs), C.POINTER(SequenceArgs)]
    L.fmc_simulate_markets_host.argtypes = [C.c_void_p, C.c_uint64] + [C.c_void_p] * 12
    L.fmc_simulate_overtime.argtypes = [C.c_void_p, C.POINTER(SimArgs), C.POINTER(OvertimeArgs)]
    L.fmc_simulate_overtime_host.argtypes = ([C.c_void_p, C.c_uint64] + [C.c_void_p] * 8 + [C.c_int32, C.c_int32] +
                                             [C.c_void_p] * 2)
    L.fmc_set_usage.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]
    L.fmc_set_start_states.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    L.fmc_pack_forest_host_dyn.restype = C.c_int64
    L.fmc_pack_forest_host_dyn.argtypes = [C.POINTER(ForestDesc), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                           C.c_void_p, C.c_int64, C.c_void_p]
    L.fmc_tree_predict.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32,
                                   C.c_int32, C.c_void_p]
    L.fmc_tree_predict_host.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32,
                                        C.c_int32, C.c_int32]
    L.fmc_packed_slots.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
    L.fmc_sync.argtypes = [C.c_void_p]
    L.fmc_debug_errors.restype = C.c_int64
    L.fmc_debug_errors.argtypes = []
    L.fmc_gather_probe.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_double)]
    L.fmc_pack_forest_host.restype = C.c_int64
    L.fmc_pack_forest_host.argtypes = [C.POINTER(ForestDesc), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                       C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    L.fmc_gather_probe_coherent.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_double)]
    L.fmc_invalidate_tables.argtypes = [C.c_void_p]
    L.fmc_tree_predict_cols_host.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                             C.c_int32, C.c_int32]
    L.fmc_predict_stats.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_int32]
    L.fmc_memo_keys_host.restype = C.c_int64
    L.fmc_memo_keys_host.argtypes = [C.POINTER(ForestDesc), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = L
    return L


EXPORTED_SYMBOLS = (
    "fmc_last_error", "fmc_abi_version", "fmc_create", "fmc_destroy", "fmc_device_info", "fmc_load_forest",
    "fmc_set_scaler", "fmc_set_active_columns", "fmc_set_params", "fmc_set_matchups", "fmc_simulate",
    "fmc_simulate_host", "fmc_tree_predict", "fmc_tree_predict_host", "fmc_packed_slots", "fmc_sync",
    "fmc_gather_probe", "fmc_debug_errors",
    "fmc_pack_forest_host", "fmc_pack_forest_host_dyn", "fmc_set_usage", "fmc_simulate_players_host",
    "fmc_set_memo", "fmc_memo_keys_host", "fmc_gather_probe_coherent", "fmc_predict_stats", "fmc_invalidate_tables", "fmc_tree_predict_cols_host",
    "fmc_set_start_states", "fmc_simulate_segments", "fmc_simulate_segments_host",
    "fmc_simulate_markets", "fmc_simulate_markets_host", "fmc_simulate_overtime", "fmc_simulate_overtime_host",
)


def _check(rc: int) -> None:
    if rc != 0:
        raise FmcError(f"libfmc_b200 error {rc}: {load_library().fmc_last_error().decode()}")


def _ptr(a: Optional[np.ndarray], t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


def forest_desc(f) -> tuple:
    """(ForestDesc, keepalive arrays) for an artifacts.Forest."""
    arrs = dict(
        feat=np.ascontiguousarray(f.feat, np.int32), thr=np.ascontiguousarray(f.thr, np.float32),
        left=np.ascontiguousarray(f.left, np.int32), right=np.ascontiguousarray(f.right, np.int32),
        dl=np.ascontiguousarray(f.default_left, np.uint8), value=np.ascontiguousarray(f.value, np.float64),
        root=np.ascontiguousarray(f.tree_root, np.int32), out=np.ascontiguousarray(f.tree_out, np.int32))
    d = ForestDesc()
    d.kind = int(f.kind); d.n_outputs = int(f.n_outputs); d.n_features = int(f.n_features)
    d.num_base = int(f.num_base); d.n_num = int(f.n_num); d.zero_is_missing = int(bool(f.zero_is_missing))
    for k in range(f.n_outputs):
        d.base[k] = float(f.base_margin[k])
    d.scale = float(f.scale)
    d.n_nodes = int(f.n_nodes); d.n_trees = int(f.n_trees)
    d.feat = _ptr(arrs["feat"], C.c_int32); d.thr = _ptr(arrs["thr"], C.c_float)
    d.left = _ptr(arrs["left"], C.c_int32); d.right = _ptr(arrs["right"], C.c_int32)
    d.default_left = _ptr(arrs["dl"], C.c_uint8); d.value = _ptr(arrs["value"], C.c_double)
    d.tree_root = _ptr(arrs["root"], C.c_int32); d.tree_out = _ptr(arrs["out"], C.c_int32)
    return d, arrs


def pack_forest_host(f, *, mode: int, cols=(-1, -1), fold_values=None, tree_begin=0, tree_end=-1, dyn=None):
    """Host-only: run the specialiser/packer and return (slots u64[], stream u64[], consts u64[], info dict)
    -- the node table, the root stream and the constants side stream of csrc/fmc_pack.hpp.
    Evaluates nothing; used by the CPU tests and for table-size accounting."""
    L = load_library()
    d, keep = forest_desc(f)
    fv = np.zeros(17, dtype=np.float64)
    if fold_values is not None:
        fv[:] = fold_values
    ns = 0
    sc = sm = ss = None
    if getattr(f, "scaler_cols", None) is not None:
        sc = np.ascontiguousarray(f.scaler_cols, np.int32)
        sm = np.ascontiguousarray(f.scaler_mean, np.float64)
        ss = np.ascontiguousarray(f.scaler_scale, np.float64)
        ns = int(sc.shape[0])
    info = np.zeros(32, dtype=np.int32)
    cap_s = 16 * int(f.n_nodes) + 64                    # pass-through chains can outnumber the original nodes
    cap_r = int(f.n_trees) + 8 * int(f.n_outputs) + 64
    cap_c = 2 * int(f.n_trees) + 64
    slots = np.zeros(cap_s, dtype=np.uint64)
    stream = np.zeros(cap_r, dtype=np.uint64)
    consts = np.zeros(cap_c, dtype=np.uint64)
    if dyn is not None:      # player mode: {model column: feature row} read per request instead of folded
        dc = np.ascontiguousarray(list(dyn.keys()), np.int32)
        dr = np.ascontiguousarray(list(dyn.values()), np.int32)
        n = L.fmc_pack_forest_host_dyn(
            C.byref(d), int(mode), int(cols[0]), int(cols[1]), fv.ctypes.data, int(dc.shape[0]),
            dc.ctypes.data if dc.shape[0] else None, dr.ctypes.data if dr.shape[0] else None,
            slots.ctypes.data, cap_s, stream.ctypes.data, cap_r, consts.ctypes.data, cap_c, info.ctypes.data)
    else:
        n = L.fmc_pack_forest_host(
            C.byref(d), int(mode), int(cols[0]), int(cols[1]), fv.ctypes.data, ns,
            None if sc is None else sc.ctypes.data, None if sm is None else sm.ctypes.data,
            None if ss is None else ss.ctypes.data, int(tree_begin), int(tree_end),
            slots.ctypes.data, cap_s, stream.ctypes.data, cap_r, consts.ctypes.data, cap_c, info.ctypes.data)
    if n < 0:
        _check(int(n))
    if n > cap_s or int(info[5]) > cap_r or int(info[6]) > cap_c:
        raise FmcError("pack_forest_host: capacity estimate too small")
    meta = dict(rounds=int(info[0]), max_depth=int(info[1]), n_outputs=int(info[2]), ilp=int(info[3]),
                ninf_row=int(info[4]), constants=int(info[7]),
                stream_off=[int(x) for x in info[8:16]], n_groups=[int(x) for x in info[16:24]],
                consts_off=[int(x) for x in info[24:32]])
    return slots[:n].copy(), stream[:int(info[5])].copy(), consts[:int(info[6])].copy(), meta


def memo_keys_host(f, family: int, states: np.ndarray, *, cols=(-1, -1), fold_values=None):
    """Host-only: exact-memo keys of `states` ([n, 5] = down, distance, yardsToGoal, score_diff, seconds) on forest `f`
    specialised like the simulation specialises it.  Returns (keys uint64[n] | None when not memoisable, info dict)."""
    L = load_library()
    d, keep = forest_desc(f)
    fv = np.zeros(17, dtype=np.float64)
    if fold_values is not None:
        fv[:] = fold_values
    ns = 0
    sc = sm = ss = None
    if getattr(f, "scaler_cols", None) is not None:
        sc = np.ascontiguousarray(f.scaler_cols, np.int32)
        sm = np.ascontiguousarray(f.scaler_mean, np.float64)
        ss = np.ascontiguousarray(f.scaler_scale, np.float64)
        ns = int(sc.shape[0])
    st = np.ascontiguousarray(states, dtype=np.float64).reshape(-1, 5)
    keys = np.zeros(st.shape[0], dtype=np.uint64)
    info = np.zeros(4, dtype=np.int32)
    rc = L.fmc_memo_keys_host(C.byref(d), int(family), int(cols[0]), int(cols[1]), fv.ctypes.data, ns,
                              None if sc is None else sc.ctypes.data, None if sm is None else sm.ctypes.data,
                              None if ss is None else ss.ctypes.data, st.shape[0], st.ctypes.data, keys.ctypes.data,
                              info.ctypes.data)
    if rc < 0:
        _check(int(rc))
    meta = dict(memoisable=bool(info[0]), n_thr_distance=int(info[1]), n_thr_ytg=int(info[2]), constants=int(info[3]),
                why=L.fmc_last_error().decode() if rc == 0 else "")
    return (keys if rc == 1 else None), meta


class Context:
    """One engine context on one GPU (fmc_create / fmc_destroy)."""

    def __init__(self, device: int = 0):
        L = load_library()
        self._L = L
        h = C.c_void_p()
        _check(L.fmc_create(int(device), C.byref(h)))
        self._h = h
        self._keep = {}
        self.device = int(device)
        sm = C.c_int32(); smem = C.c_int32(); name = C.create_string_buffer(128)
        _check(L.fmc_device_info(h, C.byref(sm), C.byref(smem), name, 128))
        self.sm_count = int(sm.value)
        self.smem_per_block = int(smem.value)
        self.device_name = name.value.decode()
        self.n_matchups = 0
        self.n_slots = 0
        self.has_usage = False

    def close(self):
        if getattr(self, "_h", None):
            self._L.fmc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- models -------------------------------------------------------------------------------
    def load_forest(self, model_id: int, f) -> None:
        d, keep = forest_desc(f)
        _check(self._L.fmc_load_forest(self._h, int(model_id), C.byref(d)))
        if getattr(f, "scaler_cols", None) is not None:
            sc = np.ascontiguousarray(f.scaler_cols, np.int32)
            sm = np.ascontiguousarray(f.scaler_mean, np.float64)
            ss = np.ascontiguousarray(f.scaler_scale, np.float64)
            _check(self._L.fmc_set_scaler(self._h, int(model_id), int(sc.shape[0]), _ptr(sc, C.c_int32),
                                          _ptr(sm, C.c_double), _ptr(ss, C.c_double)))

    def set_active_columns(self, model_id: int, col0: int, col1: int = -1) -> None:
        _check(self._L.fmc_set_active_columns(self._h, int(model_id), int(col0), int(col1)))

    def set_params(self, *, policy=0, sampler=0, stage2_mode=0, play_temp=1.0, qy_noise=0.5,
                   stage2_standin=(0.78, 0.05, 0.17), pass_class=1) -> None:
        p = Params()
        p.policy = int(policy); p.sampler = int(sampler); p.stage2_mode = int(stage2_mode)
        p.pass_class = int(pass_class)
        p.play_temp = float(play_temp); p.qy_noise = float(qy_noise)
        for k in range(3):
            p.stage2_standin[k] = float(np.float32(stage2_standin[k]))   # inplace_predict returns float32
        _check(self._L.fmc_set_params(self._h, C.byref(p)))

    def set_matchups(self, matchups) -> None:
        """matchups: iterable of dict(sp=[[r,o,d],[r,o,d]], coach_col=(c0,c1), game_begin, game_end, out_offset)."""
        ms = list(matchups)
        arr = (Matchup * len(ms))()
        for i, m in enumerate(ms):
            for t in range(2):
                for k in range(3):
                    arr[i].sp[t][k] = float(m["sp"][t][k])
            cc = m.get("coach_col", (-1, -1))
            arr[i].coach_col[0] = int(cc[0]); arr[i].coach_col[1] = int(cc[1])
            arr[i].game_begin = int(m["game_begin"]); arr[i].game_end = int(m["game_end"])
            arr[i].out_offset = int(m.get("out_offset", 0))
        _check(self._L.fmc_set_matchups(self._h, len(ms), arr))
        self.n_matchups = len(ms)
        self.n_slots = 0
        self.has_usage = False
        self.total_games = max((int(m.get("out_offset", 0)) + int(m["game_end"]) - int(m["game_begin"])) for m in ms)

    def set_usage(self, teams, n_slots: int) -> None:
        """teams: [n_matchups][2] objects with .role[r].names/.share/.slot/.col (usage.TeamUsage), or None to
        return to the shipped configuration (every name "Unknown").  fmc_set_usage."""
        if teams is None:
            _check(self._L.fmc_set_usage(self._h, 0, None, 0))
            self.n_slots, self.has_usage = 0, False
            return
        flat = [tu for pair in teams for tu in pair]
        arr = (TeamUsageC * len(flat))()
        for i, tu in enumerate(flat):
            for rname, ri in ROLE_INDEX.items():
                ru = tu.role[rname]
                u = arr[i].role[ri]
                if len(ru.names) > MAX_USAGE:
                    raise ValueError("usage table too long")
                u.n = len(ru.names)
                for e in range(MAX_USAGE):
                    u.slot[e] = -1
                    for m in range(N_MODELS):
                        u.col[m][e] = -1
                for e in range(u.n):
                    u.share[e] = float(ru.share[e])
                    u.slot[e] = int(ru.slot[e])
                    for name, cols in ru.col.items():
                        u.col[MODEL_INDEX[name]][e] = int(cols[e])
        _check(self._L.fmc_set_usage(self._h, len(teams), C.cast(arr, C.c_void_p), int(n_slots)))
        self.n_slots, self.has_usage = int(n_slots), True

    def set_start_states(self, states) -> None:
        """fmc_set_start_states: `states` = one state per matchup entry of the last set_matchups (objects with offense,
        seconds, down, score, distance, yards_to_goal, such as engine.GameState; offense by team index), or None =
        every entry starts at the kickoff."""
        if states is None:
            _check(self._L.fmc_set_start_states(self._h, self.n_matchups, None))
            return
        st = list(states)
        arr = (GameStateC * max(len(st), 1))()
        for i, g in enumerate(st):
            arr[i].offense = int(g.offense); arr[i].seconds = int(g.seconds); arr[i].down = int(g.down)
            arr[i].score[0], arr[i].score[1] = int(g.score[0]), int(g.score[1])
            arr[i].distance = float(g.distance); arr[i].yards_to_goal = float(g.yards_to_goal)
        _check(self._L.fmc_set_start_states(self._h, len(st), C.cast(arr, C.c_void_p)))

    MEMO_MODES = {"off": 0, "on": 1, "persistent": 2}

    def set_memo(self, mode="on", max_bytes: int = 0, max_trips: int = 0, break_parked: int = 0) -> None:
        """Exact rank-keyed memo in front of the tree walk (fmc_set_memo): "off" | "on" (default, cleared at every
        launch) | "persistent" (kept between launches on the same tables).  Results never depend on it."""
        m = self.MEMO_MODES[mode] if isinstance(mode, str) else int(mode)
        _check(self._L.fmc_set_memo(self._h, m, int(max_bytes), int(max_trips), int(break_parked)))

    def packed_slots(self, matchup: int = 0) -> np.ndarray:
        out = np.zeros((N_MODELS, 2), dtype=np.int32)
        _check(self._L.fmc_packed_slots(self._h, int(matchup), _ptr(out, C.c_int32)))
        return out

    # -- simulation ------------------------------------------------------------------------------
    def simulate_device(self, *, seed: int, scores=0, hist=0, counters=0, stream_in=0, trace=0, iters=0,
                        cuda_stream=0, players=0, player_hist=0, period_scores=0, segment_hist=0, sequence=0,
                        sequence_hist=0, overtime=None, ot_periods=0, ot_hist=0) -> None:
        """Asynchronous launch on raw device pointers (ints; 0 = not requested).  `period_scores` (uint32[games][3]) and
        `segment_hist` (uint32[n_matchups][2][N_SEGMENTS][BINS][BINS], zeroed by the caller) are the per-period outputs,
        `sequence` (uint32[games][2]) and `sequence_hist` (uint32[n_matchups][2][SEQ_BINS], zeroed by the caller) the
        scoring-sequence outputs of fmc_simulate_markets; without any of them the call is fmc_simulate.  `overtime` (an
        engine.OvertimeRules) plays level games to a result (fmc_simulate_overtime), with the optional outputs
        `ot_periods` (uint8[games]) and `ot_hist` (uint32[n_matchups][2][OT_MAX_PERIODS + 1][3], zeroed by the caller);
        it has no period or sequence outputs."""
        a = SimArgs()
        a.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        a.n_matchups = self.n_matchups
        a.scores_dev = scores or None; a.hist_dev = hist or None; a.counters_dev = counters or None
        a.stream_dev = stream_in or None; a.trace_dev = trace or None; a.iters_dev = iters or None
        a.stream = cuda_stream or None
        a.players_dev = players or None      # fmc_player_rec[games][2][n_slots]
        a.player_hist_dev = player_hist or None   # uint32[n_matchups][2][n_slots][PH_BINS], zeroed by the caller
        if overtime is not None:
            if period_scores or segment_hist or sequence or sequence_hist:
                raise ValueError("overtime has no period or sequence outputs")
            ot = OvertimeArgs(int(overtime.max_periods), int(overtime.snap_clock), ot_periods or None, ot_hist or None)
            _check(self._L.fmc_simulate_overtime(self._h, C.byref(a), C.byref(ot)))
        elif ot_periods or ot_hist:
            raise ValueError("ot_periods / ot_hist need overtime")
        elif period_scores or segment_hist or sequence or sequence_hist:
            sg = SegmentArgs()
            sg.period_scores_dev = period_scores or None; sg.segment_hist_dev = segment_hist or None
            sq = SequenceArgs()
            sq.sequence_dev = sequence or None; sq.sequence_hist_dev = sequence_hist or None
            _check(self._L.fmc_simulate_markets(self._h, C.byref(a), C.byref(sg), C.byref(sq)))
        else:
            _check(self._L.fmc_simulate(self._h, C.byref(a)))

    def simulate_host(self, *, seed: int, want_scores=True, want_hist=True, stream: Optional[np.ndarray] = None,
                      want_trace=False, want_iters=False, want_players=False, want_player_hist=False,
                      want_period_scores=False, want_segments=False, want_sequence=False, want_sequence_hist=False,
                      overtime=None, want_ot_periods=False, want_ot_hist=False) -> dict:
        """End-to-end call with host buffers (fmc_simulate_host / fmc_simulate_players_host, and
        fmc_simulate_segments_host when `want_period_scores` / `want_segments` ask for the per-period outputs: "period_scores"
        uint32[games][3] score words at the end of Q1..Q3 (PERIOD_NONE before the start state), "segment_hist"
        uint32[n_matchups][2][N_SEGMENTS][BINS][BINS]), and fmc_simulate_markets_host when `want_sequence` /
        `want_sequence_hist` ask for the scoring-sequence outputs: "sequence" uint32[games][2] (next-score word, drive-result
        word) and "sequence_hist" uint32[n_matchups][2][SEQ_BINS].  With `overtime` (an engine.OvertimeRules) level games
        are played to a result (fmc_simulate_overtime_host); `want_ot_periods` / `want_ot_hist` add "ot_periods"
        uint8[games] and "ot_hist" uint32[n_matchups][2][OT_MAX_PERIODS + 1][3].  Overtime has no period or sequence
        outputs."""
        n = self.total_games
        scores = np.zeros(n, dtype=np.uint32) if want_scores else None
        hist = np.zeros((self.n_matchups, 2, HIST_BINS, HIST_BINS), dtype=np.uint32) if want_hist else None
        counters = np.zeros(N_COUNTERS, dtype=np.uint64)
        trace = np.zeros((n, MAX_ITERS, TRACE_COLS), dtype=np.float64) if want_trace else None
        iters = np.zeros(n, dtype=np.uint16) if want_iters else None
        if stream is not None:
            stream = np.ascontiguousarray(stream, dtype=np.float64)
            if stream.shape != (n, MAX_ITERS, N_SLOTS):
                raise ValueError(f"stream must be [{n},{MAX_ITERS},{N_SLOTS}]")
        vp = lambda a: None if a is None else a.ctypes.data
        players = phist = None
        period = np.zeros((n, 3), dtype=np.uint32) if want_period_scores else None
        seg = (np.zeros((self.n_matchups, 2, N_SEGMENTS, HIST_BINS, HIST_BINS), dtype=np.uint32) if want_segments else None)
        if want_players or want_player_hist:
            if not self.has_usage:
                raise FmcError("want_players / want_player_hist need set_usage")
            if want_players:
                players = np.zeros((n, 2, max(self.n_slots, 1)), dtype=PLAYER_REC)
            if want_player_hist:
                phist = np.zeros((self.n_matchups, 2, max(self.n_slots, 1), PH_BINS), dtype=np.uint32)
        seq = np.zeros((n, 2), dtype=np.uint32) if want_sequence else None
        seqh = np.zeros((self.n_matchups, 2, SEQ_BINS), dtype=np.uint32) if want_sequence_hist else None
        hooks = period is not None or seg is not None or seq is not None or seqh is not None
        if overtime is None and (want_ot_periods or want_ot_hist):
            raise ValueError("want_ot_periods / want_ot_hist need overtime")
        otp = np.zeros(n, dtype=np.uint8) if want_ot_periods else None
        oth = np.zeros((self.n_matchups, 2, OT_MAX_PERIODS + 1, 3), dtype=np.uint32) if want_ot_hist else None
        if overtime is not None:
            if hooks:
                raise ValueError("overtime has no period or sequence outputs")
            _check(self._L.fmc_simulate_overtime_host(
                self._h, int(seed) & 0xFFFFFFFFFFFFFFFF, vp(scores), vp(hist), vp(counters), vp(stream), vp(trace), vp(iters),
                players.ctypes.data if (players is not None and self.n_slots) else None,
                phist.ctypes.data if (phist is not None and self.n_slots) else None,
                int(overtime.max_periods), int(overtime.snap_clock), vp(otp), vp(oth)))
        elif hooks:
            _check(self._L.fmc_simulate_markets_host(
                self._h, int(seed) & 0xFFFFFFFFFFFFFFFF, vp(scores), vp(hist), vp(counters), vp(stream), vp(trace), vp(iters),
                players.ctypes.data if (players is not None and self.n_slots) else None,
                phist.ctypes.data if (phist is not None and self.n_slots) else None, vp(period), vp(seg), vp(seq), vp(seqh)))
        elif players is not None or phist is not None:
            _check(self._L.fmc_simulate_players_host(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF, vp(scores), vp(hist),
                                                     vp(counters), vp(stream), vp(trace), vp(iters),
                                                     players.ctypes.data if (players is not None and self.n_slots) else None,
                                                     phist.ctypes.data if (phist is not None and self.n_slots) else None))
        else:
            _check(self._L.fmc_simulate_host(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF, vp(scores), vp(hist), vp(counters),
                                             vp(stream), vp(trace), vp(iters)))
        out = dict(counters={k: int(counters[i]) for i, k in enumerate(COUNTER_NAMES)})
        if players is not None:
            out["players"] = PlayerBox(players[:, :, :self.n_slots])
        if phist is not None:
            out["player_hist"] = phist[:, :, :self.n_slots]
        if scores is not None:
            # score word = points A | points B << 16: on a little-endian host the uint16 view IS the [n, 2] table
            out["scores"] = (scores.view(np.uint16).reshape(n, 2).astype(np.int32) if sys.byteorder == "little" else
                             np.stack([(scores & 0xFFFF).astype(np.int32), (scores >> 16).astype(np.int32)], axis=1))
        if hist is not None:
            out["hist"] = hist
        if trace is not None:
            out["trace"] = trace
        if iters is not None:
            out["iters"] = iters.astype(np.int32)
        if period is not None:
            out["period_scores"] = period
        if seg is not None:
            out["segment_hist"] = seg
        if seq is not None:
            out["sequence"] = seq
        if seqh is not None:
            out["sequence_hist"] = seqh
        if otp is not None:
            out["ot_periods"] = otp
        if oth is not None:
            out["ot_hist"] = oth
        return out

    # -- tree prediction -------------------------------------------------------------------------------
    def tree_predict_host(self, model_id: int, rows: np.ndarray, n_outputs: int, tree_begin=0, tree_end=-1,
                          coach_col=-1) -> np.ndarray:
        rows = np.asarray(rows, dtype=np.float64)
        full = np.zeros((rows.shape[0], 17), dtype=np.float64)
        full[:, :rows.shape[1]] = rows
        out = np.zeros((rows.shape[0], n_outputs), dtype=np.float64)
        if rows.shape[0]:
            _check(self._L.fmc_tree_predict_host(self._h, int(model_id), full.ctypes.data, rows.shape[0],
                                                 out.ctypes.data, int(tree_begin), int(tree_end), int(coach_col)))
        return out

    def tree_predict_cols_host(self, model_id: int, rows: np.ndarray, hot_cols: np.ndarray, n_outputs: int, tree_begin=0,
                               tree_end=-1) -> np.ndarray:
        """Raw margins of rows that carry their own names: hot_cols int32 [n, 2] = the one-hot columns of each row."""
        rows = np.asarray(rows, dtype=np.float64)
        full = np.zeros((rows.shape[0], 17), dtype=np.float64)
        full[:, :rows.shape[1]] = rows
        hc = np.ascontiguousarray(hot_cols, dtype=np.int32).reshape(rows.shape[0], 2)
        out = np.zeros((rows.shape[0], n_outputs), dtype=np.float64)
        if rows.shape[0]:
            _check(self._L.fmc_tree_predict_cols_host(self._h, int(model_id), full.ctypes.data, rows.shape[0], hc.ctypes.data,
                                                      out.ctypes.data, int(tree_begin), int(tree_end)))
        return out

    def tree_predict_device(self, model_id: int, rows_ptr: int, n: int, out_ptr: int, tree_begin=0, tree_end=-1,
                            coach_col=-1, cuda_stream=0) -> None:
        _check(self._L.fmc_tree_predict(self._h, int(model_id), rows_ptr, int(n), out_ptr, int(tree_begin),
                                        int(tree_end), int(coach_col), cuda_stream or None))

    def predict_stats(self, reset: bool = True) -> dict:
        """Node gathers of the tree_predict launches since the last reset (fmc_predict_stats)."""
        out = (C.c_uint64 * 2)()
        _check(self._L.fmc_predict_stats(self._h, out, 1 if reset else 0))
        return dict(warp_steps=int(out[0]), visits=int(out[1]))

    def invalidate_tables(self) -> None:
        _check(self._L.fmc_invalidate_tables(self._h))

    def sync(self) -> None:
        _check(self._L.fmc_sync(self._h))

    def gather_probe_coherent(self, table_bytes: int, window_bytes: int = 256, iters: int = 2000) -> dict:
        """Warp-coherent gather rate (lanes of a warp inside one window, like a tree level): the walk's denominator."""
        out = (C.c_double * 3)()
        _check(self._L.fmc_gather_probe_coherent(self._h, int(table_bytes), int(window_bytes), int(iters), out))
        return dict(gbs=float(out[0]), warp_gathers_per_s=float(out[1]), ms=float(out[2]))

    def gather_probe(self, table_bytes: int, iters: int = 2000) -> float:
        """GB/s of dependent 8-byte gathers through a cache-resident table (roofline denominator)."""
        v = C.c_double()
        _check(self._L.fmc_gather_probe(self._h, int(table_bytes), int(iters), C.byref(v)))
        return float(v.value)
