"""TEST INFRASTRUCTURE ONLY: the C oracle with a start record per game (tests/oracle_live.c, which compiles
oracle/fmc_oracle.c unchanged into itself).  Built on first use into a temporary directory (the tree may be read-only),
with the flags of oracle/Makefile.  Configurations, usage tables and draw streams are oracle.c_oracle's."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import c_oracle as co

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")
SOURCES = (os.path.join(HERE, "oracle_live.c"), os.path.join(ORACLE_DIR, "fmc_oracle.c"))
CFLAGS = ["-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wno-unused-function"]

_lib = None
_loaded = None


class FoStart(C.Structure):
    _fields_ = [("offense", C.c_int), ("sec", C.c_int), ("down", C.c_int), ("score", C.c_int * 2),
                ("dist", C.c_double), ("ytg", C.c_double)]


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def build() -> str:
    h = hashlib.sha1()
    for p in SOURCES:
        with open(p, "rb") as fh:
            h.update(fh.read())
    out = os.path.join(tempfile.gettempdir(), f"fmc_oracle_live_{h.hexdigest()[:16]}.so")
    if not os.path.exists(out):
        tmp = f"{out}.{os.getpid()}"
        base = ["gcc"] + CFLAGS + ["-I", ORACLE_DIR, "-o", tmp, SOURCES[0]]
        if subprocess.run(base[:1] + ["-fopenmp"] + base[1:] + ["-lm"]).returncode != 0:
            subprocess.check_call(base + ["-lm"])          # no libgomp: one thread
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def load_models(ms, play: str = "play_model") -> None:
    """The forests of `ms` into this library (its own copy of the oracle's model table), as c_oracle.load_models."""
    global _loaded
    if _loaded is ms:
        return
    L = lib()
    for name, f in ms.forests.items():
        if name in ("play_model", "play_binary") and name != play:
            continue
        mid = co.MODEL_IDS[name]
        base = np.ascontiguousarray(f.base_margin, dtype=np.float64)
        a = dict(feat=np.ascontiguousarray(f.feat, np.int32), thr=np.ascontiguousarray(f.thr, np.float32),
                 left=np.ascontiguousarray(f.left, np.int32), right=np.ascontiguousarray(f.right, np.int32),
                 dl=np.ascontiguousarray(f.default_left, np.uint8), value=np.ascontiguousarray(f.value, np.float64),
                 root=np.ascontiguousarray(f.tree_root, np.int32), out=np.ascontiguousarray(f.tree_out, np.int32))
        p = _p
        rc = L.fo_load_forest(
            mid, int(f.kind), int(f.n_outputs), int(f.n_features), int(f.num_base), int(f.n_num),
            int(bool(f.zero_is_missing)), p(base, C.c_double), C.c_double(float(f.scale)), int(f.n_nodes),
            p(a["feat"], C.c_int), p(a["thr"], C.c_float), p(a["left"], C.c_int), p(a["right"], C.c_int),
            p(a["dl"], C.c_ubyte), p(a["value"], C.c_double), int(f.n_trees), p(a["root"], C.c_int), p(a["out"], C.c_int))
        assert rc == 0, (name, rc)
        if f.scaler_cols is not None:
            cols = np.ascontiguousarray(f.scaler_cols, np.int32)
            mean = np.ascontiguousarray(f.scaler_mean, np.float64)
            sc = np.ascontiguousarray(f.scaler_scale, np.float64)
            L.fo_set_scaler(mid, int(cols.shape[0]), p(cols, C.c_int), p(mean, C.c_double), p(sc, C.c_double))
    _loaded = ms


def _starts(start, n: int):
    """A start state (any object with offense / seconds / down / distance / yards_to_goal / score, such as
    engine.GameState; offense by team index, -1 = the kickoff receiver) or a list of n of them -> (FoStart[k], k)."""
    states = list(start) if isinstance(start, (list, tuple)) else [start]
    if isinstance(start, (list, tuple)) and len(states) != n:
        raise ValueError("start: one state, or one per game")
    arr = (FoStart * len(states))()
    for i, st in enumerate(states):
        arr[i].offense = int(st.offense); arr[i].sec = int(st.seconds); arr[i].down = int(st.down)
        arr[i].score[0], arr[i].score[1] = int(st.score[0]), int(st.score[1])
        arr[i].dist = float(st.distance); arr[i].ytg = float(st.yards_to_goal)
    return arr, len(states)


def simulate(cfg, n: int, *, start, game0: int = 0, matchup: int = 0, stream: np.ndarray | None = None, seed: int = 0,
             trace: bool = False, threads: int = 0, usage=None, n_slots: int = 0):
    """c_oracle.simulate with every game starting from `start` (one state, or a list of one per game)."""
    L = lib()
    scores = np.zeros((n, 2), dtype=np.int32)
    iters = np.zeros(n, dtype=np.int32)
    tr = np.full((n, co.MAX_ITERS, co.TRACE_COLS), np.nan, dtype=np.float64) if trace else None
    counters = np.zeros(16, dtype=np.int64)
    if stream is not None:
        stream = np.ascontiguousarray(stream, dtype=np.float64)
        assert stream.shape == (n, co.MAX_ITERS, co.N_SLOTS), stream.shape
    players = None
    if usage is not None:
        players = np.zeros((n, 2, max(n_slots, 1), co.PLAYER_FIELDS), dtype=np.float64)
    st, k = _starts(start, n)
    p = _p
    rc = L.fo_live_simulate(C.byref(cfg), usage, int(max(n_slots, 1)), p(players, C.c_double) if players is not None else None,
                            st, C.c_long(k), C.c_long(n), C.c_long(game0), int(matchup), 0 if stream is not None else 1,
                            p(stream, C.c_double) if stream is not None else None, C.c_uint64(seed),
                            p(scores, C.c_int), p(iters, C.c_int), p(tr, C.c_double) if trace else None,
                            p(counters, C.c_long), int(threads))
    assert rc == 0, rc
    return dict(scores=scores, iters=iters, trace=tr, players=None if players is None else players[:, :, :n_slots, :],
                counters={name: int(counters[i]) for i, name in enumerate(co.COUNTER_NAMES)})
