"""TEST INFRASTRUCTURE ONLY: the C oracle's games played to a result under college overtime rules
(tests/oracle_overtime.c, which compiles tests/oracle_live.c and oracle/fmc_oracle.c unchanged into itself).  Built on
first use into a temporary directory (the tree may be read-only), with the flags of oracle/Makefile.  Configurations,
usage tables, draw streams and start states are those of oracle.c_oracle and tests/oracle_live.py."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_live
from oracle import c_oracle as co

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = (os.path.join(HERE, "oracle_overtime.c"),) + oracle_live.SOURCES

_lib = None
_loaded = None


def build() -> str:
    h = hashlib.sha1()
    for p in SOURCES:
        with open(p, "rb") as fh:
            h.update(fh.read())
    out = os.path.join(tempfile.gettempdir(), f"fmc_oracle_overtime_{h.hexdigest()[:16]}.so")
    if not os.path.exists(out):
        tmp = f"{out}.{os.getpid()}"
        base = ["gcc"] + oracle_live.CFLAGS + ["-I", oracle_live.ORACLE_DIR, "-I", HERE, "-o", tmp, SOURCES[0]]
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
    """The forests of `ms` into this library's own copy of the oracle's model table, as oracle_live.load_models."""
    global _loaded
    if _loaded is ms:
        return
    saved = oracle_live._lib, oracle_live._loaded
    try:
        oracle_live._lib, oracle_live._loaded = lib(), None
        oracle_live.load_models(ms, play)
    finally:
        oracle_live._lib, oracle_live._loaded = saved
    _loaded = ms


def simulate(cfg, n: int, *, start=None, max_periods: int = 16, snap_clock: int = 120, game0: int = 0, matchup: int = 0,
             stream: np.ndarray | None = None, seed: int = 0, trace: bool = False, threads: int = 0, usage=None,
             n_slots: int = 0):
    """oracle_live.simulate with overtime (start=None: the kickoff): the same outputs plus "periods" int32[n], the
    overtime periods of each game (0: decided in regulation)."""
    from fast_monte_carlo_b200.engine import KICKOFF
    L = lib()
    scores = np.zeros((n, 2), dtype=np.int32)
    iters = np.zeros(n, dtype=np.int32)
    periods = np.zeros(n, dtype=np.int32)
    tr = np.full((n, co.MAX_ITERS, co.TRACE_COLS), np.nan, dtype=np.float64) if trace else None
    counters = np.zeros(16, dtype=np.int64)
    if stream is not None:
        stream = np.ascontiguousarray(stream, dtype=np.float64)
        assert stream.shape == (n, co.MAX_ITERS, co.N_SLOTS), stream.shape
    players = None
    if usage is not None:
        players = np.zeros((n, 2, max(n_slots, 1), co.PLAYER_FIELDS), dtype=np.float64)
    st, k = oracle_live._starts(KICKOFF if start is None else start, n)
    p = oracle_live._p
    rc = L.fo_overtime_simulate(C.byref(cfg), usage, int(max(n_slots, 1)),
                                p(players, C.c_double) if players is not None else None, st, C.c_long(k), C.c_long(n),
                                C.c_long(game0), int(matchup), 0 if stream is not None else 1,
                                p(stream, C.c_double) if stream is not None else None, C.c_uint64(seed),
                                int(max_periods), int(snap_clock), p(scores, C.c_int), p(iters, C.c_int),
                                p(periods, C.c_int), p(tr, C.c_double) if trace else None, p(counters, C.c_long),
                                int(threads))
    assert rc == 0, rc
    return dict(scores=scores, iters=iters, periods=periods, trace=tr,
                players=None if players is None else players[:, :, :n_slots, :],
                counters={name: int(counters[i]) for i, name in enumerate(co.COUNTER_NAMES)})
