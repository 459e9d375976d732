"""TEST INFRASTRUCTURE ONLY: the scoring sequence of the C oracle's games (tests/oracle_sequence.c, which compiles
tests/oracle_live.c and oracle/fmc_oracle.c unchanged into itself).  Built on first use into a temporary directory (the
tree may be read-only), with the flags of oracle/Makefile.  Configurations, usage tables, draw streams and start states
are those of oracle.c_oracle and tests/oracle_live.py."""
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
SOURCES = (os.path.join(HERE, "oracle_sequence.c"),) + oracle_live.SOURCES
RACE_SETTLED = -1                 # race result of a target either team had reached at the start state

_lib = None
_loaded = None


def build() -> str:
    h = hashlib.sha1()
    for p in SOURCES:
        with open(p, "rb") as fh:
            h.update(fh.read())
    out = os.path.join(tempfile.gettempdir(), f"fmc_oracle_sequence_{h.hexdigest()[:16]}.so")
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


def simulate(cfg, n: int, *, start, game0: int = 0, matchup: int = 0, stream: np.ndarray | None = None, seed: int = 0,
             threads: int = 0, usage=None):
    """Games [game0, game0 + n) of one matchup from `start` (one state, or one per game; see oracle_live.simulate):
    {"scores" int32[n][2], "iters", "sequence" uint32[n][2] (next-score word, drive-result word, include/fmc.h),
    "race" int8[n][5] (0 A, 1 B, 2 neither, RACE_SETTLED per target of native.RACE_TARGETS)}."""
    L = lib()
    scores = np.zeros((n, 2), dtype=np.int32)
    iters = np.zeros(n, dtype=np.int32)
    seq = np.zeros((n, 2), dtype=np.uint32)
    race = np.zeros((n, 5), dtype=np.int8)
    if stream is not None:
        stream = np.ascontiguousarray(stream, dtype=np.float64)
        assert stream.shape == (n, co.MAX_ITERS, co.N_SLOTS), stream.shape
    st, k = oracle_live._starts(start, n)
    p = oracle_live._p
    rc = L.fo_sequence_simulate(C.byref(cfg), usage, st, C.c_long(k), C.c_long(n), C.c_long(game0), int(matchup),
                                0 if stream is not None else 1, p(stream, C.c_double) if stream is not None else None,
                                C.c_uint64(seed), p(scores, C.c_int), p(iters, C.c_int), p(seq, C.c_uint32),
                                p(race, C.c_byte), int(threads))
    assert rc == 0, rc
    return dict(scores=scores, iters=iters, sequence=seq, race=race)
