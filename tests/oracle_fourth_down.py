"""TEST INFRASTRUCTURE ONLY: the C oracle's games with a forced fourth-down choice at the start state
(tests/oracle_fourth_down.c, which compiles tests/oracle_overtime.c, tests/oracle_live.c and oracle/fmc_oracle.c unchanged
into itself).  Built on first use into a temporary directory (the tree may be read-only), with the flags of
oracle/Makefile.  Configurations, usage tables, draw streams and start states are those of oracle.c_oracle and
tests/oracle_live.py."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_live
import oracle_overtime
from oracle import c_oracle as co

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = (os.path.join(HERE, "oracle_fourth_down.c"),) + oracle_overtime.SOURCES
CHOICES = {None: 0, "policy": 0, "go": 1, "fg": 2, "punt": 3}     # include/fmc.h FMC_4TH_*

_lib = None
_loaded = None


def build() -> str:
    h = hashlib.sha1()
    for p in SOURCES:
        with open(p, "rb") as fh:
            h.update(fh.read())
    out = os.path.join(tempfile.gettempdir(), f"fmc_oracle_fourth_down_{h.hexdigest()[:16]}.so")
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


def simulate(cfg, n: int, *, start, choice=None, overtime: bool = False, max_periods: int = 16, snap_clock: int = 120,
             game0: int = 0, matchup: int = 0, stream: np.ndarray | None = None, seed: int = 0, trace: bool = False,
             threads: int = 0, usage=None, n_slots: int = 0):
    """oracle_overtime.simulate (overtime=True) or oracle_live.simulate (overtime=False, "periods" all 0) with the
    forced choice `choice` ("go" | "fg" | "punt" | None = the policy; one, or a list of one per start) at iteration 0."""
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
    st, k = oracle_live._starts(start, n)
    ch = list(choice) if isinstance(choice, (list, tuple)) else [choice] * k
    if len(ch) != k:
        raise ValueError("choice: one, or one per start")
    chc = np.ascontiguousarray([CHOICES[c] for c in ch], dtype=np.int32)
    p = oracle_live._p
    rc = L.fo_fourth_down_simulate(C.byref(cfg), usage, int(max(n_slots, 1)),
                                   p(players, C.c_double) if players is not None else None, st, C.c_long(k),
                                   C.c_long(n), C.c_long(game0), int(matchup), 0 if stream is not None else 1,
                                   p(stream, C.c_double) if stream is not None else None, C.c_uint64(seed),
                                   int(max_periods) if overtime else 0, int(snap_clock), p(chc, C.c_int),
                                   p(scores, C.c_int), p(iters, C.c_int), p(periods, C.c_int),
                                   p(tr, C.c_double) if trace else None, p(counters, C.c_long), int(threads))
    if rc != 0:
        raise ValueError(f"fo_fourth_down_simulate refused the arguments ({rc})")
    return dict(scores=scores, iters=iters, periods=periods, trace=tr,
                players=None if players is None else players[:, :, :n_slots, :],
                counters={name: int(counters[i]) for i, name in enumerate(co.COUNTER_NAMES)})


def branch_of(stream_u_go, state) -> str:
    """The branch the policy takes at a fourth-down `state` (offense / seconds / distance / yards_to_goal / score) for
    the draw u = stream_u_go in slot S_U_GO: handle_fourth's rule, with the oracle's fo_go_for_it_prob."""
    if float(stream_u_go) < _p_go(state):
        return "go"
    return "fg" if float(state.yards_to_goal) <= 38 else "punt"


def philox_u(seed: int, game: int, matchup: int, slot: int, iteration: int = 0) -> float:
    """The uniform draw in `slot` of (game, matchup entry, iteration) under Philox with key `seed`, as draw() forms it."""
    w = co.philox(((game & 0xFFFFFFFF), (game >> 32) & 0xFFFFFFFF, matchup, (iteration << 2) | (slot >> 2)),
                  (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    return (w[slot & 3] + 0.5) * (1.0 / 4294967296.0)


def philox_u_many(seed: int, games, matchup: int, slot: int, iteration: int = 0) -> np.ndarray:
    """philox_u for an array of game ids at once (Philox4x32-10 in numpy)."""
    g = np.asarray(games, dtype=np.uint64)
    mask = np.uint64(0xFFFFFFFF)
    c = [g & mask, g >> np.uint64(32), np.full_like(g, matchup), np.full_like(g, (iteration << 2) | (slot >> 2))]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & mask, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & mask]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & mask, (k1 + np.uint64(0xBB67AE85)) & mask
    return (c[slot & 3].astype(np.float64) + 0.5) * (1.0 / 4294967296.0)


def branches(u_go, state) -> np.ndarray:
    """branch_of for an array of S_U_GO draws: an array of "go" / "fg" / "punt"."""
    b = branch_of(2.0, state)
    return np.where(np.asarray(u_go) < _p_go(state), "go", b)


def _p_go(state) -> float:
    """min(1, 1.15 go_for_it_prob) of handle_fourth at `state`."""
    off = int(state.offense)
    sd = int(state.score[off]) - int(state.score[off ^ 1])
    return min(1.0, co.lib().fo_go_for_it_prob(float(state.yards_to_goal), float(state.distance), sd,
                                               int(state.seconds)) * 1.15)
