"""TEST INFRASTRUCTURE ONLY: the C oracle's games started inside overtime, and its overtime games with the overtime
state of every iteration (tests/oracle_overtime_live.c, which compiles tests/oracle_fourth_down.c,
tests/oracle_overtime.c, tests/oracle_live.c and oracle/fmc_oracle.c unchanged into itself).  Built on first use into a
temporary directory (the tree may be read-only), with the flags of oracle/Makefile.  Configurations, usage tables, draw
streams and start states are those of oracle.c_oracle and tests/oracle_live.py."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_fourth_down
import oracle_live
from oracle import c_oracle as co

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = (os.path.join(HERE, "oracle_overtime_live.c"),) + oracle_fourth_down.SOURCES

_lib = None
_loaded = None


class FoOtStart(C.Structure):
    """include/fmc.h fmc_overtime_state"""
    _fields_ = [("period", C.c_int), ("possession", C.c_int), ("two_point_try", C.c_int), ("reserved", C.c_int)]


def build() -> str:
    h = hashlib.sha1()
    for p in SOURCES:
        with open(p, "rb") as fh:
            h.update(fh.read())
    out = os.path.join(tempfile.gettempdir(), f"fmc_oracle_overtime_live_{h.hexdigest()[:16]}.so")
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


def _outputs(n, stream, trace, states, usage, n_slots):
    out = dict(scores=np.zeros((n, 2), dtype=np.int32), iters=np.zeros(n, dtype=np.int32),
               periods=np.zeros(n, dtype=np.int32), counters=np.zeros(16, dtype=np.int64),
               trace=np.full((n, co.MAX_ITERS, co.TRACE_COLS), np.nan, dtype=np.float64) if trace else None,
               states=np.zeros((n, co.MAX_ITERS, 3), dtype=np.int32) if states else None,
               players=np.zeros((n, 2, max(n_slots, 1), co.PLAYER_FIELDS), dtype=np.float64) if usage is not None else None)
    if stream is not None:
        stream = np.ascontiguousarray(stream, dtype=np.float64)
        assert stream.shape == (n, co.MAX_ITERS, co.N_SLOTS), stream.shape
    return out, stream


def _result(out, n_slots):
    pl = out["players"]
    return dict(scores=out["scores"], iters=out["iters"], periods=out["periods"], trace=out["trace"],
                states=out["states"], players=None if pl is None else pl[:, :, :n_slots, :],
                counters={name: int(out["counters"][i]) for i, name in enumerate(co.COUNTER_NAMES)})


def _opt(a, t):
    return oracle_live._p(a, t) if a is not None else None


def simulate_states(cfg, n: int, *, start=None, max_periods: int = 16, snap_clock: int = 120, game0: int = 0,
                    matchup: int = 0, stream: np.ndarray | None = None, seed: int = 0, trace: bool = False,
                    threads: int = 0, usage=None, n_slots: int = 0):
    """oracle_overtime.simulate plus "states" int32[n][MAX_ITERS][3]: (period, possession 1 | 2, try 0 | 1) of every
    overtime iteration, zeros in regulation."""
    from fast_monte_carlo_b200.engine import KICKOFF
    out, stream = _outputs(n, stream, trace, True, usage, n_slots)
    st, k = oracle_live._starts(KICKOFF if start is None else start, n)
    rc = lib().fo_overtime_states_simulate(
        C.byref(cfg), usage, int(max(n_slots, 1)), _opt(out["players"], C.c_double), st, C.c_long(k), C.c_long(n),
        C.c_long(game0), int(matchup), 0 if stream is not None else 1, _opt(stream, C.c_double), C.c_uint64(seed),
        int(max_periods), int(snap_clock), _opt(out["scores"], C.c_int), _opt(out["iters"], C.c_int),
        _opt(out["periods"], C.c_int), _opt(out["trace"], C.c_double), _opt(out["states"], C.c_int),
        _opt(out["counters"], C.c_long), int(threads))
    assert rc == 0, rc
    return _result(out, n_slots)


def simulate_start(cfg, n: int, *, start, choice=None, max_periods: int = 16, snap_clock: int = 120, game0: int = 0,
                   matchup: int = 0, stream: np.ndarray | None = None, seed: int = 0, trace: bool = False,
                   states: bool = False, threads: int = 0, usage=None, n_slots: int = 0):
    """Games started inside overtime: `start` = one engine.GameState with an `overtime` (OvertimeState), or a list of one
    per game; `choice` ("go" | "fg" | "punt" | None, one or one per start) at the first snap.  Outputs as
    oracle_overtime.simulate's ("periods": the last period played), plus "states" with `states=True`."""
    out, stream = _outputs(n, stream, trace, states, usage, n_slots)
    st, k = oracle_live._starts(start, n)
    sts = list(start) if isinstance(start, (list, tuple)) else [start]
    ot = (FoOtStart * k)()
    for i, g in enumerate(sts):
        ot[i].period, ot[i].possession = int(g.overtime.period), int(g.overtime.possession)
        ot[i].two_point_try = int(bool(g.overtime.two_point_try))
    ch = list(choice) if isinstance(choice, (list, tuple)) else [choice] * k
    if len(ch) != k:
        raise ValueError("choice: one, or one per start")
    chc = np.ascontiguousarray([oracle_fourth_down.CHOICES[c] for c in ch], dtype=np.int32)
    rc = lib().fo_overtime_start_simulate(
        C.byref(cfg), usage, int(max(n_slots, 1)), _opt(out["players"], C.c_double), st, ot, oracle_live._p(chc, C.c_int),
        C.c_long(k), C.c_long(n), C.c_long(game0), int(matchup), 0 if stream is not None else 1,
        _opt(stream, C.c_double), C.c_uint64(seed), int(max_periods), int(snap_clock), _opt(out["scores"], C.c_int),
        _opt(out["iters"], C.c_int), _opt(out["periods"], C.c_int), _opt(out["trace"], C.c_double),
        _opt(out["states"], C.c_int), _opt(out["counters"], C.c_long), int(threads))
    if rc != 0:
        raise ValueError(f"fo_overtime_start_simulate refused the arguments ({rc})")
    return _result(out, n_slots)


def resume_states(res, game0: int = 0, rows=None):
    """Every overtime iteration of the games of a `simulate_states` result (with trace) as a start: a list of
    (game index, iteration, engine.GameState with its OvertimeState) in game order.  `rows`: the game indices to use
    (default all).  Iterations at down 5 or more are left out: the reference plays on after an incomplete pass or a sack
    on fourth down without a change of possession, but a start state's down is 1..4."""
    from fast_monte_carlo_b200.engine import GameState, OvertimeState
    out = []
    for i in (range(len(res["iters"])) if rows is None else rows):
        first = (game0 + int(i)) & 1
        for j in range(int(res["iters"][i])):
            k, p, t = (int(x) for x in res["states"][i, j])
            if k == 0:
                continue
            tr = res["trace"][i, j]
            if tr[1] > 4:
                continue
            off = first if tr[0] == 1.0 else first ^ 1
            sc = [0, 0]
            sc[first], sc[first ^ 1] = int(tr[3]), int(tr[4])
            out.append((int(i), j, GameState(offense=off, seconds=0, down=int(tr[1]), distance=float(tr[5]),
                                              yards_to_goal=float(tr[6]), score=(sc[0], sc[1]),
                                              overtime=OvertimeState(k, p, bool(t)))))
    return out
