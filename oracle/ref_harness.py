"""ORACLE (test infrastructure only; needs the original project in the directory named by FMC_REFERENCE_DIR).

Imports the UNMODIFIED reference module fast_monte_carlo_cfb.py with
  * `xgboost` replaced by oracle/fake_xgboost.py (xgboost is not installed here),
  * the two scikit-learn 1.5.2 -> 1.9 unpickling shims (SURVEY 8c),
  * a scratch working directory that symlinks the reference artifacts and adds the one-line
    pass_stage2_classes.csv the reference reads at import (FMC:655),
and drives `simulate_game` (FMC:1428) with an injected draw stream instead of NumPy's PCG64.
Everything else -- state machine, samplers, special teams, the sklearn pipelines -- is the
reference's own code and objects.  Used by tests/golden/make_golden.py to produce the committed
golden trajectories.

Injected-stream protocol (ours; SURVEY Appendix B lists the draw sites): one record of 16 float64
slots per (game, loop iteration of FMC:1447).  Uniform slots hold u in [0,1), normal slots hold a
ready standard normal z.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import tempfile

import numpy as np

REFERENCE_DIR = os.environ.get("FMC_REFERENCE_DIR", "")     # the original project's directory; "" = not available

# slot layout (grouped so that one Philox4x32 call serves the common case)
SLOT = dict(U_call=0, U_comp=1, Z_yards=2, U_ex=3,
            U_boost=4, U_fin=5, U_s2=6, Z_int=7,
            U_go=8, U_fg=9, Z_gross=10, Z_ret=11,
            U_tb=12, U_p1=13, U_wr=14, U_yq=15)   # U_p1: passer (pass) or rusher (run); U_yq: sim_helpers sampler
N_SLOTS = 16
MAX_ITERS = 360      # 3600 s / the 10 s minimum clock cost of an iteration (FMC:35)

# (function name, line in fast_monte_carlo_cfb.py) -> slot; `choice` is resolved one frame further up
_SITES = {
    ("handle_fourth", 1395): "U_go",
    ("attempt_fg", 871): "U_fg",
    ("attempt_punt", 881): "Z_gross",
    ("attempt_punt", 882): "Z_ret",
    ("attempt_punt", 889): "U_tb",
    ("simulate_play", 1049): "U_call",
    ("simulate_play", 1157): "U_s2",
    ("simulate_play", 1158): "U_s2",
    ("sample_qb", 627): "U_p1",
    ("sample_rusher", 631): "U_p1",
    ("sample_target", 635): "U_wr",
    ("simulate_play", 1089): "U_comp",
    ("simulate_play", 1096): "U_ex",
    ("simulate_play", 1222): "U_ex",
    ("simulate_play", 1098): "U_boost",
    ("simulate_play", 1223): "U_boost",
    ("simulate_play", 1102): "U_fin",
    ("simulate_play", 1227): "U_fin",
    ("simulate_play", 1194): "Z_int",
    ("sample_pass_yards", 827): "Z_yards",
    ("sample_rush_yards", 839): "Z_yards",
    ("sample_sack_loss", 851): "Z_yards",
}


class InjectedRNG:
    """Duck-types the four numpy.random.Generator methods the reference calls (FMC:64 `RNG`)."""

    def __init__(self, stream: np.ndarray):
        self.stream = stream          # [MAX_ITERS, 16] float64 for ONE game
        self.it = -1
        self.used = []

    def begin_iteration(self):
        self.it += 1
        if self.it >= self.stream.shape[0]:
            raise RuntimeError("injected stream exhausted")

    def _slot(self, depth=2):
        f = sys._getframe(depth)
        key = (f.f_code.co_name, f.f_lineno)
        if key[0] == "sample_categorical":
            g = f.f_back
            key = (g.f_code.co_name, g.f_lineno)
        name = _SITES.get(key)
        if name is None:
            raise KeyError(f"unmapped RNG call site {key}")
        self.used.append((self.it, name))
        return float(self.stream[self.it, SLOT[name]])

    def random(self):
        return self._slot()

    def normal(self, loc=0.0, scale=1.0):
        return loc + scale * self._slot()

    def uniform(self, low=0.0, high=1.0):
        return low + (high - low) * self._slot()

    def choice(self, n, p=None):
        u = self._slot()
        cdf = np.cumsum(np.asarray(p, dtype=np.float64))
        cdf /= cdf[-1]
        return int(np.searchsorted(cdf, u, side="right"))


class _NoCache(dict):
    """Memo cache that never hits: parity is defined on cache-off semantics (SURVEY 7 'hard parts')."""

    def get(self, k, default=None):
        return default


_MOD = None


def load_reference(cache_off: bool = True):
    """Import the reference module once (fake xgboost, shims, scratch cwd)."""
    global _MOD
    if _MOD is not None:
        return _MOD
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.dirname(here))
    from fast_monte_carlo_b200.artifacts import _install_sklearn_shims
    _install_sklearn_shims()
    import oracle.fake_xgboost as fx
    sys.modules["xgboost"] = fx
    scratch = tempfile.mkdtemp(prefix="fmc_ref_")
    for fn in os.listdir(REFERENCE_DIR):
        if not fn.endswith(".py"):
            os.symlink(os.path.join(REFERENCE_DIR, fn), os.path.join(scratch, fn))
    with open(os.path.join(scratch, "pass_stage2_classes.csv"), "w") as f:
        f.write("incomplete\nintercepted\nsack\n")
    old = os.getcwd()
    os.chdir(scratch)
    try:
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            spec = importlib.util.spec_from_file_location(
                "fast_monte_carlo_cfb_reference", os.path.join(REFERENCE_DIR, "fast_monte_carlo_cfb.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
    finally:
        os.chdir(old)
    src = open(os.path.join(REFERENCE_DIR, "fast_monte_carlo_cfb.py")).read().splitlines()
    for (fn, line), name in _SITES.items():
        txt = src[line - 1]
        assert ("RNG." in txt) or ("sample_categorical" in txt) or ('p2["sack"]' in txt), (fn, line, txt)
    if cache_off:
        for nm in ("_PASS1_CACHE", "_PASS2_CACHE", "_PY_CACHE", "_RY_CACHE", "_SY_CACHE", "_PLAY_CACHE"):
            setattr(mod, nm, _NoCache())
    mod._scratch_dir = scratch
    _MOD = mod
    return mod


def team_context(mod, name: str, sp_csv: str = os.path.join(REFERENCE_DIR, "PregameSPPlus2025_1.csv")):
    sp = mod.load_sp_flex(sp_csv)
    return mod.build_team_context_from_sp_flex(name, 2025, 1, sp)


def run_game_injected(mod, off_ctx, def_ctx, stream: np.ndarray, trace: bool = True):
    """Run the reference's simulate_game(off, def) on one injected stream.

    Returns (result dict, trace array [n_iters, 8] float64):
      columns = offense_is_first, down, seconds_remaining, score_first, score_second,
                distance, yards_to_goal, going_for_it   -- sampled at the START of each iteration.
    """
    rng = InjectedRNG(stream)
    mod.RNG = rng
    rows = []
    orig = mod.__dict__.get("_orig_handle_fourth") or mod.handle_fourth
    mod._orig_handle_fourth = orig
    first = off_ctx.name

    def wrapped(gs, stats, score):
        rng.begin_iteration()
        if trace:
            rows.append((1.0 if gs.offense.name == first else 0.0, gs.down, gs.seconds_remaining,
                         score[first], score[def_ctx.name], gs.distance, gs.yards_to_goal,
                         1.0 if gs.going_for_it else 0.0))
        return orig(gs, stats, score)

    mod.handle_fourth = wrapped
    try:
        res = mod.simulate_game(off_ctx, def_ctx, seed=None)
    finally:
        mod.handle_fourth = orig
    return res, np.asarray(rows, dtype=np.float64), rng.used
