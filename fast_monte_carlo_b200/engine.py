"""Host-side engine: owns one GPU context, the compiled forests and the matchup table.

Mirrors the reference's module-level state: the models loaded at import (FMC:641-668), the play
policy switch (FMC:46, 326-328) and the per-process worker contexts (`_init_pool`, FMC:1306-1319),
but as an object so that several engines (one per GPU / rank) can coexist.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import artifacts as art
from . import native

# FMC:55-61
HEAD_COACH_MAP = {
    "Kansas State": "Chris Klieman",
    "Iowa State": "Matt Campbell",
    "Kansas": "Lance Leipold",
    "Fresno State": "Matt Entz",
}

SIM_MODELS = ("pass_stage1", "pass_stage2", "pass_yards", "run_yards", "sack_yards", "play_model")


# fmc_game_state.fourth_down (include/fmc.h FMC_4TH_POLICY)
FOURTH_DOWN_POLICY, FOURTH_DOWN_GO, FOURTH_DOWN_FG, FOURTH_DOWN_PUNT = 0, 1, 2, 3


@dataclass(frozen=True)
class OvertimeState:
    """Where in overtime a start state is (include/fmc.h fmc_overtime_state): `period` 1..16, `possession` 1 or 2 (the
    first or second possession of the period), `two_point_try` (the snap is a two-point try: always from period 3, after
    a touchdown in period 2, never in period 1)."""
    period: int
    possession: int = 1
    two_point_try: bool = False

    def __post_init__(self):
        if not (isinstance(self.period, (int, np.integer)) and 1 <= self.period <= native.OT_MAX_PERIODS):
            raise ValueError(f"OvertimeState.period must be an integer in 1..{native.OT_MAX_PERIODS}")
        if self.possession not in (1, 2):
            raise ValueError("OvertimeState.possession must be 1 or 2")
        if self.two_point_try not in (False, True):
            raise ValueError("OvertimeState.two_point_try must be a bool")
        if self.two_point_try and self.period == 1:
            raise ValueError("period 1 of overtime has no two-point try")
        if not self.two_point_try and self.period >= 3:
            raise ValueError("from period 3 of overtime every snap is a two-point try")


def overtime_margins(ot: OvertimeState) -> Tuple[int, ...]:
    """The margins (points of the team with the ball minus the opponent's) the overtime rules can reach at `ot`."""
    if not ot.two_point_try:
        if ot.possession == 1:
            return (0,)
        return (0, -3, -7) if ot.period == 1 else (0, -3, -6, -8)
    if ot.period == 2 and ot.possession == 1:
        return (6,)
    return (0,) if ot.possession == 1 else (0, -2)


@dataclass(frozen=True)
class GameState:
    """The state the games of a matchup entry start from: the rest of a game in progress (fmc_game_state).  The future of
    a game depends on nothing else: the period follows from the clock and timeouts are never spent.  `offense` is a team
    index (0 = team A, 1 = team B) or -1 = the kickoff rule (team g & 1 of game g has the ball); `score` = (points of A,
    points of B).  The default is the opening kickoff.

    `fourth_down` (FOURTH_DOWN_POLICY = 0, FOURTH_DOWN_GO, _FG, _PUNT; include/fmc.h FMC_4TH_POLICY) forces the choice
    of a fourth-down state (down 4, seconds > 0) at the first snap of every game: go for it, kick (yards_to_goal <= 38
    only, the range in which the reference kicks) or punt (yards_to_goal >= 16 only).  Every later fourth down follows
    the reference's rule.  A game whose own draw picks that branch plays the same game forced to it.

    `overtime` (an OvertimeState, None = regulation) puts the state inside overtime: the snap about to be played in that
    period and possession, played at the launch's snap clock.  It needs seconds 0 and offense 0 or 1, a try is 1st & 3 at
    the 3, and the score must be one the rules can reach there (`overtime_margins`); a forced choice is allowed at any
    overtime fourth down that is not a try.  A launch of such a state needs overtime rules with max_periods >= period."""
    offense: int = -1
    seconds: int = 3600
    down: int = 1
    distance: float = 10.0
    yards_to_goal: float = 75.0
    score: Tuple[int, int] = (0, 0)
    fourth_down: int = 0
    overtime: Optional[OvertimeState] = None

    def __post_init__(self):
        if self.offense not in (-1, 0, 1):
            raise ValueError("GameState.offense must be -1, 0 or 1")
        if not (isinstance(self.seconds, (int, np.integer)) and 0 <= self.seconds <= 3600):
            raise ValueError("GameState.seconds must be an integer in 0..3600")
        if self.down not in (1, 2, 3, 4):
            raise ValueError("GameState.down must be 1..4")
        if len(self.score) != 2 or not all(isinstance(p, (int, np.integer)) and 0 <= p <= 250 for p in self.score):
            raise ValueError("GameState.score must be two integers in 0..250")
        d, y = float(self.distance), float(self.yards_to_goal)
        if not (math.isfinite(d) and 0.0 < d <= 100.0):
            raise ValueError("GameState.distance must be finite and in (0, 100]")
        if not (0.0 < y < 100.0):
            raise ValueError("GameState.yards_to_goal must be in (0, 100)")
        c = self.fourth_down
        if not (isinstance(c, (int, np.integer)) and FOURTH_DOWN_POLICY <= c <= FOURTH_DOWN_PUNT):
            raise ValueError("GameState.fourth_down must be FOURTH_DOWN_POLICY, _GO, _FG or _PUNT (0..3)")
        ot = self.overtime
        if ot is not None and not isinstance(ot, OvertimeState):
            raise ValueError("GameState.overtime must be None or an OvertimeState")
        if c != FOURTH_DOWN_POLICY and (self.down != 4 or (ot is None and self.seconds == 0)):
            raise ValueError("a forced fourth-down choice needs a fourth down (down 4) with time left, or in overtime")
        if c != FOURTH_DOWN_POLICY and ot is not None and ot.two_point_try:
            raise ValueError("a two-point try has no fourth-down choice")
        if c == FOURTH_DOWN_FG and not y <= 38.0:
            raise ValueError("a forced field goal needs yards_to_goal <= 38")
        if c == FOURTH_DOWN_PUNT and not y >= 16.0:
            raise ValueError("a forced punt needs yards_to_goal >= 16")
        if ot is None:
            return
        if self.seconds != 0:
            raise ValueError("an overtime state has seconds 0 (regulation is over)")
        if self.offense not in (0, 1):
            raise ValueError("an overtime state names the team with the ball (offense 0 or 1)")
        if ot.two_point_try and (self.down, d, y) != (1, 3.0, 3.0):
            raise ValueError("a two-point try is down 1, distance 3, yards_to_goal 3")
        m = int(self.score[self.offense]) - int(self.score[self.offense ^ 1])
        if m not in overtime_margins(ot):
            raise ValueError(f"the overtime rules cannot reach a margin of {m} for the team with the ball at {ot} "
                             f"(possible: {overtime_margins(ot)})")


KICKOFF = GameState()


@dataclass(frozen=True)
class OvertimeRules:
    """College overtime (include/fmc.h FMC_OT_MAX_PERIODS): a game level after regulation is played on in periods of one
    possession per team from the opponent's 25 (a period-2 touchdown is followed by a two-point try; from period 3 every
    possession is a two-point try) until it has a result.  `max_periods` (1..16): a game still level after that many
    periods ends level.  `snap_clock` (1..900): the clock does not run in overtime, and every overtime snap is played
    with this many seconds left, so that the models and the fourth-down logic see end-of-game urgency."""
    max_periods: int = native.OT_MAX_PERIODS
    snap_clock: int = 120

    def __post_init__(self):
        if not (isinstance(self.max_periods, (int, np.integer)) and 1 <= self.max_periods <= native.OT_MAX_PERIODS):
            raise ValueError(f"OvertimeRules.max_periods must be an integer in 1..{native.OT_MAX_PERIODS}")
        if not (isinstance(self.snap_clock, (int, np.integer)) and 1 <= self.snap_clock <= 900):
            raise ValueError("OvertimeRules.snap_clock must be an integer in 1..900")


def overtime_rules(overtime) -> Optional[OvertimeRules]:
    """The rules an API `overtime=` argument asks for: False / None = none (the game ends at 0:00, as in the reference),
    True = the defaults, or an OvertimeRules."""
    if overtime is None or overtime is False:
        return None
    if overtime is True:
        return OvertimeRules()
    if isinstance(overtime, OvertimeRules):
        return overtime
    raise ValueError("overtime must be False, True or an OvertimeRules")


@dataclass
class MatchupSpec:
    """One team pair as the kernels see it."""
    team_a: str
    team_b: str
    sp_a: Tuple[float, float, float]     # RATING, OFFENSE, DEFENSE  (lookup_sp_flex FMC:1625-1644)
    sp_b: Tuple[float, float, float]
    games: int                           # total games of this matchup in the run (all ranks)
    game_begin: int = 0                  # this rank's slice [game_begin, game_end)
    game_end: int = 0
    out_offset: int = 0
    usage: Optional[tuple] = None        # (usage.TeamUsage of team A, of team B) or None = every name "Unknown"
    start: Optional[GameState] = None    # state every game starts from; None = the opening kickoff


class Engine:
    def __init__(self, models: Optional[art.ModelSet] = None, *, device: int = 0,
                 policy: str = "heuristic", sampler: str = "normal", stage2: str = "auto",
                 play_temp: Optional[float] = None, qy_noise: float = 0.5,
                 stage2_standin: Sequence[float] = (0.78, 0.05, 0.17), player: str = "Unknown",
                 memo: Optional[str] = None, memo_bytes: int = 0):
        """`memo`: "on" (default) | "off" | "persistent" -- the exact rank-keyed memo in front of the tree walk, the
        engine's counterpart of the reference's own memo caches (FMC:68-94); results never depend on it.  The
        environment variable FMC_MEMO overrides the default (the GPU test-suite is run under both settings)."""
        self.models = models if models is not None else art.load_default_models()
        self.ctx = native.Context(device)
        self.memo = memo if memo is not None else os.environ.get("FMC_MEMO", "on")
        self.ctx.set_memo(self.memo, max_bytes=memo_bytes,
                          max_trips=int(os.environ.get("FMC_MEMO_TRIPS", "0")),
                          break_parked=int(os.environ.get("FMC_MEMO_BREAK", "0")))
        self.player = player
        if policy == "play_json" and "play_binary" not in self.models:
            raise ValueError("policy='play_json' but the model set has no play_binary forest (play_model.json + "
                             "features.pkl + label_encoder.pkl in FMC_MODEL_DIR)")
        # the play-model slot holds ONE forest: play_model.json (policy 'play_json', what FMC:319-337 loads) or
        # play_model.xgb (policy 'play_model')
        play_name = "play_binary" if policy == "play_json" else "play_model"
        for name in SIM_MODELS[:-1] + (play_name, "run_fumble"):
            if name in self.models:
                f = self.models[name]
                mid = art.MODEL_IDS[name]
                self.ctx.load_forest(mid, f)
                cols = [-1, -1]
                if name not in ("play_model", "play_binary"):
                    for gi, g in enumerate(f.groups[:2]):
                        cols[gi] = g.column_of(player)
                self.ctx.set_active_columns(mid, cols[0], cols[1])
        if stage2 == "auto":
            stage2 = "booster" if "pass_stage2" in self.models else "standin"
        if stage2 == "booster" and "pass_stage2" not in self.models:
            raise ValueError("stage2='booster' but the model set has no pass_stage2 forest")
        if policy == "play_model" and "play_model" not in self.models:
            raise ValueError("policy='play_model' but the model set has no play_model forest")
        self.policy, self.sampler, self.stage2 = policy, sampler, stage2
        pass_class = 1
        if policy == "play_json":
            pass_class = int(self.models["play_binary"].extra["pass_class"])
            if play_temp is None:
                play_temp = float(self.models["play_binary"].extra.get("temperature", 1.0))   # calibration.json
        if play_temp is None:
            play_temp = 1.0
        self.play_temp = float(play_temp)
        self.ctx.set_params(policy={"heuristic": 0, "play_model": 1, "play_json": 1}[policy], pass_class=pass_class,
                            sampler={"normal": 0, "quantile_interp": 1}[sampler],
                            stage2_mode={"standin": 0, "booster": 1}[stage2],
                            play_temp=play_temp, qy_noise=qy_noise, stage2_standin=stage2_standin)
        self.matchups: List[MatchupSpec] = []

    # ------------------------------------------------------------------------------------------
    def coach_col(self, team: str) -> int:
        if self.policy == "play_json" or "play_model" not in self.models:
            return -1      # play_model.json: the category code the booster sees is 0 for every team (FMC:310-313)
        g = self.models["play_model"].group("coach")
        return g.column_of(HEAD_COACH_MAP.get(team)) if g is not None else -1

    def set_matchups(self, specs: Iterable[MatchupSpec]) -> None:
        self.matchups = list(specs)
        self.ctx.set_matchups([
            dict(sp=[list(m.sp_a), list(m.sp_b)], coach_col=(self.coach_col(m.team_a), self.coach_col(m.team_b)),
                 game_begin=m.game_begin, game_end=m.game_end, out_offset=m.out_offset)
            for m in self.matchups])
        # usage tables (FMC:228-249): all matchups or none; a slate mixing both gives the others the trivial table
        with_usage = [m for m in self.matchups if m.usage is not None and not (m.usage[0].trivial and m.usage[1].trivial)]
        if with_usage:
            from . import usage as _usage
            teams = []
            for m in self.matchups:
                if m.usage is None:
                    raise ValueError("player usage must be given for every matchup of a slate or for none")
                teams.append(m.usage)
            self.n_slots = max(len(tu.slots) for pair in teams for tu in pair)
            self.ctx.set_usage(teams, self.n_slots)
        else:
            self.n_slots = 0
        # start states (fmc_set_start_states): an in-game state per entry, the kickoff for the others
        if any(m.start is not None for m in self.matchups):
            self.ctx.set_start_states([m.start if m.start is not None else KICKOFF for m in self.matchups])
        else:
            self.ctx.set_start_states(None)

    def simulate_host(self, seed: int, **kw) -> dict:
        return self.ctx.simulate_host(seed=seed, **kw)

    def predict(self, name: str, rows: np.ndarray, tree_begin: int = 0, tree_end: int = -1,
                coach: Optional[str] = None, names: Optional[Sequence[Sequence[Optional[str]]]] = None,
                hot_cols: Optional[np.ndarray] = None) -> np.ndarray:
        """Raw margins of one model on [n,17] numerics.  Without `names` / `hot_cols` every row has this engine's
        `player` ("Unknown") in its name columns.  `names`: per row the values of the model's categorical inputs in the
        order of `forest.groups` (passer_name, target_name | rusher_name | coach), exactly what a DataFrame row of the
        reference carries (FMC:744, 756, 784-809); names that are not categories light nothing.  `hot_cols` gives the
        one-hot columns directly (int32 [n, 2], -1 = none)."""
        f = self.models[name]
        if names is not None:
            groups = f.groups[:2]
            hot_cols = np.full((len(names), 2), -1, dtype=np.int32)
            for i, row in enumerate(names):
                for gi, g in enumerate(groups):
                    if gi < len(row):
                        hot_cols[i, gi] = g.column_of(row[gi])
        if hot_cols is not None:
            return self.ctx.tree_predict_cols_host(art.MODEL_IDS[name], rows, hot_cols, f.n_outputs, tree_begin, tree_end)
        cc = -1
        if name == "play_model" and coach is not None:
            cc = f.group("coach").column_of(coach)
        return self.ctx.tree_predict_host(art.MODEL_IDS[name], rows, f.n_outputs, tree_begin, tree_end, cc)

    def close(self) -> None:
        self.ctx.close()
