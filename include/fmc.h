/*
 * fmc.h -- C ABI of libfmc_b200.so: the B200-native engine behind the reference's
 * fast_monte_carlo_cfb.py ("FMC") / sim_helpers.py hot path (SURVEY.md section 8).
 *
 * The reference has no FFI of its own: its boundary is the Python API
 *     simulate_upcoming_matchup(...)   FMC:1661-1715
 *     simulate_matchup(...)            FMC:1467-1521
 * plus the model objects it loads at import (FMC:641-668).  Every entry point below names the
 * reference interface it stands in for; fast_monte_carlo_b200/native.py binds them with ctypes and
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions: plain C types only; every call returns 0 on success or a negative fmc_status and
 * leaves a message retrievable with fmc_last_error() (thread-local).  One context per GPU, used
 * from one host thread at a time, with ONE fmc_simulate in flight: a second fmc_simulate (on any stream) is
 * ordered after the previous one on the device, and every call that re-specialises or re-uploads the node
 * tables first waits for the launches in flight.  Pointers named *_dev are device pointers owned by the caller
 * (e.g. torch tensors); pointers named *_host are host memory.  Calls taking `stream` are
 * asynchronous on that CUDA stream (a cudaStream_t passed as void*, NULL = default stream).
 * There is no CPU fallback: without a usable sm_100 device fmc_create fails.
 */
#ifndef FMC_H
#define FMC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FMC_ABI_VERSION 4

typedef enum {
    FMC_OK = 0,
    FMC_ERR_INVALID = -1,   /* bad argument / model not loaded */
    FMC_ERR_CUDA = -2,      /* CUDA runtime error (message has the cudaError string) */
    FMC_ERR_NO_DEVICE = -3, /* no CUDA device / not an sm_100 part */
    FMC_ERR_CAPACITY = -4,  /* a packed forest exceeds the table format limits */
} fmc_status;

/* model ids (the artifacts FMC loads at import, FMC:641-668, plus the two shipped-but-unused boosters) */
enum {
    FMC_PASS_STAGE1 = 0, /* pass_stage1_complete_vs_not.json   FMC:641, 739-747 */
    FMC_PASS_STAGE2 = 1, /* pass_stage2_notcomplete.json        FMC:642, 751-770 (optional) */
    FMC_PASS_YARDS = 2,  /* pass_yards_q{10,50,90}.joblib       FMC:658-660, 780-789 */
    FMC_RUN_YARDS = 3,   /* run_yards_q{10,50,90}.joblib        FMC:662-664, 791-800 */
    FMC_SACK_YARDS = 4,  /* sack_yards_q{10,50,90}.joblib       FMC:666-668, 802-812 */
    FMC_PLAY_MODEL = 5,  /* play_model.xgb (+ scaler.pkl, coach_label_encoder.pkl) */
    FMC_RUN_FUMBLE = 6,  /* run_fumble.json (evaluated only through fmc_tree_predict) */
    FMC_N_MODELS = 7
};

enum { FMC_KIND_XGB = 0, FMC_KIND_SKL = 1 };

/* One tree ensemble in structure-of-arrays form, as produced by the artifact compiler
 * (fast_monte_carlo_b200/artifacts.py).  Arrays are host memory and are copied.
 * Replaces: xgb.Booster().load_model(...) FMC:641-642 and joblib.load(...) FMC:651-668. */
typedef struct {
    int32_t kind;            /* FMC_KIND_XGB: f32 sums, left iff x < thr;  FMC_KIND_SKL: f64 sums, left iff f32(x) <= thr */
    int32_t n_outputs;       /* classes (xgb) or quantiles (skl family), <= 8 */
    int32_t n_features;      /* width of the model's input row */
    int32_t num_base;        /* column of the first of the 17 (12 for play_model) numerics */
    int32_t n_num;
    int32_t zero_is_missing; /* CSR-fed booster: an exact 0 takes the node's default branch */
    double base[8];          /* margin offset per output (xgb) / init constant (skl) */
    double scale;            /* skl learning rate; 1 for xgb */
    int32_t n_nodes;
    int32_t n_trees;
    const int32_t *feat;     /* [n_nodes] split column, -1 for leaves */
    const float *thr;        /* [n_nodes] */
    const int32_t *left;     /* [n_nodes] absolute child index, -1 for leaves */
    const int32_t *right;    /* [n_nodes] */
    const uint8_t *default_left; /* [n_nodes] */
    const double *value;     /* [n_nodes] leaf value */
    const int32_t *tree_root;/* [n_trees] */
    const int32_t *tree_out; /* [n_trees] output each tree adds into */
} fmc_forest_desc;

/* Engine switches.  Defaults (all zero except the doubles noted) reproduce FMC as shipped. */
typedef struct {
    int32_t policy;       /* 0: pass_prob_v1 heuristic (FMC:719-735, the path taken when play_model.json is
                                absent, FMC:326-328);  1: softmax(margins / T)[pass] of the forest loaded as
                                FMC_PLAY_MODEL (FMC:420-425): play_model.json re-laid by the artifact compiler
                                (2 classes, 16 features) or play_model.xgb (5 classes, 180 features) */
    int32_t sampler;      /* 0: Normal(q50, (q90-q10)/2.56) sampler FMC:817-852;
                                1: sim_helpers.QuantileYards.sample (sim_helpers.py:32-38) */
    int32_t stage2_mode;  /* 0: fixed raw probabilities `stage2_standin` (the booster is missing from the
                                reference snapshot);  1: evaluate FMC_PASS_STAGE2 */
    int32_t pass_class;   /* policy 1: index of "pass" among the model's classes (label_encoder.pkl order, FMC:333, 423;
                                0 for play_model.json's [pass, run], 1 for play_model.xgb) */
    double play_temp;     /* _PLAY_TEMP, FMC:50 / calibration.json FMC:335-337 (default 1.0) */
    double qy_noise;      /* sim_helpers noise (default 0.5) */
    double stage2_standin[3]; /* raw [incomplete, intercepted, sack] before the nudges of FMC:764-770 */
} fmc_params;

/* One matchup = two TeamContext objects (FMC:255-271) reduced to what the hot path reads. */
typedef struct {
    double sp[2][3];      /* [team A/B][RATING, OFFENSE, DEFENSE]   lookup_sp_flex FMC:1625-1644 */
    int32_t coach_col[2]; /* play_model.xgb one-hot column of each team's head coach (HEAD_COACH_MAP FMC:55-61), -1 = none */
    uint64_t game_begin;  /* this process simulates games [game_begin, game_end) of the matchup; */
    uint64_t game_end;    /* game g: team (g & 1) receives the opening kickoff (pairs, FMC:1321-1328) */
    uint64_t out_offset;  /* index of game_begin in the per-game output arrays */
} fmc_matchup;

/* The state a game starts from (fmc_set_start_states): the rest of a game in progress.  The future of a game depends on
 * nothing else -- the period follows from the clock (4 - (seconds - 1) / 900, as the clock derives it, FMC:956-968) and
 * timeouts are never spent (FMC:911-912).  Scores and `offense` are by team index of the matchup (0 = team A). */
typedef struct {
    int32_t offense;      /* team with the ball: 0 = A, 1 = B, -1 = team (g & 1) of game g (the kickoff rule) */
    int32_t seconds;      /* seconds remaining, 0..3600 (0: the game is over, zero iterations) */
    int32_t down;         /* 1..4 */
    int32_t score[2];     /* points of team A, team B so far, 0..250 */
    int32_t fourth_down;  /* FMC_4TH_POLICY (0), or the forced choice of a fourth-down start state: FMC_4TH_GO / _FG / _PUNT */
    double distance;      /* yards to a first down, finite, in (0, 100] */
    double yards_to_goal; /* in (0, 100) */
} fmc_game_state;

/* Fourth-down decisions (fmc_game_state.fourth_down).  A forced choice belongs to an entry whose start state is a fourth
 * down (down 4, seconds > 0, or an overtime fourth down that is not a try: fmc_overtime_state) and applies to the first
 * iteration of each of its games only, the start state's snap;
 * every later fourth down follows the reference's handle_fourth (FMC:1382-1421).
 *  - FMC_4TH_POLICY: the reference's draw, go iff u(S_U_GO) < min(1, 1.15 go_for_it_prob), else kick iff
 *    yards_to_goal <= 38, else punt.
 *  - FMC_4TH_GO: the down-4 snap is played, as when the draw says go.
 *  - FMC_4TH_FG: the field-goal branch: made iff u(S_U_FG) < field_goal_prob(yards_to_goal + 17), 12 s, change of
 *    possession.  Only with yards_to_goal <= 38, the range in which the reference kicks.
 *  - FMC_4TH_PUNT: the punt branch (S_Z_GROSS, S_Z_RET, S_U_TB), 16 s, change of possession.  Only with
 *    yards_to_goal >= 16: below that the clip of the net distance to [15, yards_to_goal - 1] is empty.
 * A forced iteration reads only the draw slots its branch reads, from the same record (game, entry, iteration 0): a game
 * whose own draws pick branch X plays, forced to X, the same game bit for bit (score, iterations, trace, box lines,
 * overtime periods, event counters).  FMC_ERR_INVALID for any other code, a non-zero code on a state that is not a
 * fourth down with time left or outside the choice's range, and forced choices with period or sequence outputs. */
enum { FMC_4TH_POLICY = 0, FMC_4TH_GO, FMC_4TH_FG, FMC_4TH_PUNT };

/* Usage table of one role of one team: TeamContext.qb_share / rush_share / target_share (FMC:262-264) as
 * the hot path reads them.  The engine samples an entry per play exactly as Generator.choice(len(df),
 * p=share) does (FMC:625-635: cdf = cumsum(share) / total, searchsorted(cdf, u, 'right')), feeds the models
 * the entry's one-hot column (the OneHotEncoder(handle_unknown='ignore') half of the preprocessors applied
 * to passer_name / target_name / rusher_name, FMC:1079-1081, 1216) and keeps a per-game box line for
 * entries whose `slot` is >= 0 (names in the team's focus track set, FMC:1062-1063, 1204). */
#define FMC_MAX_USAGE 32         /* entries per table */
#define FMC_MAX_PASSER_ROWS 4    /* passers per team that some model has a one-hot column for */
#define FMC_MAX_NAME_ROWS 8      /* same for targets and for rushers; names no model knows are not limited */
typedef struct {
    int32_t n;                   /* 1..FMC_MAX_USAGE */
    int32_t reserved;
    double share[FMC_MAX_USAGE]; /* df['share'].values, in table order */
    int32_t slot[FMC_MAX_USAGE]; /* output slot of a tracked name inside the team's box, -1 = not tracked */
    int32_t col[FMC_N_MODELS][FMC_MAX_USAGE]; /* one-hot column the name lights in model m, -1 = not a category */
} fmc_usage;
typedef struct { fmc_usage role[3]; } fmc_team_usage;   /* 0 passer (sample_qb), 1 rusher, 2 target */

/* Per-game box line of one tracked name: pstats[team][role][name] (FMC:146-166) at the end of the game.
 * counts: 10-bit fields from bit 0: att|tgt, comp|rec, td, INT, sacks.  yds is the float64 running sum in
 * play order (the reference rounds it to one decimal only when it writes the row, FMC:1276-1296). */
typedef struct {
    double yds;
    uint64_t counts;
} fmc_player_rec;

/* Per-player histograms over the games of a launch (what edge_finder.player_prop_odds reads off `players_*`,
 * edge_finder.py:168-231, without per-game rows; mergeable across GPUs by an integer all-reduce).  One record
 * of FMC_PH_BINS uint32 per (matchup, team, slot); a game counts only if the name was sampled in it (the
 * reference writes a row only then, FMC:1266-1299):
 *   [0, FMC_PH_YDS_BINS)              yards rounded to one decimal exactly like Python's round(x, 1)
 *                                     (FMC:1276, 1286, 1296): bin = tenths + FMC_PH_YDS_OFFSET, clamped
 *   then 5 x FMC_PH_CNT_BINS          att|tgt, comp|rec, td, INT, sacks: bin = min(count, FMC_PH_CNT_BINS - 1) */
#define FMC_PH_YDS_BINS 8192
#define FMC_PH_YDS_OFFSET 1000   /* bin 1000 = 0.0 yards; range -100.0 .. +719.1 */
#define FMC_PH_CNT_BINS 128
#define FMC_PH_BINS (FMC_PH_YDS_BINS + 5 * FMC_PH_CNT_BINS)

#define FMC_HIST_BINS 128        /* joint (points A, points B) histogram is FMC_HIST_BINS^2 per orientation */
#define FMC_N_COUNTERS 32
/* counters[] layout (totals over the call) */
enum {
    FMC_C_GAMES = 0, FMC_C_PLAYS, FMC_C_ITERS, FMC_C_PASS, FMC_C_COMP, FMC_C_INC, FMC_C_INT, FMC_C_SACK,
    FMC_C_RUN, FMC_C_TD, FMC_C_FGA, FMC_C_FG, FMC_C_PUNT, FMC_C_GO, FMC_C_HIST_OVERFLOW,
    FMC_C_ROUNDS, FMC_C_REQUESTS,
    FMC_C_VISITS, /* 8-byte node slots gathered for live requests (tree levels walked x lanes) */
    FMC_C_PH_OVERFLOW, /* player-histogram samples clamped into the first / last bin */
    FMC_C_WARP_STEPS,  /* warp-level node gathers of the tree walk (tree levels walked x trees per group, per warp) */
    FMC_C_MEMO_PROBES, /* requests looked up in the exact memo (fmc_set_memo) */
    FMC_C_MEMO_HITS,   /* ... of which were answered from it (the rest were walked: FMC_C_REQUESTS) */
    FMC_C_TRIPS,       /* warp-level passes of the state machine (memo kernel) */
    FMC_C_MEMO_HITS_FAM0 = 24 /* ... 29: memo hits per family (model ids 0..5); probes per family follow from the event
                                 counters: stage 1 = pass, stage 2 = pass - comp, pass yards = comp, run yards = run,
                                 sack yards = sack, play model = plays under policy 1 */,
    FMC_C_OT_GAMES = 30,      /* games that went to overtime (fmc_simulate_overtime) */
    FMC_C_OT_PERIODS = 31     /* overtime periods they played */
};

/* Periods (quarter and half markets, fmc_simulate_segments).  Quarter q (1..3) ends when the clock crosses
 * 3600 - 900 q (2700, 1800, 900): the period is 4 - (seconds - 1) / 900, as the clock derives it.  A play's points
 * count in the quarter in which it was snapped, so the score at the end of quarter q is the score after the play whose
 * clock tick crossed the boundary (the score at the next iteration start or, if the game is over, the final score).
 * Segments, in this order: Q1, Q2, Q3, Q4, H1 (= Q1 + Q2), H2 (= Q3 + Q4).  A segment's value for a game is the
 * (points A, points B) scored in it: the score at its end minus the score at its base, which is the score at its start
 * boundary or the game's start state (fmc_set_start_states) if that is later.  A segment that ends at or before the
 * start state is not counted (boundary B lies in the simulated future iff start seconds > B); one in progress counts
 * from the start state.  Q4 and H2 end at the game's end: a game that starts with the clock at 0 counts (0, 0) in Q4
 * and H2 and nothing else. */
#define FMC_N_SEGMENTS 6
enum { FMC_SEG_Q1 = 0, FMC_SEG_Q2, FMC_SEG_Q3, FMC_SEG_Q4, FMC_SEG_H1, FMC_SEG_H2 };
#define FMC_PERIOD_NONE 0xFFFFFFFFu  /* period_scores word of a quarter end at or before the start state */

/* Scoring sequence (next-score, drive-result and race-to-N markets, fmc_simulate_markets).  Everything counts from the
 * game's start state (the kickoff, or fmc_set_start_states); teams are the matchup's (0 = A).  The engine scores only
 * touchdowns (7) and made field goals (3), always by the team on offense.
 *  - Next score: the first play after the start state that adds points: (team, kind, clock at its snap = the seconds at
 *    the start of the iteration that played it).  FMC_SEQ_NONE if the game ends with the start score.
 *  - Drive result: the drive is the possession of the team on offense at the start state (g & 1 at the kickoff).  It
 *    ends at the first of: TD, FG made, FG missed, punt, interception, turnover on downs (advance_down's change of
 *    possession), end of half (the halftime change of possession when the clock crosses 1800), end of game (the clock
 *    reaches 0 with the drive on).  A play's own result comes before the end of the half its tick crosses.  A down
 *    that passes 4 without a change of possession (incomplete pass, sack) does not end it.
 *  - Race to N (N in FMC_RACE_TARGETS): won by the team whose score (start points included) first reaches N, decided
 *    at the scoring play that takes it from below N to N or more while the other team is below N; "neither" if no team
 *    reaches N.  A target either team had reached at the start state is settled and not counted. */
#define FMC_SEQ_NONE 0xFFFFFFFFu     /* sequence word 0 of a game without a score after the start state */
enum { FMC_SEQ_TD = 0, FMC_SEQ_FG = 1 };          /* kind of a scoring play */
enum { FMC_DRIVE_TD = 0, FMC_DRIVE_FG, FMC_DRIVE_MISSED_FG, FMC_DRIVE_PUNT, FMC_DRIVE_INT, FMC_DRIVE_DOWNS,
       FMC_DRIVE_HALF, FMC_DRIVE_GAME, FMC_N_DRIVE };
#define FMC_N_RACE 5
#define FMC_RACE_TARGETS {10, 15, 20, 25, 30}
enum { FMC_RACE_A = 0, FMC_RACE_B, FMC_RACE_NEITHER };
/* sequence word 0: next score team:1 | kind:1 | clock:12 (or FMC_SEQ_NONE); word 1: drive result | clock at the snap of
 * the play that ended it << 8 (0 for the end of the game) */
#define FMC_SEQ_WORD(team, kind, clock) ((uint32_t)(team) | ((uint32_t)(kind) << 1) | ((uint32_t)(clock) << 2))
#define FMC_DRIVE_WORD(code, clock) ((uint32_t)(code) | ((uint32_t)(clock) << 8))
/* bins of one orientation's sequence histogram: next score by (team, kind) and minute of regulation at its snap
 * (clock 1..3600 -> minute bin (clock - 1) / 60, aligned with the quarter ends), no further score, the drive results,
 * then the race targets x (A, B, neither) */
#define FMC_SEQ_MINUTES 60
#define FMC_SEQ_BIN_NEXT(team, kind, clock) (((team) * 2 + (kind)) * FMC_SEQ_MINUTES + ((clock) - 1) / 60)
#define FMC_SEQ_BIN_NONE (4 * FMC_SEQ_MINUTES)
#define FMC_SEQ_BIN_DRIVE(code) (FMC_SEQ_BIN_NONE + 1 + (code))
#define FMC_SEQ_BIN_RACE(target, r) (FMC_SEQ_BIN_DRIVE(FMC_N_DRIVE) + (target) * 3 + (r))
#define FMC_SEQ_BINS FMC_SEQ_BIN_RACE(FMC_N_RACE, 0)      /* 264 */

/* Overtime (fmc_simulate_overtime; opt-in: without it a game ends at 0:00, level or not, as in the reference).  The NCAA
 * rules in force since 2021, played with the reference's plays, models and fourth-down logic:
 *  - A game level when regulation ends (the clock reaches 0, or a start state at 0 s) goes to overtime.
 *  - Periods k = 1, 2, ...; each team has one possession per period.  Team (g & 1), the opening-kickoff receiver, has the
 *    first possession of period 1; the order alternates every period.
 *  - Periods 1 and 2: a possession starts at 1st & 10 at the opponent's 25 (down 1, distance 10, yards to goal 25) and
 *    is played by the reference's rules until the offense changes (TD, FG made or missed, punt, interception, turnover
 *    on downs).  A TD is 7 in period 1; in period 2 it is 6 and is followed by a two-point try.  A FG is 3.
 *  - From period 3 every possession is one two-point try.  A try is one snap at down 1, distance 3, yards to goal 3: 2
 *    points iff the snap is a TD by the reference's rules, else 0; the rest of its result is discarded and it credits
 *    no player box line (its event counters count as for any snap).
 *  - The clock does not run: every overtime snap is played with seconds = snap_clock (1..900; 120 puts it in the last
 *    two minutes of the fourth quarter, so the models and the fourth-down logic see end-of-game urgency).
 *  - The game ends as soon as the team with the second possession of a period leads (a period-2 TD that wins plays no
 *    try), after the second possession of a period if the score is not level, level after max_periods periods
 *    (1..FMC_OT_MAX_PERIODS), and as it stands when its iteration count reaches FMC_MAX_ITERS.
 *  - Every overtime snap is one iteration: the Philox counter (game, entry, iteration) keeps counting from regulation,
 *    so a game not level after regulation is the same game with overtime on or off, and the trace row of an overtime
 *    iteration holds the state after the bookkeeping of its start (possession, try, period).
 * Scores, score words, the score histogram, iteration counts, traces, counters and player boxes include overtime. */
#define FMC_OT_MAX_PERIODS 16
enum { FMC_OT_A = 0, FMC_OT_B, FMC_OT_LEVEL };    /* last index of the overtime histogram: the game's result */

/* A start state inside overtime (fmc_set_start_states_overtime): with the fmc_game_state of the entry (offense, down,
 * distance, yards_to_goal, score) it names the overtime snap about to be played, the state the trace row of an overtime
 * iteration holds.  period 0 is regulation (the other fields 0); otherwise
 *  - period k in 1..FMC_OT_MAX_PERIODS, possession 1 or 2 (the first or second possession of period k), two_point_try
 *    0 or 1.  seconds must be 0 (every snap is played at the launch's snap_clock) and offense 0 or 1; a try is down 1,
 *    distance 3, yards to goal 3.  The team with the first possession of period 1 follows from offense, possession and
 *    k (it need not be team g & 1).
 *  - d = the offense's points minus the opponent's must be one the rules can reach: 0 on the first possession of
 *    periods 1 and 2; 0, -3 or -7 on the second possession of period 1; 0, -3, -6 or -8 on the second possession of
 *    period 2; +6 on a first-possession try of period 2; 0 or -2 on a second-possession try of period 2 (a
 *    second-possession touchdown that wins plays no try); 0 on a first-possession try from period 3, 0 or -2 on a
 *    second-possession try.  No try in period 1, only tries from period 3.
 *  - A forced fourth-down choice (fmc_game_state.fourth_down) is allowed at any fourth down that is not a try, with its
 *    ranges; it applies to the first snap.
 * A launch with such an entry needs overtime with max_periods >= period (FMC_ERR_INVALID otherwise).  Draws count
 * iterations from the start state, as for every start state; the overtime histogram bin is the last period played, and
 * the overtime periods output and counters count periods, not periods from the start. */
typedef struct {
    int32_t period;
    int32_t possession;
    int32_t two_point_try;
    int32_t reserved;     /* 0 */
} fmc_overtime_state;

#define FMC_N_SLOTS 16           /* injected-draw record per (game, loop iteration); see DESIGN.md */
#define FMC_MAX_ITERS 360
#define FMC_TRACE_COLS 8

typedef struct {
    uint64_t seed;            /* Philox key; ignored when stream_dev != NULL */
    int32_t n_matchups;       /* must equal the last fmc_set_matchups */
    int32_t reserved;
    uint32_t *scores_dev;     /* optional [sum of games]: (points A) | (points B) << 16 at out_offset + (g - game_begin) */
    uint32_t *hist_dev;       /* optional [n_matchups][2][BINS][BINS], += 1 at [m][g&1][min(A,BINS-1)][min(B,BINS-1)] */
    uint64_t *counters_dev;   /* optional [FMC_N_COUNTERS], accumulated with atomics */
    const double *stream_dev; /* optional injected draws [games][FMC_MAX_ITERS][FMC_N_SLOTS] (test mode) */
    double *trace_dev;        /* optional per-iteration states [games][FMC_MAX_ITERS][FMC_TRACE_COLS] (test mode) */
    uint16_t *iters_dev;      /* optional [games] loop iterations of each game */
    void *stream;             /* cudaStream_t */
    fmc_player_rec *players_dev; /* optional, only with fmc_set_usage: [games][2 teams A/B][n_slots]; every line is written */
    uint32_t *player_hist_dev;   /* optional, only with fmc_set_usage: [n_matchups][2][n_slots][FMC_PH_BINS], += (zero it first) */
} fmc_sim_args;

typedef struct fmc_ctx fmc_ctx;

const char *fmc_last_error(void);
int fmc_abi_version(void);

/* Context on CUDA device `device`.  Fails with FMC_ERR_NO_DEVICE when there is no sm_100 GPU. */
int fmc_create(int device, fmc_ctx **out);
void fmc_destroy(fmc_ctx *ctx);
/* SM count, shared memory per block, and the resident-forest capacity the kernels were sized for. */
int fmc_device_info(fmc_ctx *ctx, int32_t *sm_count, int32_t *smem_per_block, char *name, int32_t name_len);

/* Replaces Booster.load_model / joblib.load at FMC:641-668. */
int fmc_load_forest(fmc_ctx *ctx, int32_t model_id, const fmc_forest_desc *desc);
/* StandardScaler of play_model.xgb: x[cols[i]] = (x - mean[i]) / scale[i]  (scaler.pkl). */
int fmc_set_scaler(fmc_ctx *ctx, int32_t model_id, int32_t n, const int32_t *cols, const double *mean, const double *scale);
/* Hot one-hot columns (-1 = name is not a category) every row of `model_id` uses: the
 * OneHotEncoder(handle_unknown='ignore') half of ColumnTransformer.transform, FMC:744, 756, 784-809.
 * With the shipped usage tables every player is "Unknown" (FMC:246-249). */
int fmc_set_active_columns(fmc_ctx *ctx, int32_t model_id, int32_t col0, int32_t col1);
int fmc_set_params(fmc_ctx *ctx, const fmc_params *p);
/* Replaces build_team_context_from_sp_flex x2 + _init_pool (FMC:1646-1659, 1306-1319): specialises
 * every loaded forest on the per-orientation constants and uploads the packed node tables. */
int fmc_set_matchups(fmc_ctx *ctx, int32_t n, const fmc_matchup *m);

/* Start states of the matchup entries of the last fmc_set_matchups: states[n_matchups], one per entry; every game of
 * entry m starts from states[m] instead of the opening kickoff (sec 3600, 1st & 10 at the 75, 0-0, team (g & 1) with
 * the ball).  states == NULL returns every entry to the kickoff.  fmc_set_matchups resets them to the kickoff.  Draws,
 * outputs and the score histogram are unchanged in form: the Philox counter is (game, entry, iteration), the iteration
 * count starts at 0 at the start state, histogram bin [m][g & 1] holds the final score.  Cheap: it neither
 * re-specialises nor clears the memo (fmc_set_memo mode 2 keeps it); it only rewrites the start words of the device
 * records, after the launches in flight.  FMC_ERR_INVALID for n_matchups different from the last fmc_set_matchups or a
 * field out of range (see fmc_game_state and FMC_4TH_POLICY).  While some entry has a forced fourth-down choice, a launch
 * runs the kernel instantiations with the decision rule; entries with FMC_4TH_POLICY play the same games in them. */
int fmc_set_start_states(fmc_ctx *ctx, int32_t n_matchups, const fmc_game_state *states);

/* fmc_set_start_states with an overtime state per entry: ot[n_matchups] (see fmc_overtime_state; period 0 =
 * regulation).  ot == NULL is fmc_set_start_states; states == NULL needs ot == NULL.  fmc_set_matchups and
 * fmc_set_start_states return every entry to regulation.  FMC_ERR_INVALID for a state the rules cannot reach; a launch
 * with an entry in overtime fails with FMC_ERR_INVALID without overtime, with max_periods below the entry's period, or
 * with period or sequence outputs. */
int fmc_set_start_states_overtime(fmc_ctx *ctx, int32_t n_matchups, const fmc_game_state *states,
                                  const fmc_overtime_state *ot);

/* Replaces the usage half of build_team_context_from_sp_flex (`_usage_from_focus_or_fallback`, FMC:228-249,
 * 1646-1659): teams[n_matchups][2] (team A, team B of each matchup of the last fmc_set_matchups), n_slots =
 * box lines per team in the per-game output.  teams == NULL returns to the shipped configuration (one
 * "Unknown" per role, nothing tracked; the hot columns of fmc_set_active_columns apply).  With usage set,
 * fmc_simulate runs the player instantiation of the kernel: the sampled names become extra 0/1 feature rows
 * of a request, so the node tables stay specialised per orientation only. */
int fmc_set_usage(fmc_ctx *ctx, int32_t n_matchups, const fmc_team_usage *teams, int32_t n_slots);

/* Exact memo of model outputs in front of the tree walk -- the B200 counterpart of the reference's own memo caches
 * (_PLAY_CACHE / _PASS1_CACHE / _PASS2_CACHE / _*_Q_CACHE, FMC:68-94, 343-357, 740-747, 780-812), but EXACT: the key
 * is the vector of threshold ranks of the request's features on the specialised forest, so a hit returns bit for
 * bit what the walk would (csrc/fmc_memo.hpp).  Results never depend on the mode.
 *   mode 0: off -- every request is walked (the roofline / tree-eval measurements use this);
 *   mode 1: on (default), the table is cleared at the start of every fmc_simulate;
 *   mode 2: on, the table is kept between calls for as long as the node tables stay the same.
 * max_bytes: device memory the tables may take (0 = default: up to 1/4 of the free memory, at most 16 GiB; they
 * are sized by the games of the launch).  max_trips / break_parked: scheduling knobs of the memo kernel (stage steps a
 * warp may run per round; lanes of a warp that must wait for the walk before the warp ends its round); 0 = default.
 * Entries whose forests are specialised alike (same sp and coach_col, and in player mode the same usage tables) share
 * one table set and one memo.  Player mode (fmc_set_usage) and launches of more than 1024 distinct specialisations
 * always run unmemoised. */
int fmc_set_memo(fmc_ctx *ctx, int32_t mode, uint64_t max_bytes, int32_t max_trips, int32_t break_parked);

/* Replaces simulate_matchup's pool of _run_pair workers (FMC:1467-1521): plays every game of every
 * matchup range to completion on the GPU.  Asynchronous on args->stream. */
int fmc_simulate(fmc_ctx *ctx, const fmc_sim_args *args);

/* Per-period outputs of a launch (see FMC_N_SEGMENTS for the definitions); both optional.
 *   period_scores_dev  [games][3]: score word (points A) | (points B) << 16 at the end of Q1, Q2, Q3, at
 *                      out_offset + (g - game_begin) like scores_dev; FMC_PERIOD_NONE for a quarter end at or before
 *                      the start state.
 *   segment_hist_dev   [n_matchups][2][FMC_N_SEGMENTS][BINS][BINS], += 1 at [m][g & 1][segment][min(A, BINS-1)]
 *                      [min(B, BINS-1)] with A, B the points scored in the segment (zero it first, like hist_dev).
 *                      Without period_scores_dev the library keeps the per-game rows in device scratch (12 B a game);
 *                      the first such call, and one that needs more rows than any before it, grows that scratch and
 *                      synchronises the device (grow-only, like the running player boxes). */
typedef struct {
    uint32_t *period_scores_dev;
    uint32_t *segment_hist_dev;
} fmc_segment_args;

/* fmc_simulate plus the per-period outputs.  seg == NULL, or both pointers NULL, is exactly fmc_simulate; otherwise the
 * launch runs the kernel instantiation with the period hooks (the one without them is unchanged).  Every other output,
 * draw and game is the same as without them. */
int fmc_simulate_segments(fmc_ctx *ctx, const fmc_sim_args *args, const fmc_segment_args *seg);

/* Same, with HOST result buffers (any may be NULL): allocates device scratch, runs, copies back and
 * synchronises.  This is the call the reference-facing Python API makes (end-to-end path). */
int fmc_simulate_host(fmc_ctx *ctx, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                      uint64_t *counters_host, const double *stream_host, double *trace_host,
                      uint16_t *iters_host);

/* fmc_simulate_host plus the per-game player box [games][2][n_slots] (collect_players=True, FMC:1480-1505) and / or
 * the per-player histograms [n_matchups][2][n_slots][FMC_PH_BINS]; either may be NULL.  Needs fmc_set_usage. */
int fmc_simulate_players_host(fmc_ctx *ctx, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                              uint64_t *counters_host, const double *stream_host, double *trace_host,
                              uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host);

/* fmc_simulate_players_host plus the per-period outputs: period_scores_host [games][3] and segment_hist_host
 * [n_matchups][2][FMC_N_SEGMENTS][BINS][BINS] (either may be NULL; see fmc_segment_args).  Player outputs need
 * fmc_set_usage, as there. */
int fmc_simulate_segments_host(fmc_ctx *ctx, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                               uint64_t *counters_host, const double *stream_host, double *trace_host,
                               uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host,
                               uint32_t *period_scores_host, uint32_t *segment_hist_host);

/* Scoring-sequence outputs of a launch (see FMC_SEQ_NONE for the definitions); both optional.
 *   sequence_dev       [games][2] at out_offset + (g - game_begin) like scores_dev: word 0 the next score
 *                      (FMC_SEQ_WORD or FMC_SEQ_NONE), word 1 the drive result (FMC_DRIVE_WORD).
 *   sequence_hist_dev  [n_matchups][2][FMC_SEQ_BINS], += 1 at [m][g & 1][bin] for the next score (or none), the drive
 *                      result and every race target that is not settled (zero it first, like hist_dev).
 *                      Without sequence_dev the library keeps the per-game rows in device scratch (8 B a game), grown
 *                      like the period rows of fmc_segment_args. */
typedef struct {
    uint32_t *sequence_dev;
    uint32_t *sequence_hist_dev;
} fmc_sequence_args;

/* fmc_simulate plus the per-period and the scoring-sequence outputs; seg and seq may each be NULL (or hold only NULL
 * pointers).  Neither is fmc_simulate, seg alone fmc_simulate_segments.  The launch runs the kernel instantiation with
 * the hooks it asks for; every other output, draw and game is the same as without them. */
int fmc_simulate_markets(fmc_ctx *ctx, const fmc_sim_args *args, const fmc_segment_args *seg, const fmc_sequence_args *seq);

/* fmc_simulate_segments_host plus the scoring-sequence outputs: sequence_host [games][2] and sequence_hist_host
 * [n_matchups][2][FMC_SEQ_BINS] (any output may be NULL). */
int fmc_simulate_markets_host(fmc_ctx *ctx, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                              uint64_t *counters_host, const double *stream_host, double *trace_host,
                              uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host,
                              uint32_t *period_scores_host, uint32_t *segment_hist_host, uint32_t *sequence_host,
                              uint32_t *sequence_hist_host);

/* Overtime of a launch (see FMC_OT_MAX_PERIODS for the rules).
 *   max_periods   1..FMC_OT_MAX_PERIODS: a game still level after this many periods ends level.
 *   snap_clock    1..900: the seconds every overtime snap is played with.
 *   ot_periods_dev optional [games] at out_offset + (g - game_begin) like scores_dev: overtime periods played (0: the
 *                 game was decided in regulation).
 *   ot_hist_dev   optional [n_matchups][2][FMC_OT_MAX_PERIODS + 1][3], += 1 at [m][g & 1][periods][FMC_OT_A | FMC_OT_B |
 *                 FMC_OT_LEVEL] by the final score (zero it first, like hist_dev).  Bin [.][.][0] holds the games decided
 *                 in regulation. */
typedef struct {
    int32_t max_periods;
    int32_t snap_clock;
    uint8_t *ot_periods_dev;
    uint32_t *ot_hist_dev;
} fmc_overtime_args;

/* fmc_simulate with overtime; ot == NULL is exactly fmc_simulate.  The launch runs the kernel instantiation with the
 * overtime rule.  FMC_ERR_INVALID for a field out of range.  Overtime has no period or sequence outputs (the markets of
 * fmc_simulate_markets are defined for regulation). */
int fmc_simulate_overtime(fmc_ctx *ctx, const fmc_sim_args *args, const fmc_overtime_args *ot);

/* fmc_simulate_players_host with overtime: max_periods and snap_clock as in fmc_overtime_args, ot_periods_host [games]
 * and ot_hist_host [n_matchups][2][FMC_OT_MAX_PERIODS + 1][3] (any output may be NULL; player outputs need
 * fmc_set_usage). */
int fmc_simulate_overtime_host(fmc_ctx *ctx, uint64_t seed, uint32_t *scores_host, uint32_t *hist_host,
                               uint64_t *counters_host, const double *stream_host, double *trace_host,
                               uint16_t *iters_host, fmc_player_rec *players_host, uint32_t *player_hist_host,
                               int32_t max_periods, int32_t snap_clock, uint8_t *ot_periods_host, uint32_t *ot_hist_host);

/* Raw margins of one model on n rows of the 17 numerics (play_model: first 12), NUM order of
 * FMC:676-682, float64 row-major [n][17]; out float64 [n][n_outputs].  Trees [tree_begin, tree_end)
 * (tree_end < 0: all) -- iteration_range of sim_helpers.py:22-23 / pass_outcome_infer.py:57,62.
 * Replaces Booster.inplace_predict / Booster.predict(output_margin=True) / Pipeline.predict. */
int fmc_tree_predict(fmc_ctx *ctx, int32_t model_id, const double *rows_dev, int64_t n, double *out_dev,
                     int32_t tree_begin, int32_t tree_end, int32_t coach_col, void *stream);
int fmc_tree_predict_host(fmc_ctx *ctx, int32_t model_id, const double *rows_host, int64_t n, double *out_host,
                          int32_t tree_begin, int32_t tree_end, int32_t coach_col);

/* The same for rows that carry their OWN names (a DataFrame with passer_name / target_name / rusher_name per row, FMC:744,
 * 756, 784-809): hot_cols_host = int32 [n][2], the one-hot column each of the row's (up to) two names lights in this model
 * (artifacts.OneHotGroup.column_of), -1 = the name is not a category (OneHotEncoder(handle_unknown='ignore') lights
 * nothing).  Rows are grouped by column pair, every pair gets its own specialised table; outputs are in row order. */
int fmc_tree_predict_cols_host(fmc_ctx *ctx, int32_t model_id, const double *rows_host, int64_t n, const int32_t *hot_cols_host,
                               double *out_host, int32_t tree_begin, int32_t tree_end);

/* Packed-table statistics of the last fmc_set_matchups (slots per family/orientation), for
 * DESIGN.md / roofline accounting.  out[FMC_N_MODELS][2] = 8-byte slots of matchup `m` (of the table set it shares with
 * the first entry specialised alike). */
int fmc_packed_slots(fmc_ctx *ctx, int32_t m, int32_t *out);

int fmc_sync(fmc_ctx *ctx);
/* Measurement helper: drop the specialised node tables; the next fmc_simulate specialises, packs and uploads again
 * (bench.py times the whole host path with it). */
int fmc_invalidate_tables(fmc_ctx *ctx);

/* Roofline accounting of the tree evaluator: node gathers of the fmc_tree_predict launches since the last reset.
 * out2[0] = warp-level gathers (one per warp, tree and level: what the L1 data pipe sees), out2[1] = lane-level
 * gathers of live rows (x 8 bytes = gathered bytes).  Synchronises the device. */
int fmc_predict_stats(fmc_ctx *ctx, uint64_t *out2, int32_t reset);

/* Diagnostics: out-of-range node gathers / feature offsets counted (and skipped) by a library built with
 * -DFMC_DEBUG_CHECKS since the last call; always 0 for the production build. */
int64_t fmc_debug_errors(void);

/* Measurement helper for the roofline (SURVEY 8d): achievable rate of dependent 8-byte read-only
 * gathers through a random cyclic table of `table_bytes` (L1-resident when small, L2-resident at a
 * few MiB), 8 chains per lane, one 1024-lane CTA per SM -- a tree walk with nothing around it.
 * Synchronous; returns GB/s of gathered slots (8 bytes each). */
int fmc_gather_probe(fmc_ctx *ctx, int64_t table_bytes, int32_t iters, double *gbytes_per_s);

/* The same with WARP-COHERENT lanes, the access pattern of a real tree level: the 32 lanes of a warp gather inside
 * one window of `window_bytes` (power of two; a depth-3 tree of the quantile models spans 112 bytes, a group of four
 * under 512) and all move on to the same next window.  out3 = {GB/s of gathered slots (8 bytes x lanes), warp-level
 * gathers per second, best time in ms}.  The walk's achieved gather rate (FMC_C_VISITS x 8 bytes / kernel time) is
 * reported as a fraction of this in bench.py (< 1: a walk also loads a feature and compares per level). */
int fmc_gather_probe_coherent(fmc_ctx *ctx, int64_t table_bytes, int32_t window_bytes, int32_t iters, double *out3);

/* Host-only, needs no context and no GPU: runs the forest specialiser/packer and returns the node
 * table, the root stream and the constants side stream the kernels walk (layout:
 * fast_monte_carlo_b200/csrc/fmc_pack.hpp; child offsets relative to the table start).  It
 * evaluates nothing; CPU tests walk the returned tables themselves, and DESIGN.md's table-size
 * figures come from it.  mode 0 = simulation preset (numerics 6..11 folded to fold_value17[]),
 * 1 = predict preset.  Returns the slot count (>= 0) or a negative fmc_status; buffers that are too
 * small are left untouched.  info_out[32] = {rounds, max group depth, n_outputs, trees per group,
 * "-inf" feature row, stream words, side-stream words, constant trees, stream_off[8] (8-byte words),
 * n_groups[8], consts_off[8]}. */
/* Same with dynamic one-hot columns (player mode): dyn_cols[n_dyn] are model columns whose 0/1 value is read
 * per request from feature row dyn_rows[i] instead of being folded. */
int64_t fmc_pack_forest_host_dyn(const fmc_forest_desc *desc, int32_t mode, int32_t col0, int32_t col1,
                                 const double *fold_value17, int32_t n_dyn, const int32_t *dyn_cols,
                                 const int32_t *dyn_rows, uint64_t *slots_out, int64_t slots_cap,
                                 uint64_t *stream_out, int64_t stream_cap, uint64_t *consts_out, int64_t consts_cap,
                                 int32_t *info_out);
int64_t fmc_pack_forest_host(const fmc_forest_desc *desc, int32_t mode, int32_t col0, int32_t col1,
                             const double *fold_value17, int32_t n_scaled, const int32_t *scaler_cols,
                             const double *scaler_mean, const double *scaler_scale, int32_t tree_begin,
                             int32_t tree_end, uint64_t *slots_out, int64_t slots_cap, uint64_t *stream_out,
                             int64_t stream_cap, uint64_t *consts_out, int64_t consts_cap, int32_t *info_out);

/* Host-only, needs no GPU: exact-memo keys (fmc_set_memo, csrc/fmc_memo.hpp) of n simulation states on `desc`
 * specialised as fmc_set_matchups specialises family `family` (simulation preset: numerics 6..11 folded to
 * fold_value17[], hot columns col0 / col1).  states = float64 [n][5]: down, distance, yardsToGoal, score_diff,
 * seconds_remaining (the derived flags follow from them, FMC:996-1021).  keys_out[n] = the 64-bit keys of matchup 0,
 * team 0.  Returns 1, 0 when the forest's rank vector does not fit a key (fmc_last_error says why; such a family is
 * always walked) or a negative fmc_status.  info_out[4] = {memoisable, thresholds on distance, on yardsToGoal,
 * constant trees}.  Evaluates no tree: tests group oracle margins by key to check that equal keys mean equal outputs. */
int64_t fmc_memo_keys_host(const fmc_forest_desc *desc, int32_t family, int32_t col0, int32_t col1,
                           const double *fold_value17, int32_t n_scaled, const int32_t *scaler_cols,
                           const double *scaler_mean, const double *scaler_scale, int64_t n, const double *states,
                           uint64_t *keys_out, int32_t *info_out);

#ifdef __cplusplus
}
#endif
#endif /* FMC_H */
