// Persistent play-by-play simulation kernel (one lane per simulated game).
//
// Restates, for the GPU, the reference's game engine:
//   simulate_game FMC:1428-1464, handle_fourth FMC:1382-1421, simulate_play FMC:1026-1257,
//   advance_down / change_possession / tick_clock FMC:932-968, pass_prob_v1 FMC:719-735,
//   modifiers FMC:431-472, samplers FMC:817-852 (+ sim_helpers.py:32-38), special teams FMC:858-896.
//
// Structure (DESIGN.md "simulation kernel"): one CTA of 1024 lanes per SM, each lane owns one game
// and keeps its whole state in registers.  A game is a little coroutine: it advances until it needs
// a tree model (a "request": family x orientation), parks, and resumes when the value is there.
// Per round the CTA
//   A. advances every lane to its next request (state machine, Philox draws, special teams),
//   B. compacts the requests per (family, orientation) with warp match + shared atomics and writes
//      each request's feature row into shared memory at its compacted position,
//   C. evaluates the requests: work items = (list, 32-request chunk, output) are handed to warps
//      dynamically, heaviest families first; all 32 lanes of a warp walk the same trees,
//   D. lanes read their results back and continue.
// Finished games are replaced at once from a global per-matchup game counter, so lanes stay busy
// until the matchup is exhausted (the warp-level compaction of finished games the north star asks
// for is the same mechanism: a parked lane is either refilled or absent from every request list).
//
// The game rules live here once, as step functions ("the game rules, one step at a time": new_game ... after_yards),
// and so do the pieces of a round (next_matchup, request_rank, plan_round, walk_requests).  advance_lane below and the
// trip loop of sim_memo_kernel (fmc_sim_memo.cuh) both call them: a rule is changed in one place for both kernels.
#pragma once

#include <type_traits>

#include "fmc_device.cuh"
#include "fmc_pack.hpp"

namespace fmc {

#ifndef FMC_SIM_THREADS
#define FMC_SIM_THREADS 1024
#endif
#ifndef FMC_SIM_CTAS_PER_SM
#define FMC_SIM_CTAS_PER_SM 1
#endif
constexpr int kSimThreads = FMC_SIM_THREADS;
constexpr int kSimCtasPerSm = FMC_SIM_CTAS_PER_SM;
constexpr int kNumFam = 6;           // S1, S2, PQ, RQ, SQ, PM  (== model ids 0..5)
constexpr int kNumKeys = kNumFam * 2;

struct TableRef {
    uint32_t win_lo, win_hi;    // address of the 1 MiB window the node table sits in
    uint32_t stream_off[5];     // per output: first uint4 of its root stream in the global stream buffer
    uint32_t consts_off[5];     // per output: first uint2 of its constants side stream
    uint16_t n_groups[5];
    uint8_t n_outputs;
    uint8_t max_depth;
    uint8_t multi_window;       // table larger than one window: groups carry their window index
    float base[5];              // xgb margin offsets (f32-exact) ...
    double base64[3];           // ... or sklearn init constants
};

// Usage tables of one team as the kernel reads them (include/fmc.h fmc_team_usage): role 0 passer, 1 rusher, 2 target.
struct UsageDev {
    double cdf[3][FMC_MAX_USAGE];    // cumsum(share) / total, the array Generator.choice searches (FMC:625-635)
    int8_t n[3];
    int8_t slot[3][FMC_MAX_USAGE];   // box line of a tracked name, -1 = not tracked
    int8_t row[3][FMC_MAX_USAGE];    // 0/1 feature row of a name some model has a column for, -1 = lights nothing
};

// The state every game of a matchup entry starts from (include/fmc.h fmc_game_state); kickoff unless
// fmc_set_start_states says otherwise.
struct StartDev {
    double dist, ytg;
    int32_t sec, down;
    int32_t offense;                 // -1: team (g & 1), the opening-kickoff rule; 0 / 1: that team
    int32_t score[2];
    int32_t fourth_down;             // FMC_4TH_*: the forced choice of the first iteration of every game (0: the policy)
};

struct MatchupDev {
    double bias[2], ymul[2], mz[2], tanh35[2];
    unsigned long long game_begin, game_end, out_offset;
    StartDev start;
    int32_t memo_id;                 // specialisation of this entry: index of its RankSpec set and its memo key field
    int32_t ot_start;                // overtime state every game starts from (Overtime<true>::game_start), 0: regulation
    TableRef tbl[kNumFam][2];
    UsageDev usage[2];               // player mode only
};

// Player mode: the sampled names of a play are 0/1 feature rows behind the numeric rows of a request:
// pass families: passer with name row r -> feature row kDynRow0 + r, target -> kDynRow0 + FMC_MAX_PASSER_ROWS + r;
// run yards: rusher -> kDynRow0 + r.  Only names that some model has a one-hot column for get a name row
// (UsageDev::row); every other name lights nothing (OneHotEncoder(handle_unknown='ignore')).
constexpr int kDynRow0 = kSimRows;
constexpr int kDynRows = FMC_MAX_PASSER_ROWS + FMC_MAX_NAME_ROWS;

struct SimKernelArgs {
    const MatchupDev *matchups;
    int n_matchups;
    unsigned long long *next_game;     // [n_matchups] global work counters (start at game_begin)
    const uint4 *root_stream;          // root streams of every table (fmc_pack.hpp)
    const uint2 *consts;               // constants side streams
    uint32_t seed_lo, seed_hi;
    int policy, sampler, stage2_mode;
    int pass_class;                    // index of "pass" among the play model's classes (FMC:423)
    float play_temp;
    double qy_noise;
    double standin[3];
    // play_model standardisation of the six varying numerics (rows 0..5): x = (x - mean) / scale
    double pm_mean[6], pm_scale[6];
    int pm_scaled[6];
    uint32_t *scores;
    uint32_t *hist;
    unsigned long long *counters;
    const double *stream;
    double *trace;
    uint16_t *iters;
    fmc_player_rec *players;           // player mode: [games][2][n_slots] per-game box lines (optional output)
    uint32_t *player_hist;             // player mode: [n_matchups][2][n_slots][FMC_PH_BINS] (optional output)
    fmc_player_rec *box_scratch;       // player mode: [lanes of the grid][2][n_slots] running box of each lane's game
    int n_slots;
    // player mode: name rows actually needed by the matchups of this launch (a chunk has kSimRows + name_rows rows):
    // passer rows [kDynRow0, +n_prow), target rows behind them, rusher rows [kDynRow0, +n_rrow)
    int n_prow, n_trow, n_rrow, name_rows;
    // period outputs (fmc_simulate_segments; read only by the instantiations with the period hooks): the Q1..Q3 end scores of every game
    // (never NULL there: the library supplies device scratch when the caller did not ask for them) and the optional
    // per-segment histograms
    uint32_t *period_scores;           // [games][3]
    uint32_t *segment_hist;            // [n_matchups][2][FMC_N_SEGMENTS][BINS][BINS]
    // scoring-sequence outputs (fmc_simulate_markets; read only by the instantiations with the sequence hooks): the
    // next-score and drive-result words of every game (never NULL there, device scratch like period_scores) and the
    // optional per-entry histogram
    uint32_t *sequence;                // [games][2]
    uint32_t *sequence_hist;           // [n_matchups][2][FMC_SEQ_BINS]
    // overtime (fmc_simulate_overtime; read only by the instantiations with overtime): the rules' two parameters and the
    // optional outputs
    int ot_max_periods, ot_snap_clock;
    uint8_t *ot_periods;               // [games]
    uint32_t *ot_hist;                 // [n_matchups][2][FMC_OT_MAX_PERIODS + 1][3]
};

enum Stage : int {
    ST_NEED_GAME = 0, ST_ITER, ST_WAIT_PM, ST_WAIT_S1, ST_WAIT_S2, ST_WAIT_PQ, ST_WAIT_RQ, ST_WAIT_SQ, ST_IDLE
};

// slot ids of the 16-slot draw record
enum { S_U_CALL = 0, S_U_COMP, S_Z_YARDS, S_U_EX, S_U_BOOST, S_U_FIN, S_U_S2, S_Z_INT,
       S_U_GO, S_U_FG, S_Z_GROSS, S_Z_RET, S_U_TB, S_U_P1, S_U_WR, S_U_YQ };

struct Lane {
    unsigned long long game;   // game id inside the matchup
    double dist, ytg;
    int sec, down, offense, period, going, iter;
    int score[2];
    int stage;
    int plays;                 // plays of the current game
    int p1, wr;                // player mode: usage entries sampled for the current play (passer | rusher, target)
    int home;                  // index of the running player box this game (and its successors) accumulates in
};
// The lane of the instantiations with overtime: the overtime state (Overtime<true>), 0 in regulation.  A type of its own so
// that the lane of every other instantiation keeps its layout.
struct OtLane : Lane {
    int ot;
};
template <bool OT> using LaneT = typename std::conditional<OT, OtLane, Lane>::type;

// A game's state between rounds: nine registers instead of sixteen, so that the tree walk (which runs with
// every lane's game parked) has room for its eight gather chains.
struct PackedLane {
    unsigned long long game;
    double dist, ytg;
    uint32_t a;     // sec:12 | down:10 | period:3 | offense:1 | going:1 | stage:4 | overtime:1
    uint32_t b;     // iter:10 | plays:10 | p1:5 | wr:5 (player mode)
    uint32_t c;     // score[0]:16 | score[1]:16
};
// OT: the instantiations with overtime.  In overtime the clock does not run: every snap is played at the snap clock of
// the launch, so the sec field holds the overtime state instead (bit 31 set) and unpacking restores the clock from a.
template <bool OT = false>
__device__ __forceinline__ PackedLane pack_lane(const LaneT<OT> &L) {
    PackedLane P;
    P.game = L.game; P.dist = L.dist; P.ytg = L.ytg;
    P.a = (uint32_t)L.sec | ((uint32_t)L.down << 12) | ((uint32_t)L.period << 22) | ((uint32_t)L.offense << 25) |
          ((uint32_t)L.going << 26) | ((uint32_t)L.stage << 27);
    if constexpr (OT) {
        if (L.ot) P.a = (P.a & ~0xFFFu) | (uint32_t)L.ot | 0x80000000u;
    }
    P.b = (uint32_t)L.iter | ((uint32_t)L.plays << 10) | ((uint32_t)L.p1 << 20) | ((uint32_t)L.wr << 25);
    P.c = (uint32_t)L.score[0] | ((uint32_t)L.score[1] << 16);
    return P;
}
template <bool OT = false>
__device__ __forceinline__ LaneT<OT> unpack_lane(const PackedLane &P, const SimKernelArgs &a) {
    LaneT<OT> L;
    L.game = P.game; L.dist = P.dist; L.ytg = P.ytg;
    L.sec = (int)(P.a & 0xFFFu); L.down = (int)((P.a >> 12) & 0x3FFu); L.period = (int)((P.a >> 22) & 7u);
    L.offense = (int)((P.a >> 25) & 1u); L.going = (int)((P.a >> 26) & 1u); L.stage = (int)(P.a >> 27);
    L.iter = (int)(P.b & 0x3FFu); L.plays = (int)((P.b >> 10) & 0x3FFu);
    L.p1 = (int)((P.b >> 20) & 0x1Fu); L.wr = (int)((P.b >> 25) & 0x1Fu);
    L.score[0] = (int)(P.c & 0xFFFFu); L.score[1] = (int)(P.c >> 16);
    if constexpr (OT) {
        L.stage &= 15;
        L.ot = 0;
        if (P.a >> 31) { L.ot = L.sec; L.sec = a.ot_snap_clock; }
    }
    return L;
}
// (a lane gets a new stage this way only between matchups, without a game: the overtime bit is cleared with the stage)
__device__ __forceinline__ void set_stage(PackedLane &P, int stage) { P.a = (P.a & 0x07FFFFFFu) | ((uint32_t)stage << 27); }
// the state of a lane without a game
__device__ __forceinline__ PackedLane idle_lane() {
    Lane L0;
    L0.game = 0; L0.dist = 0.0; L0.ytg = 0.0; L0.sec = 0; L0.down = 0; L0.offense = 0; L0.period = 0; L0.going = 0;
    L0.iter = 0; L0.score[0] = 0; L0.score[1] = 0; L0.plays = 0; L0.p1 = 0; L0.wr = 0; L0.home = 0;
    L0.stage = ST_IDLE;
    return pack_lane(L0);
}

// python semantics helpers (FMC:97 softclip = max(lo, min(hi, x)))
__device__ __forceinline__ double pymax(double a, double b) { return (b > a) ? b : a; }
__device__ __forceinline__ double pymin(double a, double b) { return (b < a) ? b : a; }
__device__ __forceinline__ double softclip(double x, double lo, double hi) {
    const double m = (x < hi) ? x : hi;
    return (m > lo) ? m : lo;
}

// TEST = true: the launch has an injected draw stream and/or a trace buffer (parity tests); the production
// instantiation carries neither branch.
template <bool TEST>
struct Draws {
    const SimKernelArgs &a;
    const double *rec;        // injected record base for this game (or nullptr)
    uint4 ctr;                // x,y = game; z = matchup; w = iter << 2 | block
    // ONE cached Philox block: the draw sites of an iteration visit the record block by block (play call /
    // completion / yards / explosive in block 0, boost / finish / stage 2 / return in block 1, fourth down in 2-3),
    // so a single block costs no extra Philox calls and twelve registers less than caching all four.
    int cur;
    uint4 w;
    __device__ Draws(const SimKernelArgs &a_, const MatchupDev &M, int matchup, const Lane &L) : a(a_) {
        rec = (TEST && a.stream) ? a.stream + ((size_t)(M.out_offset + (L.game - M.game_begin)) * FMC_MAX_ITERS + (size_t)L.iter) * FMC_N_SLOTS
                                 : nullptr;
        ctr = make_uint4((uint32_t)L.game, (uint32_t)(L.game >> 32), (uint32_t)matchup, (uint32_t)L.iter << 2);
        cur = -1;
    }
    __device__ __forceinline__ uint32_t word(int slot) {
        const int b = slot >> 2;
        if (b != cur) {
            uint4 c = ctr;
            c.w |= (uint32_t)b;
            w = philox4x32_10(c, make_uint2(a.seed_lo, a.seed_hi));
            cur = b;
        }
        const int j = slot & 3;
        return j == 0 ? w.x : (j == 1 ? w.y : (j == 2 ? w.z : w.w));
    }
    __device__ __forceinline__ double u(int slot) { return (TEST && rec) ? rec[slot] : u01(word(slot)); }
    __device__ __forceinline__ double z(int slot) { return (TEST && rec) ? rec[slot] : ppnd16(u01(word(slot))); }
};

// ---- state transitions -------------------------------------------------------------------------
__device__ __forceinline__ void change_possession(Lane &L, bool has_spot, double spot) {   // FMC:943-953
    L.offense ^= 1;
    L.down = 1;
    L.dist = 10.0;
    L.going = 0;
    L.ytg = has_spot ? spot : 100.0 - L.ytg;
}
__device__ __forceinline__ void advance_down(Lane &L, double gained) {                      // FMC:932-941
    L.ytg = pymax(0.0, L.ytg - gained);
    if (gained + 1e-6 >= L.dist) {
        L.down = 1;
        L.dist = 10.0;
        L.ytg = pymax(0.0, L.ytg - 0.0);
    } else {
        L.down += 1;
        L.dist -= gained;
        if (L.down > 4) change_possession(L, false, 0.0);
    }
}
// ---- period outputs (fmc_simulate_segments, include/fmc.h FMC_N_SEGMENTS) --------------------------------------------
// The hooks of the clock and of the end of a game.  Periods<false> is empty: the instantiations without period outputs
// compile to the code they had before the hooks existed.  Periods<true> keeps no lane state: the game's own
// period_scores row is its state.  The score at the end of quarter q goes to row[q - 1] when the clock crosses the
// boundary; later boundaries read the earlier words as their segment bases.  The writes and the later reads of one
// game's row are made by threads of ONE CTA in different rounds, with a __syncthreads() between them (sim_kernel moves
// games between the threads of its CTA only, at the regrouping barriers; sim_memo_kernel never moves a game, so there
// it is the same thread).
__device__ __forceinline__ uint32_t score_word(const Lane &L) { return (uint32_t)L.score[0] | ((uint32_t)L.score[1] << 16); }

template <bool SEG> struct Periods;
template <> struct Periods<false> {
    static constexpr bool kOn = false;
    __device__ __forceinline__ Periods(const SimKernelArgs &, const MatchupDev &, int) {}
    __device__ __forceinline__ void quarter_end(const Lane &, int) const {}
    __device__ __forceinline__ void game_end(const Lane &) const {}
};
template <> struct Periods<true> {
    static constexpr bool kOn = true;
    const SimKernelArgs &a;
    const MatchupDev &M;
    int matchup;
    __device__ __forceinline__ Periods(const SimKernelArgs &a_, const MatchupDev &M_, int m) : a(a_), M(M_), matchup(m) {}
    __device__ __forceinline__ uint32_t *row(const Lane &L) const {
        return a.period_scores + (size_t)(M.out_offset + (L.game - M.game_begin)) * 3;
    }
    __device__ __forceinline__ uint32_t start_word() const { return (uint32_t)M.start.score[0] | ((uint32_t)M.start.score[1] << 16); }
    // base of a segment that starts at boundary b: the score there if the game was simulated across it, else the start
    __device__ __forceinline__ uint32_t base(const uint32_t *r, int q_before) const {
        return M.start.sec > 3600 - 900 * q_before ? r[q_before - 1] : start_word();
    }
    __device__ __forceinline__ void add(const Lane &L, int seg, uint32_t end, uint32_t base) const {
        const int pa = (int)(end & 0xFFFFu) - (int)(base & 0xFFFFu), pb = (int)(end >> 16) - (int)(base >> 16);
        const int ha = pa < FMC_HIST_BINS ? pa : FMC_HIST_BINS - 1, hb = pb < FMC_HIST_BINS ? pb : FMC_HIST_BINS - 1;
        atomicAdd(a.segment_hist + ((((size_t)matchup * 2 + (L.game & 1ULL)) * FMC_N_SEGMENTS + seg) * FMC_HIST_BINS + ha) * FMC_HIST_BINS + hb, 1u);
    }
    // quarter q (1..3) ended with the play just ticked
    __device__ __forceinline__ void quarter_end(const Lane &L, int q) const {
        uint32_t *r = row(L);
        const uint32_t w = score_word(L);
        r[q - 1] = w;
        if (a.segment_hist) {
            add(L, FMC_SEG_Q1 + q - 1, w, q > 1 ? base(r, q - 1) : start_word());
            if (q == 2) add(L, FMC_SEG_H1, w, start_word());
        }
    }
    // the game is over: sentinels for the quarter ends at or before the start state; Q4 and H2 end here
    __device__ __forceinline__ void game_end(const Lane &L) const {
        uint32_t *r = row(L);
#pragma unroll
        for (int q = 1; q <= 3; ++q)
            if (M.start.sec <= 3600 - 900 * q) r[q - 1] = FMC_PERIOD_NONE;
        if (a.segment_hist) {
            const uint32_t w = score_word(L);
            add(L, FMC_SEG_Q4, w, base(r, 3));
            add(L, FMC_SEG_H2, w, base(r, 2));
        }
    }
};

// ---- scoring-sequence outputs (fmc_simulate_markets, include/fmc.h FMC_SEQ_NONE) -------------------------------------
// The hooks of the scoring plays and of the plays that end a drive, called before the play's tick so that they see the
// clock at the snap (a play's own result therefore comes before the end of the half its tick crosses).  Sequence<false>
// is empty.  Sequence<true> keeps no lane state: the game's own sequence row is its state, set at the start of the game
// (next score FMC_SEQ_NONE, drive open) and read back by the later hooks, under the same rule as the period rows.  The
// race needs no state: scores only grow, so the one play that takes a team from below N to N or more while the other is
// below N decides target N; a target either team had reached at the start state can never be decided that way, nor end
// with both teams below it, so it is counted nowhere.
constexpr uint32_t kDriveOpen = 0xFFFFFFFFu;

template <bool SEQ> struct Sequence;
template <> struct Sequence<false> {
    __device__ __forceinline__ Sequence(const SimKernelArgs &, const MatchupDev &, int) {}
    __device__ __forceinline__ void game_start(const Lane &) const {}
    __device__ __forceinline__ void scored(const Lane &, int, int, int) const {}
    __device__ __forceinline__ void drive_end(const Lane &, int, int) const {}
    __device__ __forceinline__ void game_end(const Lane &) const {}
};
template <> struct Sequence<true> {
    const SimKernelArgs &a;
    const MatchupDev &M;
    int matchup;
    __device__ __forceinline__ Sequence(const SimKernelArgs &a_, const MatchupDev &M_, int m) : a(a_), M(M_), matchup(m) {}
    __device__ __forceinline__ uint32_t *row(const Lane &L) const {
        return a.sequence + (size_t)(M.out_offset + (L.game - M.game_begin)) * 2;
    }
    __device__ __forceinline__ void count(const Lane &L, int bin) const {
        if (a.sequence_hist) atomicAdd(a.sequence_hist + ((size_t)matchup * 2 + (L.game & 1ULL)) * FMC_SEQ_BINS + bin, 1u);
    }
    __device__ __forceinline__ void game_start(const Lane &L) const {
        uint32_t *r = row(L);
        r[0] = FMC_SEQ_NONE;
        r[1] = kDriveOpen;
    }
    // `team` scored (kind FMC_SEQ_TD / FMC_SEQ_FG) on the play snapped at `clock`; L.score already holds the points
    __device__ __forceinline__ void scored(const Lane &L, int team, int kind, int clock) const {
        uint32_t *r = row(L);
        if (r[0] == FMC_SEQ_NONE) {
            r[0] = FMC_SEQ_WORD(team, kind, clock);
            count(L, FMC_SEQ_BIN_NEXT(team, kind, clock));
        }
        if (a.sequence_hist) {
            constexpr int targets[FMC_N_RACE] = FMC_RACE_TARGETS;
            const int now = L.score[team], before = now - (kind == FMC_SEQ_TD ? 7 : 3), other = L.score[team ^ 1];
#pragma unroll
            for (int t = 0; t < FMC_N_RACE; ++t)
                if (before < targets[t] && now >= targets[t] && other < targets[t]) count(L, FMC_SEQ_BIN_RACE(t, team));
        }
    }
    // the play snapped at `clock` ends the drive with result `code`, unless an earlier play ended it
    __device__ __forceinline__ void drive_end(const Lane &L, int code, int clock) const {
        uint32_t *r = row(L);
        if (r[1] == kDriveOpen) {
            r[1] = FMC_DRIVE_WORD(code, clock);
            count(L, FMC_SEQ_BIN_DRIVE(code));
        }
    }
    __device__ __forceinline__ void game_end(const Lane &L) const {
        if (row(L)[0] == FMC_SEQ_NONE) count(L, FMC_SEQ_BIN_NONE);
        drive_end(L, FMC_DRIVE_GAME, 0);
        if (a.sequence_hist) {
            constexpr int targets[FMC_N_RACE] = FMC_RACE_TARGETS;
#pragma unroll
            for (int t = 0; t < FMC_N_RACE; ++t)
                if (L.score[0] < targets[t] && L.score[1] < targets[t]) count(L, FMC_SEQ_BIN_RACE(t, FMC_RACE_NEITHER));
        }
    }
};

// ---- overtime (fmc_simulate_overtime, include/fmc.h FMC_OT_MAX_PERIODS) ------------------------------------------------
// The rule that plays a game level at the end of regulation to a result.  Overtime<false> is the reference's end of the
// game at 0:00.  Overtime<true> keeps its state in OtLane::ot: the period k (1..FMC_OT_MAX_PERIODS), whether the second
// possession of the period is on, whether the snap is a two-point try, and a period-2 touchdown whose try is still due.
// The team with the first possession of period k is (g & 1) in period 1 and alternates, or the other team when kOtFlip is
// set (a game started in overtime, fmc_set_start_states_overtime); a possession ends when the offense changes (every place
// that calls change_possession) or, for a try, after its one snap.  All bookkeeping runs at the start of an iteration
// (over), before the trace row, except the points of a touchdown, which after_yards adds.
//
// A start in overtime (MatchupDev::ot_start, written by the library) is the state before the bookkeeping of iteration 0
// that produces the start snap: k | second for a snap of a possession (offense = team()); for a try, 2 | second | kOtTd
// in period 2, (k - 1) | kOtSecond | kOtTry for the first try of period k >= 3 and k | kOtTry for its second.  Its kOtFlip
// says that team 1 had the first possession of period 1; game_start turns that into the game's own bit.
enum : int { kOtPeriod = 31, kOtSecond = 32, kOtTry = 64, kOtTd = 128, kOtFlip = 256 };

template <bool OT> struct Overtime;
template <> struct Overtime<false> {
    __device__ __forceinline__ Overtime(const SimKernelArgs &, int) {}
    __device__ __forceinline__ void game_start(const Lane &, const MatchupDev &) const {}
    // the game is over at the start of an iteration
    __device__ __forceinline__ bool over(const Lane &L) const { return L.sec <= 0; }
    // points of a touchdown just scored
    __device__ __forceinline__ int touchdown(const Lane &) const { return 7; }
    // the snap credits player box lines
    __device__ __forceinline__ bool credits(const Lane &) const { return true; }
    __device__ __forceinline__ void game_end(const Lane &, unsigned long long *, size_t) const {}
};
template <> struct Overtime<true> {
    const SimKernelArgs &a;
    int matchup;
    __device__ __forceinline__ Overtime(const SimKernelArgs &a_, int m) : a(a_), matchup(m) {}
    // the step functions see a Lane; the lanes of these instantiations are OtLanes
    __device__ __forceinline__ static int &st(Lane &L) { return static_cast<OtLane &>(L).ot; }
    __device__ __forceinline__ static int st(const Lane &L) { return static_cast<const OtLane &>(L).ot; }
    __device__ __forceinline__ void game_start(Lane &L, const MatchupDev &M) const {
        const int s = M.ot_start;
        st(L) = s ? s ^ ((int)(L.game & 1ULL) << 8) : 0;
    }
    // the team whose possession is on
    __device__ __forceinline__ static int team(const Lane &L) {
        const int o = st(L);
        return (int)(L.game & 1ULL) ^ ((o >> 8) & 1) ^ (((o & kOtPeriod) - 1) & 1) ^ ((o & kOtSecond) ? 1 : 0);
    }
    __device__ __forceinline__ static void two_point_try(Lane &L) {
        st(L) |= kOtTry;
        L.down = 1; L.dist = 3.0; L.ytg = 3.0; L.going = 0;
    }
    // the possession the state names starts: 1st & 10 at the opponent's 25 in periods 1 and 2, a two-point try from period 3
    __device__ __forceinline__ static void possession(Lane &L) {
        L.offense = team(L);
        if ((st(L) & kOtPeriod) >= 3) two_point_try(L);
        else { L.down = 1; L.dist = 10.0; L.ytg = 25.0; L.going = 0; }
    }
    __device__ __forceinline__ bool over(Lane &L) const {
        int &o = st(L);
        if (o == 0) {
            if (L.sec > 0) return false;
            if (L.score[0] != L.score[1]) return true;
            o = 1;                                             // level at 0:00: period 1, first possession
            possession(L);
        } else {
            const int t = team(L), k = o & kOtPeriod;
            if (o & kOtTd) {                                   // a period-2 touchdown: its try, unless it already won
                if ((o & kOtSecond) && L.score[t] > L.score[t ^ 1]) return true;
                o &= ~kOtTd;
                L.offense = t;
                two_point_try(L);
            } else if ((o & kOtTry) || L.offense != t) {      // the possession is over
                if (!(o & kOtSecond)) o = (o & kOtFlip) | k | kOtSecond;
                else if (L.score[0] != L.score[1] || k >= a.ot_max_periods) return true;
                else o = (o & kOtFlip) | (k + 1);
                possession(L);
            }
        }
        if (L.iter >= FMC_MAX_ITERS) return true;
        L.sec = a.ot_snap_clock;
        return false;
    }
    __device__ __forceinline__ int touchdown(Lane &L) const {
        int &o = st(L);
        if (o & kOtTry) return 2;
        if ((o & kOtPeriod) == 2) { o |= kOtTd; return 6; }
        return 7;
    }
    __device__ __forceinline__ bool credits(const Lane &L) const { return !(st(L) & kOtTry); }
    // periods played to the per-game output, the game to the overtime histogram and counters
    __device__ __forceinline__ void game_end(const Lane &L, unsigned long long *stat, size_t oi) const {
        const int k = st(L) & kOtPeriod;
        if (a.ot_periods) a.ot_periods[oi] = (uint8_t)k;
        if (a.ot_hist) {
            const int r = L.score[0] > L.score[1] ? FMC_OT_A : (L.score[1] > L.score[0] ? FMC_OT_B : FMC_OT_LEVEL);
            atomicAdd(a.ot_hist + (((size_t)matchup * 2 + (L.game & 1ULL)) * (FMC_OT_MAX_PERIODS + 1) + k) * 3 + r, 1u);
        }
        if (k) {
            atomicAdd(&stat[FMC_C_OT_GAMES], 1ULL);
            atomicAdd(&stat[FMC_C_OT_PERIODS], (unsigned long long)k);
        }
    }
};

// ---- fourth-down decisions (fmc_game_state.fourth_down, include/fmc.h FMC_4TH_POLICY) -------------------------------
// The choice fourth_down makes at a game's first iteration.  Decision<false> has none to make: fourth_down draws it, as
// the reference does.  Decision<true> reads the forced choice of the entry from the CTA's copy of its MatchupDev (the
// record new_game started the game from): no lane state.  Both kernels count the iteration before they call fourth_down,
// so the first iteration is the call that sees L.iter == 1.
template <bool DEC> struct Decision;
template <> struct Decision<false> {
    __device__ __forceinline__ Decision(const MatchupDev &) {}
    __device__ __forceinline__ int forced(const Lane &) const { return FMC_4TH_POLICY; }
};
template <> struct Decision<true> {
    const MatchupDev &M;
    __device__ __forceinline__ Decision(const MatchupDev &M_) : M(M_) {}
    __device__ __forceinline__ int forced(const Lane &L) const { return L.iter == 1 ? M.start.fourth_down : FMC_4TH_POLICY; }
};

// The hook policy of the step functions: HOOKS is a mask of the launch's optional outputs.  Hooks<0> compiles to the code
// without hooks; kOn says whether any hook is in (a hooked field goal adds its points before its tick).  OT: the overtime
// rule, DEC: the forced fourth-down choices, both instantiated with HOOKS = 0 only.  Overtime<OT> and Decision<DEC> are
// bases, so that Hooks<HOOKS, false, false> keeps the layout it had before either existed (an empty member would not).
enum { kHookPeriods = 1, kHookSequence = 2 };
template <int HOOKS, bool OT = false, bool DEC = false>
struct Hooks : Overtime<OT>, Decision<DEC> {
    static_assert(!(OT && HOOKS), "overtime has no period or sequence outputs");
    static_assert(!(DEC && HOOKS), "forced fourth-down choices have no period or sequence outputs");
    static constexpr bool kOn = HOOKS != 0;
    Periods<(HOOKS & kHookPeriods) != 0> per;
    Sequence<(HOOKS & kHookSequence) != 0> seq;
    __device__ __forceinline__ Hooks(const SimKernelArgs &a, const MatchupDev &M, int m)
        : Overtime<OT>(a, m), Decision<DEC>(M), per(a, M, m), seq(a, M, m) {}
    __device__ __forceinline__ const Overtime<OT> &ot() const { return *this; }
    __device__ __forceinline__ const Decision<DEC> &dec() const { return *this; }
    __device__ __forceinline__ void game_start(const Lane &L) const { seq.game_start(L); }
    // quarter q ended with the play snapped at `snap`; the end of the half ends the drive if nothing else did
    __device__ __forceinline__ void quarter_end(const Lane &L, int q, int snap) const {
        per.quarter_end(L, q);
        if (q == 2) seq.drive_end(L, FMC_DRIVE_HALF, snap);
    }
    __device__ __forceinline__ void scored(const Lane &L, int team, int kind, int clock) const { seq.scored(L, team, kind, clock); }
    __device__ __forceinline__ void drive_end(const Lane &L, int code, int clock) const { seq.drive_end(L, code, clock); }
    __device__ __forceinline__ void game_end(const Lane &L) const {
        per.game_end(L);
        seq.game_end(L);
    }
};

template <class Pk>
__device__ __forceinline__ void tick_clock(Lane &L, int base, const Pk &pk) {                // FMC:956-968
    const int snap = L.sec;
    const int v = L.sec - base;
    L.sec = v > 0 ? v : 0;
    const int old = L.period;
    L.period = L.sec > 0 ? 4 - ((L.sec - 1) / 900) : 4;
    if (L.period != old) pk.quarter_end(L, old, snap);
    if (L.period != old && L.period == 3) change_possession(L, true, 75.0);
}
__device__ __forceinline__ double pass_prob_v1(int down, double distance, double ytg, int sec, int sd) {  // FMC:719-735
    double base = 0.53;
    if (down == 1) base += 0.02 + 0.010 * pymax(0.0, distance - 10.0) / 10.0;
    if (down == 2) base += 0.12 + 0.020 * pymax(0.0, distance - 7.0) / 10.0;
    if (down == 3) base += 0.28 + 0.030 * pymax(0.0, distance - 5.0) / 10.0;
    if (down == 4) base += 0.45 + 0.035 * pymax(0.0, distance - 3.0) / 10.0;
    if (ytg <= 10.0) base -= 0.05;
    if (ytg <= 5.0) base -= 0.03;
    const bool two_min = (sec % 1800) <= 120;
    if (two_min && sd < 0) base += 0.22;
    if (sec < 600 && sd < 0) base += 0.06;
    return softclip(base, 0.10, 0.95);
}
__device__ __forceinline__ double explosive_prob(double mz, double ytg) {                   // FMC:467-472
    double base = 0.03 + 0.05 * mz;
    if (ytg > 60.0) base += 0.02;
    if (ytg > 40.0) base += 0.01;
    return softclip(base, 0.01, 0.12);
}
__device__ __forceinline__ double rz_finish_prob(double ytg, double tanh35, int down, bool pass) {  // FMC:444-457
    double base = (pass ? 0.32 : 0.30) + 0.30 * (pymax(0.0, 7.0 - ytg) / 7.0);
    int dl = 4 - down;
    if (dl < 0) dl = 0;
    base += (pass ? 0.03 : 0.04) * (double)dl;
    const double tilt = (pass ? 0.08 : 0.07) * tanh35;
    return pass ? softclip(base + tilt, 0.22, 0.68) : softclip(base + tilt, 0.20, 0.62);
}
__device__ __forceinline__ double field_goal_prob(double d) {                               // FMC:858-865
    if (d < 30.0) return 0.96;
    if (d < 40.0) return 0.92;
    if (d < 50.0) return 0.78;
    if (d <= 55.0) return 0.50;
    return 0.25;
}
__device__ __forceinline__ double go_for_it_prob(double ytg, double dist, int sd, int sec) {  // FMC:1336-1378
    if (sec < 300 && sd < 0) return (ytg > 38.0) ? 0.90 : 0.75;
    double p = 0.0;
    if (ytg > 80.0) { if (dist <= 1.0) p = 0.15; else if (dist <= 2.0) p = 0.05; }
    else if (ytg > 65.0) { if (dist <= 1.0) p = 0.30; else if (dist <= 2.0) p = 0.15; }
    else if (ytg > 50.0) { if (dist <= 1.0) p = 0.60; else if (dist <= 2.0) p = 0.40; else if (dist <= 3.0) p = 0.20; }
    else if (ytg > 35.0) { if (dist <= 1.0) p = 0.85; else if (dist <= 2.0) p = 0.65; else if (dist <= 3.0) p = 0.40; else if (dist <= 4.0) p = 0.25; }
    else if (ytg > 20.0) { if (dist <= 1.0) p = 0.75; else if (dist <= 2.0) p = 0.50; else if (dist <= 3.0) p = 0.30; }
    else if (ytg > 10.0) { if (dist <= 1.0) p = 0.70; else if (dist <= 2.0) p = 0.45; }
    else { if (dist <= 2.0) p = 0.85; else if (dist <= 4.0) p = 0.40; }
    if (sec < 300 && sd > 0) p *= 0.85;
    return softclip(p, 0.0, 1.0);
}

// yardage samplers FMC:817-852 / sim_helpers.py:32-38
template <bool TEST>
__device__ __forceinline__ double sample_yards(const SimKernelArgs &a, Draws<TEST> &D, const double q[3], double sig_floor,
                                               double lo, double hi) {
    if (a.sampler == 0) {
        const double sigma = pymax(sig_floor, (q[2] - q[0]) / 2.56);
        const double y = q[1] + sigma * D.z(S_Z_YARDS);
        return softclip(y, lo, hi);
    }
    const double u = D.u(S_U_YQ);
    double y = (u < 0.5) ? q[0] + (q[1] - q[0]) * (u / 0.5) : q[1] + (q[2] - q[1]) * ((u - 0.5) / 0.5);
    y = y + (0.0 + a.qy_noise * D.z(S_Z_YARDS));
    const double m = (y < lo) ? lo : y;      // np.clip
    return (m > hi) ? hi : m;
}

// matchups a slate works on at a time (see the matchup selection of the kernels)
#ifndef FMC_SLATE_WAVE
#define FMC_SLATE_WAVE 8
#endif
constexpr int kSlateWave = FMC_SLATE_WAVE;

// Shared-memory state of the rounds, common to sim_kernel (SimShared) and sim_memo_kernel (MemoShared).
struct RoundShared {
    MatchupDev M;
    int cur_matchup;
    int scan_from;                    // no matchup below this index has games left
    unsigned int cnt[2][kNumKeys];    // requests per key, double-buffered by round parity
    unsigned int off[kNumKeys];       // first position of each key's list
    unsigned int evalc[kNumKeys];     // requests of the key that are evaluated this round (the rest wait one round)
    unsigned int aged[kNumKeys];      // the key's tail was held back last round: evaluate everything now
    unsigned int item_prefix[kNumKeys + 1];
    unsigned int item_next;
    unsigned long long stat[FMC_N_COUNTERS];
};
struct SimShared : RoundShared {
    unsigned int dense_off[kNumKeys];  // first thread of each key's evaluated requests after the regrouping
    unsigned int n_eval, rest;         // evaluated requests this round; counter for the other lanes
};

// A key whose last chunk would hold fewer than this many requests holds that tail back for one round (the
// lanes re-post the same request next round, where it joins a fuller chunk); 0 disables.
#ifndef FMC_DEFER_BELOW
#define FMC_DEFER_BELOW 12
#endif
constexpr unsigned int kDeferBelow = FMC_DEFER_BELOW;

// Requests are kept in 32-request chunks, feature-major ([feature][lane]); every key's list starts on
// a chunk boundary, so at most kSimThreads/32 + kNumKeys chunks are in use.
constexpr int kSimChunks = kSimThreads / 32 + kNumKeys;
__host__ __device__ constexpr int chunk_floats(bool players) { return (kSimRows + (players ? kDynRows : 0)) * 32; }
constexpr size_t kSimSharedBytes = ((sizeof(SimShared) + 15) / 16) * 16;
__host__ __device__ constexpr size_t sim_feat_bytes(bool players) { return (size_t)kSimChunks * chunk_floats(players) * 4; }
constexpr size_t kSimResultBytes = (size_t)kSimChunks * 32 * 3 * 8;
// Regrouping: after the compaction every game moves to the thread at its request's rank, so that a warp resumes
// games of ONE (family, orientation) next round instead of six different stages.  The ten words of a game's record
// travel through shared memory: eight in the result buffer (free between the read-back and the walk), two in
// kSimXchgExtraBytes.
constexpr size_t kSimXchgExtraBytes = (size_t)2 * kSimThreads * 4;
static_assert(kSimResultBytes >= (size_t)8 * kSimThreads * 4, "the result buffer must hold eight exchange words per thread");

// keys in processing order, heaviest family first (LPT-style dynamic scheduling):
// PQ, RQ (1200 depth-3 trees x3 outputs), S2, PM, SQ, S1
__device__ __constant__ int kKeyOrder[kNumKeys] = {4, 5, 6, 7, 2, 3, 10, 11, 8, 9, 0, 1};

__device__ __forceinline__ int splits_of(int fam) { return fam == 0 ? 1 : (fam == 5 ? 5 : 3); }

// Outcome of the not-complete branch (FMC:751-770 nudges + 3-way categorical FMC:1157).
__device__ __forceinline__ int stage2_outcome(const double raw[3], double u2) {
    double p_inc = pymax(0.0, raw[0]), p_int = pymax(0.0, raw[1]), p_sck = pymax(0.0, raw[2]);
    p_sck *= 0.65;
    p_int = p_int * 1.20 + 0.004;
    double ssum = p_inc + p_int + p_sck;
    if (ssum == 0.0) ssum = 1.0;
    double b0 = p_inc / ssum, b1 = p_int / ssum, b2 = p_sck / ssum;
    const double bs = (b0 + b1) + b2;
    b0 = b0 / bs; b1 = b1 / bs; b2 = b2 / bs;
    double d0 = b0, d1 = b0 + b1;
    const double d2 = (b0 + b1) + b2;
    d0 = d0 / d2; d1 = d1 / d2;
    int o = (d0 <= u2 ? 1 : 0) + (d1 <= u2 ? 1 : 0);
    return o > 2 ? 2 : o;
}

// ---- player mode ---------------------------------------------------------------------------------
// Generator.choice(n, p=share): searchsorted(cdf, u, side='right') (FMC:625-635)
__device__ __forceinline__ int sample_usage(const UsageDev &U, int role, double u) {
    const int n = U.n[role];
    int idx = 0;
    for (int i = 0; i < n; ++i) idx += (U.cdf[role][i] <= u) ? 1 : 0;
    return idx < n ? idx : n - 1;
}
// pstats[team][role][name] of a tracked name (FMC:1073-1075, 1108-1148, 1163-1192, 1207-1249): the lane owns its
// game's box lines, so a plain read-modify-write.  counts: 10-bit fields att|tgt, comp|rec, td, INT, sacks.
enum : unsigned long long { PC_ATT = 1ULL, PC_COMP = 1ULL << 10, PC_TD = 1ULL << 20, PC_INT = 1ULL << 30, PC_SACK = 1ULL << 40 };
__device__ __forceinline__ fmc_player_rec *lane_box(const SimKernelArgs &a, int home) {
    return a.box_scratch + (size_t)(blockIdx.x * kSimThreads + home) * 2 * (size_t)a.n_slots;
}
__device__ __forceinline__ void credit(const SimKernelArgs &a, const MatchupDev &M, const Lane &L, int team, int role,
                                       int entry, unsigned long long counts, bool has_yds, double yds) {
    const int slot = M.usage[team].slot[role][entry];
    if (slot < 0) return;
    fmc_player_rec *r = lane_box(a, L.home) + team * a.n_slots + slot;
    if (has_yds) r->yds += yds;
    r->counts += counts;
}
// Python's round(x, 1) in tenths (FMC:1276, 1286, 1296): the decimal value of x correctly rounded, ties to even.
// k = floor(RN(10 x)) is the lower neighbour (or, when the product rounds up to an integer, the nearest itself);
// fma gives the exact sign of x - (2k + 1) / 20, the midpoint between k and k + 1 tenths.
__device__ __forceinline__ long long round_tenths(double x) {
    const double k = floor(x * 10.0);
    const double r = fma(x, 20.0, -(2.0 * k + 1.0));
    long long q = (long long)k;
    if (r > 0.0 || (r == 0.0 && (q & 1LL))) q += 1;
    return q;
}
// End of a game: every box line of the lane goes to the per-game output and into the per-player histograms
// (a line counts only if the name was sampled in this game), then the running box is cleared for the next game.
// (scalars by value on purpose: a reference to the lane or to the kernel arguments would force them into local memory)
__device__ __noinline__ void flush_box(fmc_player_rec *box, fmc_player_rec *out, uint32_t *hist, int lines,
                                       unsigned long long *overflow) {
    for (int i = 0; i < lines; ++i) {
        const fmc_player_rec r = box[i];
        if (out) out[i] = r;
        if (r.counts == 0ULL && r.yds == 0.0) continue;       // nothing was credited: the line is still clear
        box[i].yds = 0.0;
        box[i].counts = 0ULL;
        // `_ensure_player` ran: a pass call (attempt or sack), a target, a carry
        const bool seen = ((r.counts & 0x3FFULL) | ((r.counts >> 40) & 0x3FFULL)) != 0ULL;
        if (!hist || !seen) continue;
        uint32_t *h = hist + (size_t)i * FMC_PH_BINS;
        long long b = round_tenths(r.yds) + FMC_PH_YDS_OFFSET;
        if (b < 0 || b >= FMC_PH_YDS_BINS) { atomicAdd(overflow, 1ULL); b = b < 0 ? 0 : FMC_PH_YDS_BINS - 1; }
        atomicAdd(h + b, 1u);
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const unsigned int c = (unsigned int)((r.counts >> (10 * k)) & 0x3FFULL);
            atomicAdd(h + FMC_PH_YDS_BINS + k * FMC_PH_CNT_BINS + (c < FMC_PH_CNT_BINS ? c : FMC_PH_CNT_BINS - 1), 1u);
        }
    }
}
// FMC:420-425: float32 softmax of the play model's margins / T; returns exp of the "pass" class and the sum.
// Out of line: only the model policies reach it, and its registers stay out of the heuristic path.
__device__ __noinline__ void play_softmax(const float *m, int nc, int pass_class, float temp, float &e_pass, float &sum) {
    float zv[5], zmax = 0.f;
    sum = 0.f; e_pass = 0.f;
#pragma unroll
    for (int k = 0; k < 5; ++k)
        if (k < nc) { zv[k] = m[k] / temp; if (k == 0 || zv[k] > zmax) zmax = zv[k]; }
#pragma unroll
    for (int k = 0; k < 5; ++k)
        if (k < nc) { const float e = expf_cr(zv[k] - zmax); sum += e; if (k == pass_class) e_pass = e; }
}

// ---- the game rules, one step at a time ----------------------------------------------------------------------------
// sim_kernel (advance_lane) and sim_memo_kernel (its trip loop) schedule a game's steps differently but play them with
// these functions, so the two kernels share one copy of the rules, draws and arithmetic.  A step counts the game events
// it sees through the kernel's event sink: any type with a method hit(EV_*).

// game events, then the memo hits per family (sim_memo_kernel)
enum { EV_GO = 0, EV_FGA, EV_FG, EV_PUNT, EV_RUN, EV_PASS, EV_COMP, EV_INC, EV_INT, EV_SACK, EV_TD, EV_GAMES,
       EV_HIT0, EV_HIT1, EV_HIT2, EV_HIT3, EV_HIT4, EV_HIT5, EV_N };
__host__ __device__ constexpr int ev_counter(int ev) {      // the FMC_C_* counter of an event
    switch (ev) {
    case EV_GO: return FMC_C_GO;
    case EV_FGA: return FMC_C_FGA;
    case EV_FG: return FMC_C_FG;
    case EV_PUNT: return FMC_C_PUNT;
    case EV_RUN: return FMC_C_RUN;
    case EV_PASS: return FMC_C_PASS;
    case EV_COMP: return FMC_C_COMP;
    case EV_INC: return FMC_C_INC;
    case EV_INT: return FMC_C_INT;
    case EV_SACK: return FMC_C_SACK;
    case EV_TD: return FMC_C_TD;
    case EV_GAMES: return FMC_C_GAMES;
    default: return FMC_C_MEMO_HITS_FAM0 + (ev - EV_HIT0);
    }
}
// sim_kernel's event sink: one shared-memory atomic per event
struct StatEvents {
    unsigned long long *stat;
    __device__ __forceinline__ void hit(int ev) { atomicAdd(&stat[ev_counter(ev)], 1ULL); }
};

__device__ __forceinline__ int stage_family(int stage) {      // ST_WAIT_* -> model id
    return stage == ST_WAIT_PM ? 5 : stage - ST_WAIT_S1;      // S1, S2, PQ, RQ, SQ are consecutive
}
static_assert(ST_WAIT_S2 == ST_WAIT_S1 + 1 && ST_WAIT_PQ == ST_WAIT_S1 + 2 && ST_WAIT_RQ == ST_WAIT_S1 + 3 && ST_WAIT_SQ == ST_WAIT_S1 + 4,
              "stage_family assumes consecutive wait stages");
// key (family * 2 + team on offense) of the request a lane at a ST_WAIT_* stage waits for
__device__ __forceinline__ int request_key(const Lane &L) { return stage_family(L.stage) * 2 + L.offense; }

// game g of the matchup starts (simulate_game FMC:1428-1464) from the entry's start record: at kickoff the parity of
// its id picks the team that receives first.  The period follows from the clock as tick_clock derives it.
__device__ __forceinline__ void new_game(Lane &L, const MatchupDev &M, unsigned long long g) {
    L.game = g;
    L.offense = M.start.offense < 0 ? (int)(g & 1ULL) : M.start.offense;
    L.sec = M.start.sec; L.down = M.start.down; L.dist = M.start.dist; L.ytg = M.start.ytg;
    L.period = L.sec > 0 ? 4 - ((L.sec - 1) / 900) : 4;
    L.going = 0;
    L.score[0] = M.start.score[0]; L.score[1] = M.start.score[1]; L.iter = 0; L.plays = 0; L.p1 = 0; L.wr = 0;
    L.stage = ST_ITER;
}

// Game over (FMC:1456-1464, 1501-1503): score word, iteration count and player box to the outputs.  Returns the game's
// bin in the score histogram of its matchup ([orientation][score 0][score 1]; a score past the last bin is clamped into
// it and counted as an overflow); the kernel adds it.
template <bool PLAYERS, class Ev, class Pk>
__device__ __forceinline__ unsigned int end_game_record(const Lane &L, const SimKernelArgs &a, const MatchupDev &M, int matchup,
                                                        unsigned long long *stat, Ev &ev, const Pk &pk) {
    const size_t oi = (size_t)(M.out_offset + (L.game - M.game_begin));
    if (a.scores) a.scores[oi] = (uint32_t)L.score[0] | ((uint32_t)L.score[1] << 16);
    if (a.iters) a.iters[oi] = (uint16_t)L.iter;
    const int ha = L.score[0] < FMC_HIST_BINS ? L.score[0] : FMC_HIST_BINS - 1;
    const int hb = L.score[1] < FMC_HIST_BINS ? L.score[1] : FMC_HIST_BINS - 1;
    if (a.hist && (L.score[0] >= FMC_HIST_BINS || L.score[1] >= FMC_HIST_BINS)) atomicAdd(&stat[FMC_C_HIST_OVERFLOW], 1ULL);
    if (PLAYERS && a.n_slots > 0) {
        const int lines = 2 * a.n_slots;
        flush_box(lane_box(a, L.home), a.players ? a.players + oi * (size_t)lines : nullptr,
                  a.player_hist ? a.player_hist + (size_t)matchup * (size_t)lines * FMC_PH_BINS : nullptr, lines,
                  &stat[FMC_C_PH_OVERFLOW]);
    }
    pk.game_end(L);
    pk.ot().game_end(L, stat, oi);
    ev.hit(EV_GAMES);
    return (unsigned int)(((L.game & 1ULL) * FMC_HIST_BINS + ha) * FMC_HIST_BINS + hb);
}

// TEST: the state at the start of iteration L.iter into the per-iteration trace (parity tests)
template <bool TEST>
__device__ __forceinline__ void write_trace(const Lane &L, const SimKernelArgs &a, const MatchupDev &M) {
    if (TEST && a.trace && L.iter < FMC_MAX_ITERS) {
        const int first = (int)(L.game & 1ULL);
        double *t = a.trace + ((size_t)(M.out_offset + (L.game - M.game_begin)) * FMC_MAX_ITERS + (size_t)L.iter) * FMC_TRACE_COLS;
        t[0] = (L.offense == first) ? 1.0 : 0.0; t[1] = (double)L.down; t[2] = (double)L.sec;
        t[3] = (double)L.score[first]; t[4] = (double)L.score[first ^ 1]; t[5] = L.dist; t[6] = L.ytg;
        t[7] = (double)L.going;
    }
}

// Fourth down (handle_fourth FMC:1382-1421): go for it, kick a field goal or punt (attempt_punt FMC:876-896).  Returns
// whether a play follows; sd = score difference for the team on offense.  A forced choice (Decision<true>, the first
// iteration of a game) takes its branch without the go / kick draws; the branch reads the slots it always reads.
template <bool TEST, class Ev, class Pk>
__device__ __forceinline__ bool fourth_down(Lane &L, Draws<TEST> &D, int sd, Ev &ev, const Pk &pk) {
    if (L.down != 4) return true;
    const int team = L.offense;
    const double ytg = L.ytg, dist = L.dist;
    const int forced = pk.dec().forced(L);
    const double p_go = pymin(1.0, go_for_it_prob(ytg, dist, sd, L.sec) * 1.15);
    if (forced == FMC_4TH_GO || (forced == FMC_4TH_POLICY && D.u(S_U_GO) < p_go)) {
        L.going = 1;
        ev.hit(EV_GO);
        return true;
    }
    if (forced == FMC_4TH_FG || (forced == FMC_4TH_POLICY && ytg <= 38.0)) {
        ev.hit(EV_FGA);
        const bool good = D.u(S_U_FG) < field_goal_prob(ytg + 17.0);
        // With hooks the kick's points go on before its tick, as a touchdown's do, so that a quarter that ends on the
        // kick holds them and the scoring hook sees them.  tick_clock and change_possession read no score, so the order changes nothing else; the
        // instantiations without hooks keep the original order, which compiles to fewer spills there.
        if (Pk::kOn && good) L.score[team] += 3;
        if (good) pk.scored(L, team, FMC_SEQ_FG, L.sec);
        pk.drive_end(L, good ? FMC_DRIVE_FG : FMC_DRIVE_MISSED_FG, L.sec);
        tick_clock(L, 12, pk);
        if (good) { ev.hit(EV_FG); if (!Pk::kOn) L.score[team] += 3; change_possession(L, true, 75.0); }
        else change_possession(L, true, 100.0 - ytg);
        return false;
    }
    ev.hit(EV_PUNT);
    const double gross = pymax(30.0, 43.0 + 6.0 * D.z(S_Z_GROSS));
    const double ret = pymax(0.0, 6.0 + 3.0 * D.z(S_Z_RET));
    double net = gross - ret;
    if (ytg <= 60.0) {
        const double tb = softclip((60.0 - ytg) / 60.0, 0.10, 0.55);
        if (D.u(S_U_TB) < tb) net = ytg - 25.0;
    }
    net = softclip(net, 15.0, ytg - 1.0);
    const int inet = (int)net;
    pk.drive_end(L, FMC_DRIVE_PUNT, L.sec);
    tick_clock(L, 16, pk);
    change_possession(L, true, softclip(100.0 - (ytg - (double)inet), 1.0, 99.0));
    return false;
}

// The play call from P(pass) (FMC:1058-1075, 1203-1208; P(run) after the two normalisations of FMC:1064-1066).  Returns
// the stage the play waits at.  Player mode samples the passer and target (credits the target) or the rusher (credits
// the carry).
template <bool TEST, bool PLAYERS, class Ev, class Pk>
__device__ __forceinline__ int call_play(Lane &L, const SimKernelArgs &a, const MatchupDev &M, Draws<TEST> &D, int team,
                                         double p_pass, Ev &ev, const Pk &pk) {
    double a0 = 1.0 - p_pass, a1 = p_pass;
    const double s = a0 + a1;
    a0 = a0 / s; a1 = a1 / s;
    const double c0 = a0 / (a0 + a1);
    if (D.u(S_U_CALL) < c0) {
        ev.hit(EV_RUN);
        if (PLAYERS) {
            L.p1 = sample_usage(M.usage[team], 1, D.u(S_U_P1));
            L.wr = 0;
            if (pk.ot().credits(L)) credit(a, M, L, team, 1, L.p1, PC_ATT, false, 0.0);
        }
        return ST_WAIT_RQ;
    }
    ev.hit(EV_PASS);
    if (PLAYERS) {
        L.p1 = sample_usage(M.usage[team], 0, D.u(S_U_P1));
        L.wr = sample_usage(M.usage[team], 2, D.u(S_U_WR));
        if (pk.ot().credits(L)) credit(a, M, L, team, 2, L.wr, PC_ATT, false, 0.0);
    }
    return ST_WAIT_S1;
}

// A play starts (simulate_play FMC:1026-...).  Returns the stage it waits at: the play model's margins (policy 1), or
// the model of the play called with the heuristic P(pass).
template <bool TEST, bool PLAYERS, class Ev, class Pk>
__device__ __forceinline__ int start_play(Lane &L, const SimKernelArgs &a, const MatchupDev &M, Draws<TEST> &D, int sd, Ev &ev,
                                          const Pk &pk) {
    L.plays += 1;
    if (a.policy == 1) return ST_WAIT_PM;
    return call_play<TEST, PLAYERS>(L, a, M, D, L.offense, pass_prob_v1(L.down, L.dist, L.ytg, L.sec, sd), ev, pk);
}

// P(pass) from the play model's nc margins m (FMC:420-425): float32 softmax of m / T, clipped to [.02, .98]
__device__ __forceinline__ double p_pass_from_play_model(const float *m, int nc, const SimKernelArgs &a) {
    float e1, sum;
    play_softmax(m, nc, a.pass_class, a.play_temp, e1, sum);
    return softclip((double)(e1 / sum), 0.02, 0.98);
}

// Stage-1 result from the stage-1 model's margin m1 (FMC:1086-1087): a completed pass waits for its yards, an incomplete
// one for the stage-2 model.  Returns true when the launch has no stage-2 model: the stage stays ST_WAIT_S1 and stage 2
// is decided at once from the stand-in probabilities.
template <bool TEST, class Ev>
__device__ __forceinline__ bool after_stage1(Lane &L, const SimKernelArgs &a, const MatchupDev &M, Draws<TEST> &D, int team,
                                             float m1, Ev &ev) {
    const double p1 = (double)(1.0f / (expf_cr(-m1) + 1.0f));                 // xgboost sigmoid, float32
    const double p_complete = softclip(p1 + M.bias[team], 0.02, 0.98);
    if (D.u(S_U_COMP) < p_complete) { ev.hit(EV_COMP); L.stage = ST_WAIT_PQ; return false; }
    if (a.stage2_mode == 1) { L.stage = ST_WAIT_S2; return false; }
    return true;
}

// Stage-2 class probabilities (incomplete, interception, sack): the stage-2 model's margins m through xgboost's Softmax
// (f32 exp, double sum), or the stand-in probabilities
__device__ __forceinline__ void stage2_raw(bool model, const float *m, const SimKernelArgs &a, double raw[3]) {
    if (model) {
        float wmax = m[0];
        wmax = fmaxf(m[1], wmax); wmax = fmaxf(m[2], wmax);
        float e[3];
        double wsum = 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) { e[k] = expf_cr(m[k] - wmax); wsum += (double)e[k]; }
#pragma unroll
        for (int k = 0; k < 3; ++k) raw[k] = (double)(e[k] / (float)wsum);
    } else {
        raw[0] = a.standin[0]; raw[1] = a.standin[1]; raw[2] = a.standin[2];
    }
}

// The not-complete outcome (FMC:1157-1199): incomplete, interception, or a sack that waits for its yards
template <bool TEST, bool PLAYERS, class Ev, class Pk>
__device__ __forceinline__ void after_stage2(Lane &L, const SimKernelArgs &a, const MatchupDev &M, Draws<TEST> &D, int team,
                                             const double raw[3], Ev &ev, const Pk &pk) {
    const int outcome = stage2_outcome(raw, D.u(S_U_S2));
    if (outcome == 0) {                                   // incomplete FMC:1160-1168
        ev.hit(EV_INC);
        if (PLAYERS && pk.ot().credits(L)) credit(a, M, L, team, 0, L.p1, PC_ATT, false, 0.0);
        L.down += 1; L.going = 0;
        tick_clock(L, 10, pk);
        L.stage = ST_ITER;
    } else if (outcome == 2) {                            // sack FMC:1170-1174
        ev.hit(EV_SACK);
        if (PLAYERS && pk.ot().credits(L)) credit(a, M, L, team, 0, L.p1, PC_SACK, false, 0.0);
        L.stage = ST_WAIT_SQ;
    } else {                                              // intercepted FMC:1186-1199
        ev.hit(EV_INT);
        if (PLAYERS && pk.ot().credits(L)) credit(a, M, L, team, 0, L.p1, PC_ATT | PC_INT, false, 0.0);
        const double ret = softclip(6.0 + 5.0 * D.z(S_Z_INT), 0.0, L.ytg);
        const double spot = 100.0 - (L.ytg - ret);
        L.going = 0;
        pk.drive_end(L, FMC_DRIVE_INT, L.sec);
        change_possession(L, true, spot);
        tick_clock(L, 12, pk);
        L.stage = ST_ITER;
    }
}

// The yards of a play from the quantiles q of its yardage model: sack FMC:1170-1184, completed pass FMC:1089-1152 and
// run FMC:1201-1257 (the same steps with different constants).  The play ends.
template <bool TEST, bool PLAYERS, class Ev, class Pk>
__device__ __forceinline__ void after_yards(Lane &L, const SimKernelArgs &a, const MatchupDev &M, Draws<TEST> &D, int team,
                                            const double q[3], Ev &ev, const Pk &pk) {
    if (L.stage == ST_WAIT_SQ) {
        double loss = -sample_yards(a, D, q, 0.25, -20.0, 0.0);
        loss = pymax(0.0, loss);
        loss = pymin(loss, 100.0 - (100.0 - L.ytg));
        L.ytg += loss; L.dist += loss; L.down += 1; L.going = 0;
        tick_clock(L, 24, pk);
    } else {
        const bool pass = L.stage == ST_WAIT_PQ;
        const double ytg0 = L.ytg, mz = M.mz[team];
        double yards = sample_yards(a, D, q, pass ? 0.4 : 0.35, pass ? 0.0 : -4.0, ytg0) * M.ymul[team];
        if (ytg0 > 25.0 && D.u(S_U_EX) < (pass ? 0.60 : 0.5) * explosive_prob(mz, ytg0)) {
            const double ub = pass ? 0.35 + (0.95 - 0.35) * D.u(S_U_BOOST) : 0.2 + (0.5 - 0.2) * D.u(S_U_BOOST);
            yards *= 1.0 + ub * (1.0 + (pass ? 0.7 : 0.6) * mz);
            yards = pymin(yards, ytg0);
        }
        if (ytg0 <= (pass ? 12.0 : 9.0) && L.down <= 3) {
            if (D.u(S_U_FIN) < rz_finish_prob(ytg0, M.tanh35[team], L.down, pass)) yards = ytg0;
        }
        const bool td = yards + 1e-9 >= ytg0;
        if (PLAYERS && pk.ot().credits(L)) {      // FMC:1108-1127, 1140-1145 (pass), 1232-1234, 1246-1247 (run)
            const double y = td ? ytg0 : yards;
            const unsigned long long c_td = td ? PC_TD : 0ULL;
            if (pass) {
                credit(a, M, L, team, 0, L.p1, PC_ATT | PC_COMP | c_td, true, y);
                credit(a, M, L, team, 2, L.wr, PC_COMP | c_td, true, y);
            } else {
                credit(a, M, L, team, 1, L.p1, c_td, true, y);
            }
        }
        if (td) {
            ev.hit(EV_TD);
            L.score[team] += pk.ot().touchdown(L); L.going = 0;
            pk.scored(L, team, FMC_SEQ_TD, L.sec);
            pk.drive_end(L, FMC_DRIVE_TD, L.sec);
            tick_clock(L, pass ? 20 : 28, pk);
            change_possession(L, true, 75.0);
        } else {
            L.going = 0;
            advance_down(L, yards);
            if (L.offense != team) pk.drive_end(L, FMC_DRIVE_DOWNS, L.sec);      // turnover on downs
            tick_clock(L, pass ? 26 : 28, pk);
        }
    }
    L.stage = ST_ITER;
}

// Advance one lane until it posts a request (returns its key, family * 2 + offense) or has nothing
// left to do (returns -1).  `res` points at this lane's result record of the previous round.
template <bool TEST, bool PLAYERS, int HOOKS, bool OT, bool DEC>
__device__ __forceinline__ int advance_lane(LaneT<OT> &L, const SimKernelArgs &a, SimShared &sh, const double *res) {
    const MatchupDev &M = sh.M;
    const int matchup = sh.cur_matchup;
    StatEvents ev{sh.stat};
    const Hooks<HOOKS, OT, DEC> pk(a, M, matchup);
    for (;;) {
        if (L.stage == ST_IDLE) return -1;
        if (L.stage == ST_NEED_GAME) {
            const unsigned long long g = atomicAdd(&a.next_game[matchup], 1ULL);
            if (g >= M.game_end) { L.stage = ST_IDLE; return -1; }
            new_game(L, M, g);
            pk.game_start(L);
            pk.ot().game_start(L, M);
        }
        if (L.stage == ST_ITER) {
            // (the instantiations without overtime keep the clock test of their own: calling Overtime<false>::over here, inline
            // as it is, reorders the code of those with the sequence hooks)
            if (OT ? pk.ot().over(L) : L.sec <= 0) {
                const unsigned int bin = end_game_record<PLAYERS>(L, a, M, matchup, sh.stat, ev, pk);
                if (a.hist) atomicAdd(&a.hist[(size_t)matchup * 2 * FMC_HIST_BINS * FMC_HIST_BINS + bin], 1u);
                atomicAdd(&sh.stat[FMC_C_PLAYS], (unsigned long long)L.plays);
                atomicAdd(&sh.stat[FMC_C_ITERS], (unsigned long long)L.iter);
                L.stage = ST_NEED_GAME;
                continue;
            }
            write_trace<TEST>(L, a, M);
            Draws<TEST> D(a, M, matchup, L);
            L.iter += 1;
            const int sd = L.score[L.offense] - L.score[L.offense ^ 1];
            if (!fourth_down(L, D, sd, ev, pk)) continue;
            L.stage = start_play<TEST, PLAYERS>(L, a, M, D, sd, ev, pk);
            return request_key(L);
        }
        // ---- resuming a parked play: the iteration counter already points past this iteration
        Lane Lv = L;
        Lv.iter = L.iter - 1;
        Draws<TEST> D(a, M, matchup, Lv);
        const int team = L.offense;
        const float *mg = reinterpret_cast<const float *>(res);
        if (L.stage == ST_WAIT_PM) {
            L.stage = call_play<TEST, PLAYERS>(L, a, M, D, team, p_pass_from_play_model(mg, M.tbl[5][team].n_outputs, a), ev, pk);
            return request_key(L);
        }
        if (L.stage == ST_WAIT_S1 && !after_stage1(L, a, M, D, team, mg[0], ev)) return request_key(L);
        if (L.stage == ST_WAIT_S1 || L.stage == ST_WAIT_S2) {
            double raw[3];
            stage2_raw(L.stage == ST_WAIT_S2, mg, a, raw);
            after_stage2<TEST, PLAYERS>(L, a, M, D, team, raw, ev, pk);
            if (L.stage == ST_WAIT_SQ) return request_key(L);
            continue;
        }
        const double q[3] = {res[0], res[1], res[2]};
        after_yards<TEST, PLAYERS>(L, a, M, D, team, q, ev, pk);
    }
}

// Feature column of a request (FMC:996-1021 `_fill_row`, reduced to the numerics that vary inside one
// orientation), written feature-major: col[k * 32] is feature row k of this request.  Rows: 0 down
// 1 distance 2 yardsToGoal 3 is_red_zone 4 score_diff 5 seconds 6 goal_to_go 7 fourth_and_short
// 8 fg_range 9 half 10 two_minute 11..13 "B" views of 1, 2, 4; row 14 (-inf) is set once per chunk.
template <bool PLAYERS>
__device__ __forceinline__ void write_features(float *col, const Lane &L, int fam, const SimKernelArgs &a, const MatchupDev &M) {
    const int team = L.offense;
    if (PLAYERS && fam != 5) {
        // passer_name / target_name / rusher_name of the row (FMC:1079-1081, 1216) as 0/1 name rows
        const UsageDev &U = M.usage[team];
        if (fam == 3) {
            const int r1 = U.row[1][L.p1];
#pragma unroll
            for (int e = 0; e < FMC_MAX_NAME_ROWS; ++e)
                if (e < a.n_rrow) col[(kDynRow0 + e) * 32] = (e == r1) ? 1.f : 0.f;
        } else {
            const int r1 = U.row[0][L.p1], r2 = U.row[2][L.wr];
#pragma unroll
            for (int e = 0; e < FMC_MAX_PASSER_ROWS; ++e)
                if (e < a.n_prow) col[(kDynRow0 + e) * 32] = (e == r1) ? 1.f : 0.f;
            float *tcol = col + (kDynRow0 + a.n_prow) * 32;
#pragma unroll
            for (int e = 0; e < FMC_MAX_NAME_ROWS; ++e)
                if (e < a.n_trow) tcol[e * 32] = (e == r2) ? 1.f : 0.f;
        }
    }
    const int sd = L.score[team] - L.score[team ^ 1];
    float v[6];
    v[0] = (float)L.down; v[1] = (float)L.dist; v[2] = (float)L.ytg; v[3] = (L.ytg <= 20.0) ? 1.f : 0.f;
    v[4] = (float)sd; v[5] = (float)L.sec;
    if (fam == 5) {   // play_model.xgb: StandardScaler on everything but is_red_zone (dense rows, no missing)
        const double raw[6] = {(double)L.down, L.dist, L.ytg, (L.ytg <= 20.0) ? 1.0 : 0.0, (double)sd, (double)L.sec};
#pragma unroll
        for (int k = 0; k < 6; ++k)
            if (a.pm_scaled[k]) v[k] = (float)((raw[k] - a.pm_mean[k]) / a.pm_scale[k]);
#pragma unroll
        for (int k = 0; k < 6; ++k) col[k * 32] = v[k];
        // play_model.json also splits on goal_to_go, fourth_and_short, fg_range (features.pkl)
        col[6 * 32] = (L.dist >= (L.ytg - 0.5)) ? 1.f : 0.f;
        col[7 * 32] = (L.down == 4 && L.dist <= 2.0) ? 1.f : 0.f;
        col[8 * 32] = (L.ytg <= 33.0) ? 1.f : 0.f;
        col[9 * 32] = (L.sec > 1800) ? 1.f : 2.f;          // half / two_minute: any NUM_FEATURES name may be in features.pkl
        col[10 * 32] = ((L.sec % 1800) <= 120) ? 1.f : 0.f;
        return;
    }
    const bool zm = fam <= 1;   // CSR-fed boosters: exact zero == missing
    const float inf = __int_as_float(0x7f800000);
    col[0 * 32] = v[0];
    col[3 * 32] = v[3];
    col[5 * 32] = v[5];
    col[6 * 32] = (L.dist >= (L.ytg - 0.5)) ? 1.f : 0.f;
    col[7 * 32] = (L.down == 4 && L.dist <= 2.0) ? 1.f : 0.f;
    col[8 * 32] = (L.ytg <= 33.0) ? 1.f : 0.f;
    col[9 * 32] = (L.sec > 1800) ? 1.f : 2.f;
    col[10 * 32] = ((L.sec % 1800) <= 120) ? 1.f : 0.f;
    if (zm) {
        col[1 * 32] = v[1] == 0.f ? -inf : v[1]; col[11 * 32] = v[1] == 0.f ? inf : v[1];
        col[2 * 32] = v[2] == 0.f ? -inf : v[2]; col[12 * 32] = v[2] == 0.f ? inf : v[2];
        col[4 * 32] = v[4] == 0.f ? -inf : v[4]; col[13 * 32] = v[4] == 0.f ? inf : v[4];
    } else {
        col[1 * 32] = v[1]; col[2 * 32] = v[2]; col[4 * 32] = v[4];
    }
}

__device__ __forceinline__ double eval_output(int fam, const TableRef &T, int out, const SimKernelArgs &a,
                                              uint32_t fcol, int lane, uint32_t &levels) {
    ForestView F;
    F.win_lo = T.win_lo; F.win_hi = T.win_hi;
    F.stream = a.root_stream + T.stream_off[out];
    F.consts = a.consts + T.consts_off[out];
    F.n_groups = T.n_groups[out];
    F.multi_window = T.multi_window != 0;
    if (T.multi_window) {     // rare: a specialised table above 1 MiB
        if (fam >= 2 && fam <= 4) return walk_output<true, true>(F, fcol, lane, T.base64[out], levels);
        return walk_output<false, true>(F, fcol, lane, (double)T.base[out], levels);
    }
    if (fam >= 2 && fam <= 4) return walk_output<true, false>(F, fcol, lane, T.base64[out], levels);
    return walk_output<false, false>(F, fcol, lane, (double)T.base[out], levels);
}

// ---- the rounds of both kernels ------------------------------------------------------------------------------------

// Round state at kernel start, and the -inf feature row of every chunk (leaves keep lanes in place by testing it,
// fmc_pack.hpp).  The kernel initialises its own fields and then synchronises.
template <int THREADS>
__device__ __forceinline__ void init_rounds(RoundShared &sh, float *feats, int chunk_floats) {
    const int tid = threadIdx.x;
    for (int i = tid; i < (THREADS / 32 + kNumKeys) * 32; i += THREADS)
        feats[(size_t)(i >> 5) * chunk_floats + kSimNinfRow * 32 + (i & 31)] = __int_as_float(0xff800000);
    if (tid < FMC_N_COUNTERS) sh.stat[tid] = 0ULL;
    if (tid < kNumKeys) { sh.cnt[0][tid] = 0; sh.cnt[1][tid] = 0; sh.aged[tid] = 0; }
    if (tid == 0) { sh.cur_matchup = -1; sh.scan_from = 0; }
}

// The next matchup that still has games (-1: none), its MatchupDev copied to shared memory, its request lists empty.
// The kernel resets its own fields and then synchronises.
template <int THREADS>
__device__ __forceinline__ int next_matchup(RoundShared &sh, const SimKernelArgs &a) {
    const int tid = threadIdx.x;
    if (tid == 0) {
        // Waves: the CTAs of the grid share the kSlateWave lowest-numbered matchups that still have games (CTA b takes
        // the (b mod kSlateWave)-th of them), and move up as matchups drain -- so a slate keeps a handful of node
        // tables (and their memo entries) live at a time instead of one per CTA (720 x 0.6 MB for a season).
        int found = -1, last = -1, seen = 0;
        const int want = (int)(blockIdx.x % (unsigned)kSlateWave);
        for (int m = sh.scan_from; m < a.n_matchups; ++m) {
            if (*((volatile unsigned long long *)&a.next_game[m]) < a.matchups[m].game_end) {
                if (seen == 0) sh.scan_from = m;          // everything below is finished for good
                last = m;
                if (seen == want) { found = m; break; }
                if (++seen >= kSlateWave) break;
            }
        }
        if (found < 0) found = last;                      // fewer unfinished matchups than the wave is wide
        sh.cur_matchup = found;
    }
    __syncthreads();
    const int m = sh.cur_matchup;
    if (m < 0) return m;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(a.matchups + m);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&sh.M);
        for (int i = tid; i < (int)(sizeof(MatchupDev) / 4); i += THREADS) dst[i] = src[i];
    }
    // the last round of the previous matchup leaves its counts in one of the two buffers (the loop ends
    // before it would clear them): start every matchup from empty lists
    if (tid < kNumKeys) { sh.cnt[0][tid] = 0; sh.cnt[1][tid] = 0; sh.aged[tid] = 0; }
    return m;
}

// B: rank of the lane's request in the list of its key (key < 0: no request); warp match, one shared atomic per key
__device__ __forceinline__ unsigned int request_rank(unsigned int *cnt, int key, int lane) {
    const unsigned int peers = __match_any_sync(0xFFFFFFFFu, key);
    const int leader = __ffs(peers) - 1;
    unsigned int base = 0;
    if (key >= 0 && lane == leader) base = atomicAdd(&cnt[key], (unsigned int)__popc(peers));
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    return base + (unsigned int)__popc(peers & ((1u << lane) - 1u));
}

// Thread 0 plans the walk of a round from the request counts: the requests of each key walked now (evalc; the tail
// hold-back), the first position of each key's list (off) and the work items of each key (item_prefix).
__device__ __forceinline__ void plan_round(RoundShared &sh, int parity) {
    unsigned int o = 0, it = 0;
    for (int j = 0; j < kNumKeys; ++j) {
        const int k = kKeyOrder[j];
        unsigned int c = sh.cnt[parity][k];
        const unsigned int tail = c & 31u;
        if (tail != 0 && tail < kDeferBelow && !sh.aged[k]) { c -= tail; sh.aged[k] = 1; }
        else sh.aged[k] = 0;
        sh.evalc[k] = c;
        sh.off[k] = o;
        o += (c + 31u) & ~31u;          // lists start on chunk boundaries
        sh.item_prefix[j] = it;
        it += ((c + 31u) >> 5) * (unsigned int)splits_of(k >> 1);
    }
    sh.item_prefix[kNumKeys] = it;
    sh.item_next = 0;
}

// C: walk the planned requests.  Work item = (key, chunk of 32 requests, output), handed to warps dynamically in key
// order; each output goes to the request's result record.  Returns the node slots gathered for live requests.
__device__ __forceinline__ void walk_requests(RoundShared &sh, const SimKernelArgs &a, uint32_t feats_saddr,
                                                            int chunk_floats, double *results, int lane, unsigned long long &visits) {
    const unsigned int n_items = sh.item_prefix[kNumKeys];
    for (;;) {
        unsigned int it = 0;
        if (lane == 0) it = atomicAdd(&sh.item_next, 1u);
        it = __shfl_sync(0xFFFFFFFFu, it, 0);
        if (it >= n_items) break;
        int j = 0;
        while (it >= sh.item_prefix[j + 1]) ++j;
        const int k = kKeyOrder[j];
        const int fam = k >> 1;
        const unsigned int local = it - sh.item_prefix[j];
        const int ns = splits_of(fam);
        const unsigned int chunk = local / (unsigned int)ns;
        const int out = (int)(local - chunk * (unsigned int)ns);
        const unsigned int c = sh.evalc[k];
        const unsigned int idx = chunk * 32u + (unsigned int)lane;
        const bool live = idx < c;
        const unsigned int p = sh.off[k] + idx;      // idle lanes walk whatever their column holds
        uint32_t levels;
        const double v = eval_output(fam, sh.M.tbl[fam][k & 1], out, a,
                                     feats_saddr + (p >> 5) * (uint32_t)(chunk_floats * 4) + (uint32_t)lane * 4u, lane, levels);
        visits += (unsigned long long)levels * (live ? kIlp : 0);
        if (live) {
            if (fam >= 2 && fam <= 4) results[(size_t)p * 3 + out] = v;
            else reinterpret_cast<float *>(results + (size_t)p * 3)[out] = (float)v;
        }
    }
}

// PLAYERS = true: usage tables are set (fmc_set_usage): names are sampled per play, requests carry kDynRows
// more feature rows, tracked names get per-game box lines.  The shipped configuration (every name "Unknown")
// runs the PLAYERS = false instantiation, which carries none of it.  HOOKS: the optional outputs of the launch
// (kHookPeriods: fmc_simulate_segments, Periods<true>; kHookSequence: fmc_simulate_markets, Sequence<true>); the
// HOOKS = 0 instantiations are the code without the hooks.  OT: overtime (fmc_simulate_overtime, Overtime<true>), DEC:
// forced fourth-down choices (fmc_game_state.fourth_down, Decision<true>), both with HOOKS = 0 only.
template <bool TEST, bool PLAYERS, int HOOKS, bool OT = false, bool DEC = false>
__global__ void __launch_bounds__(kSimThreads, kSimCtasPerSm) sim_kernel(const SimKernelArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // player mode sizes a chunk by the name rows the launch needs (runtime); the shipped configuration is compile-time
    const int kChunkFloats = PLAYERS ? (kSimRows + a.name_rows) * 32 : chunk_floats(false);
    const size_t kSimFeatBytes = (size_t)kSimChunks * (size_t)kChunkFloats * 4;
    SimShared &sh = *reinterpret_cast<SimShared *>(smem_raw);
    float *feats = reinterpret_cast<float *>(smem_raw + kSimSharedBytes);
    double *results = reinterpret_cast<double *>(smem_raw + kSimSharedBytes + kSimFeatBytes);

    const uint32_t feats_saddr = (uint32_t)__cvta_generic_to_shared(feats);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    init_rounds<kSimThreads>(sh, feats, kChunkFloats);
    __syncthreads();

    PackedLane P = idle_lane();
    unsigned long long rounds = 0, requests = 0, visits = 0;
    int home = tid;        // running player box of the game this thread holds (travels with the game when games regroup)
    uint32_t *xchg = reinterpret_cast<uint32_t *>(results);                                   // words 0..7
    uint32_t *xchg2 = reinterpret_cast<uint32_t *>(smem_raw + kSimSharedBytes + kSimFeatBytes + kSimResultBytes);   // words 8..9

    for (;;) {
        // ---- the next matchup that still has games; CTAs start at different matchups so that a slate is spread over
        // the SMs and each CTA drains only when its matchup runs dry
        const int m = next_matchup<kSimThreads>(sh, a);
        if (m < 0) break;
        __syncthreads();
        set_stage(P, ST_NEED_GAME);
        int pos = 0;
        int parity = 0;
        int held = -1;                 // key of a request that was held back last round
        for (;;) {
            // ---- A: advance to the next request (a held-back lane re-posts the one it has)
            LaneT<OT> L = unpack_lane<OT>(P, a);
            L.home = home;
            const int key = held >= 0 ? held : advance_lane<TEST, PLAYERS, HOOKS, OT, DEC>(L, a, sh, results + (size_t)pos * 3);
            __syncwarp();
            // ---- B: compaction
            const unsigned int rank = request_rank(sh.cnt[parity], key, lane);
            const int total = __syncthreads_count(key >= 0);
            if (total == 0) break;
            if (tid == 0) {
                plan_round(sh, parity);
                unsigned int dn = 0;
                for (int j = 0; j < kNumKeys; ++j) {
                    const int k = kKeyOrder[j];
                    sh.dense_off[k] = dn;
                    dn += sh.evalc[k];
                }
                sh.n_eval = dn;
                sh.rest = 0;
            }
            if (tid < kNumKeys) sh.cnt[parity ^ 1][tid] = 0;
            __syncthreads();
            // ---- B2: regroup.  The game goes to thread dense_off[key] + rank (evaluated requests, key-major in the
            // order the keys are walked), every other game to the threads behind them.
            bool evald = key >= 0 && rank < sh.evalc[key];
            {
                const unsigned int slot = evald ? sh.dense_off[key] + rank : sh.n_eval + atomicAdd(&sh.rest, 1u);
                const unsigned int npos = evald ? sh.off[key] + rank : 0u;
                P = pack_lane<OT>(L);
                xchg[0 * kSimThreads + slot] = (uint32_t)P.game;
                xchg[1 * kSimThreads + slot] = (uint32_t)(P.game >> 32);
                xchg[2 * kSimThreads + slot] = (uint32_t)__double2loint(P.dist);
                xchg[3 * kSimThreads + slot] = (uint32_t)__double2hiint(P.dist);
                xchg[4 * kSimThreads + slot] = (uint32_t)__double2loint(P.ytg);
                xchg[5 * kSimThreads + slot] = (uint32_t)__double2hiint(P.ytg);
                xchg[6 * kSimThreads + slot] = P.a;
                xchg[7 * kSimThreads + slot] = P.b;
                xchg2[0 * kSimThreads + slot] = P.c;
                xchg2[1 * kSimThreads + slot] = npos | ((uint32_t)(key + 1) << 11) | ((evald ? 1u : 0u) << 16) | ((uint32_t)home << 17);
            }
            __syncthreads();
            int mykey;
            {
                P.game = (unsigned long long)xchg[0 * kSimThreads + tid] | ((unsigned long long)xchg[1 * kSimThreads + tid] << 32);
                P.dist = __hiloint2double((int)xchg[3 * kSimThreads + tid], (int)xchg[2 * kSimThreads + tid]);
                P.ytg = __hiloint2double((int)xchg[5 * kSimThreads + tid], (int)xchg[4 * kSimThreads + tid]);
                P.a = xchg[6 * kSimThreads + tid];
                P.b = xchg[7 * kSimThreads + tid];
                P.c = xchg2[0 * kSimThreads + tid];
                const uint32_t w = xchg2[1 * kSimThreads + tid];
                pos = (int)(w & 0x7FFu);
                mykey = (int)((w >> 11) & 31u) - 1;
                evald = ((w >> 16) & 1u) != 0u;
                home = (int)(w >> 17);
            }
            held = (!evald && mykey >= 0) ? mykey : -1;
            if (evald) {
                const LaneT<OT> Ln = unpack_lane<OT>(P, a);
                write_features<PLAYERS>(feats + (size_t)(pos >> 5) * kChunkFloats + (pos & 31), Ln, mykey >> 1, a, sh.M);
            }
            __syncthreads();
            // ---- C: evaluate
            walk_requests(sh, a, feats_saddr, kChunkFloats, results, lane, visits);
            __syncthreads();
            parity ^= 1;
            rounds += 1;
            requests += evald ? 1ULL : 0ULL;
        }
    }
    // ---- flush counters
    atomicAdd(&sh.stat[FMC_C_REQUESTS], requests);
    atomicAdd(&sh.stat[FMC_C_VISITS], visits);
    if (lane == 0) atomicAdd(&sh.stat[FMC_C_WARP_STEPS], visits);      // lane 0 of a walking warp is always live
    if (tid == 0) sh.stat[FMC_C_ROUNDS] = rounds;
    __syncthreads();
    if (a.counters && tid < FMC_N_COUNTERS && sh.stat[tid]) atomicAdd(&a.counters[tid], sh.stat[tid]);
}

inline size_t sim_smem_bytes(bool players = false) { return kSimSharedBytes + sim_feat_bytes(players) + kSimResultBytes + kSimXchgExtraBytes; }
// player mode with `name_rows` name rows per chunk (<= kDynRows)
inline size_t sim_smem_bytes_players(int name_rows) {
    return kSimSharedBytes + (size_t)kSimChunks * (size_t)(kSimRows + name_rows) * 32 * 4 + kSimResultBytes + kSimXchgExtraBytes;
}

}  // namespace fmc
