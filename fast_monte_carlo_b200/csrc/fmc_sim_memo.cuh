// Persistent simulation kernel with the exact rank-keyed memo (fmc_memo.hpp) in front of the tree walk.
//
// The game rules are sim_kernel's own code: the trip loop calls the step functions of fmc_sim.cuh (new_game ...
// after_yards) and its rounds use the same matchup pick, compaction, round plan and walk.  Results are bit-identical
// to sim_kernel's; the parity tests run both.  What changes is the schedule:
//
//   * a request first computes its memo key (threshold ranks of its features on the specialised forest) and
//     probes the table in HBM/L2; a hit continues the play at once, so a lane plays several plays per round;
//     only misses are compacted per (family, orientation), walked warp-cooperatively exactly as before, and
//     inserted;
//   * the state machine runs in TRIPS: one trip takes every lane of the warp through the stages of one play in
//     program order (game over / next game -> iteration start and play call -> stage-1 result -> stage-2 result
//     -> yardage), each stage executed once by the warp under a predicate.  Lanes stay converged per stage
//     without moving games between threads (sim_kernel regroups them through shared memory every round);
//   * new games are handed out per warp (one global atomic per warp and trip), event counters are reduced over
//     the warp with REDUX and kept per warp in shared memory, finished games enter the score histogram through
//     a warp match on the bin (one atomic per distinct bin).
#pragma once

#include "fmc_memo.hpp"
#include "fmc_sim.cuh"

namespace fmc {

// ---- 128-bit single-copy accesses at gpu scope (L2; the table is written while it is read) ---------------
__device__ __forceinline__ void memo_ld(unsigned long long addr, unsigned long long &k, unsigned long long &v) {
    asm volatile("{\n\t.reg .b128 r;\n\tld.relaxed.gpu.global.b128 r, [%2];\n\tmov.b128 {%0, %1}, r;\n\t}"
                 : "=l"(k), "=l"(v) : "l"(addr) : "memory");
}
__device__ __forceinline__ void memo_st(unsigned long long addr, unsigned long long k, unsigned long long v) {
    asm volatile("{\n\t.reg .b128 r;\n\tmov.b128 r, {%1, %2};\n\tst.relaxed.gpu.global.b128 [%0], r;\n\t}"
                 :: "l"(addr), "l"(k), "l"(v) : "memory");
}

// Key of the request (family, team on offense) a lane is about to post.  The feature values are formed exactly as
// write_features forms them (same float conversions, same play-model standardisation).
// `memo_id` is the entry's specialisation (MatchupDev::memo_id): entries that share one share their memo entries.
template <bool XGB>
__device__ __forceinline__ unsigned long long lane_memo_key(const RankSpec *rs, int fam, int team, int memo_id, const Lane &L,
                                                            const SimKernelArgs &a) {
    const int sd = L.score[team] - L.score[team ^ 1];
    float v1 = (float)L.dist, v2 = (float)L.ytg;
    if (fam == 5) {
        if (a.pm_scaled[1]) v1 = (float)((L.dist - a.pm_mean[1]) / a.pm_scale[1]);
        if (a.pm_scaled[2]) v2 = (float)((L.ytg - a.pm_mean[2]) / a.pm_scale[2]);
    }
    return memo_key<XGB>(rs, fam, team, memo_id, L.down, L.dist, L.ytg, sd, L.sec, v1, v2);
}

__device__ __forceinline__ unsigned long long memo_slot_addr(const MemoRegion &R, unsigned long long key) {
    unsigned long long h = (key ^ (key >> 31)) * 0x9E3779B97F4A7C15ULL;
    h ^= h >> 29;
    return R.base + ((unsigned long long)((uint32_t)(h >> 20) & R.slot_mask) << R.slot_shift);
}

// Probe: true and r[] = payloads when every unit of the entry carries the key.
template <int UNITS>
__device__ __forceinline__ bool memo_probe(unsigned long long addr, unsigned long long key, unsigned long long (&r)[3]) {
    unsigned long long k[3];
#pragma unroll
    for (int u = 0; u < UNITS; ++u) memo_ld(addr + 16ull * u, k[u], r[u]);
    bool hit = true;
#pragma unroll
    for (int u = 0; u < UNITS; ++u) hit = hit && (k[u] == (key | (unsigned long long)u));
    return hit;
}
__device__ __forceinline__ void memo_insert(unsigned long long addr, unsigned long long key, int units, const unsigned long long (&r)[3]) {
#pragma unroll
    for (int u = 0; u < 3; ++u)
        if (u < units) memo_st(addr + 16ull * u, key | (unsigned long long)u, r[u]);
}

// warp-level event tally of one trip: four words of five 6-bit fields each (a lane adds at most one per field and
// trip, a field's warp sum is at most 32) -- except the probe count, which has a word of its own
constexpr int kEvWords = (EV_N + 4) / 5;
constexpr int kWstat = 24;             // EV_N event totals, then plays, iters, probes
static_assert(EV_N + 3 <= kWstat && EV_N + 3 <= 32, "one lane per tally");
struct EvTally {
    uint32_t w[kEvWords];
    __device__ __forceinline__ EvTally() {
#pragma unroll
        for (int i = 0; i < kEvWords; ++i) w[i] = 0u;
    }
    __device__ __forceinline__ void hit(int ev) { w[ev / 5] += 1u << (6 * (ev % 5)); }
};

// CTA shape of the memo kernel (independent of sim_kernel's): with most requests answered by the memo the walk no
// longer dominates, and the CTA-wide barriers around it cost less when fewer warps share them.
#ifndef FMC_MEMO_THREADS
#define FMC_MEMO_THREADS 1024
#endif
#ifndef FMC_MEMO_CTAS_PER_SM
#define FMC_MEMO_CTAS_PER_SM 1
#endif
constexpr int kMemoThreads = FMC_MEMO_THREADS;
constexpr int kMemoCtasPerSm = FMC_MEMO_CTAS_PER_SM;
constexpr int kMemoChunks = kMemoThreads / 32 + kNumKeys;        // every key's list starts on a chunk boundary
constexpr size_t kMemoFeatBytes = (size_t)kMemoChunks * chunk_floats(false) * 4;
constexpr size_t kMemoResultBytes = (size_t)kMemoChunks * 32 * 3 * 8;

struct MemoShared : RoundShared {
    unsigned int alive[2];
    unsigned int waiting[2];             // warps that have left the trip loop this round (by round parity)
    unsigned long long wstat[kMemoThreads / 32][kWstat];  // per-warp event totals (EV_*, then plays, iters, probes), no atomics
};
constexpr size_t kMemoSharedBytes = ((sizeof(MemoShared) + 15) / 16) * 16;
constexpr size_t kMemoKeyBytes = (size_t)kMemoThreads * 8;
inline size_t sim_memo_smem_bytes() { return kMemoSharedBytes + kMemoFeatBytes + kMemoResultBytes + kMemoKeyBytes; }

// (bounds of a full CTA whatever kMemoThreads: builds of this kernel with __launch_bounds__(512 | 768, ...) die on the B200
// with "an illegal instruction was encountered" at the first launch; the same source with bounds 1024 and a 512-thread
// launch is fine -- ptxas 12.9)
// HOOKS, OT, DEC: the optional outputs of the launch, overtime and forced fourth-down choices (sim_kernel's)
template <bool TEST, int HOOKS, bool OT = false, bool DEC = false>
__global__ void __launch_bounds__(1024, 1) sim_memo_kernel(const SimKernelArgs a, const MemoArgs mm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int kChunkFloats = chunk_floats(false);
    constexpr size_t kFeatBytes_ = kMemoFeatBytes;
    MemoShared &sh = *reinterpret_cast<MemoShared *>(smem_raw);
    float *feats = reinterpret_cast<float *>(smem_raw + kMemoSharedBytes);
    double *results = reinterpret_cast<double *>(smem_raw + kMemoSharedBytes + kFeatBytes_);
    unsigned long long *mkey = reinterpret_cast<unsigned long long *>(smem_raw + kMemoSharedBytes + kFeatBytes_ + kMemoResultBytes);
    const unsigned int FULL = 0xFFFFFFFFu;

    const uint32_t feats_saddr = (uint32_t)__cvta_generic_to_shared(feats);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    init_rounds<kMemoThreads>(sh, feats, kChunkFloats);
    for (int i = tid; i < (kMemoThreads / 32) * kWstat; i += kMemoThreads) (&sh.wstat[0][0])[i] = 0ULL;
    if (tid == 0) { sh.alive[0] = 0; sh.alive[1] = 0; sh.waiting[0] = 0; sh.waiting[1] = 0; }
    __syncthreads();

    PackedLane P = idle_lane();
    unsigned long long visits = 0;
    unsigned int rounds = 0, requests = 0, trips = 0;

    for (;;) {
        const int m = next_matchup<kMemoThreads>(sh, a);
        if (m < 0) break;
        if (tid == 0) { sh.alive[0] = 0; sh.alive[1] = 0; sh.waiting[0] = 0; sh.waiting[1] = 0; }
        __syncthreads();
        const MatchupDev &M = sh.M;
        const Hooks<HOOKS, OT, DEC> pk(a, M, m);
        const RankSpec *specs = mm.specs + (size_t)M.memo_id * kMemoFams * 2;
        set_stage(P, ST_NEED_GAME);
        bool parked = false;           // the lane's request missed the memo and waits for the walk
        int pos = -1;                  // position of its request among this round's walked requests, -1 = not walked
        int parity = 0;
        for (;;) {
            LaneT<OT> L = unpack_lane<OT>(P, a);
            unsigned long long r[3] = {0ULL, 0ULL, 0ULL};
            bool have = false;         // r[] holds the outputs the lane's stage waits for
            // ---- D: walked requests come back; they also enter the memo
            if (parked && pos >= 0) {
                const unsigned long long *src = reinterpret_cast<const unsigned long long *>(results) + (size_t)pos * 3;
                r[0] = src[0]; r[1] = src[1]; r[2] = src[2];
                const int fam = stage_family(L.stage);
                const unsigned long long key = mkey[tid];
                if (key != 0ULL) memo_insert(memo_slot_addr(mm.region[fam], key), key, memo_units(fam), r);
                have = true;
                parked = false;
            }
            pos = -1;
            // ---- A: trips
            for (int trip = 0; trip < mm.max_trips; ++trip) {
                trips += 1;
                EvTally ev;
                uint32_t fin_plays = 0, fin_iters = 0, n_probes = 0;
                // -- game over
                const bool over = !parked && L.stage == ST_ITER && pk.ot().over(L);
                const unsigned int over_mask = __ballot_sync(FULL, over);
                if (over) {
                    const unsigned int bin = end_game_record<false>(L, a, M, m, sh.stat, ev, pk);
                    if (a.hist) {
                        // warp-level reduce: lanes finishing in the same bin add once
                        const unsigned int peers = __match_any_sync(over_mask, bin);
                        if (lane == __ffs(peers) - 1)
                            atomicAdd(&a.hist[(size_t)m * 2 * FMC_HIST_BINS * FMC_HIST_BINS + bin], (unsigned int)__popc(peers));
                    }
                    fin_plays = (uint32_t)L.plays; fin_iters = (uint32_t)L.iter;
                    L.stage = ST_NEED_GAME;
                }
                // -- next game: one global atomic per warp
                {
                    const bool need = !parked && L.stage == ST_NEED_GAME;
                    const unsigned int nm = __ballot_sync(FULL, need);
                    if (nm) {
                        unsigned long long base = 0ULL;
                        const int leader = __ffs(nm) - 1;
                        if (lane == leader) base = atomicAdd(&a.next_game[m], (unsigned long long)__popc(nm));
                        base = __shfl_sync(FULL, base, leader);
                        if (need) {
                            const unsigned long long g = base + (unsigned long long)__popc(nm & ((1u << lane) - 1u));
                            if (g >= M.game_end) L.stage = ST_IDLE;
                            else { new_game(L, M, g); pk.game_start(L); pk.ot().game_start(L, M); }
                        }
                    }
                }
                // draws of the iteration this trip works on: a lane that enters at ST_ITER starts iteration L.iter,
                // one that resumes a parked play is inside iteration L.iter - 1
                Lane Lv = L;
                Lv.iter = (L.stage == ST_ITER) ? L.iter : L.iter - 1;
                Draws<TEST> D(a, M, m, Lv);
                const int team = L.offense;
                const int sd = L.score[team] - L.score[team ^ 1];
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                // -- iteration start: fourth down and the play call (a game that starts with the clock at 0 has none)
                if (!parked && L.stage == ST_ITER && L.sec > 0) {
                    write_trace<TEST>(L, a, M);
                    L.iter += 1;
                    if (fourth_down(L, D, sd, ev, pk)) L.stage = start_play<TEST, false>(L, a, M, D, sd, ev, pk);
                }
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                // -- play model (policy 1): probe, then the play call
                if (a.policy == 1) {
                    if (!parked && !have && L.stage == ST_WAIT_PM) {
                        const RankSpec *rs = specs + 5 * 2 + team;
                        unsigned long long key = 0ULL;
                        bool hit = false;
                        if (mm.enabled && __ldg(&rs->enabled)) {
                            key = lane_memo_key<true>(rs, 5, team, M.memo_id, L, a);
                            hit = memo_probe<3>(memo_slot_addr(mm.region[5], key), key, r);
                            n_probes += 1; if (hit) ev.hit(EV_HIT5);
                        }
                        if (hit) have = true; else { parked = true; mkey[tid] = key; }
                    }
                    if (have && L.stage == ST_WAIT_PM) {
                        float mg[6];
                        mg[0] = __uint_as_float((uint32_t)r[0]); mg[1] = __uint_as_float((uint32_t)(r[0] >> 32));
                        mg[2] = __uint_as_float((uint32_t)r[1]); mg[3] = __uint_as_float((uint32_t)(r[1] >> 32));
                        mg[4] = __uint_as_float((uint32_t)r[2]); mg[5] = 0.f;
                        L.stage = call_play<TEST, false>(L, a, M, D, team, p_pass_from_play_model(mg, M.tbl[5][team].n_outputs, a), ev, pk);
                        have = false;
                    }
                }
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                // -- stage 1: probe, then the result
                if (!parked && !have && L.stage == ST_WAIT_S1) {
                    const RankSpec *rs = specs + 0 * 2 + team;
                    unsigned long long key = 0ULL;
                    bool hit = false;
                    if (mm.enabled && __ldg(&rs->enabled)) {
                        key = lane_memo_key<true>(rs, 0, team, M.memo_id, L, a);
                        hit = memo_probe<1>(memo_slot_addr(mm.region[0], key), key, r);
                        n_probes += 1; if (hit) ev.hit(EV_HIT0);
                    }
                    if (hit) have = true; else { parked = true; mkey[tid] = key; }
                }
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                bool s2_standin = false;
                if (have && L.stage == ST_WAIT_S1) {
                    have = false;
                    s2_standin = after_stage1(L, a, M, D, team, __uint_as_float((uint32_t)r[0]), ev);
                }
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                // -- stage 2: probe, then the not-complete outcome
                if (!parked && !have && L.stage == ST_WAIT_S2) {
                    const RankSpec *rs = specs + 1 * 2 + team;
                    unsigned long long key = 0ULL;
                    bool hit = false;
                    if (mm.enabled && __ldg(&rs->enabled)) {
                        key = lane_memo_key<true>(rs, 1, team, M.memo_id, L, a);
                        hit = memo_probe<2>(memo_slot_addr(mm.region[1], key), key, r);
                        n_probes += 1; if (hit) ev.hit(EV_HIT1);
                    }
                    if (hit) have = true; else { parked = true; mkey[tid] = key; }
                }
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                if ((have && L.stage == ST_WAIT_S2) || s2_standin) {
                    const float mg[3] = {__uint_as_float((uint32_t)r[0]), __uint_as_float((uint32_t)(r[0] >> 32)),
                                         __uint_as_float((uint32_t)r[1])};
                    double raw[3];
                    stage2_raw(!s2_standin, mg, a, raw);
                    have = false;
                    after_stage2<TEST, false>(L, a, M, D, team, raw, ev, pk);
                }
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                // -- yardage families: probe, then the outcome
                if (!parked && !have && L.stage >= ST_WAIT_PQ && L.stage <= ST_WAIT_SQ) {
                    const int fam = stage_family(L.stage);
                    const RankSpec *rs = specs + fam * 2 + team;
                    unsigned long long key = 0ULL;
                    bool hit = false;
                    if (mm.enabled && __ldg(&rs->enabled)) {
                        key = lane_memo_key<false>(rs, fam, team, M.memo_id, L, a);
                        hit = memo_probe<3>(memo_slot_addr(mm.region[fam], key), key, r);
                        n_probes += 1; if (hit) ev.w[(EV_HIT0 + fam) / 5] += 1u << (6 * ((EV_HIT0 + fam) % 5));
                    }
                    if (hit) have = true; else { parked = true; mkey[tid] = key; }
                }
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                if (have && L.stage >= ST_WAIT_PQ && L.stage <= ST_WAIT_SQ) {
                    const double q[3] = {__longlong_as_double((long long)r[0]), __longlong_as_double((long long)r[1]),
                                         __longlong_as_double((long long)r[2])};
                    have = false;
                    after_yards<TEST, false>(L, a, M, D, team, q, ev, pk);
                }
                __syncwarp();      // every stage of the trip is entered by the whole warp together
                // -- warp tallies of this trip
                {
                    const uint32_t t0 = __reduce_add_sync(FULL, ev.w[0]), t1 = __reduce_add_sync(FULL, ev.w[1]),
                                   t2 = __reduce_add_sync(FULL, ev.w[2]), t3 = __reduce_add_sync(FULL, ev.w[3]);
                    const uint32_t tp = __reduce_add_sync(FULL, fin_plays), ti = __reduce_add_sync(FULL, fin_iters),
                                   tq = __reduce_add_sync(FULL, n_probes);
                    if (lane < EV_N) {
                        const uint32_t wv = lane < 5 ? t0 : (lane < 10 ? t1 : (lane < 15 ? t2 : t3));
                        const uint32_t c = (wv >> (6 * (lane % 5))) & 63u;
                        if (c) sh.wstat[warp][lane] += (unsigned long long)c;
                    } else if (lane == EV_N) { if (tp) sh.wstat[warp][EV_N] += (unsigned long long)tp; }
                    else if (lane == EV_N + 1) { if (ti) sh.wstat[warp][EV_N + 1] += (unsigned long long)ti; }
                    else if (lane == EV_N + 2) { if (tq) sh.wstat[warp][EV_N + 2] += (unsigned long long)tq; }
                }
                // -- stop when the warp has little left to do this round
                const unsigned int busy = __ballot_sync(FULL, !parked && L.stage != ST_IDLE);
                if (__popc(busy) <= 32 - mm.break_parked) break;
                // ... or when enough of the other warps already wait at the barrier for this one
                if (*((volatile unsigned int *)&sh.waiting[parity]) >= (unsigned int)mm.break_waiting) break;
            }
            if (lane == 0) atomicAdd(&sh.waiting[parity], 1u);
            // ---- B: compact the requests that missed
            const int key = parked ? request_key(L) : -1;
            const unsigned int rank = request_rank(sh.cnt[parity], key, lane);
            if (__any_sync(FULL, L.stage != ST_IDLE) && lane == 0) sh.alive[parity] = 1u;
            P = pack_lane<OT>(L);
            const int total = __syncthreads_count(key >= 0);
            const bool alive = sh.alive[parity] != 0u;
            if (total == 0 && !alive) break;   // every game of the matchup is played
            if (total == 0) {
                // nobody missed: nothing to walk; clear the other parity's round state and go on
                if (tid < kNumKeys) sh.cnt[parity ^ 1][tid] = 0;
                if (tid == 0) { sh.alive[parity ^ 1] = 0u; sh.waiting[parity ^ 1] = 0u; }
                __syncthreads();
                parity ^= 1;
                rounds += 1;
                continue;
            }
            if (tid == 0) {
                plan_round(sh, parity);
                sh.alive[parity ^ 1] = 0u;
                sh.waiting[parity ^ 1] = 0u;
            }
            if (tid < kNumKeys) sh.cnt[parity ^ 1][tid] = 0;
            __syncthreads();
            if (key >= 0 && rank < sh.evalc[key]) {
                pos = (int)(sh.off[key] + rank);
                write_features<false>(feats + (size_t)(pos >> 5) * kChunkFloats + (pos & 31), L, key >> 1, a, sh.M);
                requests += 1;
            }
            __syncthreads();
            // ---- C: walk
            walk_requests(sh, a, feats_saddr, kChunkFloats, results, lane, visits);
            __syncthreads();
            parity ^= 1;
            rounds += 1;
        }
    }
    // ---- flush counters
    atomicAdd(&sh.stat[FMC_C_REQUESTS], (unsigned long long)requests);
    atomicAdd(&sh.stat[FMC_C_VISITS], visits);
    if (lane == 0) atomicAdd(&sh.stat[FMC_C_WARP_STEPS], visits);     // lane 0 of a walking warp is always live
    if (lane == 0) atomicAdd(&sh.stat[FMC_C_TRIPS], (unsigned long long)trips);
    if (tid == 0) sh.stat[FMC_C_ROUNDS] = (unsigned long long)rounds;
    __syncthreads();
    if (tid < EV_N + 3) {
        unsigned long long s = 0ULL;
        for (int w = 0; w < kMemoThreads / 32; ++w) s += sh.wstat[w][tid];
        const int ci = tid < EV_N ? ev_counter(tid) : (tid == EV_N ? FMC_C_PLAYS : (tid == EV_N + 1 ? FMC_C_ITERS : FMC_C_MEMO_PROBES));
        sh.stat[ci] += s;
    }
    __syncthreads();
    if (tid == 0) {
        unsigned long long h = 0ULL;
        for (int f = 0; f < kMemoFams; ++f) h += sh.stat[FMC_C_MEMO_HITS_FAM0 + f];
        sh.stat[FMC_C_MEMO_HITS] = h;
    }
    __syncthreads();
    if (a.counters && tid < FMC_N_COUNTERS && sh.stat[tid]) atomicAdd(&a.counters[tid], sh.stat[tid]);
}

}  // namespace fmc
