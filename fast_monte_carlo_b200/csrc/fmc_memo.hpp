// Exact memo of tree-ensemble outputs, keyed on threshold ranks.
//
// The reference memoises its model calls on coarse state bins (FMC:68-94, 343-357, 740-747, 780-789), which
// makes its outputs depend on visiting order.  This memo is EXACT instead: on the per-orientation specialised
// forest (fmc_pack.hpp) the output of a request depends on its feature values only through the side of every
// split threshold they fall on.  For each feature row the packer records the distinct thresholds of the walked
// nodes; a request's key is the vector of per-feature RANKS among them (plus an "is exactly zero" code where a
// zero means "missing" for the CSR-fed boosters).  Two requests with the same key take the same branch at every
// node of every tree, hence reach the same leaves and get bit-identical sums -- so a hit returns exactly what
// the walk would have computed.  The full 64-bit key is stored and compared: a hash collision can only evict,
// never alias.
//
// Table: one region per family, direct mapped, overwritten on conflict (a cache, not a map).  A region is an
// array of slots of 1, 2 or 4 UNITS of 16 bytes; unit u of an entry is {key | u, payload u} and is written /
// read with one 128-bit access, so every unit is self-identifying: a reader accepts an entry only if every
// unit carries its key, and since equal keys always carry equal payloads no ordering between units (or
// between racing writers) is needed.
//     pass stage 1      1 unit : float32 margin
//     pass stage 2      2 units: 3 float32 margins
//     pass / run / sack 3 units: q10, q50, q90 as float64           (slot = 4 units)
//     play model        3 units: up to 5 float32 margins            (slot = 4 units)
#pragma once

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "fmc_pack.hpp"

namespace fmc {

constexpr int kMemoFams = 6;
constexpr int kMemoThrMax = 127;        // thresholds of a searched (continuous) feature
constexpr int kMemoKeyBits = 47;        // rank bits available in the key
constexpr int kMemoSdOffset = 256, kMemoSdLut = 512, kMemoSecLut = 3604, kMemoDownLut = 16;

// What the kernel needs to turn a request of one (family, orientation) into its key.  Lives in global memory
// (read through L1); one per (specialisation, family, orientation): entries of a launch whose forests are specialised
// alike share one set.
struct RankSpec {
    uint32_t enabled;                   // 0: this forest's ranks do not fit the key -> its requests are always walked
    uint32_t xgb;                       // compare: 1 -> right iff x >= t (xgboost), 0 -> right iff x > t (sklearn)
    uint32_t zm;                        // exact zero == missing (rows 1, 2, 4 get the extra "zero" code)
    uint32_t n_thr[2];                  // searched features: 0 distance (row 1), 1 yardsToGoal (row 2)
    uint32_t shift[2];
    uint32_t shift_sd, shift_sec;
    float thr[2][kMemoThrMax + 1];      // ascending, padded with +inf
    uint64_t lut_down[kMemoDownLut];    // min(down, 15) -> code << shift
    uint64_t lut_flags[64];             // rz | gtg << 1 | f&s << 2 | fg << 3 | two_minute << 4 | (half == 2) << 5 -> codes << shifts
    uint8_t lut_sd[kMemoSdLut];         // clamp(score_diff + 256, 0, 511) -> code
    uint8_t lut_sec[kMemoSecLut];       // seconds 0..3600 -> code
};

struct MemoRegion {
    unsigned long long base;            // device address of the region, 0 = family not memoised
    uint32_t slot_mask;                 // slots - 1 (power of two)
    uint32_t slot_shift;                // log2(bytes per slot): 4, 5 or 6
};

struct MemoArgs {
    MemoRegion region[kMemoFams];
    const RankSpec *specs;              // [specialisations][kMemoFams][2], indexed by MatchupDev::memo_id
    int enabled;
    int max_trips;                      // stage steps a warp may run per round
    int break_parked;                   // a warp leaves the trip loop once this many of its lanes wait for the walk (or are idle)
    int break_waiting;                  // ... or once this many warps of the CTA have left it
};

__host__ __device__ inline int memo_units(int fam) { return fam == 0 ? 1 : (fam == 1 ? 2 : 3); }
__host__ __device__ inline int memo_slot_shift(int fam) { return fam == 0 ? 4 : (fam == 1 ? 5 : 6); }

#ifdef __CUDA_ARCH__
#define FMC_MEMO_LD(p) __ldg(p)
#else
#define FMC_MEMO_LD(p) (*(p))
#endif

// Rank of x among the ascending thresholds (padded with +inf to 128): #{t : x goes right of t}.
template <bool XGB>
__host__ __device__ __forceinline__ uint32_t memo_rank(const float *thr, float x) {
    uint32_t pos = 0;
#pragma unroll
    for (int s = 64; s >= 1; s >>= 1) {
        const float t = FMC_MEMO_LD(thr + pos + s - 1);
        const bool right = XGB ? (x >= t) : (x > t);
        pos += right ? (uint32_t)s : 0u;
    }
    return pos;
}

// Key of a request of (family, team on offense) in the state (down, distance, yardsToGoal, score_diff, seconds) on the
// specialisation `memo_id` (10 bits: at most 1024 specialisations per launch are memoised).
// v1 / v2 are the distance / yardsToGoal FEATURE values as write_features forms them (float conversion, play-model
// standardisation); the flags are derived exactly as `_fill_row` derives them (FMC:996-1021).  One implementation
// for the kernel and for the host-side check (fmc_memo_keys_host).
template <bool XGB>
__host__ __device__ __forceinline__ unsigned long long memo_key(const RankSpec *rs, int fam, int team, int memo_id, int down,
                                                                double dist, double ytg, int sd, int sec, float v1, float v2) {
    const uint32_t fl = (ytg <= 20.0 ? 1u : 0u) | (dist >= (ytg - 0.5) ? 2u : 0u) | ((down == 4 && dist <= 2.0) ? 4u : 0u) |
                        (ytg <= 33.0 ? 8u : 0u) | (((sec % 1800) <= 120) ? 16u : 0u) | (sec > 1800 ? 0u : 32u);
    int sdi = sd + kMemoSdOffset;
    sdi = sdi < 0 ? 0 : (sdi > kMemoSdLut - 1 ? kMemoSdLut - 1 : sdi);
    const int dn = down < 0 ? 0 : (down < kMemoDownLut - 1 ? down : kMemoDownLut - 1);
    const int si = sec < 0 ? 0 : (sec > 3600 ? 3600 : sec);
    unsigned long long k = FMC_MEMO_LD(rs->lut_down + dn) | FMC_MEMO_LD(rs->lut_flags + fl);
    k |= (unsigned long long)FMC_MEMO_LD(rs->lut_sd + sdi) << FMC_MEMO_LD(&rs->shift_sd);
    k |= (unsigned long long)FMC_MEMO_LD(rs->lut_sec + si) << FMC_MEMO_LD(&rs->shift_sec);
    const uint32_t n1 = FMC_MEMO_LD(&rs->n_thr[0]), n2 = FMC_MEMO_LD(&rs->n_thr[1]);
    const bool zm = FMC_MEMO_LD(&rs->zm) != 0u;
    uint32_t c1 = memo_rank<XGB>(rs->thr[0], v1), c2 = memo_rank<XGB>(rs->thr[1], v2);
    if (zm && v1 == 0.f) c1 = n1 + 1u;
    if (zm && v2 == 0.f) c2 = n2 + 1u;
    k |= (unsigned long long)c1 << FMC_MEMO_LD(&rs->shift[0]);
    k |= (unsigned long long)c2 << FMC_MEMO_LD(&rs->shift[1]);
    return (1ULL << 63) | (k << 16) | ((unsigned long long)memo_id << 6) | ((unsigned long long)fam << 3) | ((unsigned long long)team << 2);
}

// ---- host: build the rank spec of one specialised forest ---------------------------------------------
struct RankSpecInput {
    bool xgb = false, zm = false, play_model = false;
    // play model: standardisation of the six varying numerics (rows 0..5), as write_features applies it
    int pm_scaled[6] = {0, 0, 0, 0, 0, 0};
    double pm_mean[6] = {0, 0, 0, 0, 0, 0}, pm_scale[6] = {1, 1, 1, 1, 1, 1};
};

namespace memo_detail {
inline bool goes_right(bool xgb, float x, float t) { return xgb ? (x >= t) : (x > t); }
inline uint32_t bits_for(uint32_t max_code) { uint32_t b = 0; while ((1u << b) <= max_code) ++b; return max_code == 0 ? 0 : b; }
}  // namespace memo_detail

// row_thr: PackedForest::row_thr of the simulation preset (rows 0..10 A views, 11..13 B views of 1, 2, 4).
// Returns "" and fills `rs` (enabled = 1), or the reason the forest cannot be memoised (rs.enabled = 0).
inline std::string build_rank_spec(const std::vector<std::vector<float>> &row_thr, const RankSpecInput &in, RankSpec &rs) {
    using namespace memo_detail;
    std::memset(&rs, 0, sizeof(rs));
    rs.xgb = in.xgb ? 1u : 0u;
    rs.zm = in.zm ? 1u : 0u;
    std::vector<float> T[11];
    for (size_t r = 0; r < row_thr.size(); ++r) {
        if (row_thr[r].empty()) continue;
        size_t base = r;
        if (r == 11) base = 1; else if (r == 12) base = 2; else if (r == 13) base = 4;
        else if (r > 10) return "a feature row outside the numeric rows is split on (player mode)";
        T[base].insert(T[base].end(), row_thr[r].begin(), row_thr[r].end());
    }
    for (auto &v : T) {
        std::sort(v.begin(), v.end());
        v.erase(std::unique(v.begin(), v.end()), v.end());
        for (float t : v) if (!(std::fabs(t) < 1e30f)) return "non-finite threshold";
    }
    auto value = [&](int row, double raw) -> float {      // feature value as write_features forms it
        if (in.play_model && row < 6 && in.pm_scaled[row]) return (float)((raw - in.pm_mean[row]) / in.pm_scale[row]);
        return (float)raw;
    };
    if (in.play_model)
        for (int k = 0; k < 6; ++k) if (in.pm_scaled[k] && !(in.pm_scale[k] > 0.0)) return "non-positive scaler scale";
    auto zero_row = [&](int row) { return in.zm && (row == 1 || row == 2 || row == 4); };
    auto code = [&](int row, float x) -> uint32_t {
        if (zero_row(row) && x == 0.0f) return (uint32_t)T[row].size() + 1u;
        uint32_t c = 0;
        for (float t : T[row]) c += goes_right(in.xgb, x, t) ? 1u : 0u;
        return c;
    };
    auto max_code = [&](int row) -> uint32_t { return T[row].empty() ? 0u : (uint32_t)T[row].size() + (zero_row(row) ? 1u : 0u); };
    uint32_t shift[11], pos = 0;
    for (int r = 0; r < 11; ++r) { shift[r] = pos; pos += bits_for(max_code(r)); }
    if (pos > (uint32_t)kMemoKeyBits) return "rank vector needs " + std::to_string(pos) + " bits";
    // searched features
    for (int j = 0; j < 2; ++j) {
        const int row = 1 + j;
        if (T[row].size() > (size_t)kMemoThrMax) return "too many thresholds on a searched feature";
        rs.n_thr[j] = (uint32_t)T[row].size();
        rs.shift[j] = shift[row];
        for (int i = 0; i <= kMemoThrMax; ++i) rs.thr[j][i] = i < (int)T[row].size() ? T[row][i] : INFINITY;
    }
    // table features; the clamps of the kernel must not change a code
    for (int r : {0, 4, 5}) if (max_code(r) > 255u) return "too many thresholds on a tabulated feature";
    for (int d = 0; d < kMemoDownLut; ++d) rs.lut_down[d] = (uint64_t)code(0, value(0, (double)d)) << shift[0];
    // every threshold must lie below the clamp value, so that down >= 15 behaves like 15
    if (!T[0].empty() && T[0].back() >= value(0, (double)(kMemoDownLut - 1))) return "a down threshold beyond the table";
    for (int i = 0; i < kMemoSdLut; ++i) rs.lut_sd[i] = (uint8_t)code(4, value(4, (double)(i - kMemoSdOffset)));
    if (!T[4].empty() && (T[4].front() <= value(4, (double)-kMemoSdOffset) || T[4].back() >= value(4, (double)(kMemoSdLut - 1 - kMemoSdOffset))))
        return "a score_diff threshold beyond the table";
    for (int i = 0; i < kMemoSecLut; ++i) rs.lut_sec[i] = (uint8_t)code(5, value(5, (double)(i > 3600 ? 3600 : i)));
    rs.shift_sd = shift[4];
    rs.shift_sec = shift[5];
    for (int f = 0; f < 64; ++f) {
        const float rz = (float)(f & 1), gtg = (float)((f >> 1) & 1), fs = (float)((f >> 2) & 1), fg = (float)((f >> 3) & 1),
                    tm = (float)((f >> 4) & 1), half = ((f >> 5) & 1) ? 2.f : 1.f;
        uint64_t k = 0;
        k |= (uint64_t)code(3, value(3, rz)) << shift[3];
        k |= (uint64_t)code(6, gtg) << shift[6];
        k |= (uint64_t)code(7, fs) << shift[7];
        k |= (uint64_t)code(8, fg) << shift[8];
        k |= (uint64_t)code(9, half) << shift[9];
        k |= (uint64_t)code(10, tm) << shift[10];
        rs.lut_flags[f] = k;
    }
    rs.enabled = 1;
    return "";
}

}  // namespace fmc
