// wf_common.cuh -- shared device-side definitions of libwildfire_b200 (sm_100a).
//
// State layout in HBM (both kernel families)
// ------------------------------------------
// Every per-cell flag of the reference's env[x, y, layer] array (environment.py:38-50)
// that can change is a BIT-PLANE: one uint32 word holds 32 consecutive y of one row x.
//     word(plane, env, x, w) = planes[((plane * N + env) * RS + x) * HW + w]
// with HW = ceil(H / 32) words per row and RS = row stride (warp family: lanes per env,
// tile family: W).  Planes (one-hot cell type + the two flags type cannot express, Q7):
//     G grass  F fire(type==1)  BT burnt  D dirt  WT water  B burning_cells  I fire_mobility==inf
//     FU0.. fuel, bit-sliced (FB planes)     S0/S1 heat-source mask, ping-pong (tile family)
//     HC0.. total hits per cell, bit-sliced (HB planes; warp family with direction-independent quanta only)
// The `temp` layer is kept as exact per-direction hit counters, one uint32 per cell:
//     hits[(env * W + x) * H + y] = n_N | n_S << 8 | n_E << 16 | n_W << 24
// (temp = sum_d n_d * coef[d], environment.py:286-290), touched only where heat arrives.
// `gray` is a pure function of type; heat/threshold/agent_mobility never change -> scalars.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/wildfire.h"
#include "wf_philox.cuh"

namespace wf {

// Internal observation format of wf_step_host: the bit stream itself (1 bit per element), one record of
// ceil(envs_per_warp * W*H*3 / 32) words per warp; expanded to bytes by the host thread pool (wf_hostpool.cpp).
constexpr int kObsPacked = 100;
// The step-server session's format: every record is followed by ONE status word, 16 bits per env of the record
// (env sub-index 0 in the low half): bits 0-2 reward kind, bit 3 done, bits 4-14 grass-cell count of a burn-out reward.
constexpr int kObsPackedStatus = 101;
enum RewardKind : uint32_t { RK_ZERO = 0, RK_DEFAULT = 1, RK_DEATH = 2, RK_CONTAINED = 3, RK_BURNOUT = 4 };
// Self-validating transport of the session's records (SrvCtl::sectors): a record travels as 32-byte SECTORS of seven
// payload words + one tag word = sequence number of the step ^ hash of the seven words.  The host accepts a sector when
// the tag fits what it reads, so it needs no completion flag -- and the GPU no system-scope fence -- and can expand the
// first records while the last are still on the PCIe link; a torn or stale sector simply does not validate yet.
constexpr int kSectorPayload = 7;
__host__ __device__ __forceinline__ uint32_t sector_hash(const uint32_t* w) {
    uint32_t h = 0x9E3779B9u;
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
    for (int i = 0; i < kSectorPayload; ++i) h = (h + w[i]) * 0x9E3779B1u;
    return h ^ (h >> 15);
}

// Step-server session: the mapped host buffer holds the step's actions PACKED AND TAGGED, six per 32-bit word: bits 4k..4k+3
// action k of the word (15: none), bits 24-30 the step's sequence number mod 128, bit 31 "every record in full".  CTA 0 polls
// the buffer itself, so it is kept small: 2.7 KB per poll for 4096 envs.  srv_action_chunks: 16-byte chunks of the buffer.
constexpr uint32_t kSrvTagMask = 0x7fu;
__host__ __device__ __forceinline__ int srv_action_chunks(int n_envs) { return ((n_envs + 5) / 6 + 3) / 4; }

// Change-list blocks of a step-server session with a persistent observation array (wf_host_session mode 2): one block of
// kDeltaBlockWords words per CTA (= 4 records): word 0 = number of entries | mask of the records sent in full << 8, words
// 1-4 = the records' status words, then up to 4 * kDeltaEntries 16-bit entries (element index within the CTA's envs << 1 |
// new value).  A record (warp) with more than kDeltaEntries changed elements has its complete bit stream in
// SrvCtl::full_area instead (its bit of the mask; also kDeltaFullBit of its status word).
constexpr int kDeltaBlockWords = 32, kDeltaEntries = 13, kDeltaFirstEntry = 10 /* 16-bit units */;
constexpr uint32_t kDeltaFullBit = 0x8000u;

// Bytes per observation element of a public obs_dtype (WF_OBS_U8 / WF_OBS_F32 / WF_OBS_BF16).
__host__ __device__ __forceinline__ int obs_elem_bytes(int dtype) { return dtype == WF_OBS_F32 ? 4 : dtype == WF_OBS_BF16 ? 2 : 1; }
// WF_OBS_BITS: uint32 words per env (include/wildfire.h: element k = (x*H + y)*3 + c is bit k % 32 of word k / 32).
__host__ __device__ __forceinline__ int64_t obs_bits_words(int W, int H) { return ((int64_t)W * H * 3 + 31) / 32; }
// Bytes of one step's observation block of N envs in a public obs_dtype (WF_OBS_U8 / F32 / BF16 / BITS).
__host__ __device__ __forceinline__ size_t obs_step_bytes(int64_t N, int W, int H, int dtype) {
    return dtype == WF_OBS_BITS ? (size_t)N * obs_bits_words(W, H) * 4 : (size_t)N * W * H * 3 * obs_elem_bytes(dtype);
}
constexpr uint16_t kBf16One = 0x3F80u;  // 1.0 in bfloat16

enum Plane : int { P_G = 0, P_F, P_BT, P_D, P_WT, P_B, P_I, P_FU0 };  // + FB fuel planes (+ S0, S1, R for tiles)

constexpr int kMaxWind = 27;  // 3 speeds x 9 vectors (environment.py:189-190) or 1 fixed entry

// Read-only per-handle table, one entry per distinct wind the handle can meet.
struct WindTable {
    double coef[kMaxWind][4];  // heat quantum for displacement d: 0 N(0,-1) 1 S(0,+1) 2 E(+1,0) 3 W(-1,0)
    int32_t kmin[kMaxWind];    // uniform winds: hits needed to ignite (sequential float64 sum, as the reference adds)
    int32_t uniform[kMaxWind]; // all four quanta bit-identical
    double speed[kMaxWind];
    int32_t wx[kMaxWind], wy[kMaxWind];
};

// Device-side global statistics (int64 counters).
enum Stat : int { ST_STEPS = 0, ST_EPISODES, ST_DEATHS, ST_CONTAINED, ST_BURNOUTS, ST_TICKS, ST_N = 8 };

struct DevState {
    uint32_t* planes;   // [NP][N][RS][HW]
    uint32_t* hits;     // [N][W][H]
    int32_t* scal;      // [N][WF_NSCALARS]
    const WindTable* wind;
    unsigned long long* stats;  // [ST_N]
    int32_t N, W, H, RS, HW, FB, NP;
    int32_t HB;         // warp family, every wind of the handle uniform: total hit count per cell kept as HB bit planes
                        // (planes P_FU0 + FB ...) instead of the `hits` array; 0 otherwise
    uint32_t* fuel;     // tile family: [N][RS * HW][kFuelRec] -- the FB fuel bit-slices of ONE word side by side, so that
                        // a burning word's fuel is one 32-byte sector in and out instead of FB sectors in FB planes
                        // (`planes` then has no fuel planes).  nullptr: fuel lives in planes P_FU0 .. P_FU0 + FB - 1
};
constexpr int kFuelRec = 8;  // words per fuel record (FB = 5 or 8 used)

struct StepCfg {
    int32_t n_actions, a_speed, allow_dig_toggle, make_rivers, wind_random, fuel, extra_ignitions, auto_reset;
    double death_penalty, contained_bonus, default_reward, threshold;
    uint32_t key0, key1;
    int64_t env_id_base;
};

__device__ __forceinline__ size_t word_index(const DevState& s, int plane, int env, int x, int w) {
    return (((size_t)plane * s.N + env) * s.RS + x) * s.HW + w;
}
// Bit-slice q of the fuel of word (env, x, w), whichever layout the family uses.
__device__ __forceinline__ uint32_t* fuel_slice(const DevState& s, int q, int env, int x, int w) {
    return s.fuel ? s.fuel + ((((size_t)env * s.RS + x) * s.HW + w) * kFuelRec + q) : s.planes + word_index(s, P_FU0 + q, env, x, w);
}

// circle_points(0, 0, r) for r = 1, 2, 3 -- Simulation/utility.py:8-52, in the reference's
// list order (checked against the oracle's literal restatement in tests/test_parity_gpu.py).
__constant__ const int8_t kCircle[3][16][2] = {
    {{1, 0}, {-1, 0}, {0, -1}, {0, 1}, {1, 1}, {-1, 1}, {1, -1}, {-1, -1}},
    {{2, 0}, {-2, 0}, {0, -2}, {0, 2}, {2, 1}, {-2, 1}, {2, -1}, {-2, -1}, {1, 2}, {-1, 2}, {1, -2}, {-1, -2}},
    {{3, 0}, {-3, 0}, {0, -3}, {0, 3}, {3, 1}, {-3, 1}, {3, -1}, {-3, -1}, {1, 3}, {-1, 3}, {1, -3}, {-1, -3},
     {2, 2}, {-2, 2}, {2, -2}, {-2, -2}}};
__constant__ const int32_t kCircleLen[3] = {8, 12, 16};

// Sequential reader of the RESET stream (oracle/philox.py: stream 0, draw k = word k&3 of block k>>2).
struct ResetDraws {
    uint32_t env, episode, key0, key1, k;
    uint32_t blk[4];
    __device__ __forceinline__ ResetDraws(uint32_t env_, uint32_t ep_, uint32_t k0, uint32_t k1)
        : env(env_), episode(ep_), key0(k0), key1(k1), k(0) {}
    __device__ __forceinline__ uint32_t next() {
        if ((k & 3u) == 0u) philox4x32_10(env, episode, k >> 2, kStreamReset, key0, key1, blk);
        uint32_t r = (k & 3u) == 0u ? blk[0] : (k & 3u) == 1u ? blk[1] : (k & 3u) == 2u ? blk[2] : blk[3];
        ++k;
        return r;
    }
};

// Ignition test of a heated grass cell -- World.apply_heat_from_to, environment.py:286-294.
__device__ __forceinline__ bool ignites(uint32_t hits, const WindTable* wt, int wid, double threshold) {
    const int n0 = hits & 255u, n1 = (hits >> 8) & 255u, n2 = (hits >> 16) & 255u, n3 = hits >> 24;
    if (wt->uniform[wid]) return (n0 + n1 + n2 + n3) >= wt->kmin[wid];
    const double* c = wt->coef[wid];
    double t = __dmul_rn((double)n0, c[0]);
    t = __dadd_rn(t, __dmul_rn((double)n1, c[1]));
    t = __dadd_rn(t, __dmul_rn((double)n2, c[2]));
    t = __dadd_rn(t, __dmul_rn((double)n3, c[3]));
    return t > threshold;
}

// Fill every run of set bits of `free` that contains a bit of `seed` (seed must be a subset of free).
// (free + seed) carries through a run from the seed upwards; the brev pair does the same downwards.
__device__ __forceinline__ uint32_t hfill(uint32_t seed, uint32_t free_) {
    uint32_t up = ((free_ + seed) ^ free_) & free_;
    uint32_t rf = __brev(free_), rs = __brev(seed);
    uint32_t dn = __brev(((rf + rs) ^ rf) & rf);
    return seed | up | dn;
}

}  // namespace wf
