// wf_learn.cu -- wf_replay_fit / wf_replay_fit_many (include/wildfire.h): n_replays consecutive DQN.replay / fit_batch
// updates (DQN.py:156-185, DQN_SARSA.py:103-132; the rule agents.py pins to tests/golden/agents/n1_replay.npz) for each of
// up to 64 independent learners in ONE launch: one thread-block cluster per learner (learner = cluster index).  A
// cluster reads only its learner's descriptor, so its result does not depend on the other learners; with the same
// cluster size it is bit-identical to a launch of that learner alone (wf_replay_fit is the one-learner case).
//
// Work split.  The network's hidden units (hidden, or 2 * hidden for the dueling head: advantage units first, then value
// units) are dealt out to the CTAs of the cluster in contiguous slices.  A CTA reads and writes only its own units' first-
// layer rows, biases and second-layer columns (model, target, m and v), straight from global memory (L1 / L2 resident:
// no other CTA touches them).  Per replay, the only exchange is the second layer's partial sums: each CTA writes
// [3 passes][batch][n_actions + 1] sums over its units to shared memory, and after one cluster barrier every CTA adds the
// slices of all CTAs in rank order through DSMEM.  Every CTA therefore holds bit-identical Q-values, targets and output
// gradients (no floating-point atomics: the result is deterministic), and the small shared parameters (dense_2.bias,
// dense_4.bias and their Adam moments) are kept in every CTA's shared memory and updated redundantly and identically.
// The partial-sum buffer is double-buffered, so one cluster barrier per replay suffices: a CTA overwrites buffer r & 1 in
// replay r + 2 only after the barrier of replay r + 1, which every peer reaches after it has read replay r's sums.
//
// The first layer reads the observation bits directly: a sum of weight-row entries over the set bits.
#include <cooperative_groups.h>
#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <string>

#include "wf_common.cuh"

namespace cg = cooperative_groups;

namespace wf {
int api_fail(int code, const std::string& msg);  // wf_api.cu: sets wf_last_error
}
using wf::api_fail;

namespace {

constexpr int kThreads = 512;
constexpr int kMaxBatch = 256, kMaxHidden = 64, kMaxActions = 8, kOut = kMaxActions + 1;
constexpr int kMaxUnits = 16;  // units per CTA: 2 * kMaxHidden over a cluster of at least 8 CTAs
constexpr int kMaxLearners = 64;

struct FitLearner {  // one learner's buffers and hyper-parameters (wf_fit_learner, scalars prepared for the kernel)
    float* P;  // model
    float* T;  // target
    float* M;  // Adam m
    float* V;  // Adam v
    const int64_t* s_row;
    const int64_t* sp_row;
    const int32_t* action;
    const int32_t* next_action;
    const float* reward;
    const uint8_t* done;
    float* loss;
    float gamma, b1, omb1, b2, omb2, eps, clip;
    double lr, beta_1, beta_2;
    int64_t adam_t;
    int target_every, phase;
};

struct FitArgs {  // in the kernel's parameter block (~10 KB of the 32 KB limit)
    const uint32_t* frames;
    int64_t n_frames;
    int n_replays;
    int n_in, words, hid, A, duel, B;
    int off_b1, off_w2, off_b2, off_w3, off_b3, off_w4, off_b4;
    FitLearner learner[kMaxLearners];
};

struct Smem {
    float part[2][3][kMaxBatch][kOut];  // this CTA's second-layer partial sums (double-buffered, read by peers)
    float q[3][kMaxBatch][kOut];        // summed over the cluster + bias: model(s), target(s), target(s')
    float dout[kMaxBatch][kOut];        // dLoss / d(second-layer output); column A = value output of the dueling head
    float h[kMaxBatch][kMaxUnits];      // model hidden activations of this CTA's units on s
    float dz[kMaxBatch][kMaxUnits];     // dLoss / d(first-layer pre-activation)
    float sqerr[kMaxBatch];
    int64_t row[2][kMaxBatch];          // s, s'
    int32_t act[kMaxBatch], nact[kMaxBatch];
    float rew[kMaxBatch];
    uint8_t dn[kMaxBatch];
    float ob[4][kOut];                  // output biases (dense_2.bias, dense_4.bias): model, target, m, v
};

__device__ __forceinline__ float sigmoidf(float z) { return 1.0f / (1.0f + expf(-z)); }

// Keras 2 Adam on one element (agents.KerasAdam.step): clip, moments, p -= lr_t * m / (sqrt(v) + epsilon).
__device__ __forceinline__ float adam(const FitLearner& a, float lr_t, float p, float g, float& m, float& v) {
    g = fminf(fmaxf(g, -a.clip), a.clip);
    m = m * a.b1 + a.omb1 * g;
    v = v * a.b2 + a.omb2 * g * g;
    return p + (-lr_t) * (m / (sqrtf(v) + a.eps));
}

__global__ void __launch_bounds__(kThreads) replay_fit_kernel(const __grid_constant__ FitArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& S = *reinterpret_cast<Smem*>(smem_raw);
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank(), cs = (int)cluster.num_blocks();
    const FitLearner& l = a.learner[blockIdx.x / cs];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kThreads / 32;
    const int A = a.A, A1 = A + 1, B = a.B, hid = a.hid, n_in = a.n_in;
    const int n_units = hid * (a.duel ? 2 : 1);
    const int upc = (n_units + cs - 1) / cs;
    const int g0 = min(rank * upc, n_units), nu = min(n_units, g0 + upc) - g0;

    // offsets of unit u (global unit g0 + u) of this CTA: first-layer row, bias, stream (0 advantage / plain, 1 value)
    auto w1_off = [&](int g) { return g < hid ? g * n_in : a.off_w3 + (g - hid) * n_in; };
    auto b1_off = [&](int g) { return g < hid ? a.off_b1 + g : a.off_b3 + (g - hid); };
    auto w2_off = [&](int g, int o) { return g < hid ? a.off_w2 + o * hid + g : a.off_w4 + (g - hid); };

    if (tid < A1) {
        const int o = tid;
        const bool has = o < A || a.duel;
        const int off = o < A ? a.off_b2 + o : a.off_b4;
        S.ob[0][o] = has ? l.P[off] : 0.0f;
        S.ob[1][o] = has ? l.T[off] : 0.0f;
        S.ob[2][o] = has ? l.M[off] : 0.0f;
        S.ob[3][o] = has ? l.V[off] : 0.0f;
    }
    int until_sync = l.phase;

    for (int r = 0; r < a.n_replays; ++r) {
        const int buf = r & 1;
        const int64_t i0 = (int64_t)r * B;
        for (int b = tid; b < B; b += kThreads) {
            S.row[0][b] = l.s_row[i0 + b];
            S.row[1][b] = l.sp_row[i0 + b];
            S.act[b] = l.action[i0 + b];
            S.nact[b] = l.next_action ? l.next_action[i0 + b] : 0;
            S.rew[b] = l.reward[i0 + b];
            S.dn[b] = l.done[i0 + b];
        }
        __syncthreads();

        // ---- forward: model(s), target(s), target(s'); one warp per (pass, sample), lanes over the input bits
        for (int item = warp; item < 3 * B; item += nwarps) {
            const int p = item / B, b = item - p * B;
            const float* W = p == 0 ? l.P : l.T;
            const int64_t row = S.row[p == 2 ? 1 : 0][b];
            const bool ok = row >= 0 && row < a.n_frames;
            const uint32_t* bits = a.frames + (ok ? row : 0) * a.words;
            float acc[kMaxUnits];
#pragma unroll
            for (int u = 0; u < kMaxUnits; ++u) acc[u] = 0.0f;
            if (ok) {
                for (int w = 0; w < a.words; ++w) {
                    const int f = w * 32 + lane;
                    if (((__ldg(bits + w) >> lane) & 1u) && f < n_in) {
#pragma unroll
                        for (int u = 0; u < kMaxUnits; ++u)
                            if (u < nu) acc[u] += W[w1_off(g0 + u) + f];
                    }
                }
            }
            float part = 0.0f;  // lane o < A1: this CTA's share of output o
#pragma unroll
            for (int u = 0; u < kMaxUnits; ++u) {
                if (u < nu) {
                    float z = acc[u];
#pragma unroll
                    for (int s = 16; s > 0; s >>= 1) z += __shfl_xor_sync(0xffffffffu, z, s);
                    const int g = g0 + u;
                    const float hv = sigmoidf(z + W[b1_off(g)]);
                    if (p == 0 && lane == 0) S.h[b][u] = hv;
                    if (g < hid ? lane < A : lane == A) part += hv * W[w2_off(g, lane)];
                }
            }
            if (lane < A1) S.part[buf][p][b][lane] = part;
        }
        cluster.sync();

        // ---- every CTA adds the slices of all CTAs in rank order (identical everywhere), then the output bias
        for (int k = tid; k < 3 * B * A1; k += kThreads) {
            const int p = k / (B * A1), rem = k - p * B * A1, b = rem / A1, o = rem - b * A1;
            float s = 0.0f;
            for (int c = 0; c < cs; ++c) s += cluster.map_shared_rank(&S, c)->part[buf][p][b][o];
            S.q[p][b][o] = s + S.ob[p == 0 ? 0 : 1][o];
        }
        __syncthreads();

        // ---- targets, squared errors and the output gradient, one thread per sample
        const float inv_n = 1.0f / (float)(B * A);
        for (int b = tid; b < B; b += kThreads) {
            float qv[3][kMaxActions];
            for (int p = 0; p < 3; ++p) {
                float mean = 0.0f;
                if (a.duel) {
                    for (int o = 0; o < A; ++o) mean += S.q[p][b][o];
                    mean /= (float)A;
                }
                for (int o = 0; o < A; ++o) qv[p][o] = a.duel ? S.q[p][b][A] + (S.q[p][b][o] - mean) : S.q[p][b][o];
            }
            const int act = S.act[b], nact = S.nact[b];
            float upd = S.rew[b];
            if (!S.dn[b]) {
                if (l.next_action) {
                    if (nact >= 0 && nact < A) upd = S.rew[b] + l.gamma * qv[2][nact];
                } else {
                    float best = qv[2][0];
                    for (int o = 1; o < A; ++o) best = fmaxf(best, qv[2][o]);
                    upd = S.rew[b] + l.gamma * best;
                }
            }
            float se = 0.0f, dsum = 0.0f, dq[kMaxActions];
            for (int o = 0; o < A; ++o) {
                const float y = (o == act) ? upd : qv[1][o];
                const float e = qv[0][o] - y;
                se += e * e;
                dq[o] = 2.0f * e * inv_n;
                dsum += dq[o];
            }
            S.sqerr[b] = se;
            if (a.duel) {  // q = v + a - mean(a): dL/da_o = dq_o - mean(dq), dL/dv = sum(dq)
                const float dmean = dsum / (float)A;
                for (int o = 0; o < A; ++o) S.dout[b][o] = dq[o] - dmean;
                S.dout[b][A] = dsum;
            } else {
                for (int o = 0; o < A; ++o) S.dout[b][o] = dq[o];
                S.dout[b][A] = 0.0f;
            }
        }
        __syncthreads();

        if (rank == 0 && tid == 0 && l.loss) {
            float s = 0.0f;
            for (int b = 0; b < B; ++b) s += S.sqerr[b];
            l.loss[r] = s * inv_n;
        }
        // ---- back through the second layer into this CTA's units (reads the second layer before it is updated)
        for (int k = tid; k < B * nu; k += kThreads) {
            const int b = k / nu, u = k - b * nu, g = g0 + u;
            float dh = 0.0f;
            if (g < hid) {
                for (int o = 0; o < A; ++o) dh += S.dout[b][o] * l.P[w2_off(g, o)];
            } else {
                dh = S.dout[b][A] * l.P[w2_off(g, A)];
            }
            const float hv = S.h[b][u];
            S.dz[b][u] = dh * hv * (1.0f - hv);
        }
        __syncthreads();

        // ---- Adam on every parameter this CTA owns (+ the shared output biases, redundantly), then the target copy
        const int64_t t = l.adam_t + r + 1;
        const float lr_t = (float)(l.lr * sqrt(1.0 - pow(l.beta_2, (double)t)) / (1.0 - pow(l.beta_1, (double)t)));
        const bool sync = --until_sync == 0;
        if (sync) until_sync = l.target_every;
        for (int k = tid; k < nu * n_in; k += kThreads) {  // first-layer rows
            const int u = k / n_in, f = k - u * n_in;
            const int off = w1_off(g0 + u) + f;
            const int w = f >> 5;
            const uint32_t bit = 1u << (f & 31);
            float g = 0.0f;
            for (int b = 0; b < B; ++b) {
                const int64_t row = S.row[0][b];
                if (row >= 0 && row < a.n_frames && (__ldg(a.frames + row * a.words + w) & bit)) g += S.dz[b][u];
            }
            float m = l.M[off], v = l.V[off];
            const float p = adam(l, lr_t, l.P[off], g, m, v);
            l.P[off] = p;
            l.M[off] = m;
            l.V[off] = v;
            if (sync) l.T[off] = p;
        }
        for (int k = tid; k < nu * (1 + A1); k += kThreads) {  // first-layer biases and second-layer columns
            const int u = k / (1 + A1), c = k - u * (1 + A1), g = g0 + u;
            int off;
            float gr = 0.0f;
            if (c == 0) {
                off = b1_off(g);
                for (int b = 0; b < B; ++b) gr += S.dz[b][u];
            } else {
                const int o = c - 1;
                if (g < hid ? o >= A : o != A) continue;
                off = w2_off(g, o);
                for (int b = 0; b < B; ++b) gr += S.dout[b][o] * S.h[b][u];
            }
            float m = l.M[off], v = l.V[off];
            const float p = adam(l, lr_t, l.P[off], gr, m, v);
            l.P[off] = p;
            l.M[off] = m;
            l.V[off] = v;
            if (sync) l.T[off] = p;
        }
        if (tid < A1 && (tid < A || a.duel)) {  // output biases: every CTA, identically
            const int o = tid;
            float gr = 0.0f;
            for (int b = 0; b < B; ++b) gr += S.dout[b][o];
            S.ob[0][o] = adam(l, lr_t, S.ob[0][o], gr, S.ob[2][o], S.ob[3][o]);
            if (sync) S.ob[1][o] = S.ob[0][o];
        }
        __syncthreads();
    }

    if (rank == 0 && tid < A1 && (tid < A || a.duel)) {
        const int o = tid, off = o < A ? a.off_b2 + o : a.off_b4;
        l.P[off] = S.ob[0][o];
        l.T[off] = S.ob[1][o];
        l.M[off] = S.ob[2][o];
        l.V[off] = S.ob[3][o];
    }
    cluster.sync();  // no CTA leaves while a peer may still read its partial sums
}

// The cluster size wf_replay_fit launches with on `device`: 16 CTAs where the GPU can hold such a cluster of this kernel,
// else 8 (0: neither).  Sets the kernel's shared-memory and cluster-size attributes for that device first.  Computed once
// per device; concurrent first calls only repeat the same idempotent work.
int cluster_size_for(int device, size_t smem, cudaError_t* err) {
    constexpr int kMaxDevices = 64;
    static std::atomic<int> cached[kMaxDevices];
    if (device >= 0 && device < kMaxDevices) {
        const int c = cached[device].load(std::memory_order_relaxed);
        if (c > 0) return c;
    }
    *err = cudaFuncSetAttribute(replay_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (*err == cudaSuccess) *err = cudaFuncSetAttribute(replay_fit_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (*err != cudaSuccess) return 0;
    for (int cs : {16, 8}) {
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = cs;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.gridDim = dim3(cs);
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, replay_fit_kernel, &cfg) == cudaSuccess && n > 0) {
            if (device >= 0 && device < kMaxDevices) cached[device].store(cs, std::memory_order_relaxed);
            return cs;
        }
        cudaGetLastError();
    }
    return 0;
}

// ---- wf_replay_fit_large: the same replays for any grid, spread over the whole GPU ----------------------------------
// One cooperatively launched grid of as many CTAs as are co-resident.  The first layer's input columns are cut into
// `nc` chunks of `cw` whole observation words (a function of the shape only); CTA k owns chunks k, k + grid, ... for the
// whole launch.  Per replay:
//   forward  each CTA sums, for its chunks, the first-layer rows of the set bits of s (model and target) and s'
//            (target) in feature order, staging `sub` words of both weight matrices at a time in shared memory, and
//            writes one partial [3][B][units] per chunk to scratch;
//   -- grid barrier --
//   reduce   one CTA per sample adds the partials over chunks in a fixed tree (kSegs segments of consecutive chunks,
//            each summed in chunk order, then the segments in order), then computes the sigmoid, the second layer, the
//            target, the output gradient dout and the first-layer gradient dz of that sample;
//   -- grid barrier --
//   update   each CTA runs Adam on the first-layer entries of its chunks, g = sum over b of dz[b][u] * x[b][f] in b
//            order (the sum wf_replay_fit forms); every small parameter (first-layer biases, second layer, output
//            biases) has one owner thread of the grid; global thread 0 writes the loss.
// A CTA reads and writes only its own chunks' first-layer weights, so no barrier is needed between one replay's update
// and the next replay's forward; and the reduce of replay r + 1 starts only after every CTA has left update r, so the
// scratch needs no second buffer.  Every sum runs in an order fixed by the shape and no floating-point atomic is used:
// the result is bit-identical from run to run and whatever the number of CTAs (WF_FIT_CTAS forces it).
constexpr int kLThreads = 512;
constexpr int kMaxChunks = 128;                 // chunks of the first layer's columns
constexpr int64_t kPartBudget = int64_t(1) << 23;  // floats of the chunk partials: at most 32 MB of scratch
constexpr int kSegs = 8;                        // chunk segments of the reduction tree
constexpr int kWsFloats = 24576;                // staged first-layer weights per sub-tile: 96 KB
constexpr int kMaxSub = 8;                      // words per sub-tile
constexpr int kSlots = 4;                       // units per lane in the forward: 128 = 2 * kMaxHidden units
constexpr int kBatch = 4;                       // first-layer entries a thread loads before it uses them

struct LargeArgs {
    FitLearner l;
    const uint32_t* frames;
    int64_t n_frames;
    int n_replays;
    int n_in, words, hid, A, duel, B;
    int off_b1, off_w2, off_b2, off_w3, off_b3, off_w4, off_b4;
    int units, cw, nc, sub;
    float* part;  // [nc][3][B][units]: model(s), target(s), target(s') pre-activations of each chunk
    float* h;     // [B][units]: model hidden activations on s
    float* dz;    // [B][units]: dLoss / d(first-layer pre-activation)
    float* dout;  // [B][kOut]: dLoss / d(second-layer output)
    float* sq;    // [B]: squared error of each sample
};

// Word w of row `row` of the frames table: 0 for a row outside [0, n_frames), and bits past n_in cleared.
__device__ __forceinline__ uint32_t frame_word(const LargeArgs& a, int64_t row, int w) {
    if (row < 0 || row >= a.n_frames) return 0u;
    const uint32_t x = __ldg(a.frames + row * a.words + w);
    const int tail = a.n_in - w * 32;
    return tail >= 32 ? x : x & ((1u << tail) - 1u);
}

__global__ void __launch_bounds__(kLThreads) replay_fit_large_kernel(const __grid_constant__ LargeArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* fs = reinterpret_cast<float*>(smem_raw);
    cg::grid_group grid = cg::this_grid();
    const FitLearner& l = a.l;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kLThreads / 32;
    const int A = a.A, A1 = A + 1, B = a.B, hid = a.hid, U = a.units, n_in = a.n_in, sub = a.sub;
    const int blk = blockIdx.x, nblk = gridDim.x;
    const float inv_n = 1.0f / (float)(B * A);

    auto w1_off = [&](int g) { return g < hid ? (int64_t)g * n_in : a.off_w3 + (int64_t)(g - hid) * n_in; };
    auto b1_off = [&](int g) { return g < hid ? a.off_b1 + g : a.off_b3 + (g - hid); };
    auto w2_off = [&](int g, int o) { return g < hid ? a.off_w2 + o * hid + g : a.off_w4 + (g - hid); };

    int until_sync = l.phase;
    for (int r = 0; r < a.n_replays; ++r) {
        const int64_t i0 = (int64_t)r * B;

        // ---- forward: partial pre-activations of this CTA's chunks; warp job (j, b): j 0 = model and target on s,
        //      j 1 = target on s'; lane owns units lane + 32 * s
        float* Ws = fs;                                                      // [2][sub * 32][U]: model, target
        uint32_t* sb = reinterpret_cast<uint32_t*>(fs + 2 * sub * 32 * U);  // [2][B][sub]
        for (int c = blk; c < a.nc; c += nblk) {
            const int cw0 = c * a.cw, cw1 = min(a.words, cw0 + a.cw);
            for (int w0 = cw0; w0 < cw1; w0 += sub) {
                const int nw = min(sub, cw1 - w0), nf = nw * 32, f0 = w0 * 32;
                __syncthreads();
                for (int k0 = 0; k0 < 2 * U * nf; k0 += kBatch * kLThreads) {
                    float x[kBatch];
                    int at[kBatch];
#pragma unroll
                    for (int i = 0; i < kBatch; ++i) {
                        const int k = k0 + i * kLThreads + tid;
                        const int net = k / (U * nf), rem = k - net * U * nf, u = rem / nf, f = rem - u * nf;
                        at[i] = k < 2 * U * nf ? (net * nf + f) * U + u : -1;
                        x[i] = at[i] >= 0 && f0 + f < n_in ? (net ? l.T : l.P)[w1_off(u) + f0 + f] : 0.0f;
                    }
#pragma unroll
                    for (int i = 0; i < kBatch; ++i)
                        if (at[i] >= 0) Ws[at[i]] = x[i];
                }
                for (int k = tid; k < 2 * B * nw; k += kLThreads) {
                    const int j = k / (B * nw), rem = k - j * B * nw, b = rem / nw, w = rem - b * nw;
                    sb[(j * B + b) * sub + w] = frame_word(a, (j ? l.sp_row : l.s_row)[i0 + b], w0 + w);
                }
                __syncthreads();
                for (int job = warp; job < 2 * B; job += nwarps) {
                    const int j = job / B, b = job - j * B;
                    float* pm = a.part + ((int64_t)c * 3 * B + b) * U + lane;  // + q * B * U: pass q
                    float* p1 = pm + (j ? 2 : 1) * B * U;                        // target on s (j 0) or s' (j 1)
                    float acc0[kSlots], acc1[kSlots];
#pragma unroll
                    for (int s = 0; s < kSlots; ++s) {
                        const bool on = lane + 32 * s < U && w0 > cw0;
                        acc0[s] = on && !j ? pm[32 * s] : 0.0f;
                        acc1[s] = on ? p1[32 * s] : 0.0f;
                    }
                    for (int w = 0; w < nw; ++w) {
                        uint32_t bits = sb[(j * B + b) * sub + w];
                        while (bits) {
                            const int f = w * 32 + __ffs(bits) - 1;
                            bits &= bits - 1u;
                            const float* wm = Ws + f * U + lane;
                            const float* wt = wm + nf * U;
#pragma unroll
                            for (int s = 0; s < kSlots; ++s) {
                                if (lane + 32 * s < U) {
                                    if (!j) acc0[s] += wm[32 * s];
                                    acc1[s] += wt[32 * s];
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int s = 0; s < kSlots; ++s) {
                        if (lane + 32 * s < U) {
                            if (!j) pm[32 * s] = acc0[s];
                            p1[32 * s] = acc1[s];
                        }
                    }
                }
            }
        }
        grid.sync();

        // ---- reduce and head, one CTA per sample
        for (int b = blk; b < B; b += nblk) {
            float* seg = fs;                  // [kSegs][3][U]
            float* hq = seg + kSegs * 3 * U;  // [3][U]: hidden activations of model(s), target(s), target(s')
            float* q = hq + 3 * U;            // [3][kOut]
            float* dout = q + 3 * kOut;       // [kOut]
            const int per = (a.nc + kSegs - 1) / kSegs;
            for (int k = tid; k < kSegs * 3 * U; k += kLThreads) {
                const int s = k / (3 * U), pu = k - s * 3 * U, p = pu / U, u = pu - p * U;
                const int c1 = min(a.nc, (s + 1) * per);
                float z = 0.0f;
#pragma unroll 8
                for (int c = s * per; c < c1; ++c) z += __ldcg(a.part + (((int64_t)c * 3 + p) * B + b) * U + u);
                seg[k] = z;
            }
            __syncthreads();
            for (int k = tid; k < 3 * U; k += kLThreads) {
                const int p = k / U, u = k - p * U;
                float z = 0.0f;
                for (int s = 0; s < kSegs; ++s) z += seg[s * 3 * U + k];
                hq[k] = sigmoidf(z + __ldcg((p ? l.T : l.P) + b1_off(u)));
            }
            __syncthreads();
            if (tid < 3 * A1) {
                const int p = tid / A1, o = tid - p * A1;
                const float* W = p ? l.T : l.P;
                float s = 0.0f;
                if (o < A) {
                    for (int u = 0; u < hid; ++u) s += hq[p * U + u] * __ldcg(W + a.off_w2 + o * hid + u);
                    s += __ldcg(W + a.off_b2 + o);
                } else if (a.duel) {
                    for (int u = 0; u < hid; ++u) s += hq[p * U + hid + u] * __ldcg(W + a.off_w4 + u);
                    s += __ldcg(W + a.off_b4);
                }
                q[p * kOut + o] = s;
            }
            __syncthreads();
            if (tid == 0) {  // target, squared error and output gradient (as replay_fit_kernel)
                float qv[3][kMaxActions];
                for (int p = 0; p < 3; ++p) {
                    float mean = 0.0f;
                    if (a.duel) {
                        for (int o = 0; o < A; ++o) mean += q[p * kOut + o];
                        mean /= (float)A;
                    }
                    for (int o = 0; o < A; ++o) qv[p][o] = a.duel ? q[p * kOut + A] + (q[p * kOut + o] - mean) : q[p * kOut + o];
                }
                const int act = l.action[i0 + b], nact = l.next_action ? l.next_action[i0 + b] : 0;
                const float rew = l.reward[i0 + b];
                float upd = rew;
                if (!l.done[i0 + b]) {
                    if (l.next_action) {
                        if (nact >= 0 && nact < A) upd = rew + l.gamma * qv[2][nact];
                    } else {
                        float best = qv[2][0];
                        for (int o = 1; o < A; ++o) best = fmaxf(best, qv[2][o]);
                        upd = rew + l.gamma * best;
                    }
                }
                float se = 0.0f, dsum = 0.0f, dq[kMaxActions];
                for (int o = 0; o < A; ++o) {
                    const float e = qv[0][o] - ((o == act) ? upd : qv[1][o]);
                    se += e * e;
                    dq[o] = 2.0f * e * inv_n;
                    dsum += dq[o];
                }
                const float dmean = dsum / (float)A;
                for (int o = 0; o < A; ++o) dout[o] = a.duel ? dq[o] - dmean : dq[o];
                dout[A] = a.duel ? dsum : 0.0f;
                a.sq[b] = se;
                for (int o = 0; o < A1; ++o) a.dout[b * kOut + o] = dout[o];
            }
            __syncthreads();
            for (int u = tid; u < U; u += kLThreads) {  // back through the second layer (before it is updated)
                float dh = 0.0f;
                if (u < hid) {
                    for (int o = 0; o < A; ++o) dh += dout[o] * __ldcg(l.P + w2_off(u, o));
                } else {
                    dh = dout[A] * __ldcg(l.P + w2_off(u, A));
                }
                const float hv = hq[u];
                a.h[b * U + u] = hv;
                a.dz[b * U + u] = dh * hv * (1.0f - hv);
            }
            __syncthreads();
        }
        grid.sync();

        // ---- Adam
        const int64_t t = l.adam_t + r + 1;
        const float lr_t = (float)(l.lr * sqrt(1.0 - pow(l.beta_2, (double)t)) / (1.0 - pow(l.beta_1, (double)t)));
        const bool sync = --until_sync == 0;
        if (sync) until_sync = l.target_every;
        const int n_small = U * (1 + A1) + A1;  // per unit: bias, second-layer column; then the output biases
        for (int k = blk * kLThreads + tid; k < n_small; k += nblk * kLThreads) {
            int off;
            float gr = 0.0f;
            if (k < U * (1 + A1)) {
                const int g = k / (1 + A1), c = k - g * (1 + A1);
                if (c == 0) {
                    off = b1_off(g);
                    for (int b = 0; b < B; ++b) gr += __ldcg(a.dz + b * U + g);
                } else {
                    const int o = c - 1;
                    if (g < hid ? o >= A : o != A) continue;
                    off = w2_off(g, o);
                    for (int b = 0; b < B; ++b) gr += __ldcg(a.dout + b * kOut + o) * __ldcg(a.h + b * U + g);
                }
            } else {
                const int o = k - U * (1 + A1);
                if (o == A && !a.duel) continue;
                off = o < A ? a.off_b2 + o : a.off_b4;
                for (int b = 0; b < B; ++b) gr += __ldcg(a.dout + b * kOut + o);
            }
            float m = l.M[off], v = l.V[off];
            const float p = adam(l, lr_t, l.P[off], gr, m, v);
            l.P[off] = p;
            l.M[off] = m;
            l.V[off] = v;
            if (sync) l.T[off] = p;
        }
        if (blk == 0 && tid == 0 && l.loss) {
            float s = 0.0f;
            for (int b = 0; b < B; ++b) s += __ldcg(a.sq + b);
            l.loss[r] = s * inv_n;
        }
        // first layer of this CTA's chunks; mk[bb][f]: which samples 32 * bb .. 32 * bb + 31 have bit f set
        const int nbb = (B + 31) / 32;
        float* dzs = fs;                                                // [B][U]
        uint32_t* ub = reinterpret_cast<uint32_t*>(fs + B * U);        // [B][sub]
        uint32_t* mk = ub + B * sub;                                    // [nbb][sub * 32]
        if (blk < a.nc) {
            __syncthreads();
            for (int k = tid; k < B * U; k += kLThreads) dzs[k] = __ldcg(a.dz + k);
        }
        for (int c = blk; c < a.nc; c += nblk) {
            const int cw0 = c * a.cw, cw1 = min(a.words, cw0 + a.cw);
            for (int w0 = cw0; w0 < cw1; w0 += sub) {
                const int nw = min(sub, cw1 - w0), nf = nw * 32, f0 = w0 * 32;
                __syncthreads();
                for (int k = tid; k < B * nw; k += kLThreads) {
                    const int b = k / nw, w = k - b * nw;
                    ub[b * sub + w] = frame_word(a, l.s_row[i0 + b], w0 + w);
                }
                __syncthreads();
                for (int k = tid; k < nbb * nf; k += kLThreads) {
                    const int bb = k / nf, f = k - bb * nf;
                    uint32_t m = 0u;
                    for (int i = 0; i < 32 && bb * 32 + i < B; ++i) m |= ((ub[(bb * 32 + i) * sub + (f >> 5)] >> (f & 31)) & 1u) << i;
                    mk[bb * sub * 32 + f] = m;
                }
                __syncthreads();
                for (int k0 = 0; k0 < U * nf; k0 += kBatch * kLThreads) {  // kBatch entries per thread: loads in flight
                    float g[kBatch], p[kBatch], m[kBatch], v[kBatch];
                    int64_t off[kBatch];
                    bool ok[kBatch];
#pragma unroll
                    for (int i = 0; i < kBatch; ++i) {
                        const int k = k0 + i * kLThreads + tid, u = k / nf, f = k - u * nf;
                        ok[i] = k < U * nf && f0 + f < n_in;
                        g[i] = 0.0f;
                        off[i] = ok[i] ? w1_off(u) + f0 + f : 0;
                        if (ok[i]) {
                            for (int bb = 0; bb < nbb; ++bb) {
                                const float* d = dzs + bb * 32 * U + u;
                                for (uint32_t mb = mk[bb * sub * 32 + f]; mb; mb &= mb - 1u) g[i] += d[(__ffs(mb) - 1) * U];
                            }
                        }
                    }
#pragma unroll
                    for (int i = 0; i < kBatch; ++i) {
                        if (ok[i]) {
                            p[i] = l.P[off[i]];
                            m[i] = l.M[off[i]];
                            v[i] = l.V[off[i]];
                        }
                    }
#pragma unroll
                    for (int i = 0; i < kBatch; ++i) {
                        if (ok[i]) {
                            p[i] = adam(l, lr_t, p[i], g[i], m[i], v[i]);
                            l.P[off[i]] = p[i];
                            l.M[off[i]] = m[i];
                            l.V[off[i]] = v[i];
                            if (sync) l.T[off[i]] = p[i];
                        }
                    }
                }
            }
        }
    }
}

// Refuses a learner whose pointers or hyper-parameters wf_replay_fit would refuse; `who` prefixes the message.
int check_learner(const std::string& who, const wf_fit_learner& l) {
    if (!l.params || !l.target || !l.adam_m || !l.adam_v || !l.s_row || !l.sp_row || !l.action || !l.reward || !l.done)
        return api_fail(WF_ERR_INVALID, who + ": null argument");
    const wf_fit_params* hp = &l.hp;
    if (hp->target_every < 1 || hp->phase < 1 || hp->phase > hp->target_every)
        return api_fail(WF_ERR_INVALID, who + ": need target_every >= 1 and 1 <= phase <= target_every");
    if (hp->adam_t < 0) return api_fail(WF_ERR_INVALID, who + ": adam_t must be >= 0");
    if (!(hp->clipvalue > 0.0) || !std::isfinite(hp->gamma) || !std::isfinite(hp->lr) || !(hp->beta_1 >= 0.0 && hp->beta_1 < 1.0) ||
        !(hp->beta_2 >= 0.0 && hp->beta_2 < 1.0) || !(hp->epsilon >= 0.0))
        return api_fail(WF_ERR_INVALID, who + ": bad hyper-parameter (need clipvalue > 0, 0 <= beta < 1, epsilon >= 0)");
    for (const void* p : {(const void*)l.params, (const void*)l.target, (const void*)l.adam_m, (const void*)l.adam_v,
                          (const void*)l.action, (const void*)l.next_action, (const void*)l.reward, (const void*)l.loss})
        if (reinterpret_cast<uintptr_t>(p) & 3u) return api_fail(WF_ERR_INVALID, who + ": buffers must be 4-byte aligned");
    if ((reinterpret_cast<uintptr_t>(l.s_row) | reinterpret_cast<uintptr_t>(l.sp_row)) & 7u)
        return api_fail(WF_ERR_INVALID, who + ": s_row and sp_row must be 8-byte aligned");
    return WF_OK;
}

// The shape and call checks wf_replay_fit and wf_replay_fit_large share (the grid is checked by the caller).
int check_fit_args(const std::string& fn, const wf_mlp_shape& sh, int32_t n_replays, const uint32_t* frames_dev,
                   int64_t n_frames) {
    if (sh.hidden < 1 || sh.hidden > kMaxHidden) return api_fail(WF_ERR_INVALID, fn + ": hidden must be in 1..64");
    if (sh.n_actions < 1 || sh.n_actions > kMaxActions) return api_fail(WF_ERR_INVALID, fn + ": n_actions must be in 1..8");
    if (sh.dueling != 0 && sh.dueling != 1) return api_fail(WF_ERR_INVALID, fn + ": dueling must be 0 or 1");
    if (sh.batch < 1 || sh.batch > kMaxBatch) return api_fail(WF_ERR_INVALID, fn + ": batch must be in 1..256");
    if (n_replays < 1) return api_fail(WF_ERR_INVALID, fn + ": n_replays must be >= 1");
    if (n_frames < 0) return api_fail(WF_ERR_INVALID, fn + ": n_frames must be >= 0");
    if (reinterpret_cast<uintptr_t>(frames_dev) & 3u) return api_fail(WF_ERR_INVALID, fn + ": buffers must be 4-byte aligned");
    return WF_OK;
}

// The flat layout of include/wildfire.h in a kernel's arguments (FitArgs, LargeArgs).
template <class Args>
void set_layout(Args& a, const wf_mlp_shape& sh) {
    a.n_in = sh.width * sh.height * 3;
    a.words = (int)wf::obs_bits_words(sh.width, sh.height);
    a.hid = sh.hidden, a.A = sh.n_actions, a.duel = sh.dueling, a.B = sh.batch;
    a.off_b1 = a.hid * a.n_in;
    a.off_w2 = a.off_b1 + a.hid;
    a.off_b2 = a.off_w2 + a.A * a.hid;
    a.off_w3 = a.off_b2 + a.A;
    a.off_b3 = a.off_w3 + a.hid * a.n_in;
    a.off_w4 = a.off_b3 + a.hid;
    a.off_b4 = a.off_w4 + a.hid;
}

FitLearner prepare_learner(const wf_fit_learner& in) {
    const wf_fit_params* hp = &in.hp;
    FitLearner l;
    l.P = in.params, l.T = in.target, l.M = in.adam_m, l.V = in.adam_v;
    l.s_row = in.s_row, l.sp_row = in.sp_row, l.action = in.action, l.next_action = in.next_action;
    l.reward = in.reward, l.done = in.done, l.loss = in.loss;
    // scalars as torch applies them to float32 tensors (KerasAdam.step): cast once to float
    l.gamma = (float)hp->gamma;
    l.b1 = (float)hp->beta_1, l.omb1 = (float)(1.0 - hp->beta_1);
    l.b2 = (float)hp->beta_2, l.omb2 = (float)(1.0 - hp->beta_2);
    l.eps = (float)hp->epsilon, l.clip = (float)hp->clipvalue;
    l.lr = hp->lr, l.beta_1 = hp->beta_1, l.beta_2 = hp->beta_2;
    l.adam_t = hp->adam_t, l.target_every = hp->target_every, l.phase = hp->phase;
    return l;
}

// wf_replay_fit_many after the caller's null checks; `name` is the entry point the messages name.
int replay_fit_impl(const char* name, const wf_mlp_shape& sh, int32_t n_learners, const wf_fit_learner* learners,
                    int32_t n_replays, const uint32_t* frames_dev, int64_t n_frames, void* stream) {
    const std::string fn(name);
    if (n_learners < 1 || n_learners > kMaxLearners) return api_fail(WF_ERR_INVALID, fn + ": n_learners must be in 1..64");
    if (sh.height < 10 || sh.width < sh.height || sh.width > 32)
        return api_fail(WF_ERR_INVALID, fn + ": the grid must satisfy 10 <= height <= width <= 32");
    if (int rc = check_fit_args(fn, sh, n_replays, frames_dev, n_frames)) return rc;
    for (int j = 0; j < n_learners; ++j)
        if (int rc = check_learner(n_learners == 1 ? fn : fn + ": learner " + std::to_string(j), learners[j])) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return api_fail(WF_ERR_CUDA, "no CUDA device: libwildfire_b200 has no CPU fallback");

    FitArgs a{};
    a.frames = frames_dev, a.n_frames = n_frames, a.n_replays = n_replays;
    set_layout(a, sh);
    for (int j = 0; j < n_learners; ++j) a.learner[j] = prepare_learner(learners[j]);

    const size_t smem = sizeof(Smem);
    int device = 0;
    cudaError_t err = cudaGetDevice(&device);
    const int cs = err == cudaSuccess ? cluster_size_for(device, smem, &err) : 0;
    if (err != cudaSuccess) return api_fail(WF_ERR_CUDA, fn + ": " + cudaGetErrorString(err));
    if (cs == 0) return api_fail(WF_ERR_CUDA, fn + ": no thread-block cluster of 8 or 16 CTAs fits this device");
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cs;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3(cs * n_learners);  // one cluster per learner: clusters beyond what the GPU holds run in later waves
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = static_cast<cudaStream_t>(stream);
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    err = cudaLaunchKernelEx(&cfg, replay_fit_kernel, a);
    if (err != cudaSuccess) return api_fail(WF_ERR_CUDA, fn + ": " + cudaGetErrorString(err));
    return WF_OK;
}

// wf_replay_fit_large after the null checks.
int replay_fit_large_impl(const wf_mlp_shape& sh, const wf_fit_learner& learner, int32_t n_replays,
                          const uint32_t* frames_dev, int64_t n_frames, void* stream) {
    const std::string fn("wf_replay_fit_large");
    if (sh.height < 10 || sh.width < sh.height)
        return api_fail(WF_ERR_INVALID, fn + ": the grid must satisfy 10 <= height <= width");
    if (int rc = check_fit_args(fn, sh, n_replays, frames_dev, n_frames)) return rc;
    const int64_t n_in = (int64_t)sh.width * sh.height * 3;
    const int64_t n_flat = sh.hidden * (n_in + 1 + sh.n_actions) + sh.n_actions + (sh.dueling ? sh.hidden * (n_in + 2) + 1 : 0);
    if (n_flat > INT32_MAX)
        return api_fail(WF_ERR_INVALID, fn + ": the flat parameter buffer would exceed 2^31 - 1 floats");
    if (int rc = check_learner(fn, learner)) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return api_fail(WF_ERR_CUDA, "no CUDA device: libwildfire_b200 has no CPU fallback");

    LargeArgs a{};
    a.l = prepare_learner(learner);
    a.frames = frames_dev, a.n_frames = n_frames, a.n_replays = n_replays;
    set_layout(a, sh);
    a.units = a.hid * (a.duel ? 2 : 1);
    // chunks: at most kMaxChunks, and at most kPartBudget floats of partials; sub-tiles: kWsFloats staged weights
    const int64_t per_chunk = 3LL * a.B * a.units;
    const int64_t nc_max = std::max<int64_t>(1, std::min<int64_t>(kMaxChunks, kPartBudget / per_chunk));
    a.cw = (int)((a.words + nc_max - 1) / nc_max);
    a.nc = (a.words + a.cw - 1) / a.cw;
    a.sub = std::max(1, std::min(kMaxSub, kWsFloats / (64 * a.units)));
    const int nbb = (a.B + 31) / 32;
    const size_t smem = 4 * std::max({(size_t)2 * a.sub * 32 * a.units + 2 * a.B * a.sub,                  // forward
                                      (size_t)(kSegs + 1) * 3 * a.units + 4 * kOut,                       // reduce
                                      (size_t)a.B * a.units + a.B * a.sub + nbb * a.sub * 32});           // update
    const size_t scratch = 4 * ((size_t)a.nc * per_chunk + 2 * a.B * a.units + a.B * kOut + a.B);

    int device = 0, n_sm = 0, per_sm = 0;
    cudaError_t err = cudaGetDevice(&device);
    if (err == cudaSuccess) err = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(replay_fit_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err == cudaSuccess) err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, replay_fit_large_kernel, kLThreads, smem);
    if (err != cudaSuccess) return api_fail(WF_ERR_CUDA, fn + ": " + cudaGetErrorString(err));
    int ctas = n_sm * per_sm;
    if (ctas < 1) return api_fail(WF_ERR_CUDA, fn + ": the kernel does not fit this device");
    if (const char* env = std::getenv("WF_FIT_CTAS")) {  // experiments and tests: the result does not depend on it
        const int want = std::atoi(env);
        if (want > 0) ctas = std::min(ctas, want);
    }
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    void* buf = nullptr;
    err = cudaMallocAsync(&buf, scratch, st);
    if (err != cudaSuccess) return api_fail(WF_ERR_CUDA, fn + ": scratch: " + cudaGetErrorString(err));
    float* f = static_cast<float*>(buf);
    a.part = f;
    a.h = a.part + (size_t)a.nc * per_chunk;
    a.dz = a.h + a.B * a.units;
    a.dout = a.dz + a.B * a.units;
    a.sq = a.dout + a.B * kOut;
    void* args[] = {&a};
    err = cudaLaunchCooperativeKernel((const void*)replay_fit_large_kernel, dim3(ctas), dim3(kLThreads), args, smem, st);
    const cudaError_t err_free = cudaFreeAsync(buf, st);
    if (err == cudaSuccess) err = err_free;
    if (err != cudaSuccess) return api_fail(WF_ERR_CUDA, fn + ": " + cudaGetErrorString(err));
    return WF_OK;
}

}  // namespace

extern "C" int wf_replay_fit_many(const wf_mlp_shape* shape, int32_t n_learners, const wf_fit_learner* learners_host,
                                  int32_t n_replays, const uint32_t* frames_dev, int64_t n_frames, void* stream) {
    if (!shape || !learners_host || !frames_dev) return api_fail(WF_ERR_INVALID, "wf_replay_fit_many: null argument");
    return replay_fit_impl("wf_replay_fit_many", *shape, n_learners, learners_host, n_replays, frames_dev, n_frames, stream);
}

extern "C" int wf_replay_fit(const wf_mlp_shape* shape, const wf_fit_params* hp, int32_t n_replays, float* params_dev,
                             float* target_dev, float* adam_m_dev, float* adam_v_dev, const uint32_t* frames_dev,
                             int64_t n_frames, const int64_t* s_row_dev, const int64_t* sp_row_dev,
                             const int32_t* action_dev, const int32_t* next_action_dev, const float* reward_dev,
                             const uint8_t* done_dev, float* loss_dev, void* stream) {
    if (!shape || !hp || !frames_dev) return api_fail(WF_ERR_INVALID, "wf_replay_fit: null argument");
    const wf_fit_learner l{params_dev, target_dev, adam_m_dev, adam_v_dev, s_row_dev, sp_row_dev, action_dev, next_action_dev,
                           reward_dev, done_dev, loss_dev, *hp};
    return replay_fit_impl("wf_replay_fit", *shape, 1, &l, n_replays, frames_dev, n_frames, stream);
}

extern "C" int wf_replay_fit_large(const wf_mlp_shape* shape, const wf_fit_params* hp, int32_t n_replays, float* params_dev,
                                   float* target_dev, float* adam_m_dev, float* adam_v_dev, const uint32_t* frames_dev,
                                   int64_t n_frames, const int64_t* s_row_dev, const int64_t* sp_row_dev,
                                   const int32_t* action_dev, const int32_t* next_action_dev, const float* reward_dev,
                                   const uint8_t* done_dev, float* loss_dev, void* stream) {
    if (!shape || !hp || !frames_dev) return api_fail(WF_ERR_INVALID, "wf_replay_fit_large: null argument");
    const wf_fit_learner l{params_dev, target_dev, adam_m_dev, adam_v_dev, s_row_dev, sp_row_dev, action_dev, next_action_dev,
                           reward_dev, done_dev, loss_dev, *hp};
    return replay_fit_large_impl(*shape, l, n_replays, frames_dev, n_frames, stream);
}
