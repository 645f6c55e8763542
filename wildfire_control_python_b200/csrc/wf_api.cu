// wf_api.cu -- the C ABI of libwildfire_b200.so (include/wildfire.h): handle lifetime, argument
// checks, wind table, state import/export kernels and dispatch to the two kernel families.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif
#include <chrono>

#include "wf_families.cuh"


using namespace wf;

namespace wf {  // wf_hostpool.cpp
class HostPool;
HostPool* hostpool_create(int threads);
void hostpool_destroy(HostPool* p);
int hostpool_threads(const HostPool* p);
void hostpool_expand(HostPool* p, const uint32_t* packed, uint8_t* out, int64_t records, int64_t rec_words, int64_t env_bits,
                     int64_t envs_per_record, int64_t n_envs);
bool hostpool_expand_session(HostPool* p, const uint32_t* packed, uint8_t* out, int64_t records, int64_t rec_words,
                             int64_t env_bits, int64_t envs_per_record, int64_t n_envs, const volatile uint32_t* flags,
                             uint32_t seq, int64_t records_per_slice, double* reward, uint8_t* done, double default_reward,
                             double death_penalty, double contained_bonus, double cells, int64_t timeout_ns, int64_t sectors,
                             const uint32_t* full_area, int64_t full_stride, bool out_bits);
int hostpool_default_threads();
double hostpool_first_flag_seconds(const HostPool* p);
}  // namespace wf

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
namespace wf {  // the error text of the entry points in other translation units (wf_learn.cu)
int api_fail(int code, const std::string& msg) { return fail(code, msg); }
}  // namespace wf
#define WF_CUDA(expr)                                                                         \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return fail(WF_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));     \
    } while (0)

// Every entry point runs on the handle's device and leaves the caller's current device as it found it.
struct DeviceGuard {
    int prev = -1, dev;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device) : dev(device) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) err = cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
};
#define WF_ON_DEVICE(e)               \
    DeviceGuard _guard((e)->device);  \
    WF_CUDA(_guard.err)

struct wf_env {
    wf_config cfg;
    int32_t N, device;
    bool tile;
    DevState st;
    StepCfg sc;
    WindTable wind_host;
    int32_t n_wind;
    WindTable* wind_dev;
    int32_t a_iter;  // METADATA['a_speed_iter']: one per handle, not reset by reset() (Q8)
    int64_t launches;
    TileState* tstate;
    float* mlp_dev;      // WF_POLICY_MLP weights: per network w1 | base | w2 | b2 | threshold
    int32_t mlp_cap;     // network blocks mlp_dev holds
    MlpPolicy mlp;       // device pointers into mlp_dev (hid == 0: not set)
    FinalCapture fin;    // wf_set_final_capture (records == nullptr: off)
    // wf_step_host staging
    cudaStream_t hstream;
    // wf_step_host runs on its own stream: it is ordered behind everything the caller queued through the *_dev entry
    // points (reset, set_state, set_fire_to, step ...) by an event recorded on the stream of the last such call.
    cudaStream_t dev_stream;
    bool dev_pending;
    cudaEvent_t dev_event;
    bool host_direct, host_obs_direct;
    int32_t* h_actions;
    uint8_t* h_mask;   // wf_reset_host staging
    wf_init* h_init;
    void* h_obs;
    size_t h_obs_bytes;
    double* h_reward;
    uint8_t* h_done;
    // packed-observation path of wf_step_host: mapped page-locked record buffer + expansion threads
    bool host_packed;
    uint32_t* h_packed;      // host address
    uint32_t* h_packed_dev;  // device alias
    uint32_t* d_packed;      // HBM staging (WF_HOST_PACKED=dma: kernel -> HBM -> one DMA copy)
    bool packed_dma;
    size_t h_packed_words;
    HostPool* pool;
    const void* alias_host[4];  // the caller's four host buffers of the previous wf_step_host call ...
    void* alias_dev[4];         // ... and their device aliases (a caller steps with the same buffers every time)
    uint32_t alias_age;         // the cache is re-validated every 1024 calls (a buffer may have been re-allocated)
    double t_launch, t_sync, t_expand;  // WF_HOST_TIMING=1: accumulated seconds of the packed path's three parts
    int64_t t_calls;
    // WF_HOST_GRAPH=1 (experiment, off by default): the packed path's kernel + DMA copy as ONE instantiated CUDA graph,
    // re-captured when the caller's buffers change.  Only with a_speed == 1 (then every launch has the same parameters).
    bool host_graph;
    cudaGraphExec_t hg_exec;
    const void* hg_key[3];
    // wf_host_session: the warp kernel as a resident step server driven through mapped page-locked memory
    struct Session {
        bool wanted, running;
        uint32_t seq, generation;   // last sequence number rung; id of the current / last launch
        uint32_t* ctl;              // mapped host: doorbell @0, parked @16 (words), done flags @32 + 16 * slice
        uint32_t* ctl_dev;
        int32_t* actions;           // mapped host [N, padded to 4]
        int32_t* actions_dev;       // its device alias
        int32_t* actions_hbm;       // HBM copy made by the kernel's CTA 0 every step
        uint32_t* rec;              // mapped host [records][rec_words + 1]
        uint32_t* rec_dev;
        uint32_t* sync_dev;         // device: go @0, arrival counters @16 + slice
        unsigned long long* dbg_dev;  // device: the kernel's debug counters (SrvCtl::dbg)
        double t_wait;              // WF_HOST_TIMING: seconds between ringing and the last slice expanded
        int slices, ctas_per_slice;
        int sectors;                // sectors per record of the self-validating transport (0: completion flags + system fence)
        bool persistent_obs;        // wf_host_session mode 2: change-list records, the caller's array is patched in place
        uint32_t* full;             // mapped host [records][full_stride]: whole bit streams of the records flagged "full"
        uint32_t* full_dev;
        int full_stride;
        const void* frame_ptr;      // the caller's observation array as of the last step served (nullptr: not in step with it)
        int32_t frame_dtype;        // ... and its obs_dtype (WF_OBS_U8 or WF_OBS_BITS)
        int64_t full_frames;        // steps that asked for every record in full
        int64_t launches, steps, relaunch_races;
    } sess;
};
constexpr int kSessMaxSlices = 64;
extern "C" {
static int session_park(wf_env* e);
}

// ---------------------------------------------------------------------------------------------
// canonical-plane export / import (parity injection, checkpoint) -- works for both layouts
__global__ void get_state_kernel(DevState s, uint8_t* type, uint8_t* burning, uint8_t* fm_inf, uint8_t* fuel,
                                 uint8_t* hits, uint8_t* apos) {
    const size_t cells = (size_t)s.N * s.W * s.H;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < cells; i += (size_t)gridDim.x * blockDim.x) {
        const int y = (int)(i % s.H), x = (int)((i / s.H) % s.W), env = (int)(i / ((size_t)s.H * s.W));
        const int w = y >> 5, b = y & 31;
        auto bit = [&](int p) { return (s.planes[word_index(s, p, env, x, w)] >> b) & 1u; };
        if (type) type[i] = bit(P_G) ? WF_GRASS : bit(P_F) ? WF_FIRE : bit(P_BT) ? WF_BURNT : bit(P_D) ? WF_DIRT : WF_WATER;
        if (burning) burning[i] = (uint8_t)bit(P_B);
        if (fm_inf) fm_inf[i] = (uint8_t)bit(P_I);
        if (fuel) {
            uint32_t f = 0;
            for (int q = 0; q < s.FB; ++q) f |= ((*fuel_slice(s, q, env, x, w) >> b) & 1u) << q;
            fuel[i] = (uint8_t)f;
        }
        if (hits) {
            uint32_t hv;
            if (s.HB) {  // bit-sliced total (direction-independent quanta): reported in the N byte
                hv = 0u;
                for (int q = 0; q < s.HB; ++q) hv |= bit(P_FU0 + s.FB + q) << q;
            } else {
                hv = s.hits[i];
            }
            reinterpret_cast<uint32_t*>(hits)[i] = hv;
        }
        if (apos) {
            const int32_t* sc = s.scal + (size_t)env * WF_NSCALARS;
            apos[i] = (sc[WF_S_VISIBLE] && sc[WF_S_AX] == x && sc[WF_S_AY] == y) ? 1 : 0;
        }
    }
}

__global__ void set_state_kernel(DevState s, const uint8_t* type, const uint8_t* burning, const uint8_t* fm_inf,
                                 const uint8_t* fuel, const uint8_t* hits) {
    const size_t words = (size_t)s.N * s.W * s.HW;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < words; i += (size_t)gridDim.x * blockDim.x) {
        const int w = (int)(i % s.HW), x = (int)((i / s.HW) % s.W), env = (int)(i / ((size_t)s.HW * s.W));
        const int y0 = w * 32, ny = min(32, s.H - y0);
        const size_t cell0 = ((size_t)env * s.W + x) * s.H + y0;
        if (type) {
            uint32_t m[5] = {0, 0, 0, 0, 0};
            for (int b = 0; b < ny; ++b) {
                const int t = type[cell0 + b];
                m[t < 5 ? t : 0] |= 1u << b;
            }
            s.planes[word_index(s, P_G, env, x, w)] = m[0];
            s.planes[word_index(s, P_F, env, x, w)] = m[1];
            s.planes[word_index(s, P_BT, env, x, w)] = m[2];
            s.planes[word_index(s, P_D, env, x, w)] = m[3];
            s.planes[word_index(s, P_WT, env, x, w)] = m[4];
        }
        if (burning) {
            uint32_t m = 0;
            for (int b = 0; b < ny; ++b) m |= (burning[cell0 + b] ? 1u : 0u) << b;
            s.planes[word_index(s, P_B, env, x, w)] = m;
        }
        if (fm_inf) {
            uint32_t m = 0;
            for (int b = 0; b < ny; ++b) m |= (fm_inf[cell0 + b] ? 1u : 0u) << b;
            s.planes[word_index(s, P_I, env, x, w)] = m;
        }
        if (fuel) {
            for (int q = 0; q < s.FB; ++q) {
                uint32_t m = 0;
                for (int b = 0; b < ny; ++b) m |= ((uint32_t)(fuel[cell0 + b] >> q) & 1u) << b;
                *fuel_slice(s, q, env, x, w) = m;
            }
        }
        if (hits && s.HB) {
            for (int q = 0; q < s.HB; ++q) {
                uint32_t m = 0;
                for (int b = 0; b < ny; ++b) {
                    const uint32_t hv = reinterpret_cast<const uint32_t*>(hits)[cell0 + b];
                    const uint32_t tot = (hv & 255u) + ((hv >> 8) & 255u) + ((hv >> 16) & 255u) + (hv >> 24);
                    m |= ((tot >> q) & 1u) << b;
                }
                s.planes[word_index(s, P_FU0 + s.FB + q, env, x, w)] = m;
            }
        } else if (hits) {
            for (int b = 0; b < ny; ++b) s.hits[cell0 + b] = reinterpret_cast<const uint32_t*>(hits)[cell0 + b];
        }
    }
}

__global__ void set_scalars_kernel(DevState s, const int32_t* scalars) {
    const size_t n = (size_t)s.N * WF_NSCALARS;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        s.scal[i] = scalars[i];
}

// World.set_fire_to(cell), environment.py:233-246, one thread per env.
__global__ void set_fire_kernel(DevState s, const int32_t* cells) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= s.N) return;
    const int x = cells[2 * env], y = cells[2 * env + 1];
    if (x < 0 || x >= s.W || y < 0 || y >= s.H) return;
    const int w = y >> 5;
    const uint32_t bit = 1u << (y & 31);
    const bool was_burning = (s.planes[word_index(s, P_B, env, x, w)] & bit) != 0u;  // burning_cells is a set
    s.planes[word_index(s, P_G, env, x, w)] &= ~bit;
    s.planes[word_index(s, P_BT, env, x, w)] &= ~bit;
    s.planes[word_index(s, P_D, env, x, w)] &= ~bit;
    s.planes[word_index(s, P_WT, env, x, w)] &= ~bit;
    s.planes[word_index(s, P_F, env, x, w)] |= bit;
    s.planes[word_index(s, P_B, env, x, w)] |= bit;
    int32_t* sc = s.scal + (size_t)env * WF_NSCALARS;
    if (x == 0 || x == s.W - 1 || y == 0 || y == s.H - 1) sc[WF_S_FIRE_AT_BORDER] = 1;
    if (!was_burning) sc[WF_S_N_BURNING] += 1;
}

// World.get_state() without stepping, generic layout (used by wf_get_obs).
__global__ void get_obs_kernel(DevState s, void* obs, int dtype) {
    const size_t cells = (size_t)s.N * s.W * s.H;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < cells; i += (size_t)gridDim.x * blockDim.x) {
        const int y = (int)(i % s.H), x = (int)((i / s.H) % s.W), env = (int)(i / ((size_t)s.H * s.W));
        const int w = y >> 5, b = y & 31;
        const int32_t* sc = s.scal + (size_t)env * WF_NSCALARS;
        const uint32_t a = (sc[WF_S_VISIBLE] && sc[WF_S_AX] == x && sc[WF_S_AY] == y) ? 1u : 0u;
        const uint32_t f = (s.planes[word_index(s, P_F, env, x, w)] >> b) & 1u;
        const uint32_t d = ((s.planes[word_index(s, P_I, env, x, w)] >> b) & 1u) ^ 1u;
        if (dtype == WF_OBS_U8) {
            uint8_t* o = static_cast<uint8_t*>(obs) + 3 * i;
            o[0] = (uint8_t)a; o[1] = (uint8_t)f; o[2] = (uint8_t)d;
        } else if (dtype == WF_OBS_BF16) {
            uint16_t* o = static_cast<uint16_t*>(obs) + 3 * i;
            o[0] = a ? kBf16One : 0; o[1] = f ? kBf16One : 0; o[2] = d ? kBf16One : 0;
        } else {
            float* o = static_cast<float*>(obs) + 3 * i;
            o[0] = (float)a; o[1] = (float)f; o[2] = (float)d;
        }
    }
}

// wf_get_obs with WF_OBS_BITS: one thread per output word (padding bits after the env's last element stay 0).
__global__ void get_obs_bits_kernel(DevState s, uint32_t* obs) {
    const int nbits = s.W * s.H * 3;
    const int64_t wpe = obs_bits_words(s.W, s.H), words = (int64_t)s.N * wpe;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < words; i += (int64_t)gridDim.x * blockDim.x) {
        const int env = (int)(i / wpe), k0 = (int)(i - env * wpe) * 32;
        const int32_t* sc = s.scal + (size_t)env * WF_NSCALARS;
        const int aidx = sc[WF_S_VISIBLE] ? (sc[WF_S_AX] * s.H + sc[WF_S_AY]) * 3 : -1;  // the agent_pos element
        uint32_t v = 0u;
        for (int b = 0; b < 32 && k0 + b < nbits; ++b) {
            const int k = k0 + b, cell = k / 3, c = k - 3 * cell, x = cell / s.H, y = cell - x * s.H;
            uint32_t bit;
            if (c == 0) bit = k == aidx ? 1u : 0u;
            else if (c == 1) bit = (s.planes[word_index(s, P_F, env, x, y >> 5)] >> (y & 31)) & 1u;
            else bit = ((s.planes[word_index(s, P_I, env, x, y >> 5)] >> (y & 31)) & 1u) ^ 1u;
            v |= bit << b;
        }
        obs[i] = v;
    }
}

// wf_set_policy_mlp_dev / wf_set_policy_mlp_nets_dev: wf_set_policy_mlp's host repack, one thread per float of a network's
// packed block (network blockIdx.y), from nn.Linear-oriented weights (w1 [hidden][n_in], w2 [A][hidden]; network k's at
// in_stride floats after network k - 1's).  Every float of the block is written (padding 0, missing actions' bias -inf),
// and `base` is summed in float64 in the host's order, so each block is byte-identical to the host path's.
struct MlpThresholds {
    uint32_t v[kMlpMaxNets];  // explore threshold of every network (mlp_eps_threshold)
};
__global__ void pack_policy_mlp_kernel(float* __restrict__ out, const float* __restrict__ w1, const float* __restrict__ b1,
                                       const float* __restrict__ w2, const float* __restrict__ b2, size_t in_stride,
                                       int n_in, int cells, int hidden, int A, int L, const MlpThresholds eps) {
    const int hpl = 64 / L, net = blockIdx.y;
    const size_t n_w1 = (size_t)n_in * 64, total = mlp_net_floats(n_in);
    out += net * total;
    w1 += net * in_stride, b1 += net * in_stride, w2 += net * in_stride, b2 += net * in_stride;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        float v = 0.0f;
        if (i < n_w1) {  // w1 [n_in][64]: unit j sits at (j % L) * hpl + j / L
            const int f = (int)(i / 64), pos = (int)(i % 64);
            const int j = (pos % hpl) * L + pos / hpl;
            if (j < hidden) v = w1[(size_t)j * n_in + f];
        } else if (i < n_w1 + 64) {  // base: bias1 + the all-free empty map (channel 2 of every cell)
            const int j = (int)(i - n_w1);
            if (j < hidden) {
                double acc = b1[j];
                for (int cell = 0; cell < cells; ++cell) acc += w1[(size_t)j * n_in + cell * 3 + 2];
                v = (float)acc;
            }
        } else if (i < n_w1 + 64 + 512) {  // w2 [2][64][4]: action b of unit j at (b / 4) * 256 + j * 4 + b % 4
            const int k = (int)(i - n_w1 - 64), j = (k % 256) / 4, b = (k / 256) * 4 + k % 4;
            if (j < hidden && b < A) v = w2[(size_t)b * hidden + j];
        } else if (i < n_w1 + 64 + 512 + 8) {
            const int b = (int)(i - n_w1 - 64 - 512);
            v = b < A ? b2[b] : -INFINITY;
        } else if (i == n_w1 + 64 + 512 + 8) {
            v = __uint_as_float(eps.v[net]);
        }
        out[i] = v;
    }
}

// wf_unpack_obs_bits: one warp per output row.  Lane l expands 16-bit chunk c = l + 32 t of the row into 16 elements with
// 16-byte stores (uint8: two look-ups in the byte -> 8 bytes table); rows whose elements are not 16-byte aligned (e.g.
// 14x14x3 = 588 bytes) and a row's ragged tail are written element by element.
__device__ __forceinline__ uint32_t unpack_bf16_pair(uint32_t bytes, uint32_t sel) {  // two 0/1 bytes -> two bfloat16
    return __byte_perm(bytes, 0u, sel) * (uint32_t)kBf16One;
}
__global__ void unpack_obs_bits_kernel(const uint32_t* __restrict__ bits, int64_t n_rows, const int64_t* __restrict__ index,
                                       int64_t n_out, int W, int H, void* out, int dtype) {
    __shared__ uint2 tab8[256];  // bit i of the index -> byte i
    for (int v = threadIdx.x; v < 256; v += blockDim.x)
        tab8[v] = make_uint2(((v & 15u) * 0x00204081u) & 0x01010101u, (((v >> 4) & 15u) * 0x00204081u) & 0x01010101u);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int nbits = W * H * 3;
    const int64_t wpe = obs_bits_words(W, H);
    const int esz = obs_elem_bytes(dtype);
    const bool vec = ((int64_t)nbits * esz) % 16 == 0;  // every row starts 16-byte aligned (out is)
    const int nfull = vec ? nbits / 16 : 0;             // whole 16-element chunks
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t i = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); i < n_out; i += warps) {
        const int64_t r = index ? index[i] : i;
        const bool ok = r >= 0 && r < n_rows;
        const uint16_t* src = reinterpret_cast<const uint16_t*>(bits + (ok ? r : 0) * wpe);
        auto chunk = [&](int c) -> uint32_t { return ok ? (uint32_t)__ldg(src + c) : 0u; };
        auto bit = [&](int k) -> uint32_t { return ok ? (__ldg(bits + r * wpe + (k >> 5)) >> (k & 31)) & 1u : 0u; };
        if (dtype == WF_OBS_U8) {
            uint8_t* o = static_cast<uint8_t*>(out) + i * nbits;
            for (int c = lane; c < nfull; c += 32) {
                const uint32_t b = chunk(c);
                const uint2 lo = tab8[b & 255u], hi = tab8[b >> 8];
                reinterpret_cast<uint4*>(o)[c] = make_uint4(lo.x, lo.y, hi.x, hi.y);
            }
            for (int k = 16 * nfull + lane; k < nbits; k += 32) o[k] = (uint8_t)bit(k);
        } else if (dtype == WF_OBS_BF16) {  // 8 elements (one byte of bits) per 16-byte store
            uint16_t* o = static_cast<uint16_t*>(out) + i * nbits;
            const uint8_t* s8 = reinterpret_cast<const uint8_t*>(src);
            for (int c = lane; c < 2 * nfull; c += 32) {
                const uint2 t = tab8[ok ? __ldg(s8 + c) : 0];
                reinterpret_cast<uint4*>(o)[c] = make_uint4(unpack_bf16_pair(t.x, 0x4140u), unpack_bf16_pair(t.x, 0x4342u),
                                                            unpack_bf16_pair(t.y, 0x4140u), unpack_bf16_pair(t.y, 0x4342u));
            }
            for (int k = 16 * nfull + lane; k < nbits; k += 32) o[k] = bit(k) ? kBf16One : (uint16_t)0;
        } else {  // 4 elements (one nibble) per 16-byte store
            float* o = static_cast<float*>(out) + i * nbits;
            const uint8_t* s8 = reinterpret_cast<const uint8_t*>(src);
            constexpr uint32_t ONE = 0x3F800000u;
            for (int c = lane; c < 4 * nfull; c += 32) {
                const uint32_t nib = ok ? ((uint32_t)__ldg(s8 + (c >> 1)) >> ((c & 1) * 4)) : 0u;
                reinterpret_cast<uint4*>(o)[c] =
                    make_uint4((nib & 1u) ? ONE : 0u, (nib & 2u) ? ONE : 0u, (nib & 4u) ? ONE : 0u, (nib & 8u) ? ONE : 0u);
            }
            for (int k = 16 * nfull + lane; k < nbits; k += 32) o[k] = bit(k) ? 1.0f : 0.0f;
        }
    }
}

__global__ void philox_kat_kernel(const uint32_t* in, uint32_t* out) {
    philox4x32_10(in[0], in[1], in[2], in[3], in[4], in[5], out);
}

// ---------------------------------------------------------------------------------------------
static void build_wind_table(const wf_config& c, WindTable& t, int32_t& n) {
    // World.apply_heat_from_to / get_distance_and_angle, environment.py:260-290, evaluated once per
    // (wind, direction) with the same libm calls CPython makes (math.atan2, float ** -1 -> pow).
    static const int DX[4] = {0, 0, 1, -1}, DY[4] = {-1, 1, 0, 0};
    std::memset(&t, 0, sizeof(t));
    auto fill = [&](int id, double speed, int wx, int wy) {
        t.speed[id] = speed; t.wx[id] = wx; t.wy[id] = wy;
        for (int d = 0; d < 4; ++d) {
            const int cx = DX[d], cy = DY[d];
            const double angle = std::fabs(std::atan2((double)(wx * cy - wy * cx), (double)(wx * cx + wy * cy)));
            const double env_factor = std::pow(angle + 1.0, -1.0);
            t.coef[id][d] = speed * c.heat * env_factor;
        }
        const double c0 = t.coef[id][0];
        t.uniform[id] = (t.coef[id][1] == c0 && t.coef[id][2] == c0 && t.coef[id][3] == c0) ? 1 : 0;
        t.kmin[id] = 0x7fffffff;
        if (t.uniform[id] && c0 > 0.0) {  // the reference adds the quantum once per hit, in float64
            double temp = 0.0;
            for (int k = 1; k <= 1024; ++k) {
                temp += c0;
                if (temp > c.threshold) { t.kmin[id] = k; break; }
            }
        }
    };
    if (c.wind_random) {
        static const double speeds[3] = {0.0, 0.7, 0.85};  // environment.py:189
        n = 27;
        for (int si = 0; si < 3; ++si)
            for (int wx = -1; wx <= 1; ++wx)
                for (int wy = -1; wy <= 1; ++wy) fill(si * 9 + (wx + 1) * 3 + (wy + 1), speeds[si], wx, wy);
    } else {
        n = 1;
        fill(0, c.wind_speed, c.wind_x, c.wind_y);
    }
}

extern "C" {

void wf_default_config(wf_config* c, int32_t size) {  // constants.py:30-47, utility.py:94-102
    std::memset(c, 0, sizeof(*c));
    c->width = c->height = size;
    c->n_actions = 4;
    c->a_speed = 1;
    c->wind_speed = 0.54;
    c->death_penalty = -1000.0;
    c->contained_bonus = 1000.0;
    c->default_reward = -1.0;
    c->heat = 0.3;
    c->threshold = 3.0;
    c->fuel = 20;
    c->radius = 1;
}

const char* wf_last_error(void) { return g_err.c_str(); }
int wf_abi_version(void) { return WF_ABI_VERSION; }

int wf_create(const wf_config* cfg, int32_t n_envs, int32_t device, wf_env** out) {
    if (!cfg || !out) return fail(WF_ERR_INVALID, "null argument");
    *out = nullptr;
    const wf_config& c = *cfg;
    if (n_envs < 1) return fail(WF_ERR_INVALID, "n_envs must be >= 1");
    if (c.width < 10 || c.height < 10)
        return fail(WF_ERR_INVALID, "width and height must be >= 10 (get_agent_location asserts it, utility.py:68)");
    if (c.width < c.height)
        return fail(WF_ERR_INVALID, "width < height: the reference's border_points use [HEIGHT-1, y] "
                                    "(environment.py:222) and raise on such maps");
    if (c.radius != 1) return fail(WF_ERR_INVALID, "only grass radius 1 (4-neighbour stencil) is implemented");
    if (c.fuel < 1 || c.fuel > 255) return fail(WF_ERR_INVALID, "fuel must be in 1..255");
    if (c.a_speed < 1) return fail(WF_ERR_INVALID, "a_speed must be >= 1");
    if (c.n_actions < 1) return fail(WF_ERR_INVALID, "n_actions must be >= 1");
    if (c.extra_ignitions < 0) return fail(WF_ERR_INVALID, "extra_ignitions must be >= 0");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(WF_ERR_CUDA, "no CUDA device: libwildfire_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(WF_ERR_INVALID, "bad device index");
    DeviceGuard _guard(device);
    WF_CUDA(_guard.err);

    wf_env* e = new (std::nothrow) wf_env();
    if (!e) return fail(WF_ERR_INVALID, "out of host memory");
    std::memset(static_cast<void*>(e), 0, sizeof(*e));
    e->cfg = c;
    e->N = n_envs;
    e->device = device;
    e->tile = (c.width > 32 || c.height > 32);
    e->a_iter = c.a_speed;
    DevState& s = e->st;
    s.N = n_envs; s.W = c.width; s.H = c.height;
    s.HW = (c.height + 31) / 32;
    s.RS = e->tile ? c.width : (c.width <= 16 ? 16 : 32);
    s.FB = c.fuel <= 31 ? 5 : 8;
    s.HB = 0;
    StepCfg& sc = e->sc;
    sc.n_actions = c.n_actions; sc.a_speed = c.a_speed; sc.allow_dig_toggle = c.allow_dig_toggle;
    sc.make_rivers = c.make_rivers; sc.wind_random = c.wind_random; sc.fuel = c.fuel;
    sc.extra_ignitions = c.extra_ignitions; sc.auto_reset = c.auto_reset;
    sc.death_penalty = c.death_penalty; sc.contained_bonus = c.contained_bonus;
    sc.default_reward = c.default_reward; sc.threshold = c.threshold;
    sc.key0 = (uint32_t)(c.seed & 0xffffffffu); sc.key1 = (uint32_t)(c.seed >> 32);
    sc.env_id_base = c.env_id_base;
    build_wind_table(c, e->wind_host, e->n_wind);
    {   // Direction-independent heat quanta for every wind this handle can meet (e.g. the Logs/ constants:
        // wind [0.54, (0, 0)]): only the TOTAL hit count of a cell matters, and the warp family keeps it
        // bit-sliced in registers (7 planes cover 4 neighbours x (fuel - 1) <= 120 hits).
        bool all_uniform = true;
        for (int i = 0; i < e->n_wind; ++i) all_uniform = all_uniform && e->wind_host.uniform[i];
        if (!e->tile && all_uniform && s.FB == 5 && !getenv("WF_WARP_NO_BITSLICED_HITS")) s.HB = 7;
    }
    s.NP = e->tile ? 7 + tile_extra_planes() : 7 + s.FB + s.HB;  // tile family: fuel lives in its own records (s.fuel)

    const size_t plane_words = (size_t)s.NP * s.N * s.RS * s.HW;
    const size_t cells = (size_t)s.N * s.W * s.H;
    auto cleanup = [&](int code, const std::string& m) { wf_destroy(e); return fail(code, m); };
#define WF_CUDA_C(expr)                                                                   \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) return cleanup(WF_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)
    WF_CUDA_C(cudaMalloc(&s.planes, plane_words * sizeof(uint32_t)));
    WF_CUDA_C(cudaMemset(s.planes, 0, plane_words * sizeof(uint32_t)));
    if (e->tile) {
        const size_t fuel_words = (size_t)s.N * s.RS * s.HW * kFuelRec;
        WF_CUDA_C(cudaMalloc(&s.fuel, fuel_words * sizeof(uint32_t)));
        WF_CUDA_C(cudaMemset(s.fuel, 0, fuel_words * sizeof(uint32_t)));
    }
    WF_CUDA_C(cudaMalloc(&s.hits, cells * sizeof(uint32_t)));
    WF_CUDA_C(cudaMemset(s.hits, 0, cells * sizeof(uint32_t)));
    WF_CUDA_C(cudaMalloc(&s.scal, (size_t)s.N * WF_NSCALARS * sizeof(int32_t)));
    WF_CUDA_C(cudaMemset(s.scal, 0, (size_t)s.N * WF_NSCALARS * sizeof(int32_t)));
    WF_CUDA_C(cudaMalloc(&s.stats, ST_N * sizeof(unsigned long long)));
    WF_CUDA_C(cudaMemset(s.stats, 0, ST_N * sizeof(unsigned long long)));
    WF_CUDA_C(cudaMalloc(&e->wind_dev, sizeof(WindTable)));
    WF_CUDA_C(cudaMemcpy(e->wind_dev, &e->wind_host, sizeof(WindTable), cudaMemcpyHostToDevice));
    s.wind = e->wind_dev;
    if (e->tile) WF_CUDA_C(tile_create(&e->tstate, s, sc));
    // episode counter starts at -1 so that the first reset() opens episode 0 (like the oracle)
    {
        std::string init((size_t)s.N * WF_NSCALARS * sizeof(int32_t), '\0');
        int32_t* p = reinterpret_cast<int32_t*>(&init[0]);
        for (int i = 0; i < s.N; ++i) p[(size_t)i * WF_NSCALARS + WF_S_EPISODE] = -1;
        WF_CUDA_C(cudaMemcpy(s.scal, p, init.size(), cudaMemcpyHostToDevice));
    }
#undef WF_CUDA_C
    *out = e;
    return WF_OK;
}

void wf_destroy(wf_env* e) {
    if (!e) return;
    DeviceGuard _guard(e->device);
    session_park(e);
    if (e->sess.ctl) cudaFreeHost(e->sess.ctl);
    if (e->sess.actions) cudaFreeHost(e->sess.actions);
    if (e->sess.rec) cudaFreeHost(e->sess.rec);
    if (e->sess.full) cudaFreeHost(e->sess.full);
    cudaFree(e->sess.sync_dev);
    cudaFree(e->sess.actions_hbm);
    if (e->sess.steps && getenv("WF_HOST_TIMING")) {
        unsigned long long d[8] = {0};
        if (e->sess.dbg_dev) cudaMemcpy(d, e->sess.dbg_dev, sizeof(d), cudaMemcpyDeviceToHost);
        const double n = d[3] ? (double)d[3] : 1.0;
        fprintf(stderr, "wf_host_session: %lld steps in %lld launches of the step server (%lld park/ring races); host ring->expanded "
                        "%.2f us (first flag after %.2f us); CTA 0 per step: wait for the tagged actions (idle time included) %.2f us, fence + release "
                        "%.2f us, step %.2f us, CTA barrier %.2f us, block store + arrive %.2f us; system fence + flag of a slice's last CTA "
                        "%.2f us; steps that asked for every record in full (mode 2): %lld\n",
                (long long)e->sess.steps, (long long)e->sess.launches, (long long)e->sess.relaunch_races,
                1e6 * e->sess.t_wait / (double)e->sess.steps, 1e6 * hostpool_first_flag_seconds(e->pool) / (double)e->sess.steps,
                d[0] / n / 1e3, d[7] / n / 1e3, d[1] / n / 1e3, d[2] / n / 1e3, d[4] / n / 1e3, d[6] ? d[5] / (double)d[6] / 1e3 : 0.0,
                (long long)e->sess.full_frames);
    }
    cudaFree(e->sess.dbg_dev);
    if (e->tstate) tile_destroy(e->tstate);
    cudaFree(e->st.planes); cudaFree(e->st.fuel); cudaFree(e->st.hits); cudaFree(e->st.scal); cudaFree(e->st.stats);
    cudaFree(e->wind_dev);
    cudaFree(e->mlp_dev);
    cudaFree(e->h_actions); cudaFree(e->h_obs); cudaFree(e->h_reward); cudaFree(e->h_done);
    cudaFree(e->h_mask); cudaFree(e->h_init);
    if (e->t_calls && getenv("WF_HOST_TIMING"))
        fprintf(stderr, "wf_step_host (packed path), %lld calls: launch %.2f us, sync %.2f us, expand %.2f us per call\n",
                (long long)e->t_calls, 1e6 * e->t_launch / e->t_calls, 1e6 * e->t_sync / e->t_calls, 1e6 * e->t_expand / e->t_calls);
    if (e->hg_exec) cudaGraphExecDestroy(e->hg_exec);
    if (e->h_packed) cudaFreeHost(e->h_packed);
    cudaFree(e->d_packed);
    if (e->pool) hostpool_destroy(e->pool);
    if (e->hstream) cudaStreamDestroy(e->hstream);
    if (e->dev_event) cudaEventDestroy(e->dev_event);
    delete e;
}

const char* wf_kernel_family(const wf_env* e) { return e ? (e->tile ? "tile" : "warp") : ""; }
int64_t wf_launch_count(const wf_env* e) { return e ? e->launches : 0; }
int wf_tile_geometry(const wf_env* e, int32_t* threads, int32_t* cluster) {
    if (!e || !threads || !cluster) return fail(WF_ERR_INVALID, "null argument");
    *threads = *cluster = 0;
    if (e->tstate) tile_geometry(e->tstate, threads, cluster);
    return WF_OK;
}
int wf_host_threads(const wf_env* e) { return (e && e->pool) ? hostpool_threads(e->pool) : 0; }

int wf_expand_packed_obs(const uint32_t* packed_host, uint8_t* obs_host, int32_t n_envs, int32_t width, int32_t height,
                         int32_t threads) {
    if (!packed_host || !obs_host || n_envs < 1 || width < 1 || height < 1 || width > 32 || height > 32 || threads < 1)
        return fail(WF_ERR_INVALID, "wf_expand_packed_obs: bad argument");
    const int epw = width <= 16 ? 2 : 1;
    const int64_t env_bits = (int64_t)width * height * 3, records = (n_envs + epw - 1) / epw, rec_words = (epw * env_bits + 31) / 32;
    HostPool* p = hostpool_create(threads);
    hostpool_expand(p, packed_host, obs_host, records, rec_words, env_bits, epw, n_envs);
    hostpool_destroy(p);
    return WF_OK;
}
int wf_apply_change_blocks(const uint32_t* blocks_host, const uint32_t* full_area_host, int32_t full_stride, uint8_t* obs_host,
                           double* reward_host, uint8_t* done_host, int32_t n_envs, int32_t width, int32_t height,
                           double default_reward, double death_penalty, double contained_bonus, int32_t threads) {
    if (!blocks_host || !full_area_host || !obs_host || n_envs < 1 || width < 1 || height < 1 || width > 32 || height > 32 ||
        threads < 1 || full_stride < 1)
        return fail(WF_ERR_INVALID, "wf_apply_change_blocks: bad argument");
    const int epw = width <= 16 ? 2 : 1;
    const int64_t env_bits = (int64_t)width * height * 3, records = (n_envs + epw - 1) / epw, rec_words = (epw * env_bits + 31) / 32;
    if (full_stride < rec_words) return fail(WF_ERR_INVALID, "wf_apply_change_blocks: full_stride is smaller than a record");
    alignas(64) static const volatile uint32_t flag[16] = {1u};  // "the step is complete"
    HostPool* p = hostpool_create(threads);
    const bool ok = hostpool_expand_session(p, blocks_host, obs_host, records, rec_words, env_bits, epw, n_envs, flag, 1u, records,
                                            reward_host, done_host, default_reward, death_penalty, contained_bonus,
                                            (double)(width * height), 1000000000, 0, full_area_host, full_stride, false);
    hostpool_destroy(p);
    return ok ? WF_OK : fail(WF_ERR_STATE, "wf_apply_change_blocks: timed out");
}
int64_t wf_state_bytes_per_env(const wf_env* e) {
    if (!e) return 0;
    const DevState& s = e->st;
    return (int64_t)(s.NP + (s.fuel ? kFuelRec : 0)) * s.RS * s.HW * 4 + (s.HB ? 0 : (int64_t)s.W * s.H * 4) + WF_NSCALARS * 4;
}

// Ask a running step server to park (it stores the envs back to HBM and exits) and wait for it.
static int session_park(wf_env* e) {
    if (!e->sess.running) return WF_OK;
    *reinterpret_cast<volatile uint32_t*>(e->sess.ctl) = 0xffffffffu;  // doorbell: park
    cudaError_t err = cudaStreamSynchronize(e->hstream);
    e->sess.running = false;
    if (err != cudaSuccess) return fail(WF_ERR_CUDA, std::string("step-server kernel: ") + cudaGetErrorString(err));
    return WF_OK;
}
#define WF_QUIESCE(e)                            \
    do {                                         \
        if (int _rc = session_park(e)) return _rc; \
    } while (0)

// A *_dev entry point queued work on `st`: the next wf_step_host must wait for it (see wf_env::dev_stream).
static void note_dev_call(wf_env* e, cudaStream_t st) {
    if (st == e->hstream && e->hstream) return;  // wf_step_host's own launches
    e->dev_stream = st;
    e->dev_pending = true;
}

static bool public_obs_dtype(int32_t dtype) {
    return dtype == WF_OBS_U8 || dtype == WF_OBS_F32 || dtype == WF_OBS_BF16 || dtype == WF_OBS_BITS;
}
static int check_obs(const void* obs, int32_t dtype) {
    if (!public_obs_dtype(dtype) && dtype != kObsPacked)
        return fail(WF_ERR_INVALID, "obs_dtype must be WF_OBS_U8, WF_OBS_F32, WF_OBS_BF16 or WF_OBS_BITS");
    if (obs && (reinterpret_cast<uintptr_t>(obs) & 15u)) return fail(WF_ERR_INVALID, "obs pointer must be 16-byte aligned");
    return WF_OK;
}

static uint32_t magic_for(int H) { return (uint32_t)((0x100000000ull + (uint64_t)H - 1) / (uint64_t)H); }

int wf_reset(wf_env* e, const uint8_t* mask_dev, const wf_init* init_dev, void* obs_dev, int32_t obs_dtype,
             void* stream) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    if (int rc = check_obs(obs_dev, obs_dtype)) return rc;
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    note_dev_call(e, st);
    if (e->tile) {
        TileIO io{nullptr, obs_dev, nullptr, nullptr, mask_dev, init_dev, obs_dtype, 0, e->a_iter, 1, 0, nullptr};
        WF_CUDA(launch_tile_family(e->tstate, e->st, e->sc, io, st, &e->launches));
    } else {
        WarpIO io{nullptr, obs_dev, nullptr, nullptr, mask_dev, init_dev, obs_dtype, 1, e->a_iter, 1, magic_for(e->st.H), 0, nullptr,
                  MlpPolicy{}};
        WF_CUDA(launch_warp_family(e->st, e->sc, io, st));
        e->launches += 1;
    }
    return WF_OK;
}

static int advance_a_iter(wf_env* e, int k_steps) {
    int it = e->a_iter;
    for (int k = 0; k < k_steps; ++k) {
        it -= 1;
        if (it == 0) it = e->cfg.a_speed;
    }
    return it;
}

static int rollout_impl(wf_env* e, int32_t k_steps, const int32_t* actions_dev, int32_t policy, int32_t* actions_out,
                        void* obs_dev, int32_t obs_dtype, double* reward_dev, uint8_t* done_dev, void* stream) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    if (k_steps < 1) return fail(WF_ERR_INVALID, "k_steps must be >= 1");
    if (policy != WF_POLICY_STREAM && policy != WF_POLICY_WALK && policy != WF_POLICY_MLP)
        return fail(WF_ERR_INVALID, "unknown policy");
    if (policy == WF_POLICY_MLP && !actions_dev && e->mlp.hid == 0)
        return fail(WF_ERR_STATE, "WF_POLICY_MLP: call wf_set_policy_mlp first");
    if (int rc = check_obs(obs_dev, obs_dtype)) return rc;
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    note_dev_call(e, st);
    if (e->tile) {  // one thread-block cluster per env runs all K steps in one launch
        TileIO io{actions_dev, obs_dev, reward_dev, done_dev, nullptr, nullptr, obs_dtype, k_steps, e->a_iter, 0, policy,
                  actions_out, e->mlp};
        WF_CUDA(launch_tile_family(e->tstate, e->st, e->sc, io, st, &e->launches, &e->fin));
        e->a_iter = advance_a_iter(e, k_steps);
        return WF_OK;
    }
    WarpIO io{actions_dev, obs_dev, reward_dev, done_dev, nullptr, nullptr, obs_dtype, k_steps, e->a_iter, 0,
              magic_for(e->st.H), policy, actions_out, e->mlp};
    WF_CUDA(launch_warp_family(e->st, e->sc, io, st, &e->fin));
    e->launches += 1;
    e->a_iter = advance_a_iter(e, k_steps);
    return WF_OK;
}

int wf_rollout(wf_env* e, int32_t k_steps, const int32_t* actions_dev, void* obs_dev, int32_t obs_dtype,
               double* reward_dev, uint8_t* done_dev, void* stream) {
    return rollout_impl(e, k_steps, actions_dev, WF_POLICY_STREAM, nullptr, obs_dev, obs_dtype, reward_dev, done_dev, stream);
}

int wf_rollout_policy(wf_env* e, int32_t k_steps, int32_t policy, int32_t* actions_out_dev, void* obs_dev,
                      int32_t obs_dtype, double* reward_dev, uint8_t* done_dev, void* stream) {
    return rollout_impl(e, k_steps, nullptr, policy, actions_out_dev, obs_dev, obs_dtype, reward_dev, done_dev, stream);
}

// Explore threshold of eps: a 32-bit draw below it explores.
static uint32_t mlp_eps_threshold(double eps) { return eps >= 1.0 ? 0xffffffffu : (uint32_t)(eps * 4294967296.0); }

// Lanes of MlpPolicy::w1's layout: the warp family's lanes per env; the tile family's policy pass adds rows with 32 lanes.
static int mlp_lanes(const wf_env* e) { return e->tile ? 32 : e->st.RS; }

// The handle's packed buffer holds at least n_nets network blocks; network 0's pointers, one group covering every env.
static int mlp_reserve(wf_env* e, int n_nets, int hidden) {
    const int n_in = e->st.W * e->st.H * 3;
    const size_t per = mlp_net_floats(n_in);
    if (!e->mlp_dev || e->mlp_cap < n_nets) {
        cudaFree(e->mlp_dev);
        e->mlp_dev = nullptr;
        e->mlp_cap = 0;
        e->mlp = MlpPolicy{};
        WF_CUDA(cudaMalloc(&e->mlp_dev, per * n_nets * sizeof(float)));
        e->mlp_cap = n_nets;
    }
    e->mlp.w1 = e->mlp_dev;
    e->mlp.base = e->mlp_dev + (size_t)n_in * 64;
    e->mlp.w2 = e->mlp.base + 64;
    e->mlp.b2 = e->mlp.w2 + 512;
    e->mlp.hid = hidden;
    e->mlp.n_actions = e->cfg.n_actions;
    e->mlp.group_envs = 1 << 30;  // one network for every env (a multiple of any CTA's envs)
    e->mlp.net_stride = (int32_t)per;
    return WF_OK;
}

int wf_set_policy_mlp(wf_env* e, const float* k1, const float* b1, const float* k2, const float* b2, int32_t hidden,
                      double eps) {
    if (!e || !k1 || !b1 || !k2 || !b2) return fail(WF_ERR_INVALID, "null argument");
    if (hidden < 1 || hidden > 64) return fail(WF_ERR_INVALID, "hidden must be in 1..64");
    if (e->cfg.n_actions > 8) return fail(WF_ERR_INVALID, "WF_POLICY_MLP supports at most 8 actions");
    if (!(eps >= 0.0 && eps <= 1.0)) return fail(WF_ERR_INVALID, "eps must be in [0, 1]");
    if (e->tile) {  // the tile kernel's exact fixed-point first layer (include/wildfire.h)
        const double bound = 2147483648.0 / (2.0 * e->st.W * e->st.H + 1.0);
        for (size_t i = 0, n = (size_t)e->st.W * e->st.H * 3 * hidden; i < n; ++i)
            if (!(std::fabs((double)k1[i]) < bound))
                return fail(WF_ERR_INVALID, "wf_set_policy_mlp: on this grid every kernel1 entry must be finite and below "
                                            "2^31 / (2*W*H + 1) in magnitude");
    }
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    const DevState& s = e->st;
    const int n_in = s.W * s.H * 3, A = e->cfg.n_actions;
    // device layout (MlpPolicy): w1 [n_in][64] permuted for the lanes | base [64] | w2 [2][64][4] | b2 [8] | threshold [8]
    const int L = mlp_lanes(e), hpl = 64 / L;
    const size_t n_w1 = (size_t)n_in * 64, total = mlp_net_floats(n_in);
    std::vector<float> hbuf(total, 0.0f);
    float* h = hbuf.data();
    for (int f = 0; f < n_in; ++f)
        for (int j = 0; j < hidden; ++j) h[(size_t)f * 64 + (j % L) * hpl + j / L] = k1[(size_t)f * hidden + j];
    float* base = h + n_w1;
    for (int j = 0; j < hidden; ++j) {  // the empty map: every cell free (channel 2), no fire, no agent
        double acc = b1[j];
        for (int cell = 0; cell < s.W * s.H; ++cell) acc += k1[(size_t)(cell * 3 + 2) * hidden + j];
        base[j] = (float)acc;
    }
    float* w2 = base + 64;
    for (int j = 0; j < hidden; ++j)
        for (int b = 0; b < A; ++b) w2[(size_t)(b / 4) * 256 + j * 4 + (b & 3)] = k2[(size_t)j * A + b];
    float* bias2 = w2 + 512;
    for (int b = 0; b < 8; ++b) bias2[b] = b < A ? b2[b] : -INFINITY;
    const uint32_t thr = mlp_eps_threshold(eps);
    std::memcpy(bias2 + 8, &thr, sizeof(thr));
    cudaFree(e->mlp_dev);
    e->mlp_dev = nullptr;
    if (int rc = mlp_reserve(e, 1, hidden)) return rc;
    WF_CUDA(cudaMemcpy(e->mlp_dev, h, total * sizeof(float), cudaMemcpyHostToDevice));
    return WF_OK;
}

// Queues the repack of n_nets networks (network k's weights at k * in_stride floats after w1 / b1 / w2 / b2) into the
// handle's packed buffer on `stream`.
static int pack_policy_nets(wf_env* e, int n_nets, const float* w1, const float* b1, const float* w2, const float* b2,
                            size_t in_stride, int hidden, const double* eps, void* stream) {
    MlpThresholds thr{};
    for (int k = 0; k < n_nets; ++k) thr.v[k] = mlp_eps_threshold(eps[k]);
    if (int rc = mlp_reserve(e, n_nets, hidden)) return rc;
    const DevState& s = e->st;
    const int n_in = s.W * s.H * 3;
    const size_t total = mlp_net_floats(n_in);
    const dim3 grid((unsigned)std::min<size_t>((total + 255) / 256, 148 * 16), (unsigned)n_nets);
    pack_policy_mlp_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(e->mlp_dev, w1, b1, w2, b2, in_stride, n_in,
                                                                                  s.W * s.H, hidden, e->cfg.n_actions, mlp_lanes(e), thr);
    WF_CUDA(cudaGetLastError());
    return WF_OK;
}

int wf_set_policy_mlp_dev(wf_env* e, const float* w1, const float* b1, const float* w2, const float* b2, int32_t hidden,
                          double eps, void* stream) {
    if (!e || !w1 || !b1 || !w2 || !b2) return fail(WF_ERR_INVALID, "null argument");
    if (hidden < 1 || hidden > 64) return fail(WF_ERR_INVALID, "hidden must be in 1..64");
    if (e->cfg.n_actions > 8) return fail(WF_ERR_INVALID, "WF_POLICY_MLP supports at most 8 actions");
    if (!(eps >= 0.0 && eps <= 1.0)) return fail(WF_ERR_INVALID, "eps must be in [0, 1]");
    for (const float* p : {w1, b1, w2, b2})
        if (reinterpret_cast<uintptr_t>(p) & 3u) return fail(WF_ERR_INVALID, "weights must be 4-byte aligned");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    return pack_policy_nets(e, 1, w1, b1, w2, b2, 0, hidden, &eps, stream);
}

int wf_set_policy_mlp_nets_dev(wf_env* e, const wf_mlp_shape* shape, int32_t n_nets, const float* params_dev,
                               const double* eps_host, void* stream) {
    if (!e || !shape || !params_dev || !eps_host) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: null argument");
    if (n_nets < 1 || n_nets > kMlpMaxNets) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: n_nets must be in 1..64");
    const wf_mlp_shape& sh = *shape;
    if (sh.hidden < 1 || sh.hidden > 64) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: hidden must be in 1..64");
    if (sh.n_actions < 1 || sh.n_actions > 8) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: n_actions must be in 1..8");
    if (sh.dueling != 0 && sh.dueling != 1) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: dueling must be 0 or 1");
    if (sh.height < 10 || sh.width < sh.height || sh.width > 32)
        return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: the grid must satisfy 10 <= height <= width <= 32");
    for (int k = 0; k < n_nets; ++k)
        if (!(eps_host[k] >= 0.0 && eps_host[k] <= 1.0)) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: eps must be in [0, 1]");
    if (reinterpret_cast<uintptr_t>(params_dev) & 3u) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: params must be 4-byte aligned");
    if (e->tile) return fail(WF_ERR_INVALID, "WF_POLICY_MLP is implemented for grids up to 32x32 (warp family) only");
    if (sh.width != e->cfg.width || sh.height != e->cfg.height || sh.n_actions != e->cfg.n_actions)
        return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: the shape's grid and n_actions must be the handle's");
    if (e->N % n_nets != 0) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: n_envs must be a multiple of n_nets");
    const int group = e->N / n_nets;
    if (group % 8 != 0) return fail(WF_ERR_INVALID, "wf_set_policy_mlp_nets_dev: n_envs / n_nets must be a multiple of 8");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    // the flat layout of wf_replay_fit: dense_1.weight | dense_1.bias | dense_2.weight | dense_2.bias | (dueling) ...
    const int n_in = sh.width * sh.height * 3, hid = sh.hidden, A = sh.n_actions;
    const size_t P = (size_t)hid * (n_in + 1 + A) + A + (sh.dueling ? (size_t)hid * (n_in + 2) + 1 : 0);
    const float* w1 = params_dev;
    const float* b1 = w1 + (size_t)hid * n_in;
    const float* w2 = b1 + hid;
    const float* b2 = w2 + (size_t)A * hid;
    if (int rc = pack_policy_nets(e, n_nets, w1, b1, w2, b2, P, hid, eps_host, stream)) return rc;
    e->mlp.group_envs = group;
    return WF_OK;
}

int64_t wf_final_record_words(int32_t width, int32_t height) {
    if (width < 1 || height < 1) return 0;
    return final_record_words(width, height);
}

int wf_set_final_capture(wf_env* e, uint32_t* records_dev, int64_t capacity, uint32_t* count_dev) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    if (!records_dev) {
        e->fin = FinalCapture{};
        return WF_OK;
    }
    if (!count_dev) return fail(WF_ERR_INVALID, "wf_set_final_capture: count_dev is null");
    if (capacity < 0) return fail(WF_ERR_INVALID, "wf_set_final_capture: capacity must be >= 0");
    if (reinterpret_cast<uintptr_t>(records_dev) & 15u) return fail(WF_ERR_INVALID, "wf_set_final_capture: records must be 16-byte aligned");
    if (reinterpret_cast<uintptr_t>(count_dev) & 3u) return fail(WF_ERR_INVALID, "wf_set_final_capture: count must be 4-byte aligned");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);  // a resident step server is parked first: it has no capture
    e->fin.records = records_dev;
    e->fin.count = count_dev;
    e->fin.capacity = capacity;
    e->fin.words = final_record_words(e->cfg.width, e->cfg.height);
    e->fin.plane_off = final_plane_offset(e->cfg.width, e->cfg.height);
    return WF_OK;
}

int wf_step(wf_env* e, const int32_t* actions_dev, void* obs_dev, int32_t obs_dtype, double* reward_dev,
            uint8_t* done_dev, void* stream) {
    if (!actions_dev) return fail(WF_ERR_INVALID, "wf_step: actions_dev is null");
    return wf_rollout(e, 1, actions_dev, obs_dev, obs_dtype, reward_dev, done_dev, stream);
}

// Device-visible alias of a page-locked, mapped host buffer (nullptr if the memory is pageable).
static void* mapped_alias(const void* host_ptr) {
    if (!host_ptr) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host_ptr) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

// Common start of the host-buffer entry points: the handle's private stream (first call: also the WF_HOST_* switches)
// and its ordering behind the caller's earlier *_dev work.
static int host_prologue(wf_env* e) {
    if (!e->hstream) {
        WF_CUDA(cudaStreamCreateWithFlags(&e->hstream, cudaStreamNonBlocking));
        // WF_HOST_MODE: "hybrid" (default) = actions/reward/done zero-copy, obs staged + one DMA copy;
        //               "direct" = everything zero-copy; "copy" = everything staged.
        const char* m = getenv("WF_HOST_MODE");
        const std::string mode = m ? m : "hybrid";
        e->host_direct = mode != "copy";
        e->host_obs_direct = mode == "direct";
        // WF_HOST_PACKED=0 switches the packed-observation path off (uint8 array over PCIe, no host threads)
        const char* pk = getenv("WF_HOST_PACKED");
        e->host_packed = !(pk && pk[0] == '0');
        e->packed_dma = !(pk && std::string(pk) == "direct");  // default: stage in HBM, one DMA copy ("direct": zero-copy stores)
        const char* hg = getenv("WF_HOST_GRAPH");
        e->host_graph = hg && hg[0] == '1' && e->cfg.a_speed == 1;
    }
    if (e->dev_pending) {  // order this call behind the caller's earlier *_dev work on its own stream
        if (!e->dev_event) WF_CUDA(cudaEventCreateWithFlags(&e->dev_event, cudaEventDisableTiming));
        WF_CUDA(cudaEventRecord(e->dev_event, e->dev_stream));
        WF_CUDA(cudaStreamWaitEvent(e->hstream, e->dev_event, 0));
        e->dev_pending = false;
    }
    return WF_OK;
}

static int ensure_obs_staging(wf_env* e, size_t obs_bytes) {
    if (e->h_obs_bytes < obs_bytes) {
        cudaFree(e->h_obs);
        e->h_obs = nullptr;
        e->h_obs_bytes = 0;
        WF_CUDA(cudaMalloc(&e->h_obs, obs_bytes));
        e->h_obs_bytes = obs_bytes;
    }
    return WF_OK;
}

// ForestFire.reset() for a caller that only has host memory (INTEGRATION.md section 3).
int wf_reset_host(wf_env* e, const uint8_t* mask_host, const wf_init* init_host, void* obs_host, int32_t obs_dtype) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    if (!public_obs_dtype(obs_dtype)) return fail(WF_ERR_INVALID, "bad obs_dtype");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    const DevState& s = e->st;
    const size_t obs_bytes = obs_step_bytes(s.N, s.W, s.H, obs_dtype);
    if (int rc = host_prologue(e)) return rc;
    if ((mask_host || init_host) && !e->h_mask) {
        WF_CUDA(cudaMalloc(&e->h_mask, (size_t)s.N));
        WF_CUDA(cudaMalloc(&e->h_init, (size_t)s.N * sizeof(wf_init)));
    }
    if (mask_host) WF_CUDA(cudaMemcpyAsync(e->h_mask, mask_host, (size_t)s.N, cudaMemcpyHostToDevice, e->hstream));
    if (init_host) WF_CUDA(cudaMemcpyAsync(e->h_init, init_host, (size_t)s.N * sizeof(wf_init), cudaMemcpyHostToDevice, e->hstream));
    if (obs_host) {
        if (int rc = ensure_obs_staging(e, obs_bytes)) return rc;
    }
    if (int rc = wf_reset(e, mask_host ? e->h_mask : nullptr, init_host ? e->h_init : nullptr, obs_host ? e->h_obs : nullptr,
                          obs_dtype, e->hstream))
        return rc;
    if (obs_host) WF_CUDA(cudaMemcpyAsync(obs_host, e->h_obs, obs_bytes, cudaMemcpyDeviceToHost, e->hstream));
    WF_CUDA(cudaStreamSynchronize(e->hstream));
    return WF_OK;
}

// ---- step-server session ------------------------------------------------------------------------
static int session_launch(wf_env* e) {
    wf_env::Session& ss = e->sess;
    const DevState& s = e->st;
    ss.generation += 1u;
    WF_CUDA(cudaMemsetAsync(ss.sync_dev, 0, (16 + kSessMaxSlices) * sizeof(uint32_t), e->hstream));
    WarpIO io{ss.actions_hbm, ss.rec_dev, nullptr, nullptr, nullptr, nullptr, kObsPackedStatus, 1, e->a_iter, 0,
              magic_for(s.H), WF_POLICY_STREAM, nullptr, MlpPolicy{}};
    SrvCtl srv{};
    srv.doorbell = ss.ctl_dev;
    srv.parked = ss.ctl_dev + 16;
    srv.done = ss.ctl_dev + 32;
    srv.actions_host = ss.actions_dev;
    srv.actions_dev = ss.actions_hbm;
    srv.go = ss.sync_dev;
    srv.count = ss.sync_dev + 16;
    srv.seq0 = ss.seq;
    srv.generation = ss.generation;
    srv.ctas_per_slice = ss.ctas_per_slice;
    srv.sectors = ss.persistent_obs ? 0 : ss.sectors;
    srv.delta = ss.persistent_obs ? 1 : 0;
    srv.full_area = ss.full_dev;
    srv.full_stride = ss.full_stride;
    ss.frame_ptr = nullptr;  // a launch's first step sends every record in full
    const char* idle = getenv("WF_SESSION_IDLE_US");
    srv.dbg = ss.dbg_dev;
    srv.idle_ns = 1000ull * (unsigned long long)((idle && atoll(idle) > 0) ? atoll(idle) : 2000);
    WF_CUDA(launch_warp_server(s, e->sc, io, srv, e->hstream));
    e->launches += 1;
    ss.launches += 1;
    ss.running = true;
    return WF_OK;
}

static int session_step(wf_env* e, const int32_t* actions_host, void* obs_host, int32_t obs_dtype, double* reward_host,
                        uint8_t* done_host) {
    wf_env::Session& ss = e->sess;
    const DevState& s = e->st;
    const int epw = 32 / s.RS;
    const int64_t env_bits = (int64_t)s.W * s.H * 3, records = (s.N + epw - 1) / epw, rec_words = (epw * env_bits + 31) / 32;
    if (ss.seq >= 0xfffffff0u) {  // sequence numbers wrap: park and start over from 0
        WF_QUIESCE(e);
        ss.seq = 0u;
    }
    if (ss.running && reinterpret_cast<volatile uint32_t*>(ss.ctl)[16] == ss.generation) {  // the kernel parked itself (idle)
        WF_CUDA(cudaStreamSynchronize(e->hstream));
        ss.running = false;
    }
    if (!ss.running) {
        if (int rc = host_prologue(e)) return rc;  // behind the caller's earlier *_dev work
        if (!ss.ctl) {
            if (!e->pool) e->pool = hostpool_create(hostpool_default_threads());
            constexpr int kRecordsPerCta = 4;  // WF_WARPS_PER_BLOCK warps, one record each
            const int64_t ctas = (records + kRecordsPerCta - 1) / kRecordsPerCta;
            // Completion flags per step.  Every flag costs its slice's last CTA a system-scope fence (5-7 us: the GPU's
            // writes to host memory are drained), and the fences do not overlap, so splitting the batch to start expanding
            // early does not pay: ONE flag measured best (25.8 us per C2 step against 27.3 with 2 and 28.3 with 12).
            int slices = 1;
            if (const char* v = getenv("WF_SESSION_SLICES"))
                if (atoi(v) >= 1) slices = (int)std::min<int64_t>(std::min(atoi(v), kSessMaxSlices), ctas);
            ss.ctas_per_slice = (int)((ctas + slices - 1) / slices);
            ss.slices = (int)((ctas + ss.ctas_per_slice - 1) / ss.ctas_per_slice);
            WF_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ss.ctl), (32 + 16 * kSessMaxSlices) * sizeof(uint32_t), cudaHostAllocMapped));
            std::memset(ss.ctl, 0, (32 + 16 * kSessMaxSlices) * sizeof(uint32_t));
            WF_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ss.ctl_dev), ss.ctl, 0));
            const size_t act_bytes = (size_t)srv_action_chunks(s.N) * 16;  // packed and tagged (wf_common.cuh)
            WF_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ss.actions), act_bytes, cudaHostAllocMapped));
            std::memset(ss.actions, 0, act_bytes);
            // the kernel's unpacked copy: 24 actions per chunk (+ one word: the full-frame request)
            WF_CUDA(cudaMalloc(reinterpret_cast<void**>(&ss.actions_hbm), ((size_t)srv_action_chunks(s.N) * 24 + 4) * sizeof(int32_t)));
            WF_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ss.actions_dev), ss.actions, 0));
            // WF_SESSION_SECTORS=1: self-validating sectors (wf_common.cuh) instead of the completion flag + system fence.
            // Measured, not faster (C2: 27.4 against 26.4 us per step with 12 host threads, 54.7 against 42.3 with 3: the
            // host pays for validating 12 288 sectors, and the records do not arrive earlier without the fence), so opt-in.
            const char* sv = getenv("WF_SESSION_SECTORS");
            ss.sectors = (sv && sv[0] == '1') ? (int)((rec_words + 1 + 6) / 7) : 0;
            const size_t block_words = ss.sectors ? (size_t)kRecordsPerCta * ss.sectors * 8
                                                  : (size_t)(kRecordsPerCta * (rec_words + 1) + 31) / 32 * 32;  // one CTA's records, whole lines
            WF_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ss.rec), (size_t)ctas * block_words * sizeof(uint32_t), cudaHostAllocMapped));
            WF_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ss.rec_dev), ss.rec, 0));
            ss.full_stride = (int)((rec_words + 3) / 4 * 4);
            WF_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ss.full), (size_t)records * ss.full_stride * sizeof(uint32_t), cudaHostAllocMapped));
            WF_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ss.full_dev), ss.full, 0));
            WF_CUDA(cudaMalloc(reinterpret_cast<void**>(&ss.sync_dev), (16 + kSessMaxSlices) * sizeof(uint32_t)));
            WF_CUDA(cudaMalloc(reinterpret_cast<void**>(&ss.dbg_dev), 8 * sizeof(unsigned long long)));
            WF_CUDA(cudaMemset(ss.dbg_dev, 0, 8 * sizeof(unsigned long long)));
        }
        reinterpret_cast<volatile uint32_t*>(ss.ctl)[0] = ss.seq;  // doorbell: nothing requested yet
        if (int rc = session_launch(e)) {
            ss.wanted = false;  // e.g. the batch is too large for a cooperative launch: the launch-per-step path serves it
            cudaGetLastError();
            return wf_step_host(e, actions_host, obs_host, obs_dtype, reward_host, done_host);
        }
    }
    volatile uint32_t* ctl = ss.ctl;
    uint64_t db_flags = 0;
    if (ss.persistent_obs) {  // another array or dtype than last step's (or none yet): ask for every record in full
        const bool want_full = ss.frame_ptr != obs_host || ss.frame_dtype != obs_dtype;
        db_flags = want_full ? 1u : 0u;
        ss.full_frames += want_full ? 1 : 0;
        ss.frame_ptr = nullptr;  // (until this step has been delivered)
    }
    ss.seq += 1u;
    *reinterpret_cast<volatile uint64_t*>(ss.ctl) = (uint64_t)ss.seq | (db_flags << 32);  // (the doorbell word: 0xffffffff parks)
    {
        // The ring: the actions, six per word, every word tagged with the step's sequence number (wf_common.cuh; CTA 0 of the
        // kernel polls this buffer and validates every word, so it may read while this loop is writing).  The GPU reads these
        // lines all the time: ordinary stores would have to win each line back from the I/O agent first (4 us per step when
        // the buffer was 16 KB); streaming stores go past the caches.
        const uint32_t tag = ((ss.seq & kSrvTagMask) << 24) | (uint32_t)(db_flags << 31);
        const int64_t n_words = (int64_t)srv_action_chunks(s.N) * 4;
        int32_t* dst = ss.actions;
        int64_t i = 0;
        auto nib = [](int32_t a) -> uint32_t { return (uint32_t)a < 15u ? (uint32_t)a : 15u; };
        for (int64_t w = 0; w < n_words; w += 4) {
            uint32_t word[4];
            if (i + 24 <= s.N) {  // a whole chunk: no bounds tests
                const int32_t* a = actions_host + i;
                for (int q = 0; q < 4; ++q, a += 6)
                    word[q] = tag | nib(a[0]) | (nib(a[1]) << 4) | (nib(a[2]) << 8) | (nib(a[3]) << 12) | (nib(a[4]) << 16) | (nib(a[5]) << 20);
                i += 24;
            } else {
                for (int q = 0; q < 4; ++q) {
                    uint32_t v = tag;
                    for (int k = 0; k < 6; ++k, ++i) v |= (i < s.N ? nib(actions_host[i]) : 15u) << (4 * k);
                    word[q] = v;
                }
            }
#if defined(__x86_64__)
            _mm_stream_si128(reinterpret_cast<__m128i*>(dst + w), _mm_set_epi32((int)word[3], (int)word[2], (int)word[1], (int)word[0]));
#else
            for (int q = 0; q < 4; ++q) dst[w + q] = (int32_t)word[q];
#endif
        }
#if defined(__x86_64__)
        _mm_sfence();
#endif
    }
    std::atomic_thread_fence(std::memory_order_release);
    ss.steps += 1;
    const int64_t rps = (int64_t)ss.ctas_per_slice * 4;
    const auto t_start = std::chrono::steady_clock::now();
    for (;;) {
        const bool ok = hostpool_expand_session(e->pool, ss.rec, static_cast<uint8_t*>(obs_host), records, rec_words, env_bits, epw,
                                                s.N, ss.ctl + 32, ss.seq, rps, reward_host, done_host, e->cfg.default_reward,
                                                e->cfg.death_penalty, e->cfg.contained_bonus, (double)(s.W * s.H), 200000,
                                                ss.persistent_obs ? 0 : ss.sectors, ss.persistent_obs ? ss.full : nullptr, ss.full_stride,
                                                obs_dtype == WF_OBS_BITS);
        if (ok) {
            if (ss.persistent_obs) {
                ss.frame_ptr = obs_host;
                ss.frame_dtype = obs_dtype;
            }
            ss.t_wait += std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
            e->a_iter = advance_a_iter(e, 1);  // (after the step: a relaunch below must start from the phase before it)
            return WF_OK;
        }
        if (ctl[16] == ss.generation) {
            // The kernel decided to park in the instant the doorbell was rung: it did not take this step.  Start it
            // again behind the old launch; it finds the doorbell ahead of its seq0 and serves the step at once.
            ss.relaunch_races += 1;
            ss.seq -= 1u;  // seq0 of the new launch = the step before this one
            int rc = session_launch(e);
            ss.seq += 1u;
            if (rc) return rc;
            continue;
        }
        cudaError_t q = cudaStreamQuery(e->hstream);
        if (q != cudaErrorNotReady) {  // the kernel is gone without having parked: a fault
            ss.running = false;
            return fail(WF_ERR_CUDA, std::string("step-server kernel ended unexpectedly: ") + cudaGetErrorString(q));
        }
        if (std::chrono::steady_clock::now() - t_start > std::chrono::seconds(20)) {
            return fail(WF_ERR_CUDA, "step-server kernel did not answer within 20 s");
        }
    }
}

int wf_host_session(wf_env* e, int32_t on) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    WF_ON_DEVICE(e);
    if (on) {
        if (e->tile) return fail(WF_ERR_INVALID, "wf_host_session: grids up to 32x32 (warp family) only");
        if (e->fin.records) return fail(WF_ERR_STATE, "wf_host_session: final-state capture is on (wf_set_final_capture)");
        int coop = 0;
        WF_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, e->device));
        if (!coop) return fail(WF_ERR_INVALID, "wf_host_session: the device has no cooperative launch");
        if (on != 1 && on != 2) return fail(WF_ERR_INVALID, "wf_host_session: on must be 0, 1 or 2");
        if (e->sess.persistent_obs != (on == 2)) {  // another record format: the kernel is started again
            WF_QUIESCE(e);
            e->sess.persistent_obs = on == 2;
        }
        e->sess.wanted = true;
        return WF_OK;
    }
    WF_QUIESCE(e);
    e->sess.wanted = false;
    return WF_OK;
}
int wf_host_session_active(const wf_env* e) { return e ? (e->sess.wanted ? (e->sess.running ? 2 : 1) : 0) : 0; }

int wf_step_host(wf_env* e, const int32_t* actions_host, void* obs_host, int32_t obs_dtype, double* reward_host,
                 uint8_t* done_host) {
    if (!e || !actions_host) return fail(WF_ERR_INVALID, "null argument");
    if (!public_obs_dtype(obs_dtype)) return fail(WF_ERR_INVALID, "bad obs_dtype");
    if (e->fin.records) return fail(WF_ERR_STATE, "wf_step_host: final-state capture is on (wf_set_final_capture)");
    WF_ON_DEVICE(e);
    const DevState& s = e->st;
    const size_t obs_bytes = obs_step_bytes(s.N, s.W, s.H, obs_dtype);
    if (e->sess.wanted && !e->tile && obs_host && (obs_dtype == WF_OBS_U8 || obs_dtype == WF_OBS_BITS))
        return session_step(e, actions_host, obs_host, obs_dtype, reward_host, done_host);
    WF_QUIESCE(e);
    if (int rc = host_prologue(e)) return rc;

    // Zero-copy path: page-locked host buffers are addressed by the kernels themselves, so the
    // obs/reward/done stores stream over PCIe while the step is still computing and there is no
    // separate copy to launch.  Pageable buffers fall back to staged cudaMemcpyAsync.
    const void* hp[4] = {actions_host, obs_host, reward_host, done_host};
    for (int i = 0; i < 4; ++i) {  // cudaPointerGetAttributes costs ~1 us per buffer: look each buffer up once
        if (hp[i] != e->alias_host[i] || !hp[i] || (e->alias_age & 1023u) == 0u) {
            e->alias_host[i] = hp[i];
            e->alias_dev[i] = mapped_alias(hp[i]);
        }
    }
    e->alias_age += 1u;
    void* a_d = e->host_direct ? e->alias_dev[0] : nullptr;
    void* o_d = e->host_direct ? e->alias_dev[1] : nullptr;
    void* r_d = e->host_direct ? e->alias_dev[2] : nullptr;
    void* d_d = e->host_direct ? e->alias_dev[3] : nullptr;
    const bool small_direct = a_d && (r_d || !reward_host) && (d_d || !done_host);
    if (small_direct && e->host_packed && !e->tile && obs_host && obs_dtype == WF_OBS_U8) {
        // Packed path (grids up to 32x32): the kernel stores the observation BIT STREAM straight into mapped
        // page-locked memory (8x fewer bytes over PCIe than the uint8 array, no DMA to launch) and the host
        // thread pool expands it into the caller's buffer -- the compute the reference spends in np.dstack.
        const int epw = 32 / s.RS;
        const int64_t env_bits = (int64_t)s.W * s.H * 3, records = (s.N + epw - 1) / epw, rec_words = (epw * env_bits + 31) / 32;
        const size_t need = (size_t)records * rec_words;
        if (e->h_packed_words < need) {
            if (e->hg_exec) { cudaGraphExecDestroy(e->hg_exec); e->hg_exec = nullptr; }
            if (e->h_packed) cudaFreeHost(e->h_packed);
            cudaFree(e->d_packed);
            e->h_packed = nullptr;
            e->d_packed = nullptr;
            e->h_packed_words = 0;
            WF_CUDA(cudaMalloc(reinterpret_cast<void**>(&e->d_packed), need * sizeof(uint32_t)));
            WF_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&e->h_packed), need * sizeof(uint32_t), cudaHostAllocMapped));
            WF_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&e->h_packed_dev), e->h_packed, 0));
            e->h_packed_words = need;
        }
        if (!e->pool) e->pool = hostpool_create(hostpool_default_threads());
        const auto t0 = std::chrono::steady_clock::now();
        if (e->host_graph && e->packed_dma) {
            if (!e->hg_exec || e->hg_key[0] != a_d || e->hg_key[1] != r_d || e->hg_key[2] != d_d) {
                if (e->hg_exec) { cudaGraphExecDestroy(e->hg_exec); e->hg_exec = nullptr; }
                const int64_t launches0 = e->launches;
                cudaGraph_t g = nullptr;
                WF_CUDA(cudaStreamBeginCapture(e->hstream, cudaStreamCaptureModeThreadLocal));
                int rc = wf_step(e, static_cast<const int32_t*>(a_d), e->d_packed, kObsPacked, static_cast<double*>(r_d),
                                 static_cast<uint8_t*>(d_d), e->hstream);
                cudaError_t ce = cudaMemcpyAsync(e->h_packed, e->d_packed, need * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->hstream);
                cudaError_t ee = cudaStreamEndCapture(e->hstream, &g);
                e->launches = launches0;  // nothing ran yet
                if (rc != WF_OK) { if (g) cudaGraphDestroy(g); return rc; }
                WF_CUDA(ce);
                WF_CUDA(ee);
                cudaError_t ie = cudaGraphInstantiate(&e->hg_exec, g, 0);
                cudaGraphDestroy(g);
                WF_CUDA(ie);
                e->hg_key[0] = a_d; e->hg_key[1] = r_d; e->hg_key[2] = d_d;
            }
            WF_CUDA(cudaGraphLaunch(e->hg_exec, e->hstream));
            e->launches += 1;
        } else {
            int rc = wf_step(e, static_cast<const int32_t*>(a_d), e->packed_dma ? e->d_packed : e->h_packed_dev, kObsPacked,
                             static_cast<double*>(r_d), static_cast<uint8_t*>(d_d), e->hstream);
            if (rc != WF_OK) return rc;
            if (e->packed_dma)
                WF_CUDA(cudaMemcpyAsync(e->h_packed, e->d_packed, need * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->hstream));
        }
        const auto t1 = std::chrono::steady_clock::now();
        WF_CUDA(cudaStreamSynchronize(e->hstream));
        const auto t2 = std::chrono::steady_clock::now();
        hostpool_expand(e->pool, e->h_packed, static_cast<uint8_t*>(obs_host), records, rec_words, env_bits, epw, s.N);
        const auto t3 = std::chrono::steady_clock::now();
        e->t_launch += std::chrono::duration<double>(t1 - t0).count();
        e->t_sync += std::chrono::duration<double>(t2 - t1).count();
        e->t_expand += std::chrono::duration<double>(t3 - t2).count();
        e->t_calls += 1;
        return WF_OK;
    }
    if (small_direct) {
        // The SMs' stores over PCIe reach ~39 GB/s, a DMA copy ~48 GB/s (measured, tools/e2e_ab.py):
        // the 16-36 KB of actions/reward/done go zero-copy (no per-copy latency), the observation block
        // is written to HBM and moved by ONE cudaMemcpyAsync unless WF_HOST_MODE=direct.
        const bool obs_direct = e->host_obs_direct && o_d && (reinterpret_cast<uintptr_t>(o_d) & 15u) == 0;
        void* obs_target = nullptr;
        if (obs_host) {
            if (obs_direct) {
                obs_target = o_d;
            } else {
                if (int rc = ensure_obs_staging(e, obs_bytes)) return rc;
                obs_target = e->h_obs;
            }
        }
        int rc = wf_step(e, static_cast<const int32_t*>(a_d), obs_target, obs_dtype, static_cast<double*>(r_d),
                         static_cast<uint8_t*>(d_d), e->hstream);
        if (rc != WF_OK) return rc;
        if (obs_host && !obs_direct)
            WF_CUDA(cudaMemcpyAsync(obs_host, e->h_obs, obs_bytes, cudaMemcpyDeviceToHost, e->hstream));
        WF_CUDA(cudaStreamSynchronize(e->hstream));
        return WF_OK;
    }
    if (!e->h_actions) {
        WF_CUDA(cudaMalloc(&e->h_actions, (size_t)s.N * sizeof(int32_t)));
        WF_CUDA(cudaMalloc(&e->h_reward, (size_t)s.N * sizeof(double)));
        WF_CUDA(cudaMalloc(&e->h_done, (size_t)s.N));
    }
    if (obs_host) {
        if (int rc = ensure_obs_staging(e, obs_bytes)) return rc;
    }
    WF_CUDA(cudaMemcpyAsync(e->h_actions, actions_host, (size_t)s.N * sizeof(int32_t), cudaMemcpyHostToDevice, e->hstream));
    int rc = wf_step(e, e->h_actions, obs_host ? e->h_obs : nullptr, obs_dtype, e->h_reward, e->h_done, e->hstream);
    if (rc != WF_OK) return rc;
    if (obs_host) WF_CUDA(cudaMemcpyAsync(obs_host, e->h_obs, obs_bytes, cudaMemcpyDeviceToHost, e->hstream));
    if (reward_host) WF_CUDA(cudaMemcpyAsync(reward_host, e->h_reward, (size_t)s.N * sizeof(double), cudaMemcpyDeviceToHost, e->hstream));
    if (done_host) WF_CUDA(cudaMemcpyAsync(done_host, e->h_done, (size_t)s.N, cudaMemcpyDeviceToHost, e->hstream));
    WF_CUDA(cudaStreamSynchronize(e->hstream));
    return WF_OK;
}

static int grid_for(size_t n) { return (int)std::min<size_t>((n + 255) / 256, 148 * 16); }

int wf_get_state(wf_env* e, uint8_t* type, uint8_t* burning, uint8_t* fm_inf, uint8_t* fuel, uint8_t* hits,
                 uint8_t* apos, int32_t* scalars, void* stream) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const DevState& s = e->st;
    if (hits && (reinterpret_cast<uintptr_t>(hits) & 3u)) return fail(WF_ERR_INVALID, "hits must be 4-byte aligned");
    note_dev_call(e, st);
    if (type || burning || fm_inf || fuel || hits || apos) {
        get_state_kernel<<<grid_for((size_t)s.N * s.W * s.H), 256, 0, st>>>(s, type, burning, fm_inf, fuel, hits, apos);
        WF_CUDA(cudaGetLastError());
        e->launches += 1;
    }
    if (scalars)
        WF_CUDA(cudaMemcpyAsync(scalars, s.scal, (size_t)s.N * WF_NSCALARS * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    return WF_OK;
}

int wf_set_state(wf_env* e, const uint8_t* type, const uint8_t* burning, const uint8_t* fm_inf, const uint8_t* fuel,
                 const uint8_t* hits, const int32_t* scalars, void* stream) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const DevState& s = e->st;
    if (hits && (reinterpret_cast<uintptr_t>(hits) & 3u)) return fail(WF_ERR_INVALID, "hits must be 4-byte aligned");
    note_dev_call(e, st);
    if (type || burning || fm_inf || fuel || hits) {
        set_state_kernel<<<grid_for((size_t)s.N * s.W * s.HW), 256, 0, st>>>(s, type, burning, fm_inf, fuel, hits);
        WF_CUDA(cudaGetLastError());
        e->launches += 1;
    }
    if (scalars) {
        set_scalars_kernel<<<grid_for((size_t)s.N * WF_NSCALARS), 256, 0, st>>>(s, scalars);
        WF_CUDA(cudaGetLastError());
        e->launches += 1;
    }
    if (e->tile) WF_CUDA(tile_after_set_state(e->tstate, e->st, e->sc, st, &e->launches));
    return WF_OK;
}

int wf_get_a_iter(const wf_env* e, int32_t* out) {
    if (!e || !out) return fail(WF_ERR_INVALID, "null argument");
    *out = e->a_iter;
    return WF_OK;
}

int wf_set_a_iter(wf_env* e, int32_t a_iter) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    if (a_iter < 1 || a_iter > e->cfg.a_speed) return fail(WF_ERR_INVALID, "a_iter must be in 1..a_speed");
    e->a_iter = a_iter;
    return WF_OK;
}

int wf_set_fire_to(wf_env* e, const int32_t* cells_dev, void* stream) {
    if (!e || !cells_dev) return fail(WF_ERR_INVALID, "null argument");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    note_dev_call(e, st);
    set_fire_kernel<<<(e->N + 127) / 128, 128, 0, st>>>(e->st, cells_dev);
    WF_CUDA(cudaGetLastError());
    e->launches += 1;
    if (e->tile) WF_CUDA(tile_after_set_state(e->tstate, e->st, e->sc, st, &e->launches));
    return WF_OK;
}

int wf_get_obs(wf_env* e, void* obs_dev, int32_t obs_dtype, void* stream) {
    if (!e || !obs_dev) return fail(WF_ERR_INVALID, "null argument");
    if (int rc = check_obs(obs_dev, obs_dtype)) return rc;
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    const DevState& s = e->st;
    note_dev_call(e, static_cast<cudaStream_t>(stream));
    if (obs_dtype == WF_OBS_BITS)
        get_obs_bits_kernel<<<grid_for((size_t)s.N * obs_bits_words(s.W, s.H)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            s, static_cast<uint32_t*>(obs_dev));
    else
        get_obs_kernel<<<grid_for((size_t)s.N * s.W * s.H), 256, 0, static_cast<cudaStream_t>(stream)>>>(s, obs_dev, obs_dtype);
    WF_CUDA(cudaGetLastError());
    e->launches += 1;
    return WF_OK;
}

int wf_unpack_obs_bits(const uint32_t* bits_dev, int64_t n_rows, const int64_t* index_dev, int64_t n_out, int32_t width,
                       int32_t height, void* out_dev, int32_t out_dtype, void* stream) {
    if (out_dtype != WF_OBS_U8 && out_dtype != WF_OBS_F32 && out_dtype != WF_OBS_BF16)
        return fail(WF_ERR_INVALID, "wf_unpack_obs_bits: out_dtype must be WF_OBS_U8, WF_OBS_F32 or WF_OBS_BF16");
    if (width < 1 || height < 1) return fail(WF_ERR_INVALID, "wf_unpack_obs_bits: width and height must be >= 1");
    if (n_out < 0 || n_rows < 0) return fail(WF_ERR_INVALID, "wf_unpack_obs_bits: n_out and n_rows must be >= 0");
    if (n_out > 0 && (!out_dev || (n_rows > 0 && !bits_dev)))
        return fail(WF_ERR_INVALID, "wf_unpack_obs_bits: null argument");
    if (reinterpret_cast<uintptr_t>(out_dev) & 15u) return fail(WF_ERR_INVALID, "wf_unpack_obs_bits: out must be 16-byte aligned");
    if (reinterpret_cast<uintptr_t>(bits_dev) & 3u) return fail(WF_ERR_INVALID, "wf_unpack_obs_bits: bits must be 4-byte aligned");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(WF_ERR_CUDA, "no CUDA device: libwildfire_b200 has no CPU fallback");
    if (n_out == 0) return WF_OK;
    constexpr int kRowsPerBlock = 8;  // one warp per row
    const int64_t blocks = std::min<int64_t>((n_out + kRowsPerBlock - 1) / kRowsPerBlock, 148 * 16);
    unpack_obs_bits_kernel<<<(int)blocks, 32 * kRowsPerBlock, 0, static_cast<cudaStream_t>(stream)>>>(
        bits_dev, n_rows, index_dev, n_out, width, height, out_dev, out_dtype);
    WF_CUDA(cudaGetLastError());
    return WF_OK;
}

int wf_get_wind_table(const wf_env* e, double* coef_host, double* speed_host, int32_t* vec_host, int32_t* n_wind) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    if (n_wind) *n_wind = e->n_wind;
    for (int i = 0; i < e->n_wind; ++i) {
        if (coef_host) for (int d = 0; d < 4; ++d) coef_host[4 * i + d] = e->wind_host.coef[i][d];
        if (speed_host) speed_host[i] = e->wind_host.speed[i];
        if (vec_host) { vec_host[2 * i] = e->wind_host.wx[i]; vec_host[2 * i + 1] = e->wind_host.wy[i]; }
    }
    return WF_OK;
}

int wf_philox_kat(int32_t device, const uint32_t ctr_key_host[6], uint32_t out_host[4]) {
    if (!ctr_key_host || !out_host) return fail(WF_ERR_INVALID, "null argument");
    DeviceGuard _guard(device);
    WF_CUDA(_guard.err);
    uint32_t* buf = nullptr;
    WF_CUDA(cudaMalloc(&buf, 10 * sizeof(uint32_t)));
    WF_CUDA(cudaMemcpy(buf, ctr_key_host, 6 * sizeof(uint32_t), cudaMemcpyHostToDevice));
    philox_kat_kernel<<<1, 1>>>(buf, buf + 6);
    cudaError_t err = cudaMemcpy(out_host, buf + 6, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    cudaFree(buf);
    WF_CUDA(err);
    return WF_OK;
}

int wf_stats(wf_env* e, int64_t out_host[8], void* stream) {
    if (!e || !out_host) return fail(WF_ERR_INVALID, "null argument");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    WF_CUDA(cudaMemcpyAsync(out_host, e->st.stats, ST_N * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    WF_CUDA(cudaStreamSynchronize(st));
    return WF_OK;
}

int wf_stats_reset(wf_env* e, void* stream) {
    if (!e) return fail(WF_ERR_INVALID, "null handle");
    WF_ON_DEVICE(e);
    WF_QUIESCE(e);
    WF_CUDA(cudaMemsetAsync(e->st.stats, 0, ST_N * sizeof(unsigned long long), static_cast<cudaStream_t>(stream)));
    return WF_OK;
}

}  // extern "C"
