// wf_warp.cu -- "warp" kernel family: grids with W <= 32 and H <= 32.
//
// One environment is held by L = 16 or 32 lanes of a warp (two 14x14 envs per warp): lane x owns
// row x of every bit-plane as ONE 32-bit register (bit y = cell (x, y)), so a whole env lives in
// the register file.  The reference's per-burning-cell Python loop (forest_fire.py:85-106) becomes
// word-parallel boolean algebra; the 4-neighbour stencil is two shifts (y +- 1) and two warp
// shuffles (x +- 1); the A* containment search (environment.py:342-377, pyastar/astar.cpp) becomes
// a bitboard flood fill from the border; per-env reductions are warp ballots.  wf_rollout keeps
// the planes in registers across K steps, so HBM only sees actions in and obs/reward/done out.
#include "wf_families.cuh"

namespace wf {

// Row x of every plane, one register each (constant indices only, so it never leaves the RF).
constexpr int kHitBits = 7;  // bit-sliced total hit count per cell (<= 4 neighbours x (31 - 1) hits)

template <int FB>
struct Rows {
    uint32_t G, F, BT, D, WT, B, I;
    uint32_t FU[FB];
    uint32_t HC[kHitBits];  // only live in the UNI instantiations (dead registers otherwise)
    __device__ __forceinline__ uint32_t get(int p) const {
        switch (p) {
            case P_G: return G; case P_F: return F; case P_BT: return BT; case P_D: return D;
            case P_WT: return WT; case P_B: return B; case P_I: return I;
            default: return p < P_FU0 + FB ? FU[p - P_FU0] : HC[p - P_FU0 - FB];
        }
    }
    __device__ __forceinline__ void set(int p, uint32_t v) {
        switch (p) {
            case P_G: G = v; break; case P_F: F = v; break; case P_BT: BT = v; break; case P_D: D = v; break;
            case P_WT: WT = v; break; case P_B: B = v; break; case P_I: I = v; break;
            default: if (p < P_FU0 + FB) FU[p - P_FU0] = v; else HC[p - P_FU0 - FB] = v;
        }
    }
};

struct Agent {
    int ax, ay, alive, dead, digging, vis, running, fab, latched, wid, nburn;
    int kmin;  // uniform wind: total hits that ignite a cell; -1 = direction-dependent quanta
    uint32_t episode, t;
    __device__ __forceinline__ void refresh_wind(const WindTable* wt) { kmin = wt->uniform[wid] ? wt->kmin[wid] : -1; }
};

#ifndef WF_WARPS_PER_BLOCK
#define WF_WARPS_PER_BLOCK 4
#endif
constexpr int kWarpsPerBlock = WF_WARPS_PER_BLOCK;  // small CTAs balance 2048 warps over 148 SMs better

template <int FB>
__device__ __forceinline__ void dig(Rows<FB>& r, int x, int ax, int ay) {  // Agent.dig, environment.py:123-133
    if (x == ax) {
        const uint32_t bit = 1u << ay;
        if (!(r.D & bit)) {
            r.G &= ~bit; r.F &= ~bit; r.BT &= ~bit; r.WT &= ~bit;
            r.D |= bit;
            r.I |= bit;
        }
    }
}

template <int FB>
__device__ __forceinline__ void set_fire(Rows<FB>& r, int x, int fx, int fy) {  // World.set_fire_to, environment.py:233-246
    if (x == fx) {
        const uint32_t bit = 1u << fy;
        r.G &= ~bit; r.BT &= ~bit; r.D &= ~bit; r.WT &= ~bit;
        r.F |= bit;
        r.B |= bit;
    }
}

// World.reset -- environment.py:186-212 (+ reset_map :59-95, Agent.__init__ :100-113,
// get_agent_location utility.py:66-78).  Runs per env group; no warp collectives inside.
template <int L, int FB, bool UNI>
__device__ void reset_rows(Rows<FB>& r, Agent& a, const DevState& s, const StepCfg& c, const wf_init* init,
                           int env, int x, uint32_t validmask) {
    const int W = s.W, H = s.H;
    a.episode += 1u;
    a.t = 0u;
    ResetDraws dr((uint32_t)(c.env_id_base + env), a.episode, c.key0, c.key1);
    if (c.wind_random) {  // :188-190
        const int si = dr.next() % 3u, wx = dr.next() % 3u, wy = dr.next() % 3u;
        a.wid = si * 9 + wx * 3 + wy;
    } else {
        a.wid = 0;
    }
    r.G = validmask;
    r.F = r.BT = r.D = r.WT = r.B = r.I = 0u;
#pragma unroll
    for (int k = 0; k < FB; ++k) r.FU[k] = ((c.fuel >> k) & 1) ? validmask : 0u;
    if (UNI) {  // temp layer := 0
#pragma unroll
        for (int q = 0; q < kHitBits; ++q) r.HC[q] = 0u;
    } else {
        uint32_t* hits = s.hits + (size_t)env * W * H;
        for (int i = x; i < W * H; i += L) hits[i] = 0u;
    }

    const int cx = W / 2, cy = H / 2;  // get_fire_location, utility.py:61-64
    if (c.make_rivers) {               // reset_map :69-95; every lane replays the same draws
        int river_x = dr.next() % (uint32_t)W;
        int river_y = 1 + dr.next() % 3u;
        while (river_y < H - (1 + (int)(dr.next() % 3u))) {
            if (x == river_x) {
                const uint32_t bit = 1u << river_y;
                r.G &= ~bit;
                r.WT |= bit;
                r.I |= bit;
            }
            const int new_y = river_y + 1;
            int new_x = river_x + ((dr.next() % 2u) ? -1 : 1);
            for (;;) {  // `not a <= new_x < b and not (new_x, new_y) == fire`; the chain short-circuits b
                const int lo = 1 + dr.next() % 3u;
                bool chain = false;
                if (lo <= new_x) chain = new_x < W - (1 + (int)(dr.next() % 3u));
                if (chain || (new_x == cx && new_y == cy)) break;
                new_x = river_x + ((dr.next() % 2u) ? -1 : 1);
            }
            river_x = new_x;
            river_y = new_y;
        }
    }
    set_fire(r, x, cx, cy);  // :203
    int ax, ay;
    if (init != nullptr && init[env].ax >= 0) {
        ax = init[env].ax;
        ay = init[env].ay;
    } else {
        const int rad = dr.next() % 3u;  // radius - 1, utility.py:70
        const int idx = dr.next() % (uint32_t)kCircleLen[rad];
        ax = cx + kCircle[rad][idx][0];
        ay = cy + kCircle[rad][idx][1];
    }
    a.ax = ax; a.ay = ay;
    a.alive = 1; a.dead = 0; a.digging = 1; a.vis = 1;
    dig(r, x, ax, ay);  // Agent.__init__ digs its start cell, :112-113
    a.running = 1;
    a.latched = 0;  // reset_border_points(), :211
    a.fab = 0;      // :212
    for (int k = 0; k < c.extra_ignitions; ++k) {  // World.set_fire_to after reset (IGNITE stream)
        uint32_t w[4];
        philox4x32_10((uint32_t)(c.env_id_base + env), a.episode, (uint32_t)k, kStreamIgnite, c.key0, c.key1, w);
        const int ix = w[0] % (uint32_t)W, iy = w[1] % (uint32_t)H;
        set_fire(r, x, ix, iy);
        if (ix == 0 || ix == W - 1 || iy == 0 || iy == H - 1) a.fab = 1;
    }
}

// World.get_state -- environment.py:399-402: [agent_pos, type == fire, fire_mobility != inf].
// Output element e = (x*H + y)*3 + ch of an env is ONE BIT, so the env's whole [W][H][3] block is a
// bit stream: row x contributes 3H bits (its three masks interleaved bit by bit) at bit offset 3H*x.
// Each lane interleaves its row with a 256-entry "spread by 3" table, ORs it into the env's stream in
// shared memory, and then consecutive lanes expand consecutive nibbles of the stream into consecutive
// 4-byte words of the output (coalesced 64/128-byte stores, ~7 instructions per word).
constexpr int kStreamWords = 100;  // 3*32*32/32 = 96 words + spill-over of the last row's funnel shift

// OB: the WF_OBS_BITS instantiation (dtype == WF_OBS_BITS); the other element types never see its code.
template <int L, bool SRV = false, bool OB = false>
__device__ __forceinline__ void emit_obs(void* obs_step, int dtype, uint32_t arow, uint32_t frow, uint32_t freerow,
                                         uint32_t* stream, const uint32_t* spread3, const uint2* tab8, int lane, int sub,
                                         int x, int W, int H, int env0, int n_valid, uint32_t status16 = 0u) {
    // obs_step: start of this step's [N][W][H][3] block; env0: first env of the warp; n_valid: how many
    // of the warp's envs exist.  The warp's envs are adjacent in memory, so they share ONE bit stream.
    const int nbits = W * H * 3;
    const int tbits = n_valid * nbits;
    const int nw = (tbits + 31) >> 5;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < (L == 16 ? 2 : 4); ++i)  // 16-lane envs: <= 2 * 16 * 16 * 3 bits = 48 words (+ 4 of spill-over)
        if (lane + 32 * i < kStreamWords) stream[lane + 32 * i] = 0u;
    __syncwarp();
    if (x < W && sub < n_valid) {
        auto piece = [&](int p) -> uint32_t {  // cells 8p..8p+7 of this row -> 24 interleaved bits
            // (the agent_pos mask is one bit of one row; setting that bit under a branch instead of spreading the mask
            //  measured slower: 2.11 against 2.05 us per C2 step)
            return spread3[(arow >> (8 * p)) & 255u] | (spread3[(frow >> (8 * p)) & 255u] << 1) |
                   (spread3[(freerow >> (8 * p)) & 255u] << 2);
        };
        const uint32_t p0 = piece(0), p1 = piece(1);
        uint32_t r0 = p0 | (p1 << 24), r1 = p1 >> 8, r2 = 0u;
        if (L == 32 && H > 16) {
            const uint32_t p2 = piece(2), p3 = piece(3);
            r1 |= p2 << 16;
            r2 = (p2 >> 16) | (p3 << 8);
        }
        const int start = sub * nbits + 3 * H * x, w0 = start >> 5, sh = start & 31;
        const uint32_t c0 = r0 << sh, c1 = __funnelshift_l(r0, r1, sh), c2 = __funnelshift_l(r1, r2, sh),
                       c3 = __funnelshift_l(r2, 0u, sh);
        atomicOr(&stream[w0], c0);  // (the first two words of a row are hardly ever empty: no test, no branch)
        atomicOr(&stream[w0 + 1], c1);
        atomicOr(&stream[w0 + 2], c2);
        if (L == 32 && c3) atomicOr(&stream[w0 + 3], c3);
    }
    __syncwarp();
    if (n_valid <= 0) return;
    if (SRV || dtype == kObsPacked) {  // the stream as it is: 8x fewer bytes over PCIe, expanded on the host
        constexpr int EPW = 32 / L;
        const int rec_words = (EPW * nbits + 31) >> 5;
        if (SRV) {  // kObsPackedStatus: + one status word per record: reward kind / done / burn-out count of each env
            uint32_t st = __shfl_sync(0xffffffffu, status16, 0);
            if (EPW == 2) st |= __shfl_sync(0xffffffffu, status16, L & 31) << 16;
            uint32_t* rec = static_cast<uint32_t*>(obs_step);  // this warp's slot of the CTA's block in shared memory
            for (int w = lane; w < nw; w += 32) rec[w] = stream[w];
            if (lane == 0) rec[rec_words] = st;
        } else {
            uint32_t* rec = static_cast<uint32_t*>(obs_step) + (size_t)(env0 / EPW) * rec_words;
            for (int w = lane; w < nw; w += 32) rec[w] = stream[w];
        }
        return;
    }
    if constexpr (OB) {
        // The public format starts every env on a word boundary: output word j of env e (e = 0 or 1) is stream bits
        // e * nbits + 32 j ..., with the bits past the env's last element cleared.  The warp's envs are n_valid * wpe
        // consecutive output words, stored coalesced.
        const int wpe = (nbits + 31) >> 5, tail = nbits & 31;
        uint32_t* o = static_cast<uint32_t*>(obs_step) + (size_t)env0 * wpe;
        for (int w = lane; w < n_valid * wpe; w += 32) {
            const int e = w >= wpe ? 1 : 0, j = w - e * wpe, b = e * nbits + 32 * j;
            uint32_t v = __funnelshift_r(stream[b >> 5], stream[(b >> 5) + 1], b & 31);
            if (j == wpe - 1 && tail) v &= (1u << tail) - 1u;
            o[w] = v;
        }
        return;
    }
    if (dtype == WF_OBS_U8) {
        uint8_t* o8 = static_cast<uint8_t*>(obs_step) + (size_t)env0 * nbits;
        if ((tbits & 7) == 0 && (reinterpret_cast<uintptr_t>(o8) & 7u) == 0) {
            uint2* o64 = reinterpret_cast<uint2*>(o8);  // output bytes 8j..8j+7 = stream bits 8j..8j+7
            const uint8_t* stream8 = reinterpret_cast<const uint8_t*>(stream);
            // byte of 8 stream bits -> 8 bytes; fully unrolled under a predicate, so that all the look-ups are in flight together
            constexpr int kMaxIt = (L == 16) ? 6 : 12;  // (2 x 16 x 16 x 3 or 32 x 32 x 3 bits) / 8 / 32 lanes
            const int n8 = tbits >> 3;
#pragma unroll
            for (int i = 0; i < kMaxIt; ++i) {
                const int j = lane + 32 * i;
                if (j < n8) o64[j] = tab8[stream8[j]];
            }
        } else if ((tbits & 3) == 0 && (reinterpret_cast<uintptr_t>(o8) & 3u) == 0) {
            uint32_t* o32 = reinterpret_cast<uint32_t*>(o8);
            for (int j = lane; j < (tbits >> 2); j += 32) {
                const uint32_t nib = (stream[j >> 3] >> ((j & 7) * 4)) & 15u;
                o32[j] = (nib * 0x00204081u) & 0x01010101u;
            }
        } else {
            for (int b = lane; b < tbits; b += 32) o8[b] = (uint8_t)((stream[b >> 5] >> (b & 31)) & 1u);
        }
    } else if (dtype == WF_OBS_BF16) {  // 1.0 = 0x3F80: two elements per 32-bit store where the block allows it
        uint16_t* oh = static_cast<uint16_t*>(obs_step) + (size_t)env0 * nbits;
        if ((tbits & 1) == 0 && (reinterpret_cast<uintptr_t>(oh) & 3u) == 0) {
            uint32_t* o32 = reinterpret_cast<uint32_t*>(oh);
            for (int j = lane; j < (tbits >> 1); j += 32) {
                const uint32_t two = (stream[j >> 4] >> ((j & 15) * 2)) & 3u;
                o32[j] = ((two & 1u) ? (uint32_t)kBf16One : 0u) | ((two & 2u) ? (uint32_t)kBf16One << 16 : 0u);
            }
        } else {
            for (int b = lane; b < tbits; b += 32) oh[b] = ((stream[b >> 5] >> (b & 31)) & 1u) ? kBf16One : (uint16_t)0;
        }
    } else {
        float* of = static_cast<float*>(obs_step) + (size_t)env0 * nbits;
        for (int b = lane; b < tbits; b += 32) of[b] = ((stream[b >> 5] >> (b & 31)) & 1u) ? 1.0f : 0.0f;
    }
}

// Final-state capture: one section of the records of the warp's envs.  Row x's `nrow` bits (r0, then r1, r2) belong at
// bit x * nrow of env `sub`'s section, which is `nw` words long and starts on a word boundary; the warp assembles the
// sections in its stream buffer and stores env e's to dst[e] (nullptr: that env writes no record).
template <int L>
__device__ __forceinline__ void fin_section(uint32_t* stream, int lane, int sub, int x, int W, int nrow, int nw, uint32_t r0,
                                            uint32_t r1, uint32_t r2, uint32_t* dst0, uint32_t* dst1) {
    constexpr int EPW = 32 / L;
    __syncwarp();
    for (int i = lane; i < kStreamWords; i += 32) stream[i] = 0u;
    __syncwarp();
    if (x < W) {
        const int start = sub * nw * 32 + x * nrow, w0 = start >> 5, sh = start & 31;
        atomicOr(&stream[w0], r0 << sh);
        if (sh + nrow > 32) atomicOr(&stream[w0 + 1], __funnelshift_l(r0, r1, sh));
        if (sh + nrow > 64) atomicOr(&stream[w0 + 2], __funnelshift_l(r1, r2, sh));
        if (sh + nrow > 96) atomicOr(&stream[w0 + 3], __funnelshift_l(r2, 0u, sh));
    }
    __syncwarp();
    for (int w = lane; w < EPW * nw; w += 32) {
        const int e = w >= nw ? 1 : 0;
        uint32_t* d = e ? dst1 : dst0;
        if (d != nullptr) d[w - e * nw] = stream[w];
    }
}

// The record of every env of the warp that returns done this step (`rec`), taken before the auto-reset; include/wildfire.h
// has the layout.  Returns the header of this lane's env's record, or nullptr (no record, or past the capacity).
template <int L, int FB>
__device__ __forceinline__ uint32_t* capture_final(const Rows<FB>& r, const Agent& a, const FinalCapture& fin, bool rec, int k, int env,
                                                int lane, int sub, int x, int W, int H, uint32_t validmask, uint32_t* stream,
                                                const uint32_t* spread3) {
    constexpr uint32_t FULL = 0xffffffffu;
    uint32_t slot = 0xffffffffu;
    if (rec && x == 0) slot = atomicAdd(fin.count, 1u);
    slot = __shfl_sync(FULL, slot, sub * L);
    uint32_t* const mine = (rec && (int64_t)slot < fin.capacity) ? fin.records + (size_t)slot * fin.words : nullptr;
    uint32_t* const d0 = reinterpret_cast<uint32_t*>(__shfl_sync(FULL, reinterpret_cast<uintptr_t>(mine), 0));
    uint32_t* const d1 = L == 16 ? reinterpret_cast<uint32_t*>(__shfl_sync(FULL, reinterpret_cast<uintptr_t>(mine), 16)) : nullptr;
    if (mine != nullptr && x == 0) {
        const int flags = (a.alive ? WF_FINAL_ALIVE : 0) | (a.vis ? WF_FINAL_VISIBLE : 0) | (a.dead ? WF_FINAL_DEAD : 0) |
                          (a.digging ? WF_FINAL_DIGGING : 0);
        uint4* h = reinterpret_cast<uint4*>(mine);
        h[0] = make_uint4((uint32_t)k, (uint32_t)env, a.episode, a.t);
        h[1] = make_uint4((uint32_t)a.ax, (uint32_t)a.ay, (uint32_t)flags, 0xffffffffu);
        h[2] = make_uint4(0xffffffffu, 0u, 0u, 0u);
        h[3] = make_uint4(0u, 0u, 0u, 0u);
    }
    // the terminal observation (World.get_state, as emit_obs builds it) ...
    const uint32_t arow = (a.vis && x == a.ax) ? (1u << a.ay) : 0u, freerow = ~r.I & validmask;
    auto piece = [&](int p) -> uint32_t {
        return spread3[(arow >> (8 * p)) & 255u] | (spread3[(r.F >> (8 * p)) & 255u] << 1) | (spread3[(freerow >> (8 * p)) & 255u] << 2);
    };
    const uint32_t p0 = piece(0), p1 = piece(1);
    uint32_t o0 = p0 | (p1 << 24), o1 = p1 >> 8, o2 = 0u;
    if (L == 32 && H > 16) {
        const uint32_t p2 = piece(2), p3 = piece(3);
        o1 |= p2 << 16;
        o2 = (p2 >> 16) | (p3 << 8);
    }
    const int pw = final_plane_words(W, H), po = fin.plane_off;
    // (the section runs up to the planes, so the padding words after the observation are written as zeros too)
    fin_section<L>(stream, lane, sub, x, W, 3 * H, po - WF_FINAL_OBS, o0, o1, o2, d0 ? d0 + WF_FINAL_OBS : nullptr,
                   d1 ? d1 + WF_FINAL_OBS : nullptr);
    // ... the type planes, and the zero padding at the end of the record
    const uint32_t planes[4] = {r.F, r.BT, r.D, r.WT};
#pragma unroll
    for (int p = 0; p < 4; ++p)
        fin_section<L>(stream, lane, sub, x, W, H, pw, planes[p], 0u, 0u, d0 ? d0 + po + p * pw : nullptr,
                       d1 ? d1 + po + p * pw : nullptr);
    if (mine != nullptr)
        for (int w = po + 4 * pw + x; w < fin.words; w += L) mine[w] = 0u;
    __syncwarp();
    return mine;
}

// UNI: every wind of the handle has direction-independent heat quanta (e.g. wind vector (0, 0)): a cell
// ignites when its TOTAL hit count reaches kmin, so `temp` is a 7-bit counter per cell, bit-sliced in
// registers (planes HC0..HC6); heat transfer + ignition test are ~40 word-parallel logic instructions
// per tick instead of a data-dependent loop over hit counters in memory.
// MLP: the Q-network of WF_POLICY_MLP is evaluated in here (DQN.choose_action, DQN.py:188-196).  Its inputs
// are the observation bits, so the first layer is a SUM OF WEIGHT ROWS: every lane keeps a few hidden
// pre-activations in float64 and, per step, only adds / subtracts the rows of the bits that changed
// (agent cell, dug cell, ignitions, burn-outs; everything after a reset).
constexpr int kHidMax = 64, kActMax = 8;

// SRV: step-server session (wf_host_session).  The kernel stays resident; per step, thread 0 of CTA 0 waits for the
// host's doorbell in mapped page-locked memory and releases the other CTAs through a flag in HBM; every warp reads its
// actions from the mapped buffer, steps, stores its packed observation record (+ status word) straight into mapped host
// memory; the last CTA of every slice of the grid to finish tells the host thread that expands that slice.
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// FIN: final-state capture (`fin`): the record of every episode that ends is written before the auto-reset.
template <int L, int FB, bool UNI, bool MLP, bool SRV, bool OB, bool FIN = false>
__device__ __forceinline__ void warp_body(const DevState& s, const StepCfg& c, const WarpIO& io, const SrvCtl& srv) {
    constexpr int EPW = 32 / L;  // envs per warp
    constexpr uint32_t FULL = 0xffffffffu;
    constexpr uint32_t GMASK = (L == 32) ? 0xffffffffu : ((1u << L) - 1u);
    __shared__ __align__(16) uint32_t stream_all[kWarpsPerBlock][kStreamWords];
    __shared__ uint32_t spread3[256];  // bit i of the index -> bit 3i
    __shared__ uint2 tab8[256];        // bit i of the index -> byte i
    __shared__ uint32_t srv_cmd, srv_flags;
    __shared__ unsigned long long cta_stats[2];  // env-steps and fire ticks of this CTA's envs in this launch
    if (threadIdx.x < 2) cta_stats[threadIdx.x] = 0ull;
    // SRV: the CTA's records (one per warp: up to 96 words of observation bits + the status word) are collected here and
    // leave for host memory as ONE 128-byte-aligned block of 16-byte stores -- whole PCIe write transactions instead of
    // the 4-byte-per-lane stores of unaligned 152-byte records (which cost ~25 us per step on the link)
    __shared__ __align__(16) uint32_t srv_block[SRV ? kWarpsPerBlock * 97 + 31 + 96 : 1];  // (+ slack: the sector copy reads 7-word groups)
    __shared__ float4 mlp_w2[MLP ? 2 * kHidMax : 1];  // second layer (MlpPolicy::w2), read every step
    __shared__ float mlp_b2[MLP ? kActMax + 1 : kActMax];  // + the explore threshold (uint32 bits)
    // WF_POLICY_MLP: this CTA's envs all act with one network (MlpPolicy::group_envs is a multiple of the CTA's envs)
    const size_t mlp_off = MLP ? (size_t)((int)blockIdx.x * (kWarpsPerBlock * (32 / L)) / io.mlp.group_envs) * io.mlp.net_stride : 0;
    for (int v = threadIdx.x; v < 256; v += blockDim.x) {
        uint32_t o = 0u;
#pragma unroll
        for (int i = 0; i < 8; ++i) o |= ((v >> i) & 1u) << (3 * i);
        spread3[v] = o;
        tab8[v] = make_uint2(((v & 15u) * 0x00204081u) & 0x01010101u, (((v >> 4) & 15u) * 0x00204081u) & 0x01010101u);
    }
    if (MLP) {
        for (int v = threadIdx.x; v < 2 * kHidMax; v += blockDim.x) mlp_w2[v] = reinterpret_cast<const float4*>(io.mlp.w2 + mlp_off)[v];
        if (threadIdx.x <= kActMax) mlp_b2[threadIdx.x] = io.mlp.b2[mlp_off + threadIdx.x];
    }
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane / L, x = lane % L;
    const int env0 = (blockIdx.x * kWarpsPerBlock + warp) * EPW;  // first env of this warp
    const int env = env0 + sub;
    const bool valid_env = env < s.N;
    const int n_valid = min(EPW, s.N - env0);
    const int W = s.W, H = s.H;
    const uint32_t colmask = (H == 32) ? 0xffffffffu : ((1u << H) - 1u);
    const uint32_t validmask = (valid_env && x < W) ? colmask : 0u;
    // Literal border_points (environment.py:215-222): rows x == 0 and x == HEIGHT-1, columns 0 and H-1.
    const uint32_t seedmask = (x == 0 || x == H - 1) ? validmask : (validmask & (1u | (1u << (H - 1))));
    const uint32_t edgemask = (x == 0 || x == W - 1) ? validmask : (validmask & (1u | (1u << (H - 1))));
    auto group_bits = [&](uint32_t ballot) -> uint32_t { return (ballot >> (sub * L)) & GMASK; };
    uint32_t* stream_warp = stream_all[warp];

    // ---------------- load ----------------
    Rows<FB> r;
    Agent a;
    {
#pragma unroll
        for (int p = 0; p < 7 + FB + (UNI ? kHitBits : 0); ++p) r.set(p, valid_env ? s.planes[word_index(s, p, env, x, 0)] : 0u);
        int4 v0 = make_int4(0, 0, 0, 0), v1 = v0, v2 = v0, v3 = v0;
        if (valid_env) {
            const int4* sp = reinterpret_cast<const int4*>(s.scal + (size_t)env * WF_NSCALARS);
            v0 = sp[0]; v1 = sp[1]; v2 = sp[2]; v3 = sp[3];
        }
        a.alive = v0.x; a.ax = v0.y; a.ay = v0.z; a.dead = v0.w;
        a.digging = v1.x; a.vis = v1.y; a.running = v1.z; a.fab = v1.w;
        a.latched = v2.x; a.episode = (uint32_t)v2.y; a.t = (uint32_t)v2.z; a.wid = v2.w;
        a.nburn = v3.z;
    }
    if (!valid_env) { a.running = 0; a.alive = 0; a.ax = a.ay = 0; a.wid = 0; }
    a.refresh_wind(s.wind);

    long long n_steps_done = 0, n_ticks_done = 0;

    // WF_POLICY_MLP: hidden pre-activations of units j = x + L*i, and the observation they were computed from
    constexpr int HPL = kHidMax / L;
    double hacc[MLP ? HPL : 1];
    uint32_t pA = 0u, pF = 0u, pFree = validmask;  // the empty map: what `base` stands for
    if (MLP) {
#pragma unroll
        for (int i = 0; i < HPL; ++i) hacc[i] = (double)io.mlp.base[mlp_off + x + L * i];
    }

    if (io.reset_mode) {
        // ---------------- ForestFire.reset() ----------------
        const bool doit = valid_env && (io.mask == nullptr || io.mask[env] != 0);
        if (doit) {
            reset_rows<L, FB, UNI>(r, a, s, c, io.init, env, x, validmask);
            a.refresh_wind(s.wind);
        }
        __syncwarp();
        if (io.obs != nullptr) {
            emit_obs<L, false, OB>(io.obs, io.obs_dtype, (a.vis && x == a.ax) ? (1u << a.ay) : 0u, r.F, ~r.I & validmask,
                        stream_warp, spread3, tab8, lane, sub, x, W, H, env0, n_valid);
        }
    } else {
        // ---------------- K x ForestFire.step(action) ----------------
        int it = io.a_iter0;
        uint32_t ablk[4] = {0u, 0u, 0u, 0u}, ablk_ep = 0xffffffffu, ablk_idx = 0xffffffffu;  // cached ACTION block
        uint32_t reach = 0u;    // row x of the reach mask, valid while reach_ok (group-uniform)
        bool reach_ok = false;
        uint32_t srv_step = 0u;  // SRV: steps served by this launch
        int srv_want_full = 0;   // SRV, change-list records: the host asks for every record in full this step
        unsigned long long srv_t0 = 0ull, srv_t0b = 0ull, srv_t1 = 0ull;  // CTA 0, thread 0: time stamps of the debug counters
        for (int kk = 0; SRV || kk < io.K; ++kk) {
            const int k = SRV ? 0 : kk;  // row of the output arrays
            if (SRV) {
                if (blockIdx.x == 0) {
                    // CTA 0 waits for the step's actions and brings them into HBM; only then are the other CTAs released.
                    // The mapped host buffer holds the actions packed and TAGGED (wf_common.cuh: six 4-bit actions + the
                    // step's sequence number in every word).  The whole CTA polls the buffer itself with batched 16-byte
                    // loads until every word carries this step's tag, so the actions arrive with the poll that notices
                    // them: one PCIe round trip instead of one for a doorbell plus one for the actions (and 2048 warps each
                    // fetching its own action from host memory was ~80 us per step).  Thread 0 also reads the doorbell
                    // word -- the host writes 0xffffffff there to park the kernel -- and keeps the idle clock.
                    const uint32_t want_tag = (srv.seq0 + srv_step + 1u) & kSrvTagMask;
                    const int n16 = srv_action_chunks(s.N);
                    const int4* src = reinterpret_cast<const int4*>(srv.actions_host);
                    int4* dst = reinterpret_cast<int4*>(srv.actions_dev);  // [24 * n16] unpacked actions
                    unsigned long long t0 = 0ull;
                    if (threadIdx.x == 0) {
                        t0 = global_timer_ns();
                        srv_t0 = t0;
                        srv_cmd = srv_step + 1u;
                    }
                    auto tag_ok = [&](int w) { return (((uint32_t)w >> 24) & kSrvTagMask) == want_tag; };
                    auto unpack = [](int w, int k) { const int a = (w >> (4 * k)) & 15; return a == 15 ? -1 : a; };
                    constexpr int kBatch = 4;  // chunks a thread polls at once (4 x 128 threads x 24 = 12 288 envs per pass)
                    bool parked = false;
                    for (int base = 0; base < n16 && !parked; base += kBatch * (int)blockDim.x) {
                        for (;;) {
                            int4 v[kBatch];
                            bool ok = true;
#pragma unroll
                            for (int u = 0; u < kBatch; ++u) {
                                const int j = base + (int)threadIdx.x + u * (int)blockDim.x;
                                if (j < n16) v[u] = __ldcv(src + j);
                            }
                            uint32_t cmd = 0u;
                            if (base == 0 && threadIdx.x == 0) cmd = *srv.doorbell;
#pragma unroll
                            for (int u = 0; u < kBatch; ++u) {
                                const int j = base + (int)threadIdx.x + u * (int)blockDim.x;
                                if (j < n16) ok = ok && tag_ok(v[u].x) && tag_ok(v[u].y) && tag_ok(v[u].z) && tag_ok(v[u].w);
                            }
                            if (__syncthreads_and(ok)) {
                                if (base == 0 && threadIdx.x == 0) srv_flags = (uint32_t)v[0].x >> 31;
#pragma unroll
                                for (int u = 0; u < kBatch; ++u) {
                                    const int j = base + (int)threadIdx.x + u * (int)blockDim.x;
                                    if (j < n16) {
                                        const int w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
                                        for (int q = 0; q < 6; ++q) {  // 24 actions = 6 stores of 16 bytes
                                            int o[4];
#pragma unroll
                                            for (int i = 0; i < 4; ++i) o[i] = unpack(w[(4 * q + i) / 6], (4 * q + i) % 6);
                                            dst[6 * j + q] = make_int4(o[0], o[1], o[2], o[3]);
                                        }
                                    }
                                }
                                break;
                            }
                            if (base == 0) {  // not (all) there yet: asked to park, or idle for too long?
                                if (threadIdx.x == 0 && (cmd == 0xffffffffu || global_timer_ns() - t0 > srv.idle_ns)) {
                                    *srv.parked = srv.generation;
                                    srv_cmd = 0xffffffffu;
                                }
                                __syncthreads();
                                if (srv_cmd == 0xffffffffu) { parked = true; break; }
                            }
                        }
                    }
                    if (threadIdx.x == 0) srv_t0b = global_timer_ns();
                    if (!parked) __threadfence();
                    __syncthreads();
                    if (threadIdx.x == 0) {
                        srv_t1 = global_timer_ns();
                        if (srv.delta && !parked) srv.actions_dev[24 * srv_action_chunks(s.N)] = (int32_t)(srv_flags & 1u);  // the host's full-frame request
                        st_release_gpu(srv.go, srv_cmd);
                    }
                } else {
                    if (threadIdx.x == 0) {
                        uint32_t go;
                        do { go = ld_acquire_gpu(srv.go); } while (go == srv_step);
                        srv_cmd = go;
                    }
                    __syncthreads();
                }
                if (srv_cmd == 0xffffffffu) break;
            }
            const bool act = valid_env && a.running;  // finished envs are frozen (reward 0, done 1)
            int action;
            if (io.actions != nullptr) {
                if (SRV) {
                    action = valid_env ? __ldcg(&io.actions[env]) : -1;  // HBM copy, rewritten every step (L2, not L1)
                    if (srv.delta) srv_want_full = __ldcg(&io.actions[24 * srv_action_chunks(s.N)]);  // (needed after the step: the load is hidden)
                }
                else action = valid_env ? io.actions[(size_t)k * s.N + env] : -1;
            } else if (MLP) {
                // ---- first layer, incrementally: the weight rows of the observation bits that changed since the last
                // evaluation.  Per round the first lane of the env that still has a changed bit announces one of them
                // (input index and its new value, one shuffle); every lane then adds or subtracts its HPL weights of
                // that row (one vector load: MlpPolicy::w1 keeps them adjacent).
                const uint32_t cA = (a.vis && x == a.ax) ? (1u << a.ay) : 0u, cF = r.F, cFree = ~r.I & validmask;
                uint32_t dA = cA ^ pA, dF = cF ^ pF, dFree = cFree ^ pFree;
                pA = cA; pF = cF; pFree = cFree;
                for (;;) {
                    const uint32_t pending = __ballot_sync(FULL, (dA | dF | dFree) != 0u);
                    if (pending == 0u) break;
                    const uint32_t mine = group_bits(pending);
                    const int owner = mine ? __ffs(mine) - 1 : 0;
                    uint32_t code = 0u;
                    if (mine != 0u && x == owner) {
                        const int ch = dA ? 0 : dF ? 1 : 2;
                        const uint32_t m = dA ? dA : dF ? dF : dFree;
                        const uint32_t now = dA ? cA : dF ? cF : cFree;
                        const uint32_t low = m & (0u - m);
                        const int y = __ffs(m) - 1;
                        if (ch == 0) dA ^= low;
                        else if (ch == 1) dF ^= low;
                        else dFree ^= low;
                        code = ((uint32_t)((x * H + y) * 3 + ch) << 1) | ((now & low) ? 1u : 0u);
                    }
                    code = __shfl_sync(FULL, code, sub * L + owner);
                    if (mine) {
                        const float* wrow = io.mlp.w1 + mlp_off + (size_t)(code >> 1) * kHidMax + x * HPL;
                        const uint32_t flip = (code & 1u) ? 0u : 0x80000000u;  // bit cleared: subtract the row
                        float wv[HPL];
                        if (HPL == 4) {
                            const float4 v = __ldg(reinterpret_cast<const float4*>(wrow));
                            wv[0] = v.x; wv[1] = v.y; wv[HPL > 2 ? 2 : 0] = v.z; wv[HPL > 3 ? 3 : 0] = v.w;
                        } else {
                            const float2 v = __ldg(reinterpret_cast<const float2*>(wrow));
                            wv[0] = v.x; wv[1] = v.y;
                        }
#pragma unroll
                        for (int i = 0; i < HPL; ++i) hacc[i] += (double)__uint_as_float(__float_as_uint(wv[i]) ^ flip);
                    }
                }
                // ---- sigmoid and second layer: 8 partial Q values per lane (padded units and actions carry zero weights)
                float q[kActMax];
#pragma unroll
                for (int b = 0; b < kActMax; ++b) q[b] = 0.0f;
#pragma unroll
                for (int i = 0; i < HPL; ++i) {
                    const int j = x + L * i;
                    const float sj = __fdividef(1.0f, 1.0f + __expf(-(float)hacc[i]));
                    const float4 wa = mlp_w2[j], wb = mlp_w2[kHidMax + j];
                    q[0] = fmaf(sj, wa.x, q[0]); q[1] = fmaf(sj, wa.y, q[1]); q[2] = fmaf(sj, wa.z, q[2]); q[3] = fmaf(sj, wa.w, q[3]);
                    q[4] = fmaf(sj, wb.x, q[4]); q[5] = fmaf(sj, wb.y, q[5]); q[6] = fmaf(sj, wb.z, q[6]); q[7] = fmaf(sj, wb.w, q[7]);
                }
                // ---- sum over the env's lanes, transposing on the way: every butterfly step halves the values a lane
                // carries (it keeps the half its lane bit selects and adds the partner's copy of it), so 8 values cost
                // 4 + 2 + 1 shuffles and lane x ends with Q of action (x >> (log2 L - 3)) & 7 ...
                const bool h3 = (x & (L / 2)) != 0, h2 = (x & (L / 4)) != 0, h1 = (x & (L / 8)) != 0;
                float q4[4], q2[2], qv;
#pragma unroll
                for (int b = 0; b < 4; ++b)
                    q4[b] = (h3 ? q[b + 4] : q[b]) + __shfl_xor_sync(FULL, h3 ? q[b] : q[b + 4], L / 2, L);
#pragma unroll
                for (int b = 0; b < 2; ++b)
                    q2[b] = (h2 ? q4[b + 2] : q4[b]) + __shfl_xor_sync(FULL, h2 ? q4[b] : q4[b + 2], L / 4, L);
                qv = (h1 ? q2[1] : q2[0]) + __shfl_xor_sync(FULL, h1 ? q2[0] : q2[1], L / 8, L);
#pragma unroll
                for (int o = L / 16; o > 0; o >>= 1) qv += __shfl_xor_sync(FULL, qv, o, L);
                int greedy = (h3 ? 4 : 0) | (h2 ? 2 : 0) | (h1 ? 1 : 0);
                qv += mlp_b2[greedy];  // -inf for actions the network does not have
                // ... and the argmax (np.argmax: the first maximum) is a butterfly over those three lane bits (the first
                // partner's action index is known without a shuffle)
#pragma unroll
                for (int bit = 0; bit < 3; ++bit) {
                    const float other = __shfl_xor_sync(FULL, qv, (L / 8) << bit, L);
                    const int other_a = bit == 0 ? (greedy ^ 1) : __shfl_xor_sync(FULL, greedy, (L / 8) << bit, L);
                    if (other > qv || (other == qv && other_a < greedy)) { qv = other; greedy = other_a; }
                }
                // ---- eps-greedy: EXPLORE stream, one Philox block serves two consecutive steps
                if ((a.t & 1u) == 0u || ablk_ep != a.episode || ablk_idx != (a.t >> 1)) {
                    philox4x32_10((uint32_t)(c.env_id_base + env), a.episode, a.t >> 1, kStreamExplore, c.key0, c.key1, ablk);
                    ablk_ep = a.episode;
                    ablk_idx = a.t >> 1;
                }
                const uint32_t u0 = (a.t & 1u) ? ablk[2] : ablk[0], u1 = (a.t & 1u) ? ablk[3] : ablk[1];
                action = (u0 < __float_as_uint(mlp_b2[kActMax])) ? (int)(u1 % (uint32_t)c.n_actions) : greedy;
            } else if (io.policy == WF_POLICY_WALK) {
                // DQN.choose_randomwalk_action (DQN.py:353-389): walk clockwise round the fire origin,
                // re-draw (at most 11 times) while the move would step onto a burning cell.
                const int mx = W / 2, my = H / 2;
                int a0 = 0, a1 = 0;
                if (a.ax >= mx && a.ay > my) { a0 = 1; a1 = 3; }  // ["S", "W"]
                if (a.ax > mx && a.ay <= my) { a0 = 1; a1 = 2; }  // ["S", "E"]
                if (a.ax <= mx && a.ay < my) { a0 = 0; a1 = 2; }  // ["N", "E"]
                if (a.ax < mx && a.ay >= my) { a0 = 0; a1 = 3; }  // ["N", "W"]
                bool chosen = !(act && a.alive);  // `if not self.sim.W.agents: return 0`
                int count = 0;
                action = 0;
                uint32_t pw[4] = {0u, 0u, 0u, 0u};
                for (int j = 0; j < 12; ++j) {
                    if ((j & 3) == 0)
                        philox4x32_10((uint32_t)(c.env_id_base + env), a.episode, 3u * a.t + (uint32_t)(j >> 2), kStreamPolicy,
                                      c.key0, c.key1, pw);
                    const uint32_t u = (j & 3) == 0 ? pw[0] : (j & 3) == 1 ? pw[1] : (j & 3) == 2 ? pw[2] : pw[3];
                    const int cand = (u & 1u) ? a1 : a0;
                    const int nx = a.ax + (cand == 2 ? 1 : cand == 3 ? -1 : 0);
                    const int ny = a.ay + (cand == 1 ? 1 : cand == 0 ? -1 : 0);
                    const bool inb = nx >= 0 && nx < W && ny >= 0 && ny < H;
                    const uint32_t frow = __shfl_sync(FULL, r.F, sub * L + (inb ? nx : 0));
                    if (!chosen) {
                        action = cand;
                        const bool fire_at_loc = inb && ((frow >> ny) & 1u);  // Agent.fire_in_direction :158-160
                        if (!fire_at_loc || count > 10) chosen = true;
                        else count++;
                    }
                    if (__all_sync(FULL, chosen)) break;
                }
            } else {
                // one Philox block serves 4 consecutive steps of an episode
                if ((a.t & 3u) == 0u || ablk_ep != a.episode || ablk_idx != (a.t >> 2)) {
                    philox4x32_10((uint32_t)(c.env_id_base + env), a.episode, a.t >> 2, kStreamAction, c.key0, c.key1, ablk);
                    ablk_ep = a.episode;
                    ablk_idx = a.t >> 2;
                }
                const uint32_t aw = (a.t & 3u) == 0u ? ablk[0] : (a.t & 3u) == 1u ? ablk[1] : (a.t & 3u) == 2u ? ablk[2] : ablk[3];
                const uint32_t na = (uint32_t)c.n_actions;
                action = (na & (na - 1u)) == 0u ? (int)(aw & (na - 1u)) : (int)(aw % na);
            }
            if (io.actions_out != nullptr && valid_env && x == 0) io.actions_out[(size_t)k * s.N + env] = action;
            // ---- action: Agent.move :141-155 / toggle_digging :136-138 (agents[0] exists while alive)
            {
                const bool mv = act && a.alive && action >= 0 && action < 4;
                const int nx = a.ax + (action == 2 ? 1 : action == 3 ? -1 : 0);
                const int ny = a.ay + (action == 1 ? 1 : action == 0 ? -1 : 0);
                const bool inb = nx >= 0 && nx < W && ny >= 0 && ny < H;
                const int src_lane = sub * L + (inb ? nx : 0);
                const uint32_t wrow = __shfl_sync(FULL, r.WT, src_lane);
                const uint32_t frow = __shfl_sync(FULL, r.F, src_lane);
                bool do_dig = false;  // Agent.dig (environment.py:123-133) on cell (dgx, dgy) this step
                int dgx = 0, dgy = 0;
                if (mv) {
                    a.vis = 0;  // agent_pos cleared before the validity test (Q1)
                    if (inb && !((wrow >> ny) & 1u)) {
                        a.ax = nx; a.ay = ny; a.vis = 1;
                        const bool onfire = (frow >> ny) & 1u;
                        if (a.digging && !onfire) { do_dig = true; dgx = nx; dgy = ny; }
                        if (onfire) a.dead = 1;
                    }
                }
                if (act && a.alive && c.allow_dig_toggle && action == 4) {
                    a.digging ^= 1;
                    if (a.digging) { do_dig = true; dgx = a.ax; dgy = a.ay; }
                }
                // The reach mask (cells with a finite path to a finite border point: what the A* searches of get_reward
                // establish) is kept across steps.  A dug cell simply leaves it when its free 4-neighbours stay connected
                // through the ring of the 8 cells around it ("simple point"); only otherwise is it flooded again.
                if (__any_sync(FULL, do_dig && reach_ok)) {
                    const uint32_t free_now = ~r.I & validmask;
                    const int base = sub * L;
                    const uint32_t f0 = __shfl_sync(FULL, free_now, base + dgx);
                    uint32_t fm = __shfl_sync(FULL, free_now, base + max(dgx - 1, 0));
                    uint32_t fp = __shfl_sync(FULL, free_now, base + min(dgx + 1, L - 1));
                    const uint32_t rr = __shfl_sync(FULL, reach, base + dgx);
                    if (do_dig && reach_ok && ((f0 >> dgy) & 1u) && ((rr >> dgy) & 1u)) {
                        if (dgx == 0) fm = 0u;
                        if (dgx + 1 >= W) fp = 0u;
                        if (x == dgx) reach &= ~(1u << dgy);
                        // ring of the 8 neighbours, clockwise from N: N NE E SE S SW W NW (N = y - 1, E = x + 1).  Bit y - 1 of a
                        // row is bit y of (row << 1), bit y + 1 is bit y of (row >> 1); rows are zero outside the grid.
                        auto at = [&](uint32_t v) -> uint32_t { return (v >> dgy) & 1u; };
                        const uint32_t ring = at(f0 << 1) | at(fp << 1) << 1 | at(fp) << 2 | at(fp >> 1) << 3 | at(f0 >> 1) << 4 |
                                              at(fm >> 1) << 5 | at(fm) << 6 | at(fm << 1) << 7;
                        const uint32_t rot1 = ((ring << 1) | (ring >> 7)) & 255u, rot2 = ((ring << 2) | (ring >> 6)) & 255u;
                        const int n4 = __popc(ring & 0x55u);
                        int groups = n4 - __popc(ring & rot1 & rot2 & 0x55u);  // a 4-neighbour joined to the previous one through the corner
                        if (n4 == 4 && groups == 0) groups = 1;
                        const bool on_seed = dgx == 0 || dgx == H - 1 || dgy == 0 || dgy == H - 1;  // a literal border point
                        if (on_seed ? n4 > 0 : groups > 1) reach_ok = false;
                    }
                }
                if (do_dig) dig(r, x, dgx, dgy);
            }
            // ---- fire tick: ForestFire.update, forest_fire.py:85-106 (every a_speed steps)
            it -= 1;
            const bool do_tick = (it == 0);
            if (do_tick) it = c.a_speed;
            uint32_t ign_edge = 0u;
            if (do_tick) {
                // Agent.is_dead :116-120 -- dead flag or standing on a type==fire cell
                const uint32_t frow = __shfl_sync(FULL, r.F, sub * L + a.ax);
                if (act && a.alive && (a.dead || ((frow >> a.ay) & 1u))) {
                    a.vis = 0;
                    a.alive = 0;
                    if (x == 0) atomicAdd(&s.stats[ST_DEATHS], 1ull);
                }
                const uint32_t Bt = act ? r.B : 0u;  // burning set as of tick start (:90)
                // reduce_fuel :297-307 on every burning cell: bit-sliced decrement with borrow
                uint32_t borrow = Bt;
#pragma unroll
                for (int q = 0; q < FB; ++q) {
                    const uint32_t f = r.FU[q];
                    r.FU[q] = f ^ borrow;
                    borrow &= ~f;
                }
                uint32_t nz = 0u;
#pragma unroll
                for (int q = 0; q < FB; ++q) {
                    r.FU[q] &= ~borrow;  // fuel was already 0: stays 0 (<= 0 -> burnt)
                    nz |= r.FU[q];
                }
                const uint32_t out = Bt & ~nz;  // burnt out this tick
                const uint32_t src = Bt & nz;   // still burning: heats its neighbours
                r.BT |= out;
                r.F &= ~out; r.D &= ~out; r.WT &= ~out; r.G &= ~out;
                r.B &= ~out;
                // get_neighbours :311-326 (radius 1) + apply_heat_from_to :278-294
                uint32_t up = __shfl_up_sync(FULL, src, 1, L);
                uint32_t dn = __shfl_down_sync(FULL, src, 1, L);
                if (x == 0) up = 0u;
                if (x == L - 1) dn = 0u;
                const uint32_t h0 = r.G & (src >> 1);  // d = N (0,-1): source at y+1
                const uint32_t h1 = r.G & (src << 1);  // d = S (0,+1): source at y-1
                const uint32_t h2 = r.G & up;          // d = E (+1,0): source at x-1
                const uint32_t h3 = r.G & dn;          // d = W (-1,0): source at x+1
                uint32_t m = h0 | h1 | h2 | h3, ign = 0u;
                if (UNI) {
                    // hits this tick, per cell: h0 + h1 + h2 + h3 as a 3-bit number (s2 s1 s0) ...
                    const uint32_t x01 = h0 ^ h1, s0 = x01 ^ h2 ^ h3;
                    const uint32_t c01 = h0 & h1, c23 = h2 & h3, cx = x01 & (h2 ^ h3);
                    const uint32_t s1 = c01 ^ c23 ^ cx, s2 = c01 & c23;
                    // ... added to the 7-bit counter (ripple carry) ...
                    uint32_t k = r.HC[0] & s0;
                    r.HC[0] ^= s0;
                    uint32_t t1 = r.HC[1];
                    r.HC[1] = t1 ^ s1 ^ k;
                    k = (t1 & s1) | (k & (t1 ^ s1));
                    t1 = r.HC[2];
                    r.HC[2] = t1 ^ s2 ^ k;
                    k = (t1 & s2) | (k & (t1 ^ s2));
#pragma unroll
                    for (int q = 3; q < kHitBits; ++q) {
                        t1 = r.HC[q];
                        r.HC[q] = t1 ^ k;
                        k &= t1;
                    }
                    // ... and compared with kmin: count >= kmin  <=>  count + (2^7 - kmin) carries out of bit 6; the carry
                    // chain of adding a constant is one majority (a single LOP3) per bit-slice
                    const uint32_t addc = (uint32_t)(1 << kHitBits) - (uint32_t)min(a.kmin, (1 << kHitBits) - 1);
                    uint32_t carry = 0u;
#pragma unroll
                    for (int q = 0; q < kHitBits; ++q) {
                        const uint32_t cb = 0u - ((addc >> q) & 1u);
                        carry = (r.HC[q] & cb) | (carry & (r.HC[q] | cb));
                    }
                    ign = m & carry;  // only cells heated this tick can cross the threshold
                    m = 0u;
                }
                uint32_t* hrow = s.hits + ((size_t)(valid_env ? env : 0) * W + x) * H;
                while (m) {
                    const int y = __ffs(m) - 1;
                    m &= m - 1u;
                    const uint32_t v = hrow[y] + (((h0 >> y) & 1u) | (((h1 >> y) & 1u) << 8) |
                                                  (((h2 >> y) & 1u) << 16) | (((h3 >> y) & 1u) << 24));
                    hrow[y] = v;
                    const bool ig = a.kmin >= 0 ? (int)__dp4a(v, 0x01010101u, 0u) >= a.kmin
                                                : ignites(v, s.wind, a.wid, c.threshold);
                    if (ig) ign |= 1u << y;
                }
                r.G &= ~ign;  // set_fire_to :233-246
                r.F |= ign;
                r.B |= ign;
                ign_edge = ign & edgemask;
            }
            __syncwarp();
            const uint32_t any_edge = group_bits(__ballot_sync(FULL, ign_edge != 0u));
            const uint32_t anyB = group_bits(__ballot_sync(FULL, r.B != 0u));
            if (do_tick && act) {
                if (any_edge) a.fab = 1;
                if (!a.alive || !anyB) a.running = 0;  // :105-106
            }
            // ---- World.get_reward, environment.py:342-390
            const bool check = act && !a.fab && !a.latched && anyB;
            bool contained = false;
            if (__any_sync(FULL, check)) {
                const uint32_t free_ = ~r.I & validmask;
                const uint32_t seeds = free_ & seedmask;  // finite border points: the goals of the A* searches
                auto flood = [&](uint32_t reach) -> uint32_t {  // cells with a finite-cost 4-connected path to a source
                    for (;;) {
                        uint32_t n = hfill(reach, free_);
                        uint32_t u = __shfl_up_sync(FULL, n, 1, L), d = __shfl_down_sync(FULL, n, 1, L);
                        if (x == 0) u = 0u;
                        if (x == L - 1) d = 0u;
                        n |= (u | d) & free_;
                        const bool changed = (n != reach);
                        reach = n;
                        if (!__any_sync(FULL, changed)) return reach;
                    }
                };
                auto neighbours = [&](uint32_t m) -> uint32_t {
                    uint32_t u = __shfl_up_sync(FULL, m, 1, L), d = __shfl_down_sync(FULL, m, 1, L);
                    if (x == 0) u = 0u;
                    if (x == L - 1) d = 0u;
                    return (m << 1) | (m >> 1) | u | d;
                };
                // A* ignores the start cell's own cost (astar.cpp:89-90, Q5) and astar_path returns an EMPTY path when
                // start == goal (pyastar.py:53-62): a burning cell reaches the border iff one of its 4 NEIGHBOURS is a
                // finite border point or connected to one -- where a burning border point does not count for ITSELF.
                // Burning border points exist off the rim only (W > H maps: the literal [HEIGHT-1, y] column, else
                // fire_at_border has switched the search off), so the second flood is normally skipped.
                uint32_t touch;
                if (__any_sync(FULL, check && (seeds & r.B) != 0u)) {  // (`check`: the warp's other env may burn at its rim)
                    const uint32_t from_cold = flood(seeds & ~r.B);
                    touch = r.B & neighbours(from_cold | seeds);
                    const uint32_t from_burning = flood(seeds & r.B);
                    // (two burning border points joined only through unburnt cells, with no other burning cell and no
                    //  cold border point in their pocket, would still count as contained here: not reproduced)
                    touch |= r.B & ~seedmask & neighbours(from_burning);
                } else {
                    // the usual case: no border point burns, so the search goals are all finite border points and the
                    // region connected to them is the persistent reach mask (flooded when it is not valid)
                    if (__any_sync(FULL, check && !reach_ok)) {
                        reach = flood(seeds);
                        reach_ok = true;
                    }
                    touch = r.B & neighbours(reach);
                }
                contained = !group_bits(__ballot_sync(FULL, touch != 0u));
            }
            double rew = 0.0;
            uint32_t rkind = RK_ZERO, rcnt = 0u;  // SRV: the reward as a code (the host evaluates the same expressions)
            if (act) {
                if (check && contained) {
                    a.latched = 1;  // border_points left empty: bonus is paid once (Q4)
                    rew = c.contained_bonus;
                    rkind = RK_CONTAINED;
                    if (x == 0) atomicAdd(&s.stats[ST_CONTAINED], 1ull);
                } else if (!a.alive) {
                    rew = c.death_penalty;
                    rkind = RK_DEATH;
                } else if (!anyB) {
                    rew = 1.0;  // placeholder: burn-out fraction computed below
                    rkind = RK_BURNOUT;
                } else {
                    rew = c.default_reward;
                    rkind = RK_DEFAULT;
                }
            }
            const bool burnout = act && !(check && contained) && a.alive && !anyB;
            if (__any_sync(FULL, burnout)) {  // np.count_nonzero(type == grass) / (W * H), :385-387
                int cnt = __popc(r.G);
#pragma unroll
                for (int o = L / 2; o > 0; o >>= 1) cnt += __shfl_xor_sync(FULL, cnt, o, L);
                if (burnout) rew = __dmul_rn(c.contained_bonus, __ddiv_rn((double)cnt, (double)(W * H)));
                if (burnout) rcnt = (uint32_t)cnt;
            }
            const bool done = valid_env && !a.running;
            if (act) {
                a.t += 1u;
                n_steps_done += 1;
                n_ticks_done += do_tick ? 1 : 0;
                if (done && x == 0) {
                    atomicAdd(&s.stats[ST_EPISODES], 1ull);
                    if (a.alive) atomicAdd(&s.stats[ST_BURNOUTS], 1ull);
                }
            }
            if (valid_env && x == 0) {
                if (io.reward != nullptr) io.reward[(size_t)k * s.N + env] = rew;
                if (io.done != nullptr) io.done[(size_t)k * s.N + env] = done ? 1 : 0;
            }
            if constexpr (FIN) {
                // ---- final-state capture, then the auto-reset and the next episode's start cell in the record
                uint32_t* fin_rec = nullptr;
                if (__any_sync(FULL, act && done))
                    fin_rec = capture_final<L, FB>(r, a, static_cast<const WarpFinIO&>(io).fin, act && done, k, env, lane, sub, x,
                                                   W, H, validmask, stream_warp, spread3);
                if (c.auto_reset && act && done) {
                    reset_rows<L, FB, UNI>(r, a, s, c, nullptr, env, x, validmask);
                    a.refresh_wind(s.wind);
                    reach_ok = false;
                    if (fin_rec != nullptr && x == 0) {
                        fin_rec[WF_F_NEXT_AX] = (uint32_t)a.ax;
                        fin_rec[WF_F_NEXT_AY] = (uint32_t)a.ay;
                    }
                }
            } else if (c.auto_reset && act && done) {
                // ---- auto-reset (batched-env convention: the returned obs is the new episode's first)
                reset_rows<L, FB, UNI>(r, a, s, c, nullptr, env, x, validmask);
                a.refresh_wind(s.wind);
                reach_ok = false;
            }
            __syncwarp();
            if (SRV && srv.delta) {
                // ---- persistent observation array: send what changed since the last step this warp sent
                const uint32_t cA = (a.vis && x == a.ax) ? (1u << a.ay) : 0u, cF = r.F, cFree = ~r.I & validmask;
                uint32_t dA = cA ^ pA, dF = cF ^ pF, dFree = cFree ^ pFree;
                pA = cA; pF = cF; pFree = cFree;
                const bool want_full = srv_step == 0u || srv_want_full != 0;
                // this warp's list: status word, count, then its entries (16-bit units from index 4); the CTA merges the four
                uint32_t* const cw = srv_block + kDeltaBlockWords + warp * 12;
                int total = want_full ? kDeltaEntries + 1 : 0;
                while (total <= kDeltaEntries) {
                    const bool has = (dA | dF | dFree) != 0u;
                    const uint32_t pend = __ballot_sync(FULL, has);
                    if (pend == 0u) break;
                    if (has) {
                        const int ch = dA ? 0 : dF ? 1 : 2;
                        const uint32_t m = dA ? dA : dF ? dF : dFree;
                        const uint32_t now = dA ? cA : dF ? cF : cFree;
                        const uint32_t low = m & (0u - m);
                        const int y = __ffs(m) - 1;
                        if (ch == 0) dA ^= low;
                        else if (ch == 1) dF ^= low;
                        else dFree ^= low;
                        const int slot = total + __popc(pend & ((1u << lane) - 1u));
                        const uint32_t elem = (uint32_t)(sub * (W * H * 3) + (x * H + y) * 3 + ch);
                        if (slot < kDeltaEntries)
                            reinterpret_cast<uint16_t*>(cw)[4 + slot] = (uint16_t)((elem << 1) | ((now & low) ? 1u : 0u));
                    }
                    total += __popc(pend);
                }
                const bool full = total > kDeltaEntries;  // warp-uniform
                {
                    const uint32_t status16 = rkind | (done ? 8u : 0u) | (rcnt << 4);
                    uint32_t st = __shfl_sync(FULL, status16, 0);
                    if (EPW == 2) st |= __shfl_sync(FULL, status16, L & 31) << 16;
                    if (lane == 0) {
                        cw[0] = st | (full ? kDeltaFullBit : 0u);
                        cw[1] = (full || n_valid <= 0) ? 0u : (uint32_t)total;
                    }
                }
                if (full && n_valid > 0) {  // the whole stream, as aligned 16-byte stores straight into the host's full area
                    // (emit_obs leaves the stream in stream_warp; the copy it makes into the warp's slot of the CTA's block
                    //  -- behind the change-list records -- is not used)
                    emit_obs<L, true>(srv_block + kDeltaBlockWords + 48 + warp * (((EPW * W * H * 3 + 31) >> 5) + 1), kObsPackedStatus,
                                      cA, cF, cFree, stream_warp, spread3, tab8, lane, sub, x, W, H, env0, n_valid, 0u);
                    __syncwarp();
                    const int n4 = (((EPW * W * H * 3 + 31) >> 5) + 3) >> 2;
                    uint4* dst = reinterpret_cast<uint4*>(srv.full_area + (size_t)(env0 / EPW) * srv.full_stride);
                    if (lane < n4) dst[lane] = reinterpret_cast<const uint4*>(stream_warp)[lane];
                }
            } else if (io.obs != nullptr) {
                const size_t step_bytes =
                    io.obs_dtype == kObsPacked ? (size_t)((s.N + EPW - 1) / EPW) * ((EPW * W * H * 3 + 31) >> 5) * 4
                    : OB ? obs_step_bytes(s.N, W, H, WF_OBS_BITS) : (size_t)s.N * W * H * 3 * obs_elem_bytes(io.obs_dtype);
                const int srv_stride = ((EPW * W * H * 3 + 31) >> 5) + 1;  // words per record incl. the status word
                emit_obs<L, SRV, OB>(SRV ? static_cast<void*>(srv_block + warp * srv_stride) : static_cast<char*>(io.obs) + (size_t)k * step_bytes,
                                 io.obs_dtype, (a.vis && x == a.ax) ? (1u << a.ay) : 0u, r.F, ~r.I & validmask, stream_warp, spread3, tab8,
                                 lane, sub, x, W, H, env0, n_valid, SRV ? (rkind | (done ? 8u : 0u) | (rcnt << 4)) : 0u);
            }
            if (SRV) {
                unsigned long long srv_t2 = 0ull, srv_t2b = 0ull;
                if (blockIdx.x == 0 && threadIdx.x == 0) srv_t2 = global_timer_ns();
                __syncthreads();  // the CTA's records are complete in shared memory
                const int srv_stride = ((EPW * W * H * 3 + 31) >> 5) + 1;
                if (srv.sectors) {
                    // self-validating sectors: output word 8 * sec + slot of the CTA's block = payload word 7 * (sec % nsec) + slot
                    // of record sec / nsec, slot 7 = step's sequence number ^ hash of the sector's seven payload words
                    const int nsec = (srv_stride + kSectorPayload - 1) / kSectorPayload;
                    const uint32_t seq = srv.seq0 + srv_step + 1u;
                    uint4* dst = reinterpret_cast<uint4*>(static_cast<uint32_t*>(io.obs) + (size_t)blockIdx.x * (kWarpsPerBlock * nsec * 8));
                    for (int j = threadIdx.x; j < kWarpsPerBlock * nsec * 2; j += blockDim.x) {
                        const int sec = j >> 1, rec = sec / nsec, p0 = (sec - rec * nsec) * kSectorPayload;
                        const uint32_t* rw = srv_block + rec * srv_stride;
                        uint32_t w[kSectorPayload];
#pragma unroll
                        for (int i = 0; i < kSectorPayload; ++i) w[i] = p0 + i < srv_stride ? rw[p0 + i] : 0u;
                        dst[j] = (j & 1) ? make_uint4(w[4], w[5], w[6], seq ^ sector_hash(w)) : make_uint4(w[0], w[1], w[2], w[3]);
                    }
                } else if (srv.delta) {
                    // merge the four warps' lists into the CTA's block: header, status words, entries back to back
                    const uint32_t* pw = srv_block + kDeltaBlockWords;
                    const int t = threadIdx.x;
                    const int c0 = (int)pw[1], c1 = c0 + (int)pw[13], c2 = c1 + (int)pw[25], c3 = c2 + (int)pw[37];
                    if (t == 0) {
                        const uint32_t fullmask = ((pw[0] >> 15) & 1u) | (((pw[12] >> 15) & 1u) << 1) | (((pw[24] >> 15) & 1u) << 2) |
                                                  (((pw[36] >> 15) & 1u) << 3);
                        srv_block[0] = (uint32_t)c3 | (fullmask << 8);
                    } else if (t < 5) {
                        srv_block[t] = pw[(t - 1) * 12];
                    }
                    if (t < kWarpsPerBlock * kDeltaEntries) {
                        const int w = (t >= c0) + (t >= c1) + (t >= c2);
                        const int first = w == 0 ? 0 : w == 1 ? c0 : w == 2 ? c1 : c2;
                        uint32_t e = 0xffffu;
                        if (t < c3) e = (uint32_t)reinterpret_cast<const uint16_t*>(pw + w * 12)[4 + t - first] + (uint32_t)(w * EPW * W * H * 3) * 2u;
                        reinterpret_cast<uint16_t*>(srv_block)[kDeltaFirstEntry + t] = (uint16_t)e;
                    }
                    __syncthreads();
                    uint4* dst = reinterpret_cast<uint4*>(static_cast<uint32_t*>(io.obs) + (size_t)blockIdx.x * kDeltaBlockWords);
                    if (t < kDeltaBlockWords / 4) dst[t] = reinterpret_cast<const uint4*>(srv_block)[t];
                } else {
                    const int block_words = (kWarpsPerBlock * srv_stride + 31) & ~31;  // whole 128-byte lines
                    uint4* dst = reinterpret_cast<uint4*>(static_cast<uint32_t*>(io.obs) + (size_t)blockIdx.x * block_words);
                    const uint4* src = reinterpret_cast<const uint4*>(srv_block);
                    for (int j = threadIdx.x; j < (block_words >> 2); j += blockDim.x) dst[j] = src[j];
                }
                __syncthreads();  // every thread of the CTA has issued its stores to mapped host memory ...
                if (blockIdx.x == 0 && threadIdx.x == 0) srv_t2b = global_timer_ns();
                srv_step += 1u;
                if (threadIdx.x == 0 && srv.sectors) {
                    if (blockIdx.x == 0 && srv.dbg != nullptr) {
                        srv.dbg[0] += srv_t0b - srv_t0;
                        srv.dbg[7] += srv_t1 - srv_t0b;
                        srv.dbg[1] += srv_t2 - srv_t1;
                        srv.dbg[2] += srv_t2b - srv_t2;
                        srv.dbg[3] += 1ull;
                    }
                } else if (threadIdx.x == 0) {
                    // ... and are ordered before this CTA's arrival at GPU scope.  System-scope fences are expensive (each
                    // one drains the GPU's writes to host memory: ~100 us per step when all 512 CTAs issued one), so only
                    // the LAST CTA of a slice issues one -- it is cumulative over the stores it has observed through the
                    // arrival counter -- before it raises the slice's flag.
                    __threadfence();
                    const uint32_t slice = blockIdx.x / (uint32_t)srv.ctas_per_slice;
                    const uint32_t n_in = min((uint32_t)srv.ctas_per_slice, gridDim.x - slice * (uint32_t)srv.ctas_per_slice);
                    const uint32_t old = atomicAdd(&srv.count[slice], 1u);
                    if (old + 1u == n_in * srv_step) {  // the slice's last CTA of this step
                        const unsigned long long tf = global_timer_ns();
                        __threadfence_system();
                        srv.done[slice * 16u] = srv.seq0 + srv_step;
                        if (srv.dbg != nullptr) {
                            atomicAdd(&srv.dbg[5], global_timer_ns() - tf);
                            atomicAdd(&srv.dbg[6], 1ull);
                        }
                    }
                    if (blockIdx.x == 0 && srv.dbg != nullptr) {
                        const unsigned long long t3 = global_timer_ns();
                        srv.dbg[0] += srv_t0b - srv_t0;
                        srv.dbg[7] += srv_t1 - srv_t0b;
                        srv.dbg[1] += srv_t2 - srv_t1;
                        srv.dbg[2] += srv_t2b - srv_t2;
                        srv.dbg[4] += t3 - srv_t2b;
                        srv.dbg[3] += 1ull;
                    }
                }
            }
        }
    }

    // ---------------- store ----------------
    {
        int nb = __popc(r.B);
#pragma unroll
        for (int o = L / 2; o > 0; o >>= 1) nb += __shfl_xor_sync(FULL, nb, o, L);
        a.nburn = nb;
    }
    if (valid_env) {
#pragma unroll
        for (int p = 0; p < 7 + FB + (UNI ? kHitBits : 0); ++p) s.planes[word_index(s, p, env, x, 0)] = r.get(p);
        if (x == 0) {
            int4* sp = reinterpret_cast<int4*>(s.scal + (size_t)env * WF_NSCALARS);
            sp[0] = make_int4(a.alive, a.ax, a.ay, a.dead);
            sp[1] = make_int4(a.digging, a.vis, a.running, a.fab);
            sp[2] = make_int4(a.latched, (int)a.episode, (int)a.t, a.wid);
            sp[3] = make_int4(s.wind->wx[a.wid], s.wind->wy[a.wid], a.nburn, 0);
        }
    }
    // Step / tick counters: summed over the CTA in shared memory, one pair of global atomics per CTA (one pair per ENV was
    // 8192 atomics on two addresses per launch -- microseconds of a one-step launch).
    if (valid_env && x == 0) {
        if (n_steps_done) atomicAdd(&cta_stats[0], (unsigned long long)n_steps_done);
        if (n_ticks_done) atomicAdd(&cta_stats[1], (unsigned long long)n_ticks_done);
    }
    __syncthreads();
    if (threadIdx.x < 2 && cta_stats[threadIdx.x]) atomicAdd(&s.stats[threadIdx.x == 0 ? ST_STEPS : ST_TICKS], cta_stats[threadIdx.x]);
}

// The C2 kernel must stay at 128 registers (16 warps per SM: all 2048 warps of a 4096-env batch resident; at 164
// registers a step costs 3.3 instead of 2.3 us).  ptxas lands there by itself and schedules better that way than under an
// explicit cap (__launch_bounds__(128, 4): 115 registers, 2.52 us per step; A/B on one box, tools/build_variant.sh
// -DWF_WARP_MINBLOCKS); the build checks the register count (csrc/Makefile, `make check-regs`).
// OB: WF_OBS_BITS observations -- a separate instantiation, because any extra code in the observation path of the C2 kernel
// moves ptxas's schedule (with the bits path behind a run-time test the uint8 step took 2.15 instead of 1.97 us, same box).
template <int L, int FB, bool UNI, bool MLP, bool OB>
#ifdef WF_WARP_MINBLOCKS
__global__ void __launch_bounds__(kWarpsPerBlock * 32, (MLP && !UNI) ? 8 / kWarpsPerBlock : 16 / kWarpsPerBlock)
#else
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
#endif
warp_kernel(DevState s, StepCfg c, WarpIO io) {
    warp_body<L, FB, UNI, MLP, false, OB>(s, c, io, SrvCtl{});
}
// The same with final-state capture (wf_set_final_capture): a kernel of its own, so that warp_kernel keeps its code.
template <int L, int FB, bool UNI, bool MLP, bool OB>
__global__ void __launch_bounds__(kWarpsPerBlock * 32) warp_fin_kernel(DevState s, StepCfg c, WarpFinIO io) {
    warp_body<L, FB, UNI, MLP, false, OB, true>(s, c, io, SrvCtl{});
}
// The step server must be resident as a whole (cooperative launch): 128 registers at most.
template <int L, int FB, bool UNI>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, 16 / kWarpsPerBlock) warp_server_kernel(DevState s, StepCfg c, WarpIO io, SrvCtl srv) {
    warp_body<L, FB, UNI, false, true, false>(s, c, io, srv);
}

// ---------------------------------------------------------------------------------------------
// host launcher (called from wf_api.cu)
cudaError_t launch_warp_family(const DevState& s, const StepCfg& c, const WarpIO& io, cudaStream_t stream, const FinalCapture* fin) {
    const int L = s.RS;
    const int epw = 32 / L;
    const int envs_per_block = kWarpsPerBlock * epw;
    const dim3 grid((s.N + envs_per_block - 1) / envs_per_block), block(kWarpsPerBlock * 32);
    if (s.HB != 0 && (s.HB != kHitBits || s.FB != 5)) return cudaErrorInvalidValue;
    const bool mlp = io.policy == WF_POLICY_MLP && io.actions == nullptr && !io.reset_mode;
    if (mlp && (io.mlp.hid < 1 || io.mlp.hid > kHidMax || io.mlp.n_actions > kActMax || io.mlp.group_envs < 1 ||
                io.mlp.group_envs % envs_per_block != 0))
        return cudaErrorInvalidValue;
    const bool ob = io.obs != nullptr && io.obs_dtype == WF_OBS_BITS;
    const bool capture = fin != nullptr && fin->records != nullptr && !io.reset_mode;
    WarpFinIO fio;
    static_cast<WarpIO&>(fio) = io;
    if (capture) fio.fin = *fin;
#define WF_LAUNCH(LL, FF, UU, MM)                                                                         \
    do {                                                                                                  \
        if (capture) {                                                                                    \
            if (ob) warp_fin_kernel<LL, FF, UU, MM, true><<<grid, block, 0, stream>>>(s, c, fio);         \
            else warp_fin_kernel<LL, FF, UU, MM, false><<<grid, block, 0, stream>>>(s, c, fio);           \
        } else if (ob) warp_kernel<LL, FF, UU, MM, true><<<grid, block, 0, stream>>>(s, c, io);           \
        else warp_kernel<LL, FF, UU, MM, false><<<grid, block, 0, stream>>>(s, c, io);                    \
    } while (0)
    if (mlp) {
        if (L == 16 && s.FB == 5 && s.HB) WF_LAUNCH(16, 5, true, true);
        else if (L == 32 && s.FB == 5 && s.HB) WF_LAUNCH(32, 5, true, true);
        else if (L == 16 && s.FB == 5) WF_LAUNCH(16, 5, false, true);
        else if (L == 16 && s.FB == 8) WF_LAUNCH(16, 8, false, true);
        else if (L == 32 && s.FB == 5) WF_LAUNCH(32, 5, false, true);
        else if (L == 32 && s.FB == 8) WF_LAUNCH(32, 8, false, true);
        else return cudaErrorInvalidValue;
    } else if (L == 16 && s.FB == 5 && s.HB) WF_LAUNCH(16, 5, true, false);
    else if (L == 32 && s.FB == 5 && s.HB) WF_LAUNCH(32, 5, true, false);
    else if (L == 16 && s.FB == 5) WF_LAUNCH(16, 5, false, false);
    else if (L == 16 && s.FB == 8) WF_LAUNCH(16, 8, false, false);
    else if (L == 32 && s.FB == 5) WF_LAUNCH(32, 5, false, false);
    else if (L == 32 && s.FB == 8) WF_LAUNCH(32, 8, false, false);
    else return cudaErrorInvalidValue;
#undef WF_LAUNCH
    return cudaGetLastError();
}

// The step server: the same kernel, launched cooperatively (all CTAs resident, or the launch fails).
cudaError_t launch_warp_server(const DevState& s, const StepCfg& c, const WarpIO& io, const SrvCtl& srv, cudaStream_t stream) {
    const int L = s.RS;
    const int epw = 32 / L;
    const int envs_per_block = kWarpsPerBlock * epw;
    const dim3 grid((s.N + envs_per_block - 1) / envs_per_block), block(kWarpsPerBlock * 32);
    if (s.HB != 0 && (s.HB != kHitBits || s.FB != 5)) return cudaErrorInvalidValue;
    const void* fn = nullptr;
    if (L == 16 && s.FB == 5 && s.HB) fn = (const void*)warp_server_kernel<16, 5, true>;
    else if (L == 32 && s.FB == 5 && s.HB) fn = (const void*)warp_server_kernel<32, 5, true>;
    else if (L == 16 && s.FB == 5) fn = (const void*)warp_server_kernel<16, 5, false>;
    else if (L == 16 && s.FB == 8) fn = (const void*)warp_server_kernel<16, 8, false>;
    else if (L == 32 && s.FB == 5) fn = (const void*)warp_server_kernel<32, 5, false>;
    else if (L == 32 && s.FB == 8) fn = (const void*)warp_server_kernel<32, 8, false>;
    else return cudaErrorInvalidValue;
    void* args[4] = {const_cast<DevState*>(&s), const_cast<StepCfg*>(&c), const_cast<WarpIO*>(&io), const_cast<SrvCtl*>(&srv)};
    return cudaLaunchCooperativeKernel(fn, grid, block, args, 0, stream);
}

}  // namespace wf
