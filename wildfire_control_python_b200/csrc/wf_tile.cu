// wf_tile.cu -- "tile" kernel family: grids wider or taller than 32 cells (256x256, 1024x1024 ...).
//
// Same bit-plane state as the warp family (wf_common.cuh) but resident in HBM: a row x of H cells is
// HW = ceil(H/32) words.  ONE thread-block cluster (1..8 CTAs, chosen so that all envs together fill
// the 148 SMs; 16 with the non-portable opt-in) owns one environment for a whole K-step rollout;
// CTA r of the cluster owns the r-th contiguous slice of the env's words.  Everything the reference
// does in ForestFire.step happens in this one kernel, per step:
//
//   agent phase   thread 0 of every CTA (redundantly, from identical inputs): action, Agent.move /
//                 toggle_digging / is_dead (environment.py:116-171), local articulation test for the
//                 reach plane.  Reads only; the dig is applied by the thread that owns the word.
//                 (Runs while the other warps still emit the previous step's observation.)
//   barrier X     (cluster)  nobody writes a plane before everybody has read the agent's surroundings
//   tick          every warp on its own: stream G, B and the heat-source mask S (1 bit/cell: burning and
//                 fuel >= 2) of 128 words; words that burn or are heated are compacted into the warp's
//                 queue in shared memory and handed one per lane to the active path (fuel planes, hit
//                 counters, ignition, burn-out -- forest_fire.py:85-106, environment.py:278-307); S is
//                 ping-ponged (parity bit per env) so the in-place update of every other plane is
//                 race-free across warps and CTAs.
//   barrier Y     (cluster)  per-env reductions exchanged through distributed shared memory
//   finish        RUNNING, World.get_reward (environment.py:342-390: containment = no burning cell next
//                 to the border-connected reach plane R), done, statistics; auto-reset
//   observation   World.get_state (environment.py:399-402): 2 plane words in, 96 bytes out per word
//
// WF_POLICY_MLP (the MLP instantiations) adds a policy pass after every step and before step 0: the Q-network's first
// layer over the observation the step left (mlp_action), summed exactly in int64 fixed point, exchanged through DSMEM;
// the agent phase of the next step then runs after it instead of during the observation.
//
// The A* containment search (pyastar/astar.cpp) is the persistent reach plane R (cells with a finite
// 4-connected path to a finite border point), re-flooded by the cluster only when a dig may disconnect
// it; burning cells that are border points themselves (W > H maps) get a scratch flood (seed_cells_touch).
#include <cstdio>
#include <cstdlib>

#include "wf_families.cuh"

#include <type_traits>

namespace wf {

struct TileState {
    int32_t P_S0, P_S1, P_R;
    int32_t T, CS;  // threads per CTA, CTAs per cluster (one cluster per env)
};

struct TilePar {  // launch constants, precomputed on the host so the kernel re-reads them from the constant bank
    int32_t P_S0, P_S1, P_R, hw_shift;
    uint32_t hw_magic;   // ceil(2^32 / HW): row = umulhi(word, hw_magic) when HW is not a power of two
    int32_t wpc;         // words of an env owned by one CTA (multiple of 32)
    int32_t T;           // threads per CTA
    int32_t nwords;      // W * HW
    int32_t cells;       // W * H
    size_t pstride;      // words between consecutive planes (N * RS * HW)
    size_t env_words;    // words between consecutive envs within a plane (RS * HW)
    size_t step_bytes;   // bytes of one step's observation block [N][W][H][3]
};

// Block-wide scratch of the env a CTA is working on (every CTA of the cluster holds the same values).
struct StepShared {
    int32_t act;          // env was running at step start (finished envs are frozen)
    int32_t dig_word;     // word index of the cell dug this step, or -1
    uint32_t dig_bit;
    int32_t dig_clear_R;  // the dug cell leaves the reach plane
    int32_t need_flood;   // ... and may disconnect it: re-flood before the tick
    int32_t tot[8];       // cluster totals: burning cells, grass cells, ignition on edge, burning touches reach,
                          // a burning cell is a border point (W > H maps only); 5..7 unused
    int32_t reset_now;
    int32_t obs_ctr;                  // next 128-word observation group of this CTA (dynamic distribution)
    uint32_t stat[ST_N];  // this launch's contribution to the handle's statistics (flushed once, at the end)
    int32_t obs_agent[2][3];  // agent_pos layer (visible, x, y) after the action of step k, in slot k & 1
    int32_t slow;             // this step's reward needs the whole cluster (seed_cells_touch) before it is known
    int32_t keep[3];          // ... and the step's totals (burning, grass, ignition on edge) kept meanwhile
};

int tile_extra_planes() { return 3; }

constexpr int kRed = 8;  // per-env reductions exchanged per step (power of two; T >= kRed * kMaxCluster)
constexpr int kMaxCluster = 16;  // CTAs per cluster: 8 is the portable limit, 16 needs the non-portable opt-in

// Phase timing of one probe CTA (debug builds only: -DWF_TILE_TIMING; read with wf_debug_tile_timing).
#ifdef WF_TILE_TIMING
__device__ unsigned long long g_tile_timing[16];
#define WF_TSTAMP(slot)                                                      \
    do {                                                                     \
        if (blockIdx.x == gridDim.x / 2 && threadIdx.x == 0) {               \
            unsigned long long _t;                                           \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_t));           \
            g_tile_timing[slot] += _t - t_last;                              \
            t_last = _t;                                                     \
        }                                                                    \
    } while (0)
#else
#define WF_TSTAMP(slot) do { } while (0)
#endif

// ---------------------------------------------------------------------------------------------
// cluster primitives
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_barrier() {  // release/acquire at cluster scope (also orders global memory)
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void st_shared_cluster(int* local_ptr, uint32_t peer, int v) {  // DSMEM store
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(local_ptr);
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(peer));
    asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(ra), "r"(v) : "memory");
}
__device__ __forceinline__ void st_shared_cluster(long long* local_ptr, uint32_t peer, long long v) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(local_ptr);
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(peer));
    asm volatile("st.shared::cluster.s64 [%0], %1;" ::"r"(ra), "l"(v) : "memory");
}
template <bool CL>
__device__ __forceinline__ void sync_env() {
    if (CL) cluster_barrier();
    else __syncthreads();
}

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t valid_word(int H, int w) {
    const int rem = H - 32 * w;
    return rem >= 32 ? 0xffffffffu : (rem <= 0 ? 0u : ((1u << rem) - 1u));
}
// Literal border_points (environment.py:215-222): (x,0) (x,H-1) for all x; (0,y) (H-1,y) for all y.
__device__ __forceinline__ uint32_t seed_word(int W, int H, int x, int w) {
    const uint32_t v = valid_word(H, w);
    if (x == 0 || x == H - 1) return v;
    uint32_t m = 0u;
    if (w == 0) m |= 1u;
    if (w == (H - 1) >> 5) m |= 1u << ((H - 1) & 31);
    return m & v;
}
__device__ __forceinline__ uint32_t edge_word(int W, int H, int x, int w) {
    const uint32_t v = valid_word(H, w);
    if (x == 0 || x == W - 1) return v;
    uint32_t m = 0u;
    if (w == 0) m |= 1u;
    if (w == (H - 1) >> 5) m |= 1u << ((H - 1) & 31);
    return m & v;
}

// Everything a device function needs to address the env this CTA works on.
struct Env {
    uint32_t* P0;    // word 0 of plane 0 of this env
    size_t pstride;  // words between consecutive planes
    uint32_t* hits;  // hit counters of this env
    uint32_t* FU;    // fuel records of this env: kFuelRec words per plane word
    int env, W, H, HW, nwords, hw_shift;
    uint32_t hw_magic;
    int lo, hi;      // this CTA's slice of the env's words
    int rank, CS, tid, T;
    __device__ __forceinline__ uint32_t* plane(int p) const { return P0 + (size_t)p * pstride; }
    __device__ __forceinline__ int row_of(int i) const {
        return hw_shift >= 0 ? (i >> hw_shift) : (int)__umulhi((uint32_t)i, hw_magic);
    }
    __device__ __forceinline__ bool bit(int p, int x, int y) const {
        return (plane(p)[x * HW + (y >> 5)] >> (y & 31)) & 1u;
    }
};

// Sum the CTAs' partial reductions red[0..3] over the cluster into ss.tot[0..3] (and clear red).
// Call with red[] complete (after a __syncthreads); returns with ss.tot visible to the whole CTA.
template <bool CL>
__device__ __forceinline__ void exchange(const Env& e, int* red, int (*xch)[kMaxCluster][kRed], int& par, StepShared& ss) {
    if (CL) {
        if (e.tid < kRed * e.CS) st_shared_cluster(&xch[par][e.rank][e.tid & (kRed - 1)], (uint32_t)(e.tid / kRed), red[e.tid & (kRed - 1)]);
        cluster_barrier();
        if (e.tid < kRed) {
            int v = 0;
            for (int r = 0; r < e.CS; ++r) v += xch[par][r][e.tid];
            ss.tot[e.tid] = v;
            red[e.tid] = 0;
        }
        par ^= 1;
    } else {
        if (e.tid < kRed) {
            ss.tot[e.tid] = red[e.tid];
            red[e.tid] = 0;
        }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// Reach plane: R = finite cells 4-connected to a finite border point (flood from the border over
// ~fm_inf).  Whole cluster; in-place monotone relaxation until a full sweep changes nothing anywhere.
// `plane`: where the result goes (the persistent reach plane, or a scratch plane); `cold_only`: burning border
// points are not sources (see seed_cells_touch).
template <bool CL>
__device__ void flood(const Env& e, const TilePar& t, int* red, int (*xch)[kMaxCluster][kRed], int& par, StepShared& ss,
                      int plane = -1, bool cold_only = false) {
    const int W = e.W, H = e.H, HW = e.HW;
    uint32_t* R = e.plane(plane < 0 ? t.P_R : plane);
    const uint32_t* I = e.plane(P_I);
    const uint32_t* Bp = e.plane(P_B);
    for (int i = e.lo + e.tid; i < e.hi; i += e.T) {
        const int x = e.row_of(i), w = i - x * HW;
        R[i] = seed_word(W, H, x, w) & ~I[i] & (cold_only ? ~Bp[i] : 0xffffffffu);
    }
    sync_env<CL>();
    for (;;) {
        int changed = 0;
        for (int i = e.lo + e.tid; i < e.hi; i += e.T) {
            const int x = e.row_of(i), w = i - x * HW;
            const uint32_t free_ = ~I[i] & valid_word(H, w);
            if (!free_) continue;
            const uint32_t old = R[i];
            uint32_t n = old;
            if (x > 0) n |= R[i - HW];
            if (x < W - 1) n |= R[i + HW];
            if (w > 0) n |= R[i - 1] >> 31;
            if (w < HW - 1) n |= R[i + 1] << 31;
            n = hfill(n & free_, free_);
            if (n != old) {
                R[i] = n;
                changed = 1;
            }
        }
        if (changed) red[0] = 1;
        __syncthreads();
        exchange<CL>(e, red, xch, par, ss);
        if (!ss.tot[0]) break;
    }
}

// ---------------------------------------------------------------------------------------------
// Everything the agent phase needs to know about a cell and its 8 neighbours, fetched with loads
// that do not depend on each other (one memory round trip instead of one per question).
struct Around {
    uint32_t wt, f, d, i, r;  // bits of the cell itself: water, type == fire, dirt, fm_inf, reach
    bool free8[8];            // free (in bounds and finite fire mobility) neighbours N, NE, E, SE, S, SW, W, NW
};
__device__ __forceinline__ Around load_around(const Env& e, const TilePar& t, int x, int y) {
    const int W = e.W, H = e.H, HW = e.HW;
    const int w = y >> 5, b = y & 31, wi = x * HW + w;
    const uint32_t WTw = e.plane(P_WT)[wi], Fw = e.plane(P_F)[wi], Dw = e.plane(P_D)[wi], Rw = e.plane(t.P_R)[wi];
    const uint32_t* I = e.plane(P_I);
    uint32_t rows[3][3];  // fm_inf words [x-1, x, x+1][w-1, w, w+1]; out of bounds reads as blocked
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx)
#pragma unroll
        for (int dw = -1; dw <= 1; ++dw) {
            const int xx = x + dx, ww = w + dw;
            const bool ok = xx >= 0 && xx < W && ww >= 0 && ww < HW && (dw == 0 || (dw < 0 ? b == 0 : b == 31));
            rows[dx + 1][dw + 1] = ok ? I[xx * HW + ww] : 0xffffffffu;
        }
    Around a;
    a.wt = (WTw >> b) & 1u; a.f = (Fw >> b) & 1u; a.d = (Dw >> b) & 1u; a.r = (Rw >> b) & 1u;
    a.i = (rows[1][1] >> b) & 1u;
    auto blocked = [&](int dx, int dy) -> bool {  // fm_inf (or outside the grid) at (x + dx, y + dy)
        const int yy = y + dy;
        if (yy < 0 || yy >= H) return true;
        const int dw = (yy >> 5) - w;
        return (rows[dx + 1][dw + 1] >> (yy & 31)) & 1u;
    };
    const int dx8[8] = {0, 1, 1, 1, 0, -1, -1, -1}, dy8[8] = {-1, -1, 0, 1, 1, 1, 0, -1};  // screen: N = y-1, E = x+1
#pragma unroll
    for (int k = 0; k < 8; ++k) a.free8[k] = !blocked(dx8[k], dy8[k]);
    return a;
}

// Agent.dig (environment.py:123-133), planning half: what the dig changes and whether the reach plane
// survives it.  Thread 0 only, no memory access.  Returns true iff the cell becomes dirt now.
__device__ __forceinline__ bool plan_dig(const Env& e, const Around& a, const int32_t* sc, StepShared& ss, int x, int y) {
    const int H = e.H;
    if (a.d) return false;
    ss.dig_word = x * e.HW + (y >> 5);
    ss.dig_bit = 1u << (y & 31);
    if (a.i) return true;  // the cell already had infinite fire mobility (water is never entered; kept for safety)
    // get_reward only searches for a path while `not fire_at_border and len(border_points)`
    // (environment.py:345): once either latch is set R is never read again in this episode
    // (World.reset re-floods it), so it is not maintained.
    if (sc[WF_S_FIRE_AT_BORDER] || sc[WF_S_LATCHED]) return true;
    if (!a.r) return true;  // the cell had no path to the border: nobody reached the border through it
    ss.dig_clear_R = 1;
    // Does removing this cell possibly disconnect its neighbours from the border?  Its free 4-neighbours
    // were all in R.  If they stay connected to each other through the ring of 8 surrounding cells,
    // every path through the dug cell can be re-routed and R is unchanged elsewhere ("simple point").
    const bool on_seed = (x == 0 || x == H - 1 || y == 0 || y == H - 1);
    int n4 = 0, groups = 0;
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
        if (!a.free8[k]) continue;
        n4++;
        // this 4-neighbour starts a new group unless it is ring-connected to the previous 4-neighbour
        const int pk = (k + 6) & 7, pd = (k + 7) & 7;
        if (!(a.free8[pk] && a.free8[pd])) groups++;
    }
    if (n4 == 4 && groups == 0) groups = 1;  // full ring
    if (on_seed ? n4 > 0 : groups > 1) ss.need_flood = 1;
    return true;
}

// The planned dig, applied to the planes in HBM (by the one thread that owns the word).
__device__ __forceinline__ void apply_dig(const Env& e, const TilePar& t, int wi, uint32_t bit, int clear_R) {
    atomicAnd(&e.plane(P_G)[wi], ~bit);
    atomicAnd(&e.plane(P_F)[wi], ~bit);
    atomicAnd(&e.plane(P_BT)[wi], ~bit);
    atomicAnd(&e.plane(P_WT)[wi], ~bit);
    atomicOr(&e.plane(P_D)[wi], bit);
    atomicOr(&e.plane(P_I)[wi], bit);
    if (clear_R) atomicAnd(&e.plane(t.P_R)[wi], ~bit);
}

// ForestFire.step part 1: the action (Agent.move :141-155, toggle_digging :136-138) and, on tick
// steps, Agent.is_dead (:116-120).  Thread 0 of every CTA computes the same thing; only `writer`
// (cluster rank 0) touches global memory.  MLP: the action is `mlp_act`, what mlp_action chose.
template <bool MLP>
__device__ void agent_phase_impl(const Env& e, const StepCfg& c, const TilePar& t, const TileIO& io, const DevState& s, int k,
                                 int do_tick, int32_t* sc, StepShared& ss, bool writer, int mlp_act);
template <bool MLP>
__device__ __forceinline__ void agent_phase(const Env& e, const StepCfg& c, const TilePar& t, const TileIO& io, const DevState& s,
                                            int k, int do_tick, int32_t* sc, StepShared& ss, bool writer, int mlp_act = 0) {
    agent_phase_impl<MLP>(e, c, t, io, s, k, do_tick, sc, ss, writer, mlp_act);
    // the agent_pos layer of step k's observation (nothing after the action moves the agent; a reset re-reads the scalars)
    ss.obs_agent[k & 1][0] = sc[WF_S_VISIBLE]; ss.obs_agent[k & 1][1] = sc[WF_S_AX]; ss.obs_agent[k & 1][2] = sc[WF_S_AY];
}
template <bool MLP>
__device__ void agent_phase_impl(const Env& e, const StepCfg& c, const TilePar& t, const TileIO& io, const DevState& s, int k,
                                 int do_tick, int32_t* sc, StepShared& ss, bool writer, int mlp_act) {
    ss.act = sc[WF_S_RUNNING];
    ss.dig_word = -1;
    ss.dig_bit = 0u;
    ss.dig_clear_R = 0;
    ss.need_flood = 0;
    if (!sc[WF_S_RUNNING]) return;
    const int W = e.W, H = e.H;
    int action;
    if (MLP) {
        action = mlp_act;
    } else if (io.actions != nullptr) {
        action = io.actions[(size_t)k * s.N + e.env];
    } else if (io.policy == WF_POLICY_WALK) {  // DQN.choose_randomwalk_action, DQN.py:353-389
        action = 0;
        if (sc[WF_S_ALIVE]) {
            const int mx = W / 2, my = H / 2, px = sc[WF_S_AX], py = sc[WF_S_AY];
            int a0 = 0, a1 = 0;
            if (px >= mx && py > my) { a0 = 1; a1 = 3; }
            if (px > mx && py <= my) { a0 = 1; a1 = 2; }
            if (px <= mx && py < my) { a0 = 0; a1 = 2; }
            if (px < mx && py >= my) { a0 = 0; a1 = 3; }
            uint32_t pw[4];
            for (int j = 0, count = 0;; ++j) {
                if ((j & 3) == 0)
                    philox4x32_10((uint32_t)(c.env_id_base + e.env), (uint32_t)sc[WF_S_EPISODE],
                                  3u * (uint32_t)sc[WF_S_T] + (uint32_t)(j >> 2), kStreamPolicy, c.key0, c.key1, pw);
                action = (pw[j & 3] & 1u) ? a1 : a0;
                const int nx = px + (action == 2 ? 1 : action == 3 ? -1 : 0);
                const int ny = py + (action == 1 ? 1 : action == 0 ? -1 : 0);
                const bool fire_at_loc = nx >= 0 && nx < W && ny >= 0 && ny < H && e.bit(P_F, nx, ny);
                if (!fire_at_loc || count > 10) break;
                count++;
            }
        }
    } else {
        uint32_t w[4];
        const uint32_t tt = (uint32_t)sc[WF_S_T];
        philox4x32_10((uint32_t)(c.env_id_base + e.env), (uint32_t)sc[WF_S_EPISODE], tt >> 2, kStreamAction, c.key0, c.key1, w);
        action = (int)(w[tt & 3u] % (uint32_t)c.n_actions);
    }
    if (writer && io.actions_out != nullptr) io.actions_out[(size_t)k * s.N + e.env] = action;
    if (!sc[WF_S_ALIVE]) return;
    int ax = sc[WF_S_AX], ay = sc[WF_S_AY];
    const int nx = ax + (action == 2 ? 1 : action == 3 ? -1 : 0);
    const int ny = ay + (action == 1 ? 1 : action == 0 ? -1 : 0);
    const bool is_move = action >= 0 && action < 4;
    const bool inb = is_move && nx >= 0 && nx < W && ny >= 0 && ny < H;
    // one round trip: the cell under the agent and everything about the target cell
    bool on_fire_now = e.bit(P_F, ax, ay);  // type == fire under the agent
    const Around tgt = load_around(e, t, inb ? nx : ax, inb ? ny : ay);
    if (is_move) {
        sc[WF_S_VISIBLE] = 0;  // Q1
        if (inb && !tgt.wt) {
            ax = nx; ay = ny;
            sc[WF_S_AX] = ax; sc[WF_S_AY] = ay; sc[WF_S_VISIBLE] = 1;
            const bool onfire = tgt.f != 0u;
            on_fire_now = onfire;
            if (sc[WF_S_DIGGING] && !onfire) plan_dig(e, tgt, sc, ss, nx, ny);
            if (onfire) sc[WF_S_DEAD] = 1;
        }
    }
    if (c.allow_dig_toggle && action == 4) {  // not a move: `tgt` describes the agent's own cell
        sc[WF_S_DIGGING] ^= 1;
        if (sc[WF_S_DIGGING] && plan_dig(e, tgt, sc, ss, ax, ay)) on_fire_now = false;  // dig makes the cell dirt (Q7)
    }
    if (do_tick && (sc[WF_S_DEAD] || on_fire_now)) {
        sc[WF_S_VISIBLE] = 0;
        sc[WF_S_ALIVE] = 0;
        ss.stat[ST_DEATHS] += 1u;
    }
}

// Fuel record of one plane word: its FB bit-slices side by side (one 32-byte sector).
template <int FB>
__device__ __forceinline__ void load_fuel(const uint32_t* rec, uint32_t (&FU)[FB]) {
    const uint4 a = *reinterpret_cast<const uint4*>(rec);
    FU[0] = a.x; FU[1] = a.y; FU[2] = a.z; FU[3] = a.w;
    if (FB == 5) {
        FU[4] = rec[4];
    } else {
        const uint4 b = *reinterpret_cast<const uint4*>(rec + 4);
        FU[4] = b.x; FU[FB > 5 ? 5 : 4] = b.y; FU[FB > 6 ? 6 : 4] = b.z; FU[FB > 7 ? 7 : 4] = b.w;
    }
}
template <int FB>
__device__ __forceinline__ void store_fuel(uint32_t* rec, const uint32_t (&FU)[FB]) {
    *reinterpret_cast<uint4*>(rec) = make_uint4(FU[0], FU[1], FU[2], FU[3]);
    if (FB == 5) rec[4] = FU[4];
    else *reinterpret_cast<uint4*>(rec + 4) = make_uint4(FU[4], FU[FB > 5 ? 5 : 4], FU[FB > 6 ? 6 : 4], FU[FB > 7 ? 7 : 4]);
}

// ---------------------------------------------------------------------------------------------
// The stencil.
// Active word (it burns or is heated): reduce_fuel :297-307, burn-out, apply_heat_from_to :278-294,
// set_fire_to :233-246.  Returns the word's heat sources for the next tick.  Planes this thread does
// not hold in registers are patched with fire-and-forget reductions (RED), so nothing waits on them.
template <int FB>
__device__ __forceinline__ uint32_t tick_active_word(uint32_t* P, size_t pstride, uint32_t* Frec, uint32_t& G, uint32_t& B,
                                                     uint32_t h0, uint32_t h1, uint32_t h2, uint32_t h3, const DevState& s,
                                                     const StepCfg& c, uint32_t* hrow, int wid, int kmin,
                                                     uint32_t edge, int& my_edge) {
    uint32_t m = h0 | h1 | h2 | h3;
    // issue the loads of this word together: fuel planes (only if it burns) and the first heated cells
    uint32_t FU[FB];
    if (B) load_fuel<FB>(Frec, FU);
    int y[4];
    uint32_t v[4];
    uint32_t mm = m;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        y[j] = mm ? __ffs(mm) - 1 : -1;
        mm &= mm - 1u;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = y[j] >= 0 ? hrow[y[j]] : 0u;

    uint32_t out = 0u, ge2 = 0u;
    const bool burning_word = B != 0u;
    if (B) {
        uint32_t borrow = B;
#pragma unroll
        for (int q = 0; q < FB; ++q) {
            const uint32_t f = FU[q];
            FU[q] = f ^ borrow;
            borrow &= ~f;
        }
        uint32_t nz = 0u;
#pragma unroll
        for (int q = 0; q < FB; ++q) {
            FU[q] &= ~borrow;
            nz |= FU[q];
        }
        out = B & ~nz;
        store_fuel<FB>(Frec, FU);
#pragma unroll
        for (int q = 1; q < FB; ++q) ge2 |= FU[q];  // fuel >= 2, for every cell of the word
    }
    uint32_t ign = 0u;
    auto heat_cell = [&](int yy, uint32_t old) {
        const uint32_t nv = old + (((h0 >> yy) & 1u) | (((h1 >> yy) & 1u) << 8) | (((h2 >> yy) & 1u) << 16) |
                                   (((h3 >> yy) & 1u) << 24));
        hrow[yy] = nv;
        const bool ig = kmin >= 0 ? (int)__dp4a(nv, 0x01010101u, 0u) >= kmin : ignites(nv, s.wind, wid, c.threshold);
        if (ig) ign |= 1u << yy;
    };
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (y[j] >= 0) heat_cell(y[j], v[j]);
    while (mm) {  // more than 4 heated cells in one word: rare
        const int yy = __ffs(mm) - 1;
        mm &= mm - 1u;
        heat_cell(yy, hrow[yy]);
    }
    if (out) {  // type := burnt whatever it was (a dug-while-burning cell is dirt, Q7)
        atomicOr(&P[P_BT * pstride], out);
        atomicAnd(&P[P_D * pstride], ~out);
        atomicAnd(&P[P_WT * pstride], ~out);
        atomicAnd(&P[P_F * pstride], ~out);
        G &= ~out; B &= ~out;
    }
    if (ign) {
        atomicOr(&P[P_F * pstride], ign);
        G &= ~ign; B |= ign;
        if (!burning_word) {  // heated-only word that ignites (rare): now its fuel is needed
            load_fuel<FB>(Frec, FU);
#pragma unroll
            for (int q = 1; q < FB; ++q) ge2 |= FU[q];
        }
    }
    if (ign | out) {
        P[P_G * pstride] = G;
        P[P_B * pstride] = B;
    }
    if (ign & edge) my_edge = 1;
    return B & ge2;  // sources of the next tick: burning with fuel >= 2
}

// Does a burning cell of word `wi` sit next to the border-connected region R?  Words of other
// CTAs' slices may not show this step's dig yet: the dug cell is masked out here (digw, digclr).
__device__ __forceinline__ bool touches_reach(const uint32_t* R, int wi, uint32_t B, int x, int w, int W, int HW, int digw,
                                              uint32_t digclr) {
    auto ld = [&](int j) -> uint32_t {
        const uint32_t v = R[j];
        return j == digw ? (v & ~digclr) : v;
    };
    // its 4 NEIGHBOURS (A* ignores the start cell's cost and finds no path when start == goal, pyastar.py:53-62)
    const uint32_t own = ld(wi);
    uint32_t near = (own << 1) | (own >> 1);
    if (x > 0) near |= ld(wi - HW);
    if (x < W - 1) near |= ld(wi + HW);
    if (w > 0) near |= ld(wi - 1) >> 31;
    if (w < HW - 1) near |= ld(wi + 1) << 31;
    return (B & near) != 0u;
}

// One tick (or, on non-tick steps, just the per-env counts) over this CTA's slice.  Leaves the CTA's
// partial reductions in red[0..3]; the caller synchronises.
// VW = words per thread and iteration along y: 4 (128-bit loads; needs HW % 4 == 0) or 1.
// Every WARP works on its own: it streams 32 units, compacts the ACTIVE words (burning or heated)
// into its private queue in shared memory (ballot + prefix count) and then hands one queued word to
// each lane, so the dependent loads of the active path (fuel planes, hit counters) run in parallel
// instead of serially inside the few lanes that own a fire front.  Nothing in the tick couples two
// warps (S is ping-ponged, R is only read, every other plane word has one owner), so there is no
// block-wide barrier here and a warp without fire never waits for one that has some.
template <int FB, int VW>
__device__ __forceinline__ void tick_slice(const Env& e, const DevState& s, const StepCfg& c, const TilePar& t,
                                           const int32_t* sc, const StepShared& ss, bool ticking, int digw, int* red,
                                           uint32_t* qmem) {
    const int W = e.W, H = e.H, HW = e.HW, tid = e.tid;
    const int lane = tid & 31, warp = tid >> 5, nwarps = e.T >> 5;
    constexpr int QW = 32 * VW;  // queue capacity of one warp
    constexpr int WSM = 7 * QW;  // shared words per warp: 7 queue arrays (the observation phase reuses them as staging)
    uint32_t* const q_idx = qmem + warp * WSM;
    uint32_t* const q_G = q_idx + QW;
    uint32_t* const q_B = q_idx + 2 * QW;
    uint32_t* const q_h = q_idx + 3 * QW;  // [4][QW]
    const unsigned FULL = 0xffffffffu;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const size_t pstride = e.pstride;
    const bool want_touch = !sc[WF_S_FIRE_AT_BORDER] && !sc[WF_S_LATCHED];
    const int cur = sc[WF_S_RESERVED] & 1;
    const int scur = cur ? t.P_S1 : t.P_S0, snxt = cur ? t.P_S0 : t.P_S1;
    const uint32_t digclr = ss.dig_clear_R ? ss.dig_bit : 0u;
    const int digw_R = ss.dig_word;  // R is patched in registers even after a re-flood (harmless: the bit is clear)
    const uint32_t* const Rp = e.plane(t.P_R);
    const int wid = sc[WF_S_WIND_ID];
    const int kmin = s.wind->uniform[wid] ? s.wind->kmin[wid] : -1;
    int my_nb = 0, my_ng = 0, my_edge = 0, my_touch = 0, my_bseed = 0;
    const int nu = (e.hi - e.lo + VW - 1) / VW;
    for (int ub = warp; ub * 32 < nu; ub += nwarps) {
        const int u = ub * 32 + lane;
        uint32_t G[VW], B[VW], h[4][VW];
        bool active[VW];
#pragma unroll
        for (int k = 0; k < VW; ++k) {
            G[k] = B[k] = 0u;
            h[0][k] = h[1][k] = h[2][k] = h[3][k] = 0u;
            active[k] = false;
        }
        const int i = e.lo + u * VW;  // first word of this lane's unit
        if (u < nu) {
            const int x = e.row_of(i), w0 = i - x * HW;
            uint32_t* P = e.P0 + i;
            if (VW == 4) {
                const uint4 g4 = *reinterpret_cast<const uint4*>(P + P_G * pstride);
                const uint4 b4 = *reinterpret_cast<const uint4*>(P + P_B * pstride);
                G[0] = g4.x; G[VW > 1 ? 1 : 0] = g4.y; G[VW > 2 ? 2 : 0] = g4.z; G[VW > 3 ? 3 : 0] = g4.w;
                B[0] = b4.x; B[VW > 1 ? 1 : 0] = b4.y; B[VW > 2 ? 2 : 0] = b4.z; B[VW > 3 ? 3 : 0] = b4.w;
            } else {
                G[0] = P[P_G * pstride];
                B[0] = P[P_B * pstride];
            }
            if (digw >= i && digw < i + VW) {  // Agent.dig lands in this unit: this thread owns the word
#pragma unroll
                for (int k = 0; k < VW; ++k)
                    if (digw == i + k) G[k] &= ~ss.dig_bit;
                apply_dig(e, t, digw, ss.dig_bit, ss.dig_clear_R);
            }
            if (ticking) {
                const uint32_t* Sc = P + (size_t)scur * pstride;
                uint32_t* Sn = P + (size_t)snxt * pstride;
                uint32_t S[VW + 2], Sup[VW], Sdn[VW];
                if (VW == 4) {
                    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
                    const uint4 s4 = *reinterpret_cast<const uint4*>(Sc);
                    const uint4 u4 = x > 0 ? *reinterpret_cast<const uint4*>(Sc - HW) : z;
                    const uint4 d4 = x < W - 1 ? *reinterpret_cast<const uint4*>(Sc + HW) : z;
                    S[1] = s4.x; S[VW > 1 ? 2 : 1] = s4.y; S[VW > 2 ? 3 : 1] = s4.z; S[VW > 3 ? 4 : 1] = s4.w;
                    Sup[0] = u4.x; Sup[VW > 1 ? 1 : 0] = u4.y; Sup[VW > 2 ? 2 : 0] = u4.z; Sup[VW > 3 ? 3 : 0] = u4.w;
                    Sdn[0] = d4.x; Sdn[VW > 1 ? 1 : 0] = d4.y; Sdn[VW > 2 ? 2 : 0] = d4.z; Sdn[VW > 3 ? 3 : 0] = d4.w;
                } else {
                    S[1] = Sc[0];
                    Sup[0] = x > 0 ? Sc[-HW] : 0u;
                    Sdn[0] = x < W - 1 ? Sc[HW] : 0u;
                }
                S[0] = w0 > 0 ? Sc[-1] : 0u;
                S[VW + 1] = w0 + VW < HW ? Sc[VW] : 0u;
#pragma unroll
                for (int k = 0; k < VW; ++k) {
                    h[0][k] = G[k] & ((S[k + 1] >> 1) | (S[k + 2] << 31));  // d = N (0,-1): source at y+1
                    h[1][k] = G[k] & ((S[k + 1] << 1) | (S[k] >> 31));      // d = S (0,+1): source at y-1
                    h[2][k] = G[k] & Sup[k];                                // d = E (+1,0): source at x-1
                    h[3][k] = G[k] & Sdn[k];                                // d = W (-1,0): source at x+1
                    active[k] = (B[k] | h[0][k] | h[1][k] | h[2][k] | h[3][k]) != 0u;
                    if (!active[k]) my_ng += __popc(G[k]);  // inactive words cannot burn: B == 0
                }
                // inactive words have no sources next tick; queued words overwrite their slot in phase 2
                if (VW == 4) *reinterpret_cast<uint4*>(Sn) = make_uint4(0u, 0u, 0u, 0u);
                else Sn[0] = 0u;
            } else {
#pragma unroll
                for (int k = 0; k < VW; ++k) {
                    my_nb += __popc(B[k]);
                    my_ng += __popc(G[k]);
                    if (B[k] && want_touch) {  // burning border points are judged by seed_cells_touch
                        const uint32_t sw = seed_word(W, H, x, w0 + k);
                        if (B[k] & sw) my_bseed = 1;
                        if ((B[k] & ~sw) && touches_reach(Rp, i + k, B[k] & ~sw, x, w0 + k, W, HW, digw_R, digclr)) my_touch = 1;
                    }
                }
            }
        }
        if (!ticking) continue;
        // ---- compact the warp's active words into its queue
        int nq = 0;
#pragma unroll
        for (int k = 0; k < VW; ++k) {
            const uint32_t m = __ballot_sync(FULL, active[k]);
            if (active[k]) {
                const int pos = nq + __popc(m & lt_mask);
                q_idx[pos] = (uint32_t)(i + k);
                q_G[pos] = G[k]; q_B[pos] = B[k];
                q_h[pos] = h[0][k]; q_h[QW + pos] = h[1][k]; q_h[2 * QW + pos] = h[2][k]; q_h[3 * QW + pos] = h[3][k];
            }
            nq += __popc(m);
        }
        if (nq == 0) continue;  // warp-uniform
        __syncwarp();
        // ---- phase 2: one queued active word per lane
        for (int it = lane; it < nq; it += 32) {
            const int wi = (int)q_idx[it];
            const int x = e.row_of(wi), w = wi - x * HW;
            uint32_t Gq = q_G[it], Bq = q_B[it];
            uint32_t* P = e.P0 + wi;
            const uint32_t sn = tick_active_word<FB>(P, pstride, e.FU + (size_t)wi * kFuelRec, Gq, Bq, q_h[it], q_h[QW + it],
                                                     q_h[2 * QW + it], q_h[3 * QW + it], s, c,
                                                     e.hits + ((size_t)x * H + 32 * w), wid, kmin, edge_word(W, H, x, w), my_edge);
            P[(size_t)snxt * pstride] = sn;
            my_nb += __popc(Bq);
            my_ng += __popc(Gq);
            if (Bq && want_touch) {
                const uint32_t sw = seed_word(W, H, x, w);
                if (Bq & sw) my_bseed = 1;
                if ((Bq & ~sw) && touches_reach(Rp, wi, Bq & ~sw, x, w, W, HW, digw_R, digclr)) my_touch = 1;
            }
        }
        __syncwarp();
    }
    // ---- partial reductions of this CTA: warp redux -> shared
    my_nb = __reduce_add_sync(FULL, my_nb);
    my_ng = __reduce_add_sync(FULL, my_ng);
    my_edge = __any_sync(FULL, my_edge);
    my_touch = __any_sync(FULL, my_touch);
    my_bseed = __any_sync(FULL, my_bseed);
    if (lane == 0) {
        if (my_nb) atomicAdd(&red[0], my_nb);
        if (my_ng) atomicAdd(&red[1], my_ng);
        if (my_edge) atomicOr(&red[2], 1);
        if (my_touch) atomicOr(&red[3], 1);
        if (my_bseed) atomicOr(&red[4], 1);
    }
}

// Burning cells that are border points themselves.  For the reference a border point is not a goal for the A*
// search that STARTS on it (pyastar.astar_path returns an empty path when start == goal, pyastar.py:53-62), so such
// a cell reaches the border only through a neighbour that is a finite border point or is connected to a border
// point that does not burn.  (Other burning cells simply test their neighbours against R, which is seeded by all
// finite border points.)  Off the rim such cells exist only on W > H maps -- the literal [HEIGHT-1, y] column of
// environment.py:222 -- so this rarely runs: flood a scratch plane from the cold border points, test, done.
// Whole cluster; returns (in every thread) whether one of those cells reaches the border.
template <bool CL>
__device__ bool seed_cells_touch(const Env& e, const TilePar& t, int scratch_plane, int* red, int (*xch)[kMaxCluster][kRed],
                                 int& par, StepShared& ss) {
    const int W = e.W, H = e.H, HW = e.HW;
    flood<CL>(e, t, red, xch, par, ss, scratch_plane, true);
    const uint32_t* Rc = e.plane(scratch_plane);
    const uint32_t* I = e.plane(P_I);
    const uint32_t* B = e.plane(P_B);
    int hit = 0;
    for (int i = e.lo + e.tid; i < e.hi; i += e.T) {
        const int x = e.row_of(i), w = i - x * HW;
        const uint32_t b = B[i] & seed_word(W, H, x, w);
        if (!b) continue;
        auto goal = [&](int j, int xx, int ww) -> uint32_t { return Rc[j] | (seed_word(W, H, xx, ww) & ~I[j]); };
        const uint32_t own = goal(i, x, w);
        uint32_t near = (own << 1) | (own >> 1);
        if (x > 0) near |= goal(i - HW, x - 1, w);
        if (x < W - 1) near |= goal(i + HW, x + 1, w);
        if (w > 0) near |= goal(i - 1, x, w - 1) >> 31;
        if (w < HW - 1) near |= goal(i + 1, x, w + 1) << 31;
        if (b & near) hit = 1;
    }
    if (hit) red[0] = 1;
    __syncthreads();
    exchange<CL>(e, red, xch, par, ss);
    return ss.tot[0] != 0;
}

// ---------------------------------------------------------------------------------------------
// WF_POLICY_MLP: DQN.choose_action (DQN.py:188-196) on the observation of the state the planes and scalars hold now, i.e.
// what the last step emitted (after an auto-reset: the new episode's first frame).  Whole cluster; the action is returned
// in thread 0.  Hidden unit j = base_j + [visible] w1[agent, 0] + sum_F w1[cell, 1] - sum_I w1[cell, 2] (base: the
// all-free map, MlpPolicy::base).  The sums are exact: every weight is rounded to int64 fixed point (w * 2^32: exact
// scaling, then round to nearest), so any order -- warps, shared atomics, the CTAs of any cluster size -- gives the same
// totals, and the action does not depend on the geometry or on how the steps are split into launches.  Precondition: the
// magnitudes summed into one unit stay below 2^31 (at most 2 W H + 1 rows: |w1| < 2^31 / (2 W H + 1) suffices).
// Each warp sweeps 32 words of its CTA's slice at a time; every lane with a set bit left announces its lowest one and all
// lanes add that row (lane l: packed positions 2l, 2l + 1 = units l, l + 32), four rows per round so their loads overlap.
// Then sigmoid, the second layer and the first-max argmax in float64 (warp 0), eps-greedy from the EXPLORE stream as
// in the warp family (wf_warp.cu).
template <bool CL>
__device__ int mlp_action(const Env& e, const StepCfg& c, const MlpPolicy& m, const int32_t* sc) {
    __shared__ long long part[64];                          // this CTA's sums of the 64 packed positions
    __shared__ long long xmlp[CL ? kMaxCluster : 1][64];    // every CTA's sums (written by the peers)
    constexpr unsigned FULL = 0xffffffffu;
    const int H = e.H, HW = e.HW, tid = e.tid, lane = tid & 31, warp = tid >> 5, nwarps = e.T >> 5;
    const size_t off = (size_t)(e.env / m.group_envs) * m.net_stride;
    const float2* w1 = reinterpret_cast<const float2*>(m.w1 + off);
    if (tid < 64) part[tid] = 0;
    __syncthreads();  // (also: this CTA's words of the planes are final)
    const int aw = sc[WF_S_VISIBLE] ? sc[WF_S_AX] * HW + (sc[WF_S_AY] >> 5) : -1;
    const uint32_t abit = 1u << (sc[WF_S_AY] & 31);
    const uint32_t* PF = e.plane(P_F);
    const uint32_t* PI = e.plane(P_I);
    long long acc0 = 0, acc1 = 0;
    for (int g = e.lo + warp * 32; g < e.hi; g += nwarps * 32) {  // warp-uniform
        const int i = g + lane;
        uint32_t dA = 0u, dF = 0u, dI = 0u;
        int cell0 = 0;
        if (i < e.hi) {
            const int x = e.row_of(i), w = i - x * HW;
            const uint32_t v = valid_word(H, w);
            dF = PF[i] & v;
            dI = PI[i] & v;
            dA = i == aw ? abit : 0u;
            cell0 = x * H + 32 * w;
        }
        for (;;) {
            const bool has = (dA | dF | dI) != 0u;
            int code = 0;  // (input row << 1) | subtract
            if (has) {
                const int ch = dA ? 0 : dF ? 1 : 2;
                uint32_t& d = dA ? dA : dF ? dF : dI;
                const int y = __ffs(d) - 1;
                d &= d - 1u;
                code = (((cell0 + y) * 3 + ch) << 1) | (ch == 2 ? 1 : 0);
            }
            uint32_t todo = __ballot_sync(FULL, has);
            if (todo == 0u) break;
            while (todo) {
                int cd[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int src = todo ? __ffs(todo) - 1 : -1;
                    todo &= todo - 1u;
                    cd[j] = __shfl_sync(FULL, code, src < 0 ? 0 : src);
                    if (src < 0) cd[j] = -1;
                }
                float2 wv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) wv[j] = cd[j] >= 0 ? __ldg(&w1[(size_t)(cd[j] >> 1) * 32 + lane]) : make_float2(0.0f, 0.0f);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const long long a = __float2ll_rn(wv[j].x * 0x1p32f), b = __float2ll_rn(wv[j].y * 0x1p32f);
                    if (cd[j] & 1) { acc0 -= a; acc1 -= b; }
                    else { acc0 += a; acc1 += b; }
                }
            }
        }
    }
    if (acc0) atomicAdd(reinterpret_cast<unsigned long long*>(&part[2 * lane]), (unsigned long long)acc0);
    if (acc1) atomicAdd(reinterpret_cast<unsigned long long*>(&part[2 * lane + 1]), (unsigned long long)acc1);
    __syncthreads();
    long long h0 = 0, h1 = 0;
    if (CL) {
        for (int v = tid; v < 64 * e.CS; v += e.T) st_shared_cluster(&xmlp[e.rank][v & 63], (uint32_t)(v >> 6), part[v & 63]);
        cluster_barrier();
        if (warp == 0)
            for (int r = 0; r < e.CS; ++r) { h0 += xmlp[r][2 * lane]; h1 += xmlp[r][2 * lane + 1]; }
    } else if (warp == 0) {
        h0 = part[2 * lane]; h1 = part[2 * lane + 1];
    }
    int action = 0;
    if (warp == 0) {
        const float* base = m.base + off;
        const float4* w2 = reinterpret_cast<const float4*>(m.w2 + off);  // [2][64]: actions 0..3, 4..7 of unit j
        const float* b2 = m.b2 + off;                                   // [8] (-inf: no such action), then the threshold
        const double s0 = 1.0 / (1.0 + exp(-((double)base[lane] + (double)h0 * 0x1p-32)));
        const double s1 = 1.0 / (1.0 + exp(-((double)base[lane + 32] + (double)h1 * 0x1p-32)));
        const float4 a0 = w2[lane], b0 = w2[64 + lane], a1 = w2[lane + 32], b1 = w2[96 + lane];
        double q[8] = {s0 * a0.x + s1 * a1.x, s0 * a0.y + s1 * a1.y, s0 * a0.z + s1 * a1.z, s0 * a0.w + s1 * a1.w,
                       s0 * b0.x + s1 * b1.x, s0 * b0.y + s1 * b1.y, s0 * b0.z + s1 * b1.z, s0 * b0.w + s1 * b1.w};
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int b = 0; b < 8; ++b) q[b] += __shfl_xor_sync(FULL, q[b], o);
        if (lane == 0) {
            int greedy = 0;
            double best = q[0] + (double)b2[0];
#pragma unroll
            for (int b = 1; b < 8; ++b) {
                const double v = q[b] + (double)b2[b];
                if (v > best) { best = v; greedy = b; }
            }
            uint32_t w[4];
            const uint32_t tt = (uint32_t)sc[WF_S_T];
            philox4x32_10((uint32_t)(c.env_id_base + e.env), (uint32_t)sc[WF_S_EPISODE], tt >> 1, kStreamExplore, c.key0, c.key1, w);
            const uint32_t u0 = (tt & 1u) ? w[2] : w[0], u1 = (tt & 1u) ? w[3] : w[1];
            action = (u0 < __float_as_uint(b2[8])) ? (int)(u1 % (uint32_t)c.n_actions) : greedy;
        }
    }
    return action;
}

// ---------------------------------------------------------------------------------------------
// Float observations (WF_OBS_BF16 / WF_OBS_F32) of a staged bit stream: `nelem` (a multiple of 512) stream bits
// become `nelem` elements starting at element `elem0` of the step's block, 16 bytes per lane and store.
__device__ __forceinline__ uint32_t bf16_pair(uint32_t bytes01, uint32_t sel) {  // two 0/1 bytes -> two bfloat16
    return __byte_perm(bytes01, 0u, sel) * (uint32_t)kBf16One;
}
__device__ __forceinline__ void expand_stream_float(void* obs_step, int obs_dtype, size_t elem0, const uint32_t* stage,
                                                    int nelem, const uint2* tab8, int lane) {
    const uint8_t* s8 = reinterpret_cast<const uint8_t*>(stage);
    if (obs_dtype == WF_OBS_BF16) {
        uint4* o = reinterpret_cast<uint4*>(static_cast<uint16_t*>(obs_step) + elem0);
#pragma unroll 4
        for (int c = lane; c < (nelem >> 3); c += 32) {  // 8 stream bits -> 8 x bf16
            const uint2 t = tab8[s8[c]];
            __stcs(&o[c], make_uint4(bf16_pair(t.x, 0x4140u), bf16_pair(t.x, 0x4342u), bf16_pair(t.y, 0x4140u),
                                     bf16_pair(t.y, 0x4342u)));
        }
    } else {
        uint4* o = reinterpret_cast<uint4*>(static_cast<float*>(obs_step) + elem0);
        constexpr uint32_t ONE = 0x3F800000u;
#pragma unroll 4
        for (int c = lane; c < (nelem >> 2); c += 32) {  // 4 stream bits -> 4 x float32
            const uint32_t nib = ((uint32_t)s8[c >> 1] >> ((c & 1) * 4)) & 15u;
            __stcs(&o[c], make_uint4((nib & 1u) ? ONE : 0u, (nib & 2u) ? ONE : 0u, (nib & 4u) ? ONE : 0u, (nib & 8u) ? ONE : 0u));
        }
    }
}

// World.get_state :399-402 of this CTA's slice: [agent_pos, type == fire, fire_mobility != inf].
// Output element (x*H + y)*3 + ch is ONE BIT, so a word's 32 cells are a 96-bit stream (its three masks
// interleaved bit by bit, via a 256-entry "spread by 3" table).  A warp stages the streams of 32
// consecutive words in shared memory (3 KB of output); then lane l expands the 16 stream bits of
// 16-byte chunk it*32+l with two lookups in a byte -> 8 bytes table: every store instruction writes
// 512 contiguous bytes.  2 plane words in, 96 bytes out per word.
// ctr (optional, shared, zeroed by the caller): the warps take their 128-word groups from this counter instead of
// a fixed stride, so that a warp that starts late (warp 0 runs the next step's agent phase first) does less.
// ROW (WF_OBS_BITS only): obs_step is the env's own row (a final-state record's observation), not an [N][words] block.
template <bool ROW = false>
__device__ __forceinline__ void emit_obs_slice(const Env& e, void* obs_step, int obs_dtype, const uint32_t* spread3,
                                               const uint2* tab8, uint32_t* stage_all, int vis, int ax, int ay, int* ctr = nullptr) {
    const int W = e.W, H = e.H, HW = e.HW;
    const int lane = e.tid & 31, warp = e.tid >> 5, nwarps = e.T >> 5;
    const uint32_t* PF = e.plane(P_F);
    const uint32_t* PI = e.plane(P_I);
    const int aw = vis ? ax * HW + (ay >> 5) : -1;
    // Every warp stages in its OWN region, whichever path it takes: a warp on the narrow path (a slice's tail)
    // must not write where another warp is still emitting a 128-word group (found by tools/soak.py: 130x128,
    // cluster of 2).  384 words per warp exist whenever the wide path does (HW % 4 == 0 <=> VW == 4).
    uint32_t* stage = stage_all + warp * ((HW & 3) == 0 ? 384 : 96);  // 32 words x 96 bits
    const uint16_t* stage16 = reinterpret_cast<const uint16_t*>(stage);
    // WF_OBS_BITS: the env's words.  With H % 32 == 0 word i's 96-bit stream is exactly output words 3i .. 3i+2.
    uint32_t* const obits = static_cast<uint32_t*>(obs_step) + (ROW ? (size_t)0 : (size_t)e.env * obs_bits_words(W, H));
    int g_first = e.lo;
    if ((H & 31) == 0 && (HW & 3) == 0) {
        // One instantiation per element type, so that the loop carries no per-iteration test of it.
        // kind: 0 uint8, 1 bfloat16 / float32, 2 WF_OBS_BITS
        auto wide = [&](auto kind) {
            // Wide path: a warp takes 128 consecutive words (12 KB of output) per iteration with two 128-bit
            // loads per lane, issued one iteration ahead so that the expansion never waits on HBM.
            uint32_t* stage4 = stage_all + warp * 384;  // 128 words x 96 bits
            const uint16_t* stage4_16 = reinterpret_cast<const uint16_t*>(stage4);
            const int n128 = (e.hi - e.lo) >> 7;  // full 128-word groups of this slice
            const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
            uint4 F4 = z4, I4 = z4;
            auto next_group = [&](int prev) -> int {  // warp-uniform
                if (ctr == nullptr) return prev < 0 ? warp : prev + nwarps;
                int v = 0;
                if (lane == 0) v = atomicAdd(ctr, 1);
                return __shfl_sync(0xffffffffu, v, 0);
            };
            int gi = next_group(-1);
            if (gi < n128) {
                F4 = *reinterpret_cast<const uint4*>(PF + e.lo + gi * 128 + 4 * lane);
                I4 = *reinterpret_cast<const uint4*>(PI + e.lo + gi * 128 + 4 * lane);
            }
            while (gi < n128) {
                const int g = e.lo + gi * 128;
                const uint4 Fc = F4, Ic = I4;
                const int gn = next_group(gi);
                if (gn < n128) {
                    F4 = *reinterpret_cast<const uint4*>(PF + e.lo + gn * 128 + 4 * lane);
                    I4 = *reinterpret_cast<const uint4*>(PI + e.lo + gn * 128 + 4 * lane);
                }
                const uint32_t Fw[4] = {Fc.x, Fc.y, Fc.z, Fc.w}, Iw[4] = {Ic.x, Ic.y, Ic.z, Ic.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t F = Fw[j], freerow = ~Iw[j];
                    uint32_t p[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        p[k] = (spread3[(F >> (8 * k)) & 255u] << 1) | (spread3[(freerow >> (8 * k)) & 255u] << 2);
                    if (g + 4 * lane + j == aw) p[(ay & 31) >> 3] |= 1u << (3 * (ay & 7));
                    uint32_t* st = stage4 + (4 * lane + j) * 3;
                    st[0] = p[0] | (p[1] << 24);
                    st[1] = (p[1] >> 8) | (p[2] << 16);
                    st[2] = (p[2] >> 16) | (p[3] << 8);
                }
                __syncwarp();
                if constexpr (decltype(kind)::value == 2) {
                    // the staged stream as it is: 384 words, 12 bytes per plane word (HW % 4 == 0 and the groups start at
                    // multiples of 4 words, so the destination is 16-byte aligned)
                    uint4* o = reinterpret_cast<uint4*>(obits + 3 * (size_t)g);
                    const uint4* s4 = reinterpret_cast<const uint4*>(stage4);
#pragma unroll
                    for (int it = 0; it < 3; ++it) __stcs(&o[it * 32 + lane], s4[it * 32 + lane]);
                } else if constexpr (decltype(kind)::value == 0) {
                    uint4* o = reinterpret_cast<uint4*>(static_cast<uint8_t*>(obs_step) + (((size_t)e.env * W) * H + (size_t)32 * g) * 3);
#pragma unroll 8
                    for (int it = 0; it < 24; ++it) {
                        const int cidx = it * 32 + lane;  // 16-byte chunk of the warp's 12288 bytes = 16 stream bits
                        const uint32_t bits = stage4_16[cidx];
                        const uint2 lo = tab8[bits & 255u], hi = tab8[bits >> 8];
                        __stcs(&o[cidx], make_uint4(lo.x, lo.y, hi.x, hi.y));  // streamed: not read again by this kernel
                    }
                } else {
                    expand_stream_float(obs_step, obs_dtype, (((size_t)e.env * W) * H + (size_t)32 * g) * 3, stage4, 128 * 96, tab8, lane);
                }
                __syncwarp();
                gi = gn;
            }
            g_first = e.lo + n128 * 128;  // the slice's tail (< 128 words) takes the narrow path
        };
        if (obs_dtype == WF_OBS_U8) wide(std::integral_constant<int, 0>{});
        else if (obs_dtype == WF_OBS_BITS) wide(std::integral_constant<int, 2>{});
        else wide(std::integral_constant<int, 1>{});
    }
    const bool fast_ok = (H & 31) == 0;
    for (int g = g_first + warp * 32; g < e.hi; g += nwarps * 32) {
        const int i = g + lane;
        if (i < e.hi) {
            const int x = e.row_of(i), w = i - x * HW;
            const uint32_t F = PF[i];
            const uint32_t freerow = ~PI[i] & valid_word(H, w);
            uint32_t p[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                p[k] = (spread3[(F >> (8 * k)) & 255u] << 1) | (spread3[(freerow >> (8 * k)) & 255u] << 2);
            if (i == aw) p[(ay & 31) >> 3] |= 1u << (3 * (ay & 7));  // agent_pos layer: one cell per env
            const uint32_t r0 = p[0] | (p[1] << 24), r1 = (p[1] >> 8) | (p[2] << 16), r2 = (p[2] >> 16) | (p[3] << 8);
            if (fast_ok && g + 31 < e.hi) {
                stage[3 * lane] = r0; stage[3 * lane + 1] = r1; stage[3 * lane + 2] = r2;
            } else {  // ragged rows, the slice's tail, float observations: one word per thread
                const int ncell = min(32, H - 32 * w);
                const size_t e0 = (((size_t)e.env * W + x) * H + 32 * w) * 3;  // first output element of this word
                const uint32_t r[3] = {r0, r1, r2};
                if (obs_dtype == WF_OBS_BITS) {
                    // bits [b0, b1) of the env's stream; the env's last word also clears the padding after its last
                    // element.  A word shared with a neighbouring thread -- or with another CTA of the cluster -- is
                    // updated as clear-then-set over this thread's own bits only, which is right in any order and needs
                    // no zeroed output.
                    const int b0 = (int)(e0 - (size_t)e.env * W * H * 3), sh = b0 & 31, w0 = b0 >> 5;
                    int b1 = b0 + 3 * ncell;
                    if (x == W - 1 && w == HW - 1) b1 = (b1 + 31) & ~31;
                    const int nq = ((b1 - 1) >> 5) - w0 + 1;  // <= 4 words
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if (q < nq) {
                            const uint32_t v = __funnelshift_l(q > 0 ? r[q - 1] : 0u, q < 3 ? r[q] : 0u, sh);
                            const int wb = 32 * (w0 + q), lo = max(b0, wb) - wb, n = min(b1, wb + 32) - wb - lo;
                            const uint32_t m = n == 32 ? 0xffffffffu : ((1u << n) - 1u) << lo;
                            if (m == 0xffffffffu) {
                                obits[w0 + q] = v;
                            } else {
                                atomicAnd(&obits[w0 + q], ~m);
                                atomicOr(&obits[w0 + q], v & m);
                            }
                        }
                    }
                } else if (obs_dtype == WF_OBS_U8) {
                    uint8_t* o8 = static_cast<uint8_t*>(obs_step) + e0;
                    for (int b = 0; b < 3 * ncell; ++b) o8[b] = (uint8_t)((r[b >> 5] >> (b & 31)) & 1u);
                } else if (obs_dtype == WF_OBS_BF16) {
                    uint16_t* oh = static_cast<uint16_t*>(obs_step) + e0;
                    for (int b = 0; b < 3 * ncell; ++b) oh[b] = ((r[b >> 5] >> (b & 31)) & 1u) ? kBf16One : (uint16_t)0;
                } else {
                    float* of = static_cast<float*>(obs_step) + e0;
                    for (int b = 0; b < 3 * ncell; ++b) of[b] = ((r[b >> 5] >> (b & 31)) & 1u) ? 1.0f : 0.0f;
                }
            }
        }
        if (fast_ok && g + 31 < e.hi) {  // warp-uniform
            __syncwarp();
            if (obs_dtype == WF_OBS_BITS) {  // 32 plane words = 96 output words
                uint32_t* o = obits + 3 * (size_t)g;
#pragma unroll
                for (int it = 0; it < 3; ++it) __stcs(&o[it * 32 + lane], stage[it * 32 + lane]);
            } else if (obs_dtype == WF_OBS_U8) {
                uint4* o = reinterpret_cast<uint4*>(static_cast<uint8_t*>(obs_step) + (((size_t)e.env * W) * H + (size_t)32 * g) * 3);
#pragma unroll
                for (int it = 0; it < 6; ++it) {
                    const int cidx = it * 32 + lane;  // 16-byte chunk of the warp's 3072 bytes = 16 stream bits
                    const uint32_t bits = stage16[cidx];
                    const uint2 lo = tab8[bits & 255u], hi = tab8[bits >> 8];
                    __stcs(&o[cidx], make_uint4(lo.x, lo.y, hi.x, hi.y));  // streamed: not read again by this kernel
                }
            } else {
                expand_stream_float(obs_step, obs_dtype, (((size_t)e.env * W) * H + (size_t)32 * g) * 3, stage, 32 * 96, tab8, lane);
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// World.reset (environment.py:186-212) of this cluster's env: reset_map (:59-95), fire at the centre,
// Agent.__init__ (:100-113), extra ignitions, reach plane, burning count.  Whole cluster.
template <int FB, bool CL>
__device__ void reset_env(const Env& e, const DevState& s, const StepCfg& c, const TilePar& t, const wf_init* init,
                          int32_t* sc, StepShared& ss, int* red, int (*xch)[kMaxCluster][kRed], int& par) {
    const int W = e.W, H = e.H, HW = e.HW, tid = e.tid, T = e.T;
    const size_t pstride = e.pstride;
    const uint32_t episode = (uint32_t)sc[WF_S_EPISODE] + 1u;  // every thread reads the old value ...
    const int cur = sc[WF_S_RESERVED] & 1;
    __syncthreads();                                            // ... before thread 0 overwrites it
    // ---- reset_map :59-67: every plane and the temp layer of this slice back to their defaults
    for (int i = e.lo + tid; i < e.hi; i += T) {
        const int x = e.row_of(i), w = i - x * HW;
        const uint32_t valid = valid_word(H, w);
        uint32_t* P = e.P0 + i;
        P[P_G * pstride] = valid;
        P[P_F * pstride] = 0u; P[P_BT * pstride] = 0u; P[P_D * pstride] = 0u; P[P_WT * pstride] = 0u;
        P[P_B * pstride] = 0u; P[P_I * pstride] = 0u;
        {
            uint32_t FU[FB];
#pragma unroll
            for (int q = 0; q < FB; ++q) FU[q] = ((c.fuel >> q) & 1) ? valid : 0u;
            store_fuel<FB>(e.FU + (size_t)i * kFuelRec, FU);
        }
        P[(size_t)t.P_S0 * pstride] = 0u;
        P[(size_t)t.P_S1 * pstride] = 0u;
        P[(size_t)t.P_R * pstride] = valid;  // open field: every cell reaches the border (re-flooded if rivers)
    }
    {   // hit counters (temp layer := 0) of the cells of words [lo, hi)
        auto cell_of = [&](int i) -> int {
            if (i >= e.nwords) return W * H;
            const int x = e.row_of(i), w = i - x * HW;
            return x * H + min(32 * w, H);
        };
        const int c0 = cell_of(e.lo), c1 = cell_of(e.hi);
        uint32_t* hits = e.hits;
        if ((((size_t)e.env * W * H) & 3) == 0 && (c0 & 3) == 0 && (c1 & 3) == 0) {
            uint4* h4 = reinterpret_cast<uint4*>(hits);
            for (int i = (c0 >> 2) + tid; i < (c1 >> 2); i += T) h4[i] = make_uint4(0u, 0u, 0u, 0u);
        } else {
            for (int i = c0 + tid; i < c1; i += T) hits[i] = 0u;
        }
    }
    sync_env<CL>();
    const bool writer = e.rank == 0;
    const int cx = W / 2, cy = H / 2;  // get_fire_location, utility.py:61-64
    const int scur = cur ? t.P_S1 : t.P_S0;
    if (tid == 0) {  // the draws are replayed by every CTA (identical scalars); rank 0 writes the planes
        ResetDraws dr((uint32_t)(c.env_id_base + e.env), episode, c.key0, c.key1);
        int wid = 0;
        if (c.wind_random) {  // :188-190
            const int si = dr.next() % 3u, wx = dr.next() % 3u, wy = dr.next() % 3u;
            wid = si * 9 + wx * 3 + wy;
        }
        if (c.make_rivers) {  // reset_map :69-95
            int river_x = dr.next() % (uint32_t)W;
            int river_y = 1 + dr.next() % 3u;
            while (river_y < H - (1 + (int)(dr.next() % 3u))) {
                if (writer) {
                    const uint32_t bit = 1u << (river_y & 31);
                    const int wi = river_x * HW + (river_y >> 5);
                    e.plane(P_G)[wi] &= ~bit;
                    e.plane(P_WT)[wi] |= bit;
                    e.plane(P_I)[wi] |= bit;
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
        int ax, ay;
        if (init != nullptr && init[e.env].ax >= 0) {
            ax = init[e.env].ax; ay = init[e.env].ay;
        } else {
            const int rad = dr.next() % 3u;  // radius - 1, utility.py:70
            const int idx = dr.next() % (uint32_t)kCircleLen[rad];
            ax = cx + kCircle[rad][idx][0];
            ay = cy + kCircle[rad][idx][1];
        }
        if (writer) {
            {   // World.set_fire_to(centre), :203 / :233-246 (a river cell under the origin keeps fm_inf, Q5)
                const uint32_t bit = 1u << (cy & 31);
                const int wi = cx * HW + (cy >> 5);
                e.plane(P_G)[wi] &= ~bit; e.plane(P_BT)[wi] &= ~bit; e.plane(P_D)[wi] &= ~bit; e.plane(P_WT)[wi] &= ~bit;
                e.plane(P_F)[wi] |= bit; e.plane(P_B)[wi] |= bit;
                if (c.fuel >= 2) e.plane(scur)[wi] |= bit;
            }
            {   // Agent.__init__ digs its start cell (:112-113)
                const uint32_t bit = 1u << (ay & 31);
                const int wi = ax * HW + (ay >> 5);
                if (!(e.plane(P_D)[wi] & bit)) {
                    e.plane(P_G)[wi] &= ~bit; e.plane(P_F)[wi] &= ~bit; e.plane(P_BT)[wi] &= ~bit; e.plane(P_WT)[wi] &= ~bit;
                    e.plane(P_D)[wi] |= bit; e.plane(P_I)[wi] |= bit;
                    e.plane(t.P_R)[wi] &= ~bit;
                }
            }
        }
        sc[WF_S_ALIVE] = 1; sc[WF_S_AX] = ax; sc[WF_S_AY] = ay; sc[WF_S_DEAD] = 0; sc[WF_S_DIGGING] = 1;
        sc[WF_S_VISIBLE] = 1; sc[WF_S_RUNNING] = 1; sc[WF_S_LATCHED] = 0;
        sc[WF_S_EPISODE] = (int32_t)episode; sc[WF_S_T] = 0; sc[WF_S_WIND_ID] = wid;
        sc[WF_S_WIND_X] = s.wind->wx[wid]; sc[WF_S_WIND_Y] = s.wind->wy[wid];
        sc[WF_S_FIRE_AT_BORDER] = 0;  // :212
    }
    __syncthreads();
    // extra ignitions: World.set_fire_to after reset() (IGNITE stream).  set_fire_to is idempotent and
    // commutes with itself, so the k-th ignitions run in parallel with atomics (rank 0); every CTA
    // replays the draws for the fire_at_border flag.
    int my_fab = 0;
    for (int k = tid; k < c.extra_ignitions; k += T) {
        uint32_t wd[4];
        philox4x32_10((uint32_t)(c.env_id_base + e.env), episode, (uint32_t)k, kStreamIgnite, c.key0, c.key1, wd);
        const int x = (int)(wd[0] % (uint32_t)W), y = (int)(wd[1] % (uint32_t)H);
        if (writer) {
            const int wi = x * HW + (y >> 5);
            const uint32_t bit = 1u << (y & 31);
            atomicAnd(&e.plane(P_G)[wi], ~bit);
            atomicAnd(&e.plane(P_BT)[wi], ~bit);
            atomicAnd(&e.plane(P_D)[wi], ~bit);
            atomicAnd(&e.plane(P_WT)[wi], ~bit);
            atomicOr(&e.plane(P_F)[wi], bit);
            atomicOr(&e.plane(P_B)[wi], bit);
            if (c.fuel >= 2) atomicOr(&e.plane(scur)[wi], bit);
        }
        if (x == 0 || x == W - 1 || y == 0 || y == H - 1) my_fab = 1;
    }
    const int fab = __syncthreads_or(my_fab);
    if (tid == 0 && fab) sc[WF_S_FIRE_AT_BORDER] = 1;
    sync_env<CL>();
    // Without rivers the only blocked cell is the agent's start cell, and one cell cannot cut a
    // >= 10x10 grid: R = every free cell (set above).  With rivers: flood.
    if (c.make_rivers) flood<CL>(e, t, red, xch, par, ss);
    int n = 0;
    const uint32_t* B = e.plane(P_B);
    for (int i = e.lo + tid; i < e.hi; i += T) n += __popc(B[i]);
    n = __reduce_add_sync(0xffffffffu, n);
    if ((tid & 31) == 0 && n) atomicAdd(&red[0], n);
    __syncthreads();
    exchange<CL>(e, red, xch, par, ss);
    if (tid == 0) sc[WF_S_N_BURNING] = ss.tot[0];
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// Final-state capture (`fin`, wf_set_final_capture): the record of this cluster's env, whose episode ended at step k, taken before the
// auto-reset.  Whole cluster: rank 0 takes the slot and hands it to every CTA; each CTA writes the terminal observation of
// its slice and its share of the type planes' words (gathered from any row: nothing writes a plane until the closing
// barrier).  fin_sh[1] receives the slot.
template <bool CL>
__device__ void capture_final(const Env& e, const FinalCapture& fin, int k, const int32_t* sc, int32_t* fin_sh, const uint32_t* spread3,
                              const uint2* tab8, uint32_t* qmem, int ovis, int oax, int oay) {
    if (e.rank == 0 && e.tid == 0) {
        const int slot = (int)atomicAdd(fin.count, 1u);
        if (CL) {
            for (int r = 0; r < e.CS; ++r) st_shared_cluster(&fin_sh[1], (uint32_t)r, slot);
        } else {
            fin_sh[1] = slot;
        }
    }
    sync_env<CL>();
    const uint32_t slot = (uint32_t)fin_sh[1];
    if ((int64_t)slot < fin.capacity) {
        uint32_t* const rec = fin.records + (size_t)slot * fin.words;
        const int W = e.W, H = e.H, HW = e.HW;
        if (e.rank == 0 && e.tid < WF_FINAL_HEADER_WORDS) {
            const int i = e.tid;
            const int flags = (sc[WF_S_ALIVE] ? WF_FINAL_ALIVE : 0) | (sc[WF_S_VISIBLE] ? WF_FINAL_VISIBLE : 0) |
                              (sc[WF_S_DEAD] ? WF_FINAL_DEAD : 0) | (sc[WF_S_DIGGING] ? WF_FINAL_DIGGING : 0);
            const int v = i == WF_F_K ? k : i == WF_F_ENV ? e.env : i == WF_F_EPISODE ? sc[WF_S_EPISODE] : i == WF_F_T ? sc[WF_S_T]
                        : i == WF_F_AX ? sc[WF_S_AX] : i == WF_F_AY ? sc[WF_S_AY] : i == WF_F_FLAGS ? flags
                        : (i == WF_F_NEXT_AX || i == WF_F_NEXT_AY) ? -1 : 0;
            rec[i] = (uint32_t)v;
        }
        if (e.rank == 0) {  // the padding words after the observation and after the planes
            const int pad0 = WF_FINAL_OBS + obs_bits_words(W, H), pad1 = fin.plane_off + 4 * final_plane_words(W, H);
            for (int i = e.tid; i < (fin.plane_off - pad0) + (fin.words - pad1); i += e.T)
                rec[i < fin.plane_off - pad0 ? pad0 + i : pad1 + i - (fin.plane_off - pad0)] = 0u;
        }
        // the terminal observation, straight into the record's row
        emit_obs_slice<true>(e, rec + WF_FINAL_OBS, WF_OBS_BITS, spread3, tab8, qmem, ovis, oax, oay);
        // the type planes: word j of a plane holds cells 32j .. 32j + 31 in x*H + y order
        const int pw = final_plane_words(W, H), per = (pw + e.CS - 1) / e.CS;
        const int j0 = min(pw, e.rank * per), nj = min(pw, j0 + per) - j0;
        const int src[4] = {P_F, P_BT, P_D, P_WT};
        for (int q = e.tid; q < 4 * nj; q += e.T) {
            const int p = q / nj, j = j0 + q - p * nj;
            const uint32_t* P = e.plane(src[p]);
            const int cend = min(32 * j + 32, W * H);
            uint32_t v = 0u;
            for (int cell = 32 * j; cell < cend;) {
                const int x = cell / H, y = cell - x * H;
                const int n = min(min(cend - cell, H - y), 32);
                const int wi = x * HW + (y >> 5), sh = y & 31;
                const uint32_t hi = (sh != 0 && (y >> 5) + 1 < HW) ? P[wi + 1] : 0u;
                uint32_t bits = __funnelshift_r(P[wi], hi, sh);
                if (n < 32) bits &= (1u << n) - 1u;
                v |= bits << (cell - 32 * j);
                cell += n;
            }
            rec[fin.plane_off + p * pw + j] = v;
        }
    }
    sync_env<CL>();
}

// Shared words of the capture kernels only (a kernel that never calls this has none).
__device__ __forceinline__ int32_t* fin_shared() {
    __shared__ int32_t v[2];
    return v;
}

// ---------------------------------------------------------------------------------------------
// K x ForestFire.step (forest_fire.py:30-49) or ForestFire.reset of one env per cluster.
// MLP: WF_POLICY_MLP steps (no reset mode, no action array).  FIN: final-state capture (tile_fin_kernel only).
// tid_x: threadIdx.x, read in the kernel itself (where __launch_bounds__ bounds its range).
template <int FB, int VW, bool CL, bool MLP, bool FIN>
__device__ __forceinline__ void tile_body(const DevState& s, const StepCfg& c, const TilePar& t, const TileIO& io, int tid_x,
                                          const FinalCapture& fin = FinalCapture{}) {
    extern __shared__ uint32_t qmem[];  // per-warp active-word queues (7 x 32 * VW words each); observation staging
    __shared__ int32_t sc[WF_NSCALARS];
    __shared__ int red[kRed];
    __shared__ int xch[2][kMaxCluster][kRed];
    __shared__ StepShared ss;
    __shared__ uint32_t spread3[256];  // bit i of the index -> bit 3i
    __shared__ uint2 tab8[256];        // bit i of the index -> byte i
    int32_t* const fin_sh = FIN ? fin_shared() : nullptr;  // FIN: the step ended the episode; the record's slot

    Env e;
    e.tid = tid_x; e.T = t.T;
    e.CS = CL ? (int)cluster_nctarank() : 1;
    e.rank = CL ? (int)cluster_ctarank() : 0;
    e.env = CL ? (int)cluster_id_x() : (int)blockIdx.x;
    e.W = s.W; e.H = s.H; e.HW = s.HW; e.nwords = t.nwords; e.hw_shift = t.hw_shift; e.hw_magic = t.hw_magic;
    e.lo = min(e.nwords, e.rank * t.wpc);
    e.hi = min(e.nwords, e.lo + t.wpc);
    e.pstride = t.pstride;
    e.P0 = s.planes + (size_t)e.env * t.env_words;
    e.hits = s.hits + (size_t)e.env * t.cells;
    e.FU = s.fuel + (size_t)e.env * t.env_words * kFuelRec;
    const int tid = e.tid;

    for (int v = tid; v < 256; v += e.T) {
        uint32_t o = 0u;
#pragma unroll
        for (int i = 0; i < 8; ++i) o |= ((v >> i) & 1u) << (3 * i);
        spread3[v] = o;
        uint2 b8;
        b8.x = ((v & 15u) * 0x00204081u) & 0x01010101u;
        b8.y = (((v >> 4) & 15u) * 0x00204081u) & 0x01010101u;
        tab8[v] = b8;
    }
    if (tid < WF_NSCALARS) sc[tid] = s.scal[(size_t)e.env * WF_NSCALARS + tid];
    if (tid < kRed) red[tid] = 0;
    if (tid < ST_N) ss.stat[tid] = 0u;
    __syncthreads();
    int par = 0;
    const bool writer = e.rank == 0;
    const size_t step_bytes = t.step_bytes;

#ifdef WF_TILE_TIMING
    unsigned long long t_last;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_last));
#endif
    if (io.reset_mode) {
        // ---------------- ForestFire.reset() ----------------
        if (io.mask == nullptr || io.mask[e.env] != 0) reset_env<FB, CL>(e, s, c, t, io.init, sc, ss, red, xch, par);
        if (io.obs != nullptr) emit_obs_slice(e, io.obs, io.obs_dtype, spread3, tab8, qmem, sc[WF_S_VISIBLE], sc[WF_S_AX], sc[WF_S_AY]);
    } else {
        // ---------------- K x ForestFire.step(action) ----------------
        // The agent phase of step k+1 (one thread, a few dependent loads) runs while the other warps emit the
        // observation of step k: nothing writes a plane between barrier Y of step k and barrier X of step k+1.
        int it = io.a_iter0;
        auto tick_of = [&](int& iter) -> int {  // the fire ticks once every a_speed steps (forest_fire.py:40-43)
            iter -= 1;
            const int dt = (iter == 0);
            if (dt) iter = c.a_speed;
            return dt;
        };
        int do_tick = tick_of(it);
        if (tid == 0) { ss.obs_ctr = 0; ss.slow = 0; }
        if (MLP) {
            // the policy pass: every CTA of the cluster, or none (a frozen env's action is not used).  Its DSMEM stores need
            // every CTA of the cluster to have started: one cluster barrier first (later passes follow barrier X).
            if (CL) cluster_barrier();
            const int a = sc[WF_S_RUNNING] ? mlp_action<CL>(e, c, io.mlp, sc) : 0;
            if (tid == 0) agent_phase<true>(e, c, t, io, s, 0, do_tick, sc, ss, writer, a);
        } else if (tid == 0 && io.K > 0) {
            agent_phase<false>(e, c, t, io, s, 0, do_tick, sc, ss, writer);
        }
        // ---- RUNNING (forest_fire.py:105-106), World.get_reward (environment.py:342-390), done; thread 0 only
        auto finish_step = [&](int k, int dt, int touches, int n_burning, int n_grass, int edge_ignition) {
            const int cur = sc[WF_S_RESERVED];
            if (dt) sc[WF_S_RESERVED] = cur ^ 1;  // the source mask just written becomes current
            const bool anyB = n_burning > 0;
            sc[WF_S_N_BURNING] = n_burning;
            if (dt) {
                if (edge_ignition) sc[WF_S_FIRE_AT_BORDER] = 1;
                if (!sc[WF_S_ALIVE] || !anyB) sc[WF_S_RUNNING] = 0;
            }
            double rew;
            const bool check = !sc[WF_S_FIRE_AT_BORDER] && !sc[WF_S_LATCHED] && anyB;
            if (check && !touches) {
                sc[WF_S_LATCHED] = 1;  // bonus paid once (Q4), tested before the death test
                rew = c.contained_bonus;
                ss.stat[ST_CONTAINED] += 1u;
            } else if (!sc[WF_S_ALIVE]) {
                rew = c.death_penalty;
            } else if (!anyB) {
                rew = __dmul_rn(c.contained_bonus, __ddiv_rn((double)n_grass, (double)(s.W * s.H)));
            } else {
                rew = c.default_reward;
            }
            sc[WF_S_T] += 1;
            const bool is_done = !sc[WF_S_RUNNING];
            ss.stat[ST_STEPS] += 1u;
            if (dt) ss.stat[ST_TICKS] += 1u;
            if (is_done) {
                ss.stat[ST_EPISODES] += 1u;
                if (sc[WF_S_ALIVE]) ss.stat[ST_BURNOUTS] += 1u;
            }
            if (writer) {
                if (io.reward) io.reward[(size_t)k * s.N + e.env] = rew;
                if (io.done) io.done[(size_t)k * s.N + e.env] = is_done ? 1 : 0;
            }
            ss.reset_now = c.auto_reset && is_done;
            if (FIN) fin_sh[0] = is_done;
        };
        // Per step: barrier X -> tick -> CTA barrier -> the partial sums go to the peers and every thread ARRIVES at cluster
        // barrier Y; warp 0 waits for it, adds the totals up, and thread 0 does finish + the agent phase of the next step,
        // while the other warps already emit the observation (its agent layer was fixed by this step's agent phase; they
        // wait for Y afterwards).  The observation is speculative in one respect: if the episode ends here and auto_reset
        // is on, it is emitted again after the reset.  The rare step whose reward needs a whole-cluster pass
        // (seed_cells_touch) finishes after the observation instead.
        // WF_TSTAMP slots (thread 0 of the probe CTA, in warp 0): 0 barrier X, 1 re-flood + tick, 2 CTA barrier, 3 wait for
        // Y + finish + next agent phase, 4 observation, 5 closing __syncthreads (the other warps' half of Y), 6 slow path +
        // reset.
        for (int k = 0; k < io.K; ++k) {
            sync_env<CL>();  // barrier X: agent phase k (and everything thread 0 wrote) is visible; no plane is written before
            WF_TSTAMP(0);
            const bool act = ss.act != 0;
            int digw = ss.dig_word;
            const int ovis = ss.obs_agent[k & 1][0], oax = ss.obs_agent[k & 1][1], oay = ss.obs_agent[k & 1][2];
            void* obs_k = io.obs != nullptr ? static_cast<char*>(io.obs) + (size_t)k * step_bytes : nullptr;
            const int dt = do_tick;
            do_tick = tick_of(it);  // of step k + 1
            if (ss.need_flood) {  // rare: the dig may cut the reach plane -> apply it now and re-flood R
                if (tid == 0 && digw >= e.lo && digw < e.hi) apply_dig(e, t, digw, ss.dig_bit, ss.dig_clear_R);
                digw = -1;
                sync_env<CL>();
                flood<CL>(e, t, red, xch, par, ss);
            }
            const int warp = tid >> 5;
            if (act) {
                tick_slice<FB, VW>(e, s, c, t, sc, ss, dt != 0, digw, red, qmem);
                WF_TSTAMP(1);
                const int cur = sc[WF_S_RESERVED];  // (before thread 0 flips it)
                __syncthreads();                    // red[] is complete, this CTA's planes are final
                WF_TSTAMP(2);
                if (CL) {
                    if (tid < kRed * e.CS) st_shared_cluster(&xch[par][e.rank][tid & (kRed - 1)], (uint32_t)(tid / kRed), red[tid & (kRed - 1)]);
                    cluster_arrive();  // barrier Y, first half
                }
                if (warp == 0) {
                    if (CL) cluster_wait();
                    if (tid < kRed) {
                        int v = 0;
                        if (CL) { for (int r = 0; r < e.CS; ++r) v += xch[par][r][tid]; }
                        else v = red[tid];
                        ss.tot[tid] = v;
                        red[tid] = 0;
                    }
                    __syncwarp();
                    if (tid == 0) {
                        const bool searching = !sc[WF_S_FIRE_AT_BORDER] && !sc[WF_S_LATCHED] && ss.tot[0] > 0 && !(dt && ss.tot[2]);
                        if (ss.tot[4] && searching && !ss.tot[3]) {
                            ss.slow = 1;  // rare (W > H maps): a burning cell is a border point itself
                            ss.reset_now = 0;
                            ss.keep[0] = ss.tot[0]; ss.keep[1] = ss.tot[1]; ss.keep[2] = ss.tot[2];  // (exchange reuses ss.tot)
                        } else {
                            ss.slow = 0;
                            finish_step(k, dt, ss.tot[3], ss.tot[0], ss.tot[1], ss.tot[2]);
                            if (!MLP && !ss.reset_now && k + 1 < io.K) agent_phase<false>(e, c, t, io, s, k + 1, do_tick, sc, ss, writer);
                        }
                    }
                }
                WF_TSTAMP(3);
                if (CL) par ^= 1;
                if (obs_k != nullptr) emit_obs_slice(e, obs_k, io.obs_dtype, spread3, tab8, qmem, ovis, oax, oay, &ss.obs_ctr);
                WF_TSTAMP(4);
                if (CL && warp != 0) cluster_wait();  // barrier Y, second half
                __syncthreads();  // what thread 0 decided is visible
                WF_TSTAMP(5);
                if (ss.slow) {
                    const int scratch = dt ? ((cur & 1) ? t.P_S1 : t.P_S0) : ((cur & 1) ? t.P_S0 : t.P_S1);  // not the current sources
                    const int touches = seed_cells_touch<CL>(e, t, scratch, red, xch, par, ss) ? 1 : 0;
                    if (tid == 0) finish_step(k, dt, touches, ss.keep[0], ss.keep[1], ss.keep[2]);
                    __syncthreads();
                }
            } else {
                if (tid == 0) {  // frozen env: reward 0, done 1, nothing moves
                    if (writer) {
                        if (io.reward) io.reward[(size_t)k * s.N + e.env] = 0.0;
                        if (io.done) io.done[(size_t)k * s.N + e.env] = 1;
                    }
                    ss.reset_now = 0;
                    ss.slow = 0;
                    if (FIN) fin_sh[0] = 0;
                    if (!MLP && k + 1 < io.K) agent_phase<false>(e, c, t, io, s, k + 1, do_tick, sc, ss, writer);
                }
                WF_TSTAMP(3);
                if (obs_k != nullptr) emit_obs_slice(e, obs_k, io.obs_dtype, spread3, tab8, qmem, ovis, oax, oay, &ss.obs_ctr);
                WF_TSTAMP(4);
                __syncthreads();
                WF_TSTAMP(5);
            }
            if constexpr (FIN) {
                if (fin_sh[0]) capture_final<CL>(e, fin, k, sc, fin_sh, spread3, tab8, qmem, ovis, oax, oay);
            }
            const bool late_agent = act && (ss.slow || ss.reset_now);
            if (ss.reset_now) {
                reset_env<FB, CL>(e, s, c, t, nullptr, sc, ss, red, xch, par);
                if (FIN && writer && tid == 0 && fin_sh[0] && (int64_t)(uint32_t)fin_sh[1] < fin.capacity) {  // the next start
                    uint32_t* const rec = fin.records + (size_t)(uint32_t)fin_sh[1] * fin.words;
                    rec[WF_F_NEXT_AX] = (uint32_t)sc[WF_S_AX];
                    rec[WF_F_NEXT_AY] = (uint32_t)sc[WF_S_AY];
                }
                if (tid == 0) ss.obs_ctr = 0;
                __syncthreads();
                if (obs_k != nullptr)  // the new episode's first observation replaces the speculative one
                    emit_obs_slice(e, obs_k, io.obs_dtype, spread3, tab8, qmem, sc[WF_S_VISIBLE], sc[WF_S_AX], sc[WF_S_AY], &ss.obs_ctr);
                __syncthreads();
            }
            if (tid == 0) {
                if (!MLP && late_agent && k + 1 < io.K) agent_phase<false>(e, c, t, io, s, k + 1, do_tick, sc, ss, writer);
                ss.obs_ctr = 0;
                ss.slow = 0;
            }
            if (MLP && k + 1 < io.K) {  // the policy pass on the state this step left, then the next step's agent phase
                const int a = sc[WF_S_RUNNING] ? mlp_action<CL>(e, c, io.mlp, sc) : 0;
                if (tid == 0) agent_phase<true>(e, c, t, io, s, k + 1, do_tick, sc, ss, writer, a);
            }
            WF_TSTAMP(6);
        }
    }
    __syncthreads();
    if (writer && tid < WF_NSCALARS) s.scal[(size_t)e.env * WF_NSCALARS + tid] = sc[tid];
    if (writer && tid < ST_N && ss.stat[tid]) atomicAdd(&s.stats[tid], (unsigned long long)ss.stat[tid]);
}

#ifndef WF_TILE_MAXT
#define WF_TILE_MAXT 512
#define WF_TILE_MINB 2
#endif
template <int FB, int VW, bool CL, bool MLP>
__global__ void __launch_bounds__(WF_TILE_MAXT, WF_TILE_MINB) tile_rollout_kernel(DevState s, StepCfg c, TilePar t, TileIO io) {
    tile_body<FB, VW, CL, MLP, false>(s, c, t, io, threadIdx.x);
}
// The same with final-state capture (wf_set_final_capture): a kernel of its own, so that tile_rollout_kernel keeps its code.
template <int FB, int VW, bool CL, bool MLP>
__global__ void __launch_bounds__(WF_TILE_MAXT, WF_TILE_MINB) tile_fin_kernel(DevState s, StepCfg c, TilePar t, TileIO io, FinalCapture fin) {
    tile_body<FB, VW, CL, MLP, true>(s, c, t, io, threadIdx.x, fin);
}

// S := B & (fuel >= 2) in the env's current source plane, R re-flooded, n_burning recounted
// (after wf_set_state / wf_set_fire_to).  One CTA per env.
__global__ void rebuild_kernel(DevState s, TilePar t) {
    __shared__ int red[kRed];
    __shared__ int xch[2][kMaxCluster][kRed];
    __shared__ StepShared ss;
    Env e;
    e.tid = threadIdx.x; e.T = blockDim.x; e.CS = 1; e.rank = 0; e.env = blockIdx.x;
    e.W = s.W; e.H = s.H; e.HW = s.HW; e.nwords = t.nwords; e.hw_shift = t.hw_shift; e.hw_magic = t.hw_magic;
    e.lo = 0; e.hi = e.nwords;
    e.pstride = t.pstride;
    e.P0 = s.planes + (size_t)e.env * t.env_words;
    e.hits = s.hits + (size_t)e.env * t.cells;
    e.FU = s.fuel + (size_t)e.env * t.env_words * kFuelRec;
    int32_t* sc = s.scal + (size_t)e.env * WF_NSCALARS;
    const int cur = sc[WF_S_RESERVED] & 1;
    if (e.tid < kRed) red[e.tid] = 0;
    __syncthreads();
    int n = 0;
    for (int i = e.tid; i < e.nwords; i += e.T) {
        uint32_t* P = e.P0 + i;
        uint32_t ge2 = 0u;
        for (int q = 1; q < s.FB; ++q) ge2 |= e.FU[(size_t)i * kFuelRec + q];
        const uint32_t B = P[P_B * e.pstride];
        P[(size_t)(cur ? t.P_S1 : t.P_S0) * e.pstride] = B & ge2;
        n += __popc(B);
    }
    n = __reduce_add_sync(0xffffffffu, n);
    if ((e.tid & 31) == 0 && n) atomicAdd(&red[0], n);
    __syncthreads();
    if (e.tid == 0) {
        sc[WF_S_N_BURNING] = red[0];
        red[0] = 0;
    }
    __syncthreads();
    int par = 0;
    flood<false>(e, t, red, xch, par, ss);
}

// ---------------------------------------------------------------------------------------------
// host side
static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// Threads per env so that all N envs together fill the machine (148 SMs x 1024 threads at <= 64
// registers), split into a CTA size T and a cluster size CS.  Measured on B200 (tools/geom_sweep.sh):
// 256 threads per env beat 128 even when that means two waves of CTAs (c4: 51 vs 61 us/step).
static void choose_geometry(const DevState& s, int& T, int& CS) {
    const int VW = (s.HW % 4 == 0) ? 4 : 1;
    const long nunits = ((long)s.W * s.HW + VW - 1) / VW;
    long tpe = 148L * 1024 / (s.N > 0 ? s.N : 1);
    long p = 256;
    while (p * 2 <= tpe && p < 4096) p *= 2;
    while (p > 128 && p > nunits) p /= 2;
    T = (int)(p < 512 ? p : 512);
    CS = (int)(p / T);
    // Few large envs (C5: 64 of 1024x1024): 16 CTAs of 128 threads per env rather than 8 of 256 -- 84.2-84.7 against 88.1-91.1 us
    // per C5 step in three alternating runs on one box (r02).  16 is a non-portable cluster size: tile_create falls back to
    // 256 x 8 if the device cannot hold such a cluster.
    if (p == 2048) { T = 128; CS = 16; }
    const int t_env = env_int("WF_TILE_T", 0), cs_env = env_int("WF_TILE_CS", 0);
    if (t_env == 128 || t_env == 256 || t_env == 512) T = t_env;
    if (cs_env == 1 || cs_env == 2 || cs_env == 4 || cs_env == 8 || cs_env == 16) CS = cs_env;
}

template <typename Kernel>
static cudaError_t set_smem_attr_of(Kernel k, bool cl) {
    if (cl) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (e != cudaSuccess) return e;
    }
    return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 512 * 4 * 28);
}
template <int FB, int VW, bool CL, bool MLP>
static cudaError_t set_smem_attr() {
    cudaError_t e = set_smem_attr_of(tile_rollout_kernel<FB, VW, CL, MLP>, CL);
    return e == cudaSuccess ? set_smem_attr_of(tile_fin_kernel<FB, VW, CL, MLP>, CL) : e;
}
template <bool MLP>
static cudaError_t set_smem_attrs() {
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = set_smem_attr<5, 1, false, MLP>();
    if (e == cudaSuccess) e = set_smem_attr<5, 4, false, MLP>();
    if (e == cudaSuccess) e = set_smem_attr<8, 1, false, MLP>();
    if (e == cudaSuccess) e = set_smem_attr<8, 4, false, MLP>();
    if (e == cudaSuccess) e = set_smem_attr<5, 1, true, MLP>();
    if (e == cudaSuccess) e = set_smem_attr<5, 4, true, MLP>();
    if (e == cudaSuccess) e = set_smem_attr<8, 1, true, MLP>();
    if (e == cudaSuccess) e = set_smem_attr<8, 4, true, MLP>();
    return e;
}

cudaError_t tile_create(TileState** out, const DevState& s, const StepCfg&) {
    TileState* t = new TileState();
    t->P_S0 = P_FU0;  // no fuel planes in this family: the fuel has its own records (DevState::fuel)
    t->P_S1 = P_FU0 + 1;
    t->P_R = P_FU0 + 2;
    choose_geometry(s, t->T, t->CS);
    cudaError_t e = set_smem_attrs<false>();
    if (e == cudaSuccess) e = set_smem_attrs<true>();
    if (e != cudaSuccess) {
        delete t;
        return e;
    }
    if (t->CS == 16 && env_int("WF_TILE_CS", 0) != 16) {  // chosen, not forced: only if such clusters can be resident
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(16);
        cfg.blockDim = dim3(t->T);
        cfg.dynamicSmemBytes = (size_t)t->T * 4 * 28;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 16;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int nc = 0;
        if (cudaOccupancyMaxActiveClusters(&nc, tile_rollout_kernel<5, 4, true, false>, &cfg) != cudaSuccess || nc < 1) {
            cudaGetLastError();
            t->T = 256;
            t->CS = 8;
        }
    }
    *out = t;
    return cudaSuccess;
}

void tile_destroy(TileState* t) { delete t; }
void tile_geometry(const TileState* t, int32_t* threads, int32_t* cluster) {
    *threads = t->T;
    *cluster = t->CS;
}

static TilePar make_par(const TileState* t, const DevState& s, int obs_dtype) {
    TilePar p;
    p.P_S0 = t->P_S0; p.P_S1 = t->P_S1; p.P_R = t->P_R;
    p.hw_shift = -1;
    for (int k = 0; k < 16; ++k)
        if ((1 << k) == s.HW) p.hw_shift = k;
    p.hw_magic = (uint32_t)((0x100000000ull + (uint64_t)s.HW - 1) / (uint64_t)s.HW);  // exact for word < 2^32 / HW
    const int nwords = s.W * s.HW;
    const int per = (nwords + t->CS - 1) / t->CS;
    p.wpc = (per + 31) / 32 * 32;
    p.T = t->T;
    p.nwords = nwords;
    p.cells = s.W * s.H;
    p.pstride = (size_t)s.N * s.RS * s.HW;
    p.env_words = (size_t)s.RS * s.HW;
    p.step_bytes = obs_step_bytes(s.N, s.W, s.H, obs_dtype);
    return p;
}

template <int FB, int VW, bool MLP>
static cudaError_t launch(const TileState* t, const DevState& s, const StepCfg& c, const TileIO& io, cudaStream_t st,
                          const FinalCapture* fin) {
    const TilePar p = make_par(t, s, io.obs_dtype);
    const size_t smem = (size_t)t->T * VW * 28;  // per warp: 7 queue arrays of 32 * VW words (reused as observation staging)
    const bool capture = fin != nullptr && fin->records != nullptr && !io.reset_mode;
    if (t->CS == 1) {
        if (capture) tile_fin_kernel<FB, VW, false, MLP><<<s.N, t->T, smem, st>>>(s, c, p, io, *fin);
        else tile_rollout_kernel<FB, VW, false, MLP><<<s.N, t->T, smem, st>>>(s, c, p, io);
        return cudaGetLastError();
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)s.N * t->CS);
    cfg.blockDim = dim3(t->T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = t->CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (env_int("WF_TILE_DEBUG", 0)) {  // how many clusters of this shape the GPU holds at once (waves = grid / that)
        static bool said = false;
        int nc = 0;
        if (!said && cudaOccupancyMaxActiveClusters(&nc, tile_rollout_kernel<FB, VW, true, MLP>, &cfg) == cudaSuccess)
            fprintf(stderr, "wf_tile: %d clusters of %d x %d threads in the grid, %d resident at once\n", s.N, t->CS, t->T, nc);
        said = true;
    }
    if (capture) return cudaLaunchKernelEx(&cfg, tile_fin_kernel<FB, VW, true, MLP>, s, c, p, io, *fin);
    return cudaLaunchKernelEx(&cfg, tile_rollout_kernel<FB, VW, true, MLP>, s, c, p, io);
}

template <bool MLP>
static cudaError_t launch_fb_vw(const TileState* t, const DevState& s, const StepCfg& c, const TileIO& io, cudaStream_t st,
                                const FinalCapture* fin) {
    const bool v4 = (s.HW % 4 == 0);
    if (s.FB == 5) return v4 ? launch<5, 4, MLP>(t, s, c, io, st, fin) : launch<5, 1, MLP>(t, s, c, io, st, fin);
    return v4 ? launch<8, 4, MLP>(t, s, c, io, st, fin) : launch<8, 1, MLP>(t, s, c, io, st, fin);
}

cudaError_t launch_tile_family(TileState* t, const DevState& s, const StepCfg& c, const TileIO& io,
                               cudaStream_t stream, int64_t* launches, const FinalCapture* fin) {
    *launches += 1;
    if (io.policy == WF_POLICY_MLP && io.actions == nullptr && !io.reset_mode) return launch_fb_vw<true>(t, s, c, io, stream, fin);
    return launch_fb_vw<false>(t, s, c, io, stream, fin);
}

#ifdef WF_TILE_TIMING
extern "C" int wf_debug_tile_timing(unsigned long long* out16, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out16, g_tile_timing, sizeof(unsigned long long) * 16);
    if (reset) {
        unsigned long long z[16] = {0};
        cudaMemcpyToSymbol(g_tile_timing, z, sizeof(z));
    }
    return 0;
}
#endif

cudaError_t tile_after_set_state(TileState* t, const DevState& s, const StepCfg&, cudaStream_t stream,
                                 int64_t* launches) {
    rebuild_kernel<<<s.N, s.W * s.HW >= 8192 ? 1024 : 256, 0, stream>>>(s, make_par(t, s, WF_OBS_U8));
    *launches += 1;
    return cudaGetLastError();
}

}  // namespace wf
