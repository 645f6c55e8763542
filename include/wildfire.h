/* wildfire.h -- C ABI of libwildfire_b200.so
 *
 * B200-native (sm_100a) batched replacement for the reference's environment
 * step: Simulation/forest_fire.py + Simulation/environment.py of
 * dashdeckers/Wildfire-Control-Python.  One handle owns N independent
 * environments on one GPU; every call steps / resets all of them in one launch.
 *
 * FFI precedent in the reference: pyastar/pyastar.py:9-22 binds one extern "C"
 * symbol of pyastar/astar.cpp:41-44 through ctypes with caller-allocated output
 * arrays.  This header keeps that style: plain pointers and sizes, int status
 * codes, no C++ or torch types.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - "dev" pointers are device pointers on the handle's GPU, owned by the caller
 *     (torch tensors); the library owns only the environments' internal planes.
 *   - All *_dev calls are asynchronous on `stream` (a cudaStream_t passed as void*;
 *     NULL = the legacy default stream).  A handle is not thread-safe.  The *_host calls
 *     (wf_step_host, wf_reset_host) run on a private stream of the handle and are ordered
 *     behind every *_dev call made on the handle before them (an event on that call's stream);
 *     they synchronise before returning, so later *_dev calls are ordered behind them too.
 *   - Every call runs on the handle's device and restores the caller's current device.
 *   - Grid indexing follows the reference: cell (x, y) of env n lives at
 *     [n][x][y], x is the SLOW axis (environment.py: env[x, y, layer]).
 *   - Return value: WF_OK (0) or a negative error code; wf_last_error() gives text.
 *     Nothing throws across the ABI.  There is no CPU fallback: without a CUDA
 *     device wf_create fails with WF_ERR_CUDA.
 */
#ifndef WILDFIRE_H
#define WILDFIRE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WF_ABI_VERSION 2 /* 2: + wf_reset_host, wf_host_session(_active), wf_get/set_a_iter, wf_tile_geometry, wf_apply_change_blocks;
                            later, still 2: + WF_OBS_BITS, wf_unpack_obs_bits; + wf_set_policy_mlp_dev, wf_replay_fit;
                            + wf_set_policy_mlp_nets_dev, wf_replay_fit_many; + wf_set_final_capture,
                            wf_final_record_words (additions only) */

enum {
    WF_OK = 0,
    WF_ERR_INVALID = -1, /* bad argument / unsupported configuration */
    WF_ERR_CUDA = -2,    /* CUDA runtime error (text in wf_last_error) */
    WF_ERR_STATE = -3    /* call not valid in the handle's current state */
};

/* Observation element type written by wf_reset / wf_step / wf_rollout / wf_step_host / wf_get_obs: the 0 / 1 values of
 * World.get_state (environment.py:399-402) as uint8, float32, or bfloat16 (1.0 = 0x3F80) for a bf16 learner, or packed
 * one bit per element (WF_OBS_BITS, 8x smaller than uint8):
 *   - every env takes ceil(W*H*3 / 32) little-endian uint32 words and starts on a word boundary: obs is [N][words]
 *     ([K][N][words] for a rollout) in place of [N][W][H][3];
 *   - element k = (x*H + y)*3 + c (the order of [W][H][3], i.e. Keras' Flatten) is bit k % 32 of word k / 32;
 *   - the padding bits after element W*H*3 - 1 are zero.
 * On a little-endian host np.unpackbits(obs.view(np.uint8), axis=-1, bitorder="little")[..., :W*H*3] is the uint8
 * observation; on the device wf_unpack_obs_bits gathers and expands rows. */
enum { WF_OBS_U8 = 0, WF_OBS_F32 = 1, WF_OBS_BF16 = 2, WF_OBS_BITS = 3 };

/* Cell types -- Simulation/utility.py:128-140. */
enum { WF_GRASS = 0, WF_FIRE = 1, WF_BURNT = 2, WF_DIRT = 3, WF_WATER = 4 };

/* Replaces the module-global METADATA dict (Simulation/constants.py:30-47) and the
 * `grass` cell parameters (Simulation/utility.py:94-102).  Same names, same meaning. */
typedef struct wf_config {
    int32_t width, height;     /* METADATA['width'/'height']; 10 <= W, H (utility.py:68), W >= H */
    int32_t n_actions;         /* actions 0..3 = N,S,E,W; 4 = dig toggle iff allow_dig_toggle; else no-op */
    int32_t a_speed;           /* fire ticks once every a_speed steps (forest_fire.py:40-43) */
    int32_t allow_dig_toggle;
    int32_t make_rivers;       /* reset_map river (environment.py:69-95), drawn from the RESET stream */
    int32_t containment_wins;  /* kept for parity: a no-op in the reference (environment.py:365-366) */
    int32_t wind_random;       /* METADATA['wind'] == "random" (environment.py:188-190) */
    int32_t wind_x, wind_y;    /* else METADATA['wind'] = [wind_speed, (wind_x, wind_y)] */
    int32_t fuel;              /* grass['fuel'], 1..255 */
    int32_t radius;            /* grass['radius']; only 1 (the 4-neighbour stencil) is implemented */
    int32_t extra_ignitions;   /* World.set_fire_to() calls right after reset(), IGNITE stream */
    int32_t auto_reset;        /* 1: an env that returns done is reset inside the same step */
    double wind_speed;
    double death_penalty, contained_bonus, default_reward;
    double heat, threshold;    /* grass['heat'], grass['threshold'] */
    uint64_t seed;             /* key of the shared Philox4x32-10 stream */
    int64_t env_id_base;       /* global id of env 0 (multi-GPU sharding: counter = env_id_base + n) */
} wf_config;

/* Optional per-env overrides for wf_reset (parity injection / scripted starts). */
typedef struct wf_init {
    int32_t ax, ay;            /* agent start cell; ax < 0 = draw from the RESET stream */
} wf_init;

/* Per-env scalars exposed by wf_get_scalars (int32 x WF_NSCALARS per env). */
enum {
    WF_S_ALIVE = 0,    /* len(World.agents) == 1 */
    WF_S_AX, WF_S_AY,  /* agents[0].x / .y (last position once dead) */
    WF_S_DEAD,         /* Agent.dead */
    WF_S_DIGGING,      /* Agent.digging */
    WF_S_VISIBLE,      /* agent_pos layer holds a 1 at (ax, ay) -- quirk Q1 */
    WF_S_RUNNING,      /* World.RUNNING */
    WF_S_FIRE_AT_BORDER,
    WF_S_LATCHED,      /* containment bonus already paid (border_points empty, quirk Q4) */
    WF_S_EPISODE, WF_S_T,
    WF_S_WIND_ID,      /* index into the handle's wind table */
    WF_S_WIND_X, WF_S_WIND_Y,
    WF_S_N_BURNING,    /* len(World.burning_cells) after the last step */
    WF_S_RESERVED,
    WF_NSCALARS = 16
};

typedef struct wf_env wf_env; /* opaque handle */

/* ---- lifetime ------------------------------------------------------------------ */
void wf_default_config(wf_config* cfg, int32_t size);
int wf_create(const wf_config* cfg, int32_t n_envs, int32_t device, wf_env** out);
void wf_destroy(wf_env* env);
const char* wf_last_error(void);
int wf_abi_version(void);
/* Name of the kernel family chosen for this geometry: "warp" (W,H <= 32) or "tile". */
const char* wf_kernel_family(const wf_env* env);

/* ---- ForestFire.reset() -- forest_fire.py:52-54 -> World.reset environment.py:186-212 ----
 * mask_dev: N bytes, reset env n iff mask[n] != 0 (NULL = all).  init_dev: N wf_init or NULL.
 * obs_dev (may be NULL): receives World.get_state() of every env, [N][W][H][3]. */
int wf_reset(wf_env* env, const uint8_t* mask_dev, const wf_init* init_dev,
             void* obs_dev, int32_t obs_dtype, void* stream);

/* ---- ForestFire.step(action) -- forest_fire.py:30-49 -----------------------------
 * actions_dev: N int32.  obs_dev: [N][W][H][3] (NULL = skip).  reward_dev: N float64
 * (World.get_reward, environment.py:342-390).  done_dev: N bytes (not World.RUNNING). */
int wf_step(wf_env* env, const int32_t* actions_dev, void* obs_dev, int32_t obs_dtype,
            double* reward_dev, uint8_t* done_dev, void* stream);

/* K consecutive steps in ONE launch, state resident on chip between steps (warp family).
 * actions_dev: [K][N] int32, or NULL = draw action t from the ACTION stream (what the
 * oracle's wfo_stream_action does).  obs_dev [K][N][W][H][3], reward_dev [K][N],
 * done_dev [K][N]; any of the three may be NULL.  Requires auto_reset or tolerates
 * finished envs by freezing them (reward 0, done 1). */
int wf_rollout(wf_env* env, int32_t k_steps, const int32_t* actions_dev, void* obs_dev,
               int32_t obs_dtype, double* reward_dev, uint8_t* done_dev, void* stream);

/* Action sources of wf_rollout_policy. */
enum {
    WF_POLICY_STREAM = 0, /* uniform random action from the ACTION stream (same as wf_rollout with NULL actions) */
    WF_POLICY_WALK = 1,   /* the reference's heuristic "walk round the fire" demonstration / Baseline policy:
                             DQN.choose_randomwalk_action, DQN.py:353-389 (draws from the POLICY stream) */
    WF_POLICY_MLP = 2     /* the reference's Q-network evaluated inside the step kernel, eps-greedy
                             (DQN.choose_action DQN.py:188-196 on DQN.make_network DQN.py:209-233);
                             weights from wf_set_policy_mlp(_dev) (or, up to 32x32, wf_set_policy_mlp_nets_dev);
                             both kernel families.  The action depends only on the observation, the network and the
                             EXPLORE stream: not on the launch geometry or how the steps are split into launches */
};
/* wf_rollout with the actions chosen on the device by a built-in policy (DQN.collect_memories' inner loop,
 * DQN.py:303-308: choose_randomwalk_action -> sim.step).  actions_out_dev: [K][N] int32 or NULL. */
int wf_rollout_policy(wf_env* env, int32_t k_steps, int32_t policy, int32_t* actions_out_dev, void* obs_dev,
                      int32_t obs_dtype, double* reward_dev, uint8_t* done_dev, void* stream);

/* The network of WF_POLICY_MLP: Flatten(W,H,3) -> Dense(hidden, sigmoid) -> Dense(n_actions, linear), Keras
 * orientation (kernel[in][out], in = (x*H + y)*3 + channel).  Host pointers; copied.  For the dueling
 * head (DQN_DUEL.py:18-48) pass the ADVANTAGE stream: argmax_a (V + A_a - mean A) = argmax_a A_a.
 * eps: probability of a uniformly random action instead of the greedy one (EXPLORE Philox stream:
 * step t uses words 2*(t&1), 2*(t&1)+1 of block t>>1: explore iff word < eps * 2^32, action = word' % n_actions).
 * hidden <= 64, n_actions <= 8.  Any grid: on grids larger than 32x32 (the tile family) the kernel sums the first layer
 * exactly, in int64 fixed point (each weight rounded to a multiple of 2^-32), which needs the magnitudes summed into one
 * hidden unit below 2^31: |kernel1| < 2^31 / (2*W*H + 1) suffices, and wf_set_policy_mlp refuses (WF_ERR_INVALID) a
 * kernel1 entry that is not finite and below that bound there; sigmoid, second layer and argmax are float64 there.
 * The warp family keeps float64 sums of float32 weights, updated incrementally. */
int wf_set_policy_mlp(wf_env* env, const float* kernel1_host, const float* bias1_host, const float* kernel2_host,
                      const float* bias2_host, int32_t hidden, double eps);
/* wf_set_policy_mlp from DEVICE tensors in nn.Linear orientation: weight1_dev [hidden][W*H*3], bias1_dev [hidden],
 * weight2_dev [n_actions][hidden], bias2_dev [n_actions] (float32).  The repack into the kernel's layout runs as a kernel
 * on `stream`: no host copy and no synchronisation, so a refresh queued behind a rollout on the same stream sees the
 * weights that rollout's predecessors left and the next rollout on that stream sees the new ones.  The first call of a
 * handle allocates the packed buffer (as wf_set_policy_mlp does), later calls overwrite it in place: a rollout still
 * running on ANOTHER stream must be ordered by the caller.  The packed buffer is byte-identical to wf_set_policy_mlp's
 * for the same weights (the empty-map sum is accumulated in float64 in the same order), so rollouts are too.  Both kernel
 * families, with wf_set_policy_mlp's precondition on the tile family (not checked here: the weights stay on the device).
 * On the tile family every call re-sums the all-free map over W*H cells in float64, one thread per hidden unit. */
int wf_set_policy_mlp_dev(wf_env* env, const float* weight1_dev, const float* bias1_dev, const float* weight2_dev,
                          const float* bias2_dev, int32_t hidden, double eps, void* stream);

/* ---- final states of finished episodes ----------------------------------------------------------------------------
 * With an auto-reset the state an episode ends in is overwritten inside the step that ends it.  While final-state capture
 * is on (wf_set_final_capture), the step kernels of both families write ONE RECORD for every env that returns done at
 * step k of a wf_step / wf_rollout / wf_rollout_policy launch: before the auto-reset, or at the done step itself without
 * auto_reset (a frozen env, already done, never records again).  A record is wf_final_record_words(W, H) uint32 words:
 *   header, WF_FINAL_HEADER_WORDS words of int32, indexed by WF_F_*: k (the step of the launch), env, the finished
 *     episode's WF_S_EPISODE and WF_S_T (its length), the final WF_S_AX / WF_S_AY, a flag word (WF_FINAL_ALIVE,
 *     WF_FINAL_VISIBLE, WF_FINAL_DEAD, WF_FINAL_DIGGING), and the start cell of the next episode (-1, -1 without
 *     auto_reset); the remaining header words are zero;
 *   from word WF_FINAL_OBS: the terminal observation as one WF_OBS_BITS row (ceil(W*H*3 / 32) words), what the step
 *     would have returned without the reset;
 *   from word WF_FINAL_OBS + ceil(ceil(W*H*3 / 32) / 4) * 4: four bit planes of ceil(W*H / 32) words each, in the order
 *     fire, burnt, dirt, water (WF_FINAL_PLANE_*; a cell in none of them is grass): cell (x, y) is bit (x*H + y) % 32 of
 *     word (x*H + y) / 32 of its plane, padding bits zero.
 * The record length is a multiple of 4 words.  The slot of a record is an atomicAdd on *count_dev, so the order of records
 * is unspecified while every record's content is deterministic; a record whose slot is >= capacity is counted but not
 * written, so *count_dev > capacity shows an overflow.  The counter is never reset by the library: the caller zeroes it
 * (and reads it) between calls as it likes. */
enum {
    WF_F_K = 0, WF_F_ENV, WF_F_EPISODE, WF_F_T, WF_F_AX, WF_F_AY, WF_F_FLAGS, WF_F_NEXT_AX, WF_F_NEXT_AY,
    WF_FINAL_HEADER_WORDS = 16,
    WF_FINAL_OBS = WF_FINAL_HEADER_WORDS
};
enum { WF_FINAL_ALIVE = 1, WF_FINAL_VISIBLE = 2, WF_FINAL_DEAD = 4, WF_FINAL_DIGGING = 8 };
enum { WF_FINAL_PLANE_FIRE = 0, WF_FINAL_PLANE_BURNT = 1, WF_FINAL_PLANE_DIRT = 2, WF_FINAL_PLANE_WATER = 3 };
/* uint32 words of one record for a W x H grid. */
int64_t wf_final_record_words(int32_t width, int32_t height);
/* Turn final-state capture on (records_dev: capacity records of wf_final_record_words words, device memory; count_dev:
 * one device uint32) or off (records_dev NULL).  Handle state, like the policy weights: it applies to every later
 * wf_step, wf_rollout and wf_rollout_policy until it is turned off, and the buffers must stay valid meanwhile.  While it is
 * on, wf_step_host and wf_host_session return WF_ERR_STATE (no capture there). */
int wf_set_final_capture(wf_env* env, uint32_t* records_dev, int64_t capacity, uint32_t* count_dev);

/* Host-buffer variant of wf_step (what a CPU-side caller of the reference would bind):
 * copies actions H2D, steps, copies obs/reward/done D2H and synchronises.  Buffers should
 * be page-locked for full PCIe rate; pageable memory works but is slower.
 * With page-locked buffers, uint8 observations and a grid up to 32x32 the observation crosses PCIe as a
 * bit stream and is expanded into obs_host by a small pool of host threads (WF_HOST_THREADS, default
 * min(12, cores / ranks on the host); WF_HOST_PACKED=0 sends the uint8 array instead,
 * WF_HOST_PACKED=direct stores the bit stream straight into mapped host memory instead of one DMA copy;
 * WF_HOST_TIMING=1 prints the launch / sync / expand split when the handle is destroyed; WF_HOST_GRAPH=1
 * (a_speed == 1 only) issues kernel + copy as one CUDA graph: 40.0-40.6 against 42.1 us per C2 step, tools/e2e_ab.py).
 * Fastest: wf_host_session below (23 us; 19 us with a persistent observation array), which also lifts the page-locked requirement.
 * WF_OBS_BITS (both families): the kernel writes the packed observation to a staging buffer (or, with WF_HOST_MODE=direct,
 * straight into page-locked obs_host) and one cudaMemcpyAsync brings it over; no host thread expands anything.
 * The device alias of each page-locked buffer is looked up once and re-validated every 1024 calls: a caller that
 * unpins or frees a buffer must not hand the same ADDRESS back as a different kind of memory within that window
 * (pass a new address, or destroy the handle). */
int wf_step_host(wf_env* env, const int32_t* actions_host, void* obs_host, int32_t obs_dtype,
                 double* reward_host, uint8_t* done_host);
/* Step-server session for wf_step_host (grids up to 32x32, uint8 observations).  While a session is on, the step kernel
 * stays RESIDENT on the GPU (a cooperative launch) with every env in registers and is driven through mapped page-locked
 * memory: wf_step_host writes the actions, packed six per word and tagged with the step's sequence number, into a mapped
 * buffer that CTA 0 polls;
 * CTA 0 copies them into HBM and releases the other CTAs; every CTA steps its envs and stores its records -- the observation bit
 * stream plus one status word per record (reward kind, done, burn-out count) -- straight into mapped host memory; the
 * last CTA to finish issues a system-scope fence and raises the completion flag; the library's host threads then expand
 * the records into obs_host and decode reward / done (any host memory: the caller's buffers may be pageable).  No kernel
 * launch, no copy call and no stream synchronise per step: 23 instead of 42 us per 4096-env 14x14 step.
 *   wf_host_session(env, 1)  turn it on (the kernel is started by the next wf_step_host);  (env, 0) park it.
 * Any other entry point on the handle (wf_reset, wf_step, wf_get_state, ...) parks the kernel first -- it stores the
 * envs back to HBM and exits -- and the next wf_step_host starts it again, so results never depend on the session.
 * A kernel that sees no step request for WF_SESSION_IDLE_US (default 2000) microseconds parks itself: the GPU is not held
 * hostage by a caller that stops stepping (other work on the device is delayed by at most that long).
 * A batch with more CTAs (8 envs of <= 16 rows, 4 of up to 32 rows, each) than the GPU can hold resident cannot be
 * served: the first wf_step_host then turns the session off and the launch-per-step path takes over.
 *   wf_host_session(env, 2)  session with a PERSISTENT OBSERVATION ARRAY (the convention of vectorised Gym environments
 * with copy=False): the caller passes the same obs_host on every wf_step_host and does not write to it between calls; the
 * kernel then sends, per record, only the list of elements that changed since the previous step (up to 14 per record of
 * two 14x14 envs: 32 instead of 152 bytes over PCIe) and the host threads patch those elements in place.  A record with
 * more changes (a reset env, a large fire tick) travels in full and is expanded as in mode 1.  The array is always complete
 * and equal to what mode 1 delivers after every call: the library compares obs_host with the previous call's pointer and
 * asks for every record in full whenever it differs, on the first step after the kernel was (re)started and hence after
 * every other entry point used in between.  What it cannot detect is the caller overwriting the array: then the patched
 * elements are right and the others stay as the caller left them until their record next travels in full.
 * WF_OBS_BITS calls are served by the session too (uint8 and bits calls may alternate): the host threads copy each record's
 * envs into obs_host [N][words], re-aligning the second env of a two-env record.  In mode 2 the changed elements are
 * patched as bits in place (a host thread owns whole envs, so no two threads share a word); a call whose dtype differs
 * from the previous call's asks for every record in full, like a new array.
 * Returns WF_ERR_INVALID for the tile family.  wf_host_session_active: 0 off, 1 on (kernel parked), 2 kernel resident. */
int wf_host_session(wf_env* env, int32_t on);
int wf_host_session_active(const wf_env* env);
/* Host-buffer variant of wf_reset (ForestFire.reset, forest_fire.py:52-54): mask_host / init_host as in wf_reset but in
 * host memory (NULL = all envs / draw the start cell), obs_host [N][W][H][3] receives World.get_state() (NULL = skip).
 * Synchronises.  Ordered behind every earlier call on the handle, like wf_step_host. */
int wf_reset_host(wf_env* env, const uint8_t* mask_host, const wf_init* init_host, void* obs_host, int32_t obs_dtype);
/* Host threads wf_step_host uses to expand observations (0: the packed path has not been used). */
int wf_host_threads(const wf_env* env);
/* The host half of that path on its own (no GPU needed): expand a packed observation buffer -- one record of
 * ceil(e * W*H*3 / 32) uint32 words per group of e consecutive envs (e = 2 if W <= 16 else 1), bit k of a
 * record = element k of the group's [e][W][H][3] block -- into uint8 obs_host[n_envs][W][H][3]. */
int wf_expand_packed_obs(const uint32_t* packed_host, uint8_t* obs_host, int32_t n_envs, int32_t width,
                         int32_t height, int32_t threads);
/* The host half of wf_host_session mode 2 on its own (no GPU needed): apply one step's change-list blocks to obs_host.
 * blocks_host: one block of 32 words per 4 records (a record = e consecutive envs as in wf_expand_packed_obs): word 0 =
 * number of entries | mask of the records sent in full << 8; words 1-4 = the records' status words (16 bits per env:
 * bits 0-2 reward kind -- 0 zero, 1 default, 2 death, 3 containment, 4 burn-out = contained_bonus * (count / (W * H)) --
 * bit 3 done, bits 4-14 the burn-out's grass count); then 16-bit entries (element index within the block's envs << 1 |
 * new value).  A record flagged in the mask is taken whole from full_area_host[record * full_stride] (packed as for
 * wf_expand_packed_obs).  reward_host / done_host [n_envs] may be NULL. */
int wf_apply_change_blocks(const uint32_t* blocks_host, const uint32_t* full_area_host, int32_t full_stride, uint8_t* obs_host,
                           double* reward_host, uint8_t* done_host, int32_t n_envs, int32_t width, int32_t height,
                           double default_reward, double death_penalty, double contained_bonus, int32_t threads);

/* ---- state access (parity injection, checkpointing) --------------------------------
 * Canonical planes, device pointers, any may be NULL:
 *   type/burning/fm_inf/fuel/apos: [N][W][H] uint8;  hits: [N][W][H][4] uint8 = number of
 *   heat quanta received from direction d (0 N,1 S,2 E,3 W as seen from the source), so
 *   that temp = sum_d hits[d] * coef[wind_id][d]  (environment.py:286-290);
 *   scalars: [N][WF_NSCALARS] int32. */
int wf_get_state(wf_env* env, uint8_t* type, uint8_t* burning, uint8_t* fm_inf, uint8_t* fuel,
                 uint8_t* hits, uint8_t* apos, int32_t* scalars, void* stream);
int wf_set_state(wf_env* env, const uint8_t* type, const uint8_t* burning, const uint8_t* fm_inf,
                 const uint8_t* fuel, const uint8_t* hits, const int32_t* scalars, void* stream);
/* METADATA['a_speed_iter'] (forest_fire.py:40-43; constants.py:38): steps left until the next fire tick, 1..a_speed.
 * One counter per handle, NOT reset by wf_reset (quirk Q8) and not part of the per-env scalars: a checkpoint of a handle
 * with a_speed > 1 is wf_get_state + wf_get_a_iter, restored by wf_set_state + wf_set_a_iter. */
int wf_get_a_iter(const wf_env* env, int32_t* out);
int wf_set_a_iter(wf_env* env, int32_t a_iter);
/* World.set_fire_to(cell) on selected envs: cells_dev [N][2] int32 (x, y), x < 0 = skip. */
int wf_set_fire_to(wf_env* env, const int32_t* cells_dev, void* stream);
/* World.get_state() without stepping. */
int wf_get_obs(wf_env* env, void* obs_dev, int32_t obs_dtype, void* stream);

/* Unpack WF_OBS_BITS rows to [n_out][W][H][3] u8 / f32 / bf16 (out_dtype WF_OBS_U8 / F32 / BF16): row i of out = bits row
 * index[i] of bits_dev [n_rows][ceil(W*H*3 / 32)] (index_dev: n_out int64, NULL = rows 0..n_out-1) -- a minibatch drawn
 * from a packed replay buffer.  An index outside [0, n_rows) yields an all-zero observation (never an out-of-bounds read).
 * Needs no handle: runs on the current device, asynchronously on `stream`.  out_dev 16-byte aligned. */
int wf_unpack_obs_bits(const uint32_t* bits_dev, int64_t n_rows, const int64_t* index_dev, int64_t n_out,
                       int32_t width, int32_t height, void* out_dev, int32_t out_dtype, void* stream);

/* ---- learning: n_replays consecutive DQN.replay updates (DQN.py:156-185, DQN_SARSA.py:103-132) in one launch ----
 * The Q-network is Flatten(W, H, 3) -> Dense(hidden, sigmoid) -> Dense(n_actions) (DQN.make_network, DQN.py:209-233), or
 * the dueling head (DQN_DUEL.py:18-48) with a value stream Flatten -> Dense(hidden, sigmoid) -> Dense(1) and
 * q = v + (a - mean a).  Its parameters are ONE flat float32 buffer in torch.nn.utils.parameters_to_vector(model.parameters())
 * order, nn.Linear orientation (weight[out][in]), n_in = width * height * 3:
 *   dense_1.weight [hidden][n_in] | dense_1.bias [hidden] | dense_2.weight [n_actions][hidden] | dense_2.bias [n_actions]
 *   dueling head, then: dense_3.weight [hidden][n_in] | dense_3.bias [hidden] | dense_4.weight [1][hidden] | dense_4.bias [1]
 * i.e. (hidden * (n_in + 1 + n_actions) + n_actions) floats, plus (hidden * (n_in + 2) + 1) for the dueling head.  The
 * target network and Adam's first and second moments m and v use the same layout. */
typedef struct wf_mlp_shape {
    int32_t width, height; /* observation grid of the warp family: 10 <= height <= width <= 32 */
    int32_t hidden;        /* 1..64 units per stream */
    int32_t n_actions;     /* 1..8 */
    int32_t dueling;       /* 0: plain head, 1: dueling head */
    int32_t batch;         /* transitions per replay, 1..256 */
} wf_mlp_shape;

/* Hyper-parameters of wf_replay_fit: the reference's gamma and Keras 2's Adam(lr, clipvalue) (agents.KerasAdam). */
typedef struct wf_fit_params {
    double gamma;
    double lr, beta_1, beta_2, epsilon; /* epsilon is added to sqrt(v) of the uncorrected second moment (Keras) */
    double clipvalue;                   /* every gradient element is clipped to +-clipvalue first (> 0; INFINITY: none) */
    int64_t adam_t;                     /* updates made before this call: replay r uses t = adam_t + r + 1 */
    int32_t target_every;               /* the model is copied into the target every target_every replays (>= 1) ... */
    int32_t phase;                      /* ... after the replay that brings this counter (1..target_every) to zero:
                                           the reference's until_sync */
} wf_fit_params;

/* Replay r (0 <= r < n_replays) is one fit_batch on transitions i = r * batch .. r * batch + batch - 1:
 *   s = frames row s_row[i], s' = frames row sp_row[i] (frames_dev [n_frames][ceil(W*H*3 / 32)] WF_OBS_BITS rows);
 *   target = Q_target(s) with entry action[i] replaced by reward[i] if done[i] else
 *            reward[i] + gamma * (max_a Q_target(s', a), or Q_target(s', next_action[i]) when next_action_dev != NULL);
 *   loss = mean over batch x n_actions of (Q_model(s) - target)^2; one clipped Keras Adam step on every parameter;
 *   then the model is copied into the target if the replay brings the until_sync counter to zero.
 * Out-of-range inputs never cause an out-of-bounds access: a row outside [0, n_frames) is an all-zero observation (as in
 * wf_unpack_obs_bits); an action outside [0, n_actions) replaces no entry (the sample's target is Q_target(s)); a next
 * action outside [0, n_actions) bootstraps nothing (the target entry is reward[i], as for a terminal transition).
 * loss_dev [n_replays] may be NULL.  Runs as ONE thread-block cluster on the current device, asynchronously on `stream`;
 * each CTA owns a slice of the hidden units and the result is deterministic (no floating-point atomics).
 * Needs no handle; without a CUDA device it fails with WF_ERR_CUDA (no CPU fallback). */
int wf_replay_fit(const wf_mlp_shape* shape, const wf_fit_params* params, int32_t n_replays, float* params_dev,
                  float* target_dev, float* adam_m_dev, float* adam_v_dev, const uint32_t* frames_dev, int64_t n_frames,
                  const int64_t* s_row_dev, const int64_t* sp_row_dev, const int32_t* action_dev,
                  const int32_t* next_action_dev, const float* reward_dev, const uint8_t* done_dev, float* loss_dev,
                  void* stream);

/* wf_replay_fit for any grid wf_create takes: 10 <= height <= width, no upper bound (hidden, n_actions, dueling and batch
 * as above; the flat parameter buffer must hold at most 2^31 - 1 floats).  Same arguments, update rule, target sync,
 * losses and out-of-range rules as wf_replay_fit.  Runs as ONE cooperative launch of as many CTAs as the device holds at
 * once: each CTA owns a fixed set of chunks of the first layer's input columns (the chunking is a function of the shape)
 * and every sum runs in an order fixed by the shape, so the result is deterministic (no floating-point atomics) and does
 * not depend on the number of CTAs (environment variable WF_FIT_CTAS, read on every call: at most that many).  Allocates
 * and frees its scratch (at most 32 MB + 8 * batch * (2 * hidden + 10) bytes) stream-ordered on `stream`.  Grids up to
 * 32x32 are taken too; its sums are ordered differently from wf_replay_fit's, so the two agree to rounding, not bit for
 * bit.  Needs no handle; without a CUDA device it fails with WF_ERR_CUDA (no CPU fallback). */
int wf_replay_fit_large(const wf_mlp_shape* shape, const wf_fit_params* params, int32_t n_replays, float* params_dev,
                        float* target_dev, float* adam_m_dev, float* adam_v_dev, const uint32_t* frames_dev,
                        int64_t n_frames, const int64_t* s_row_dev, const int64_t* sp_row_dev, const int32_t* action_dev,
                        const int32_t* next_action_dev, const float* reward_dev, const uint8_t* done_dev, float* loss_dev,
                        void* stream);

/* ---- populations: up to 64 independent learners in one launch -------------------------------------------------------
 * One learner of wf_replay_fit_many: its own flat model, target and Adam moments (the layout above), its own transitions
 * ([n_replays * batch] each, as for wf_replay_fit; next_action NULL = the DQN target, max_a Q_target(s', a)), its own loss
 * ([n_replays] or NULL) and its own hyper-parameters, Adam step and target-sync phase. */
typedef struct wf_fit_learner {
    float *params, *target, *adam_m, *adam_v;
    const int64_t *s_row, *sp_row;
    const int32_t *action, *next_action;
    const float* reward;
    const uint8_t* done;
    float* loss;
    wf_fit_params hp;
} wf_fit_learner;

/* wf_replay_fit for n_learners (1..64) learners of one network shape and batch size (learners_host: a host array,
 * read before the call returns), in ONE launch: one thread-block cluster per learner.  The frames table is shared and
 * its row numbers are global, so each learner may use any rows (e.g. its own demonstrations).  Every learner is checked
 * as wf_replay_fit checks its arguments (misaligned pointers included) and follows its out-of-range rules.  The
 * cluster size is the one wf_replay_fit uses on this device, so each learner's result is bit-identical to a
 * wf_replay_fit call on that learner alone; clusters beyond those the GPU holds at once run in later waves.
 * wf_replay_fit is this call with one learner. */
int wf_replay_fit_many(const wf_mlp_shape* shape, int32_t n_learners, const wf_fit_learner* learners_host,
                       int32_t n_replays, const uint32_t* frames_dev, int64_t n_frames, void* stream);

/* The in-kernel policy (WF_POLICY_MLP) with n_nets (1..64) networks: env n acts with network n / (N / n_nets).
 * N must be a multiple of n_nets and the group size N / n_nets a multiple of 8 (whole CTAs of the warp family, so each CTA
 * uses one network).  params_dev: [n_nets][P] float32 in the flat layout of wf_replay_fit above (P floats per network,
 * dueling included); the policy reads dense_1 / dense_2 (the advantage stream of a dueling head), so the buffer that
 * wf_replay_fit(_many) writes is read as it is.  eps_host: n_nets exploration rates in [0, 1] (host; read before the call
 * returns).  shape: the handle's grid and n_actions; batch is ignored.  Like wf_set_policy_mlp_dev, the repack runs as a
 * kernel on `stream` with no host copy and no synchronisation, and each network's packed block is byte-identical to the
 * one wf_set_policy_mlp(_dev) produces for the same weights and eps (those calls write network 0, one group covering every
 * env).  A call with more networks than any call before it on the handle reallocates the packed buffer (which waits for
 * the device). */
int wf_set_policy_mlp_nets_dev(wf_env* env, const wf_mlp_shape* shape, int32_t n_nets, const float* params_dev,
                               const double* eps_host, void* stream);

/* Heat quanta table: coef[wind_id][4] float64 (host pointer), n_wind entries (1 or 27). */
int wf_get_wind_table(const wf_env* env, double* coef_host, double* speed_host,
                      int32_t* vec_host, int32_t* n_wind);

/* Episode statistics accumulated on device since creation / last wf_stats_reset:
 * out_host[0]=env-steps [1]=episodes ended [2]=agent deaths [3]=containments [4]=burn-outs
 * [5]=fire ticks.  Synchronises `stream`. */
int wf_stats(wf_env* env, int64_t out_host[8], void* stream);
int wf_stats_reset(wf_env* env, void* stream);

/* Self-test hook: one Philox4x32-10 block computed ON THE DEVICE (ctr[4] then key[2] in, 4 words out),
 * so the device generator can be pinned to the Random123 known-answer vectors. */
int wf_philox_kat(int32_t device, const uint32_t ctr_key_host[6], uint32_t out_host[4]);

/* Tile family: threads per CTA and CTAs per thread-block cluster (one cluster per env) the handle launches with; chosen
 * from n_envs so that the batch fills the GPU (overridable for experiments and tests: WF_TILE_T, WF_TILE_CS, read by
 * wf_create).  Warp family: both 0. */
int wf_tile_geometry(const wf_env* env, int32_t* threads, int32_t* cluster);
/* How many kernels of this library the handle has launched (bench.py's gpu_launches). */
int64_t wf_launch_count(const wf_env* env);
/* Introspection for DESIGN.md / bench roofline: bytes of internal state per env. */
int64_t wf_state_bytes_per_env(const wf_env* env);

#ifdef __cplusplus
}
#endif
#endif /* WILDFIRE_H */
