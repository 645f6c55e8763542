// wf_families.cuh -- launch interfaces of the two kernel families (warp: W,H <= 32; tile: larger).
#pragma once
#include "wf_common.cuh"

namespace wf {

// Q-networks of WF_POLICY_MLP, device pointers into network 0's block (owned by the handle).  Everything is padded to 64
// hidden units and 8 actions (zero weights; -inf bias for the missing actions), so the kernel has no bounds tests.
// Network k's block starts net_stride floats after network k - 1's; env n acts with network n / group_envs.
struct MlpPolicy {
    const float* w1;    // [n_in][64]: hidden unit j = x + L*i of a row sits at x*(64/L) + i (L = lanes per env), i.e. the
                        // units one lane accumulates are adjacent: one 16- or 8-byte load per changed input bit
    const float* base;  // [64]: bias1 + sum over cells of w1[(cell, channel 2)] -- the all-free, no-fire, no-agent map
    const float* w2;    // [2][64] float4: actions 0..3 and 4..7 of every hidden unit
    const float* b2;    // [8], then [8]: the explore threshold (uint32 bits: explore iff a 32-bit draw is below it), 0 x 7
    int32_t hid, n_actions;
    int32_t group_envs; // envs per network: a multiple of the envs of one CTA, so a CTA's envs share one network
    int32_t net_stride; // floats per network block
};
constexpr int kMlpMaxNets = 64;
// Floats of one network's block: w1 | base [64] | w2 [2][64][4] | b2 [8] | threshold + padding [8].
__host__ __device__ inline size_t mlp_net_floats(int n_in) { return (size_t)n_in * 64 + 64 + 512 + 16; }

// Step-server session (wf_host_session): the warp kernel stays resident and is driven from the host through
// flags in mapped page-locked memory -- no launch and no stream synchronise per step.
struct SrvCtl {
    volatile uint32_t* doorbell;  // mapped host, host -> GPU: sequence number of the last step requested; 0xffffffff: park (the
                                  // request itself is the tagged action buffer)
    volatile uint32_t* parked;    // mapped host, GPU -> host: the launch's generation, once the kernel has decided to exit
    volatile uint32_t* done;      // mapped host, GPU -> host: [slices] flags 16 words apart = sequence number completed
    const int32_t* actions_host;  // mapped host [srv_action_chunks(N) * 4] words: the step's actions, packed and tagged (wf_common.cuh)
    int32_t* actions_dev;         // HBM [24 * srv_action_chunks(N) + 4]: CTA 0's unpacked copy, what the warps read (WarpIO::actions)
    uint32_t* go;                 // device: master CTA -> every CTA: index of the step to run (1, 2, ...), 0xffffffff = exit
    uint32_t* count;              // device: [slices] arrival counters
    uint32_t seq0, generation;    // sequence number already processed when the kernel starts; id of this launch
    int32_t ctas_per_slice;
    int32_t sectors;              // != 0: records travel as self-validating 32-byte sectors (wf_common.cuh), no flags / fences
    int32_t delta;                // != 0: change-list blocks (wf_common.cuh; WarpIO::obs = [CTAs][kDeltaBlockWords]); a warp whose
                                  // envs changed in more than kDeltaEntries elements -- or when the host asks for it (bit 31 of
                                  // the action tags), or on the launch's first step -- sends its whole bit stream to full_area
    uint32_t* full_area;          // mapped host [records][full_stride] words
    int32_t full_stride;          // words between two records of full_area (a multiple of 4)
    unsigned long long idle_ns;   // no doorbell for this long: the kernel parks itself (the GPU is not held hostage)
    unsigned long long* dbg;      // device, 8 counters of CTA 0 (ns, summed over steps; WF_HOST_TIMING prints them):
                                  // 0 doorbell wait + action copy, 1 go -> thread 0's warp has stepped and stored, 2 CTA
                                  // barrier (the slowest warp), 3 steps, 4 fence + arrival
};

// Final-state capture (wf_set_final_capture): one record per finished episode, layout in include/wildfire.h.
struct FinalCapture {
    uint32_t* records;   // [capacity][words], or nullptr: capture off
    uint32_t* count;     // slots taken (records past capacity are counted, not written)
    int64_t capacity;
    int32_t words;       // wf_final_record_words(W, H)
    int32_t plane_off;   // first word of the fire plane within a record
};
__host__ __device__ inline int32_t final_plane_words(int W, int H) { return (W * H + 31) / 32; }
__host__ __device__ inline int32_t final_plane_offset(int W, int H) { return WF_FINAL_OBS + ((W * H * 3 + 31) / 32 + 3) / 4 * 4; }
__host__ __device__ inline int32_t final_record_words(int W, int H) {
    return (final_plane_offset(W, H) + 4 * final_plane_words(W, H) + 3) / 4 * 4;
}

struct WarpIO {
    const int32_t* actions;  // [K][N] or nullptr (ACTION stream)
    void* obs;               // [K][N][W][H][3] or nullptr
    double* reward;          // [K][N] or nullptr
    uint8_t* done;           // [K][N] or nullptr
    const uint8_t* mask;     // reset mode: [N] or nullptr
    const wf_init* init;     // reset mode: [N] or nullptr
    int32_t obs_dtype, K, a_iter0, reset_mode;
    uint32_t magicH;         // ceil(2^32 / H)
    int32_t policy;          // actions == nullptr: WF_POLICY_STREAM, WF_POLICY_WALK or WF_POLICY_MLP
    int32_t* actions_out;    // [K][N] or nullptr: the actions the policy chose
    MlpPolicy mlp;           // WF_POLICY_MLP only
};
// fin: final-state capture (nullptr or records == nullptr: off); a separate kernel argument, so that the kernels without
// capture keep their parameters and code.
struct WarpFinIO : WarpIO {  // the kernel argument of the warp family's capture kernels
    FinalCapture fin;
};
cudaError_t launch_warp_family(const DevState& s, const StepCfg& c, const WarpIO& io, cudaStream_t stream,
                               const FinalCapture* fin = nullptr);
// The same kernel as a cooperative launch (every CTA resident) that serves steps until told to park; io.actions / io.obs
// are mapped host buffers (obs_dtype kObsPackedStatus).  cudaErrorCooperativeLaunchTooLarge if the batch does not fit.
cudaError_t launch_warp_server(const DevState& s, const StepCfg& c, const WarpIO& io, const SrvCtl& srv, cudaStream_t stream);

struct TileIO {
    const int32_t* actions;  // [K][N] or nullptr (ACTION stream / policy)
    void* obs;               // [K][N][W][H][3] or nullptr
    double* reward;          // [K][N] or nullptr
    uint8_t* done;           // [K][N] or nullptr
    const uint8_t* mask;     // reset mode: [N] or nullptr
    const wf_init* init;     // reset mode: [N] or nullptr
    int32_t obs_dtype, K, a_iter0, reset_mode;
    int32_t policy;          // actions == nullptr: WF_POLICY_STREAM, WF_POLICY_WALK or WF_POLICY_MLP
    int32_t* actions_out;    // [K][N] or nullptr
    MlpPolicy mlp;           // WF_POLICY_MLP only (packed with 32 lanes: unit j at (j % 32) * 2 + j / 32 of a w1 row)
};
struct TileState;
int tile_extra_planes();
cudaError_t tile_create(TileState** out, const DevState& s, const StepCfg& c);
void tile_destroy(TileState* t);
void tile_geometry(const TileState* t, int32_t* threads, int32_t* cluster);
cudaError_t launch_tile_family(TileState* t, const DevState& s, const StepCfg& c, const TileIO& io,
                               cudaStream_t stream, int64_t* launches, const FinalCapture* fin = nullptr);
cudaError_t tile_after_set_state(TileState* t, const DevState& s, const StepCfg& c, cudaStream_t stream,
                                 int64_t* launches);

}  // namespace wf
