// Host-side launch interface between pnr_api.cu (C-ABI) and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include <utility>
#include "pnr_device.cuh"

#define PNR_STEP_WARPS 4
#define PNR_STEP_THREADS (PNR_STEP_WARPS * 32)
#ifndef PNR_STEP_MIN_CTAS
#define PNR_STEP_MIN_CTAS 6                                                  // 24 warps / SM, <= 85 registers: no spills (8 CTAs spill)
#endif
#define PNR_STEP_BUFS 2                                                      // observation tile buffers per CTA (producer / consumer pipeline)
#ifndef PNR_STEP_MIN_CTAS_FILTER
#define PNR_STEP_MIN_CTAS_FILTER 4                                           // fused normaliser: 39.9 KB of shared memory per CTA, <= 128 registers
#endif
#define PNR_FSCRATCH_STRIDE 19                                               // raw r | cos r | sin r per env (18 floats, odd stride)
#define PNR_FSCRATCH_FLOATS (32 * PNR_FSCRATCH_STRIDE)
#define PNR_STEP_SMEM_FILTER (PNR_STEP_SMEM + PNR_STEP_BUFS * PNR_FSCRATCH_FLOATS * sizeof(float))
#define PNR_BAR_HEAD 1                                                       // named barrier ids: HEAD[2], DONE[2], FREE[2]
#define PNR_BAR_DONE 3
#define PNR_BAR_FREE 5
#define PNR_BAR_JOINT 7                                                      // obstacle variant: the three joint warps among themselves
#define PNR_PEN_FLOATS (3 * 32)                                              // obstacle variant: per-buffer partial contact depths [joint warp][env]
#define PNR_STEP_SMEM_OBST (PNR_STEP_BUFS * PNR_PEN_FLOATS * sizeof(float))
#define PNR_STEP_SMEM (PNR_STEP_BUFS * 32 * PNR_OBS_DIM * sizeof(float))     // step kernel: 17,536 B per tile buffer
#define PNR_RO_SMEM (PNR_STEP_WARPS * 32 * PNR_OBS_DIM * sizeof(float))      // reset/observe: one tile per warp
#define PNR_MAX_DEVICES 16
// The statistics accumulator of the normaliser is PNR_FILTER_SLOTS copies of double[PNR_FILTER_DELTA_LEN]; a CTA adds its
// partial sums to copy blockIdx % SLOTS.  With one copy the ~900 CTAs of a 65,536-env step queued ~900 float64 atomics on
// each of 274 addresses and the kernel's tail took 13 us (tools/fuse_probe.py: 18.5 us without statistics, 31.7 us with).
// pnr_launch_filter_fold adds copies 1.. into copy 0 (what the host and the all-reduce read) and clears them.
#define PNR_FILTER_SLOTS 64
__device__ __forceinline__ double* pnr_filter_slot(double* delta, uint32_t i) {
    return delta + (size_t)(i & (PNR_FILTER_SLOTS - 1)) * PNR_FILTER_DELTA_LEN;
}

// the SM count of `device`, queried once
int pnr_sm_count(int device);
// once per kernel and device: allow `smem` bytes of dynamic shared memory and count the CTAs of `threads` threads the whole
// GPU holds at once (at least one per SM)
cudaError_t pnr_prepare(const void* kernel, int device, int threads, size_t smem, int* resident);

// Launch with programmatic dependent launch on or off (pnr_pdl_wait / pnr_pdl_trigger in pnr_device.cuh)
template <typename Kern, typename... Args>
inline cudaError_t pnr_launch_pdl(Kern kernel, bool pdl, int64_t grid, int threads, size_t smem, cudaStream_t stream,
                                  Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// f_applied != NULL selects the fused normaliser (kinematic: a separate instantiation, float32 arithmetic and terminal
// observations only; dynamic: a run-time switch, both observation modes); f_delta may be NULL (normalise, no statistics)
cudaError_t pnr_launch_step(const PnrParams& p, int device, int arith, int obs_mode, float4* state, const float* actions,
                            float* obs, float* reward, uint8_t* done, PnrStats* stats, uint32_t tick, uint32_t domain,
                            const float* f_applied, double* f_delta, float f_clip, PnrMulti multi, cudaStream_t stream);
cudaError_t pnr_launch_step_dynamic(const PnrParams& p, int device, int obs_mode, float4* state, const float* actions,
                                    float* obs, float* reward, uint8_t* done, PnrStats* stats, uint32_t tick, uint32_t domain,
                                    const float* f_applied, double* f_delta, float f_clip, PnrMulti multi, cudaStream_t stream);
cudaError_t pnr_launch_reset_observe(const PnrParams& p, int device, int mode, float4* state, const int64_t* idx,
                                     int64_t n, const float* q0, const float* target, float* obs_out, uint32_t tick,
                                     cudaStream_t stream);
cudaError_t pnr_launch_state_io(bool set, float4* state, int64_t N, float* r, float* v, float* a, float* potential,
                                float* target, int32_t* t, float* ep_return, cudaStream_t stream);
cudaError_t pnr_launch_observe_done(const PnrParams& p, int device, float4* state, const uint8_t* done, float* obs,
                                    float* terminal_out, const float* f_applied, double* f_delta, float f_clip,
                                    cudaStream_t stream);
cudaError_t pnr_launch_box_io(bool set, float4* box_a, float* box_z, int64_t N, float* box, cudaStream_t stream);
cudaError_t pnr_launch_compact_obs(int device, const float* full, float* compact, int64_t n_rows, cudaStream_t stream);
cudaError_t pnr_launch_tick_advance(PnrStats* stats, uint32_t n, int absolute, cudaStream_t stream);
cudaError_t pnr_launch_env_steps_set(PnrStats* stats, double env_steps, cudaStream_t stream);
cudaError_t pnr_launch_stats_merge(const double* gathered, int world, int len, double* out, cudaStream_t stream);
cudaError_t pnr_launch_stats_snapshot(PnrStats* stats, double* out, int clear, cudaStream_t stream);
// pnr_iteration_sync window layout: double slots[2 parities][MAX_PEERS][288] | uint32 flags[2][MAX_PEERS] | uint32 seq | uint32 status
#define PNR_SYNC_THREADS 288                                    // >= 8 + PNR_FILTER_DELTA_LEN (283), 9 warps
#define PNR_SYNC_SLOT_STRIDE PNR_SYNC_THREADS
#define PNR_SYNC_FLAGS_OFF (2 * PNR_SYNC_MAX_PEERS * PNR_SYNC_SLOT_STRIDE * 8)
#define PNR_SYNC_SEQ_OFF (PNR_SYNC_FLAGS_OFF + 2 * PNR_SYNC_MAX_PEERS * 4)
#define PNR_SYNC_STATUS_OFF (PNR_SYNC_SEQ_OFF + 4)
// pnr_iteration_sync: the windows of all ranks as this process sees them (window[rank] is the local one); world == 1 needs none
struct PnrSyncPeers {
    unsigned char* window[PNR_SYNC_MAX_PEERS];
    int world, rank;
};
cudaError_t pnr_launch_iteration_sync(PnrStats* stats, int clear, double* filt_slots, double* filt_state, float* applied,
                                      int demean, int destd, const PnrSyncPeers& peers, unsigned long long timeout_ns,
                                      double* out, cudaStream_t stream);
cudaError_t pnr_launch_filter_fold(double* delta_slots, cudaStream_t stream);
cudaError_t pnr_launch_filter_refresh(const double* state, float* applied, int demean, int destd, cudaStream_t stream);
cudaError_t pnr_launch_filter_sync(double* slots, const double* merged, double* state, float* applied, int demean, int destd,
                                   cudaStream_t stream);
cudaError_t pnr_launch_filter(int device, const float* in, float* out, int64_t n_rows, const float* applied,
                              double* delta, float clip, int update, int normalize, cudaStream_t stream);
