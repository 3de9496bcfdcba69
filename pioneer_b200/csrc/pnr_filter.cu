// N2: fused observation normaliser (the ConcurrentMeanStdFilter -- RLlib's MeanStdFilter behind a lock -- the reference launcher configures for its rollout workers,
// pioneer/launch/pioneer_knm_train.py:66 'observation_filter': 'ConcurrentMeanStdFilter').  ONE streaming pass over the
// observation batch does what the host-side filter does in three (push statistics, demean, scale): a CTA pulls a
// tile of 32 rows into shared memory with a TMA bulk load, every thread owns one of the 137 columns -- accumulates
// sum and sum of squares of (x - applied_mean) over the tile's rows, rewrites the column as
// clip((x - mean) * inv_std) -- and the tile leaves with a TMA bulk store.  Bound: HBM, 548 B read + 548 B written
// per row.  Statistics of the rows seen since the last synchronisation accumulate in float64 on the device
// (one atomicAdd per column per CTA); pnr_filter_sync merges them into the running mean / M2 (Chan et al.
// parallel update) and refreshes the applied mean / inverse std, so between synchronisations every rank
// normalises with the SAME statistics (what RLlib's synchronised filters converge to once per iteration).
#include <cuda_runtime.h>
#include <cstdint>
#include "pnr_device.cuh"
#include "pnr_launch.h"

#define PNR_FILTER_THREADS 160                      // >= PNR_OBS_DIM columns, 5 warps
#define PNR_FILTER_ROWS 32
#define PNR_FILTER_TILE_BYTES (PNR_FILTER_ROWS * PNR_OBS_DIM * 4)

__device__ __forceinline__ void pnr_mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pnr_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void pnr_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pnr_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pnr_bulk_load(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(pnr_smem_u32(sdst)), "l"(gsrc), "r"(bytes), "r"(pnr_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void pnr_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra WAIT_LOOP;\n"
        "}\n" ::"r"(pnr_smem_u32(bar)), "r"(parity) : "memory");
}

// applied: [mean[137], inv_std[137]] float; delta: [count, sum_d[137], sumsq_d[137]] double
__global__ void __launch_bounds__(PNR_FILTER_THREADS)
pnr_filter_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t n_rows,
                  const float* __restrict__ applied, double* __restrict__ delta, float clip, int update,
                  int normalize) {
    extern __shared__ __align__(128) float tile[];
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x;
    const bool col_ok = tid < PNR_OBS_DIM;
    const float mean = col_ok ? applied[tid] : 0.f;
    const float inv_std = col_ok ? applied[PNR_OBS_DIM + tid] : 0.f;
    if (tid == 0) pnr_mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    const int64_t n_tiles = (n_rows + PNR_FILTER_ROWS - 1) / PNR_FILTER_ROWS;
    double acc_s = 0.0, acc_q = 0.0;
    uint32_t phase = 0;
    for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int64_t row0 = t * PNR_FILTER_ROWS;
        const int rows = (int)((n_rows - row0) < PNR_FILTER_ROWS ? (n_rows - row0) : PNR_FILTER_ROWS);
        const float* src = in + row0 * PNR_OBS_DIM;
        float* dst = out + row0 * PNR_OBS_DIM;
        const bool bulk = (rows & 3) == 0;                      // byte count a multiple of 16
        if (bulk) {
            if (tid == 0) {
                pnr_mbar_expect_tx(&bar, (uint32_t)(rows * PNR_OBS_DIM * 4));
                pnr_bulk_load(tile, src, (uint32_t)(rows * PNR_OBS_DIM * 4), &bar);
            }
            pnr_mbar_wait(&bar, phase);
            phase ^= 1;
        } else {
            for (int i = tid; i < rows * PNR_OBS_DIM; i += PNR_FILTER_THREADS) tile[i] = src[i];
            __syncthreads();
        }
        if (col_ok) {
            // float64 accumulation (B200 has the FP64 rate for 2 DFMA per element of an HBM-bound stream): before the
            // first synchronisation the applied mean is 0, and sum(x^2) - sum(x)^2 / n of a constant column must
            // cancel to ~0, which float32 partial sums do not deliver
            double s[4] = {0.0, 0.0, 0.0, 0.0}, q[4] = {0.0, 0.0, 0.0, 0.0};   // four independent FP64 chains
            int r = 0;
            for (; r + 3 < rows; r += 4) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float d = tile[(r + k) * PNR_OBS_DIM + tid] - mean;
                    const double dd = (double)d;
                    s[k] += dd;
                    q[k] = fma(dd, dd, q[k]);
                    if (normalize) tile[(r + k) * PNR_OBS_DIM + tid] = fminf(fmaxf(d * inv_std, -clip), clip);
                }
            }
            for (; r < rows; ++r) {
                const float d = tile[r * PNR_OBS_DIM + tid] - mean;
                const double dd = (double)d;
                s[0] += dd;
                q[0] = fma(dd, dd, q[0]);
                if (normalize) tile[r * PNR_OBS_DIM + tid] = fminf(fmaxf(d * inv_std, -clip), clip);
            }
            acc_s += (s[0] + s[1]) + (s[2] + s[3]);
            acc_q += (q[0] + q[1]) + (q[2] + q[3]);
        }
        if (normalize || out != in) {
            pnr_fence_async_smem();
            __syncthreads();
            if (bulk) {
                if (tid == 0) {
                    pnr_bulk_store(dst, tile, (uint32_t)(rows * PNR_OBS_DIM * 4));
                    pnr_bulk_commit();
                    pnr_bulk_wait_read<0>();
                }
            } else {
                for (int i = tid; i < rows * PNR_OBS_DIM; i += PNR_FILTER_THREADS) dst[i] = tile[i];
            }
        }
        __syncthreads();                                        // the tile may be overwritten
    }
    double* slot = pnr_filter_slot(delta, blockIdx.x);
    if (update && col_ok) {
        atomicAdd(&slot[1 + tid], acc_s);
        atomicAdd(&slot[1 + PNR_OBS_DIM + tid], acc_q);
    }
    if (update && blockIdx.x == 0 && tid == 0) atomicAdd(&delta[0], (double)n_rows);
}

// column j of the accumulator summed over its copies (see pnr_launch.h) in copy order, as every reader folds it
__device__ __forceinline__ double pnr_filter_fold_column(const double* slots, int j) {
    double acc = slots[j];
    for (int s = 1; s < PNR_FILTER_SLOTS; ++s) acc += slots[(size_t)s * PNR_FILTER_DELTA_LEN + j];
    return acc;
}

// copy 0 += copies 1 .. SLOTS-1, which are cleared
__global__ void pnr_filter_fold_kernel(double* __restrict__ slots) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= PNR_FILTER_DELTA_LEN) return;
    const double acc = pnr_filter_fold_column(slots, c);
    for (int s = 1; s < PNR_FILTER_SLOTS; ++s) slots[(size_t)s * PNR_FILTER_DELTA_LEN + c] = 0.0;
    slots[c] = acc;
}

// applied statistics from the running ones: mean (float) and 1 / (std + 1e-8); RunningStat.var = S / (n - 1) if n > 1 else
// mean^2 (RLlib, restated in oracle/filter_oracle.py)
__device__ __forceinline__ void pnr_filter_refresh_column(double count, double mean, double m2, float* applied, int c,
                                                          int demean, int destd) {
    if (!(count > 0.0)) {           // nothing pushed yet: identity (an RLlib filter that has seen no sample never normalises)
        applied[c] = 0.f;
        applied[PNR_OBS_DIM + c] = 1.f;
        return;
    }
    const double var = count > 1.0 ? m2 / (count - 1.0) : mean * mean;
    applied[c] = demean ? (float)mean : 0.f;
    applied[PNR_OBS_DIM + c] = destd ? (float)(1.0 / (sqrt(var) + 1e-8)) : 1.f;
}

__global__ void pnr_filter_refresh_kernel(const double* state, float* applied, int demean, int destd) {
    const int c = threadIdx.x;
    if (c < PNR_OBS_DIM) pnr_filter_refresh_column(state[0], state[1 + c], state[1 + PNR_OBS_DIM + c], applied, c, demean, destd);
}

// Chan et al. merge of one column's batch sums (relative to the APPLIED mean) into the running mean / M2, and the refreshed
// applied statistics of that column; na = running count before, nb = rows in the batch, n = count after
__device__ __forceinline__ void pnr_filter_merge_column(int c, double na, double nb, double n, double sum_d, double sum_q,
                                                        double* state, float* applied, int demean, int destd) {
    double mean = state[1 + c], m2 = state[1 + PNR_OBS_DIM + c];
    if (nb > 0.0) {
        const double applied_mean = demean ? (double)applied[c] : 0.0;
        const double mean_b = applied_mean + sum_d / nb;
        const double m2_b = sum_q - sum_d * sum_d / nb;
        const double delta = mean_b - mean;
        m2 += (m2_b > 0.0 ? m2_b : 0.0) + delta * delta * na * nb / n;
        mean += delta * nb / n;
        state[1 + c] = mean;
        state[1 + PNR_OBS_DIM + c] = m2;
    }
    pnr_filter_refresh_column(n, mean, m2, applied, c, demean, destd);
}

__device__ __forceinline__ void pnr_filter_clear_slots(double* slots, int c, bool col_ok) {
    for (int k = 0; k < PNR_FILTER_SLOTS; ++k) {
        double* sl = slots + (size_t)k * PNR_FILTER_DELTA_LEN;
        if (c == 0) sl[0] = 0.0;
        if (col_ok) { sl[1 + c] = 0.0; sl[1 + PNR_OBS_DIM + c] = 0.0; }
    }
}

// One CTA, thread = column: merge a batch (nb rows; this column's sums, relative to the applied mean) into the running
// count / mean / M2, refresh the applied statistics, clear the accumulator.  No __restrict__: one thread writes the count.
__device__ __forceinline__ void pnr_filter_merge_batch(double nb, double sum_d, double sum_q, double* slots, double* state,
                                                       float* applied, int demean, int destd) {
    const int c = threadIdx.x;
    const bool col_ok = c < PNR_OBS_DIM;
    const double na = state[0];
    const double n = nb > 0.0 ? na + nb : na;
    __syncthreads();                                            // everybody has read the old count and the accumulator
    if (col_ok) pnr_filter_merge_column(c, na, nb, n, sum_d, sum_q, state, applied, demean, destd);
    if (c == 0) state[0] = n;
    pnr_filter_clear_slots(slots, c, col_ok);
}

// Once per iteration, entirely on the device: the batch is `merged` (the merged delta of all ranks) or else this rank's
// accumulator, folded
__global__ void __launch_bounds__(PNR_FILTER_THREADS)
pnr_filter_sync_kernel(double* slots, const double* merged, double* state, float* applied, int demean, int destd) {
    const int c = threadIdx.x;
    const bool col_ok = c < PNR_OBS_DIM;
    auto batch = [&](int j) { return merged ? merged[j] : pnr_filter_fold_column(slots, j); };
    pnr_filter_merge_batch(batch(0), col_ok ? batch(1 + c) : 0.0, col_ok ? batch(1 + PNR_OBS_DIM + c) : 0.0, slots, state,
                           applied, demean, destd);
}

// ---------------------------------------------------------------------------------------------
// The path's one exchange as ONE kernel over NVLink peer memory (pnr_iteration_sync): what a rollout worker hands to
// the trainer once per iteration (episode statistics, pioneer/launch/pioneer_knm_train.py:49 + cli.py:32-38; the
// observation filter's delta, :66).  One CTA, thread = one double of the packed vector [8 statistics | 275 filter sums]:
//   1. snapshot: thread i < 8 reads statistics field i (thread 0 then clears the window), thread 8 + j folds column j of
//      the filter's accumulator copies;
//   2. publish: every thread stores its double into slot [parity][my rank] of EVERY rank's window -- plain stores to
//      peer-mapped addresses, NVLink carries them -- then one thread per peer releases flag [parity][my rank] = seq there;
//   3. wait: thread r polls its own window's flag [parity][r] (acquire, system scope) until rank r's data is in;
//   4. merge: every thread combines its double over the ranks IN RANK ORDER (identical bits on every rank): sum, or max /
//      min for the return extrema; the filter columns then go through the Chan merge into the running statistics.
// `seq` counts the calls and lives in the window, so a captured graph replays with fresh sequence numbers; two parities
// suffice because a rank can only enter call k + 2 after every rank has published call k + 1, i.e. finished call k.
// A wait that exceeds `timeout_ns` poisons the output with NaN and raises the window's status word instead of hanging.
// ---------------------------------------------------------------------------------------------
static_assert(PNR_SYNC_THREADS >= PNR_STATS_LEN + PNR_FILTER_DELTA_LEN, "one thread per packed double");
static_assert(PNR_SYNC_STATUS_OFF + 4 <= PNR_SYNC_WINDOW_BYTES, "window layout exceeds PNR_SYNC_WINDOW_BYTES");

__device__ __forceinline__ void pnr_st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t pnr_ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double pnr_ld_volatile_f64(const double* p) {
    double v;
    asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t pnr_globaltimer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__global__ void __launch_bounds__(PNR_SYNC_THREADS)
pnr_iteration_sync_kernel(PnrStats* stats, int clear, double* filt_slots, double* filt_state, float* applied, int demean,
                          int destd, const PnrSyncPeers peers, unsigned long long timeout_ns, double* out) {
    __shared__ double merged_s[PNR_SYNC_THREADS];
    const int i = threadIdx.x;
    const int len = filt_slots ? PNR_STATS_LEN + PNR_FILTER_DELTA_LEN : PNR_STATS_LEN;
    // 1. snapshot
    double v = 0.0;
    if (i < PNR_STATS_LEN) {
        v = pnr_stats_read(stats, i);
    } else if (i < len) {
        v = pnr_filter_fold_column(filt_slots, i - PNR_STATS_LEN);
    }
    __syncthreads();                                            // every field is read before the window is cleared
    if (i == 0 && clear) pnr_stats_clear(stats);
    double acc = v;
    if (peers.world > 1) {
        unsigned char* mine = peers.window[peers.rank];
        uint32_t* seq_p = reinterpret_cast<uint32_t*>(mine + PNR_SYNC_SEQ_OFF);
        const uint32_t seq = *seq_p + 1;                        // written back by thread 0 behind the barrier below
        const size_t par = seq & 1u;
        // 2. publish
        if (i < len)
            for (int r = 0; r < peers.world; ++r)
                reinterpret_cast<double*>(peers.window[r])[(par * PNR_SYNC_MAX_PEERS + peers.rank) * PNR_SYNC_SLOT_STRIDE + i] = v;
        __threadfence_system();
        __syncthreads();
        bool ok = true;
        if (i < peers.world) {
            pnr_st_release_sys(reinterpret_cast<uint32_t*>(peers.window[i] + PNR_SYNC_FLAGS_OFF) + par * PNR_SYNC_MAX_PEERS +
                                   peers.rank, seq);
            // 3. wait
            const uint32_t* flag = reinterpret_cast<const uint32_t*>(mine + PNR_SYNC_FLAGS_OFF) + par * PNR_SYNC_MAX_PEERS + i;
            const uint64_t t0 = pnr_globaltimer_ns();
            while (pnr_ld_acquire_sys(flag) != seq) {
                if (timeout_ns && pnr_globaltimer_ns() - t0 > timeout_ns) { ok = false; break; }
            }
        }
        const int all_ok = __syncthreads_and(ok ? 1 : 0);
        // 4. merge, in rank order
        if (i < len) {
            const double* sl = reinterpret_cast<const double*>(mine) + par * PNR_SYNC_MAX_PEERS * PNR_SYNC_SLOT_STRIDE + i;
            acc = pnr_ld_volatile_f64(sl);
            for (int r = 1; r < peers.world; ++r)
                acc = pnr_stats_combine(i, acc, pnr_ld_volatile_f64(sl + (size_t)r * PNR_SYNC_SLOT_STRIDE));
            if (!all_ok) acc = __longlong_as_double(0x7ff8000000000000ll);
        }
        if (i == 0) {
            *seq_p = seq;
            if (!all_ok) *reinterpret_cast<uint32_t*>(mine + PNR_SYNC_STATUS_OFF) = 1u;
        }
    }
    if (i < len) out[i] = acc;
    if (!filt_slots) return;
    merged_s[i] = acc;
    __syncthreads();
    const double* batch = merged_s + PNR_STATS_LEN;             // [count, sum_d[137], sum_q[137]]
    const bool col_ok = i < PNR_OBS_DIM;
    if (batch[0] == batch[0])
        pnr_filter_merge_batch(batch[0], col_ok ? batch[1 + i] : 0.0, col_ok ? batch[1 + PNR_OBS_DIM + i] : 0.0, filt_slots,
                               filt_state, applied, demean, destd);
    else                    // a poisoned (timed-out) exchange leaves the statistics alone; the accumulator is still cleared
        pnr_filter_clear_slots(filt_slots, i, col_ok);
}

cudaError_t pnr_launch_filter_refresh(const double* state, float* applied, int demean, int destd, cudaStream_t stream) {
    pnr_filter_refresh_kernel<<<1, PNR_FILTER_THREADS, 0, stream>>>(state, applied, demean, destd);
    return cudaGetLastError();
}

cudaError_t pnr_launch_filter_sync(double* slots, const double* merged, double* state, float* applied, int demean, int destd,
                                   cudaStream_t stream) {
    pnr_filter_sync_kernel<<<1, PNR_FILTER_THREADS, 0, stream>>>(slots, merged, state, applied, demean, destd);
    return cudaGetLastError();
}

cudaError_t pnr_launch_iteration_sync(PnrStats* stats, int clear, double* filt_slots, double* filt_state, float* applied,
                                      int demean, int destd, const PnrSyncPeers& peers, unsigned long long timeout_ns,
                                      double* out, cudaStream_t stream) {
    pnr_iteration_sync_kernel<<<1, PNR_SYNC_THREADS, 0, stream>>>(stats, clear, filt_slots, filt_state, applied, demean, destd,
                                                                  peers, timeout_ns, out);
    return cudaGetLastError();
}

cudaError_t pnr_launch_filter_fold(double* delta_slots, cudaStream_t stream) {
    pnr_filter_fold_kernel<<<(PNR_FILTER_DELTA_LEN + 127) / 128, 128, 0, stream>>>(delta_slots);
    return cudaGetLastError();
}

cudaError_t pnr_launch_filter(int device, const float* in, float* out, int64_t n_rows, const float* applied,
                              double* delta, float clip, int update, int normalize, cudaStream_t stream) {
    static int resident[PNR_MAX_DEVICES] = {};
    int& res = resident[device % PNR_MAX_DEVICES];
    if (res == 0) {
        cudaError_t e = pnr_prepare((const void*)pnr_filter_kernel, device, PNR_FILTER_THREADS, PNR_FILTER_TILE_BYTES, &res);
        if (e != cudaSuccess) return e;
    }
    if (n_rows <= 0) return cudaSuccess;
    int64_t grid = (n_rows + PNR_FILTER_ROWS - 1) / PNR_FILTER_ROWS;
    if (grid > res) grid = res;
    pnr_filter_kernel<<<(unsigned)grid, PNR_FILTER_THREADS, PNR_FILTER_TILE_BYTES, stream>>>(in, out, n_rows, applied, delta,
                                                                                            clip, update, normalize);
    return cudaGetLastError();
}
