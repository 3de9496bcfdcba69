// K2 kernel template, shared by pnr_dynamic.cu (explicit substep) and pnr_dynamic_bullet.cu (opt-in Bullet-like substep): the
// two sets of instantiations compile in parallel.
#pragma once
#include "pnr_kernels.cuh"
#include "pnr_dynamics.cuh"
#include "pnr_launch.h"

typedef void (*PnrDynKernel)(const PnrParams, float4*, const float*, float*, float*, uint8_t*, PnrStats*, uint32_t, uint32_t,
                             const float*, double*, float, const PnrMulti);
// [chain][obs_mode][obstacles] of the Bullet-like instantiations (pnr_dynamic_bullet.cu)
PnrDynKernel pnr_dynamic_bullet_kernel(int chain, int obs_mode, int obst);

// Launch shape (v6).  The substep loop is FP32-issue bound and every warp's dependent chain is long, so what matters is
// how many warps an SM holds and that a 65,536-env launch (2,048 tiles) fits in ONE wave.  v5 held 12 warps per SM (three
// 4-warp CTAs: 163 registers, and four 17.5 KB observation tiles per CTA capped shared memory at three CTAs), i.e. 1,776
// warp slots -> a second, 13 % full wave.  v6: CTAs of 2 warps, 8 per SM = 16 warps = 2,368 slots, which needs
//   * <= 128 registers per thread (ptxas gets there without a spill once the launch bound asks for it; 10 CTAs = 96
//     registers spill and measured 22 % slower), and
//   * half the staging memory per warp: the observation tile leaves in two halves of 16 rows through one 8.8 KB buffer.
// Measured on B200 (tools/ab_dynamic.py, fragments of 8 steps): 65,536 envs 41.0 -> 37.1 us per step, 131,072 envs 68.3 ->
// 66.8, 1,048,576 envs 452.5 -> 458 (the two rounds cost 1 % where the second wave does not exist).
// The packing work is not repeated for the second half: in round h the 16 envs of half h are packed by ALL 32 lanes, lane
// pair (l, l + 16) sharing one env -- its owner packs joints 0..2 and the tail, the partner lane joints 3..5 from values
// it received by ONE set of warp shuffles (shfl.xor 16 serves both rounds, the roles swap).  Same instructions per tile as
// packing 32 rows at once, same results (the per-joint pack functions are the kinematic kernel's).
#ifndef PNR_DYN_WARPS
#define PNR_DYN_WARPS 2
#endif
#ifndef PNR_DYN_MIN_CTAS
#define PNR_DYN_MIN_CTAS 8
#endif
#define PNR_DYN_THREADS (PNR_DYN_WARPS * 32)
#define PNR_HALF_ROWS 16
#define PNR_HALF_FLOATS (PNR_HALF_ROWS * PNR_OBS_DIM)             // 2,192 floats = 8,768 B = one TMA bulk store
#define PNR_DYN_SMEM (PNR_DYN_WARPS * PNR_HALF_FLOATS * sizeof(float))

template <int OBS_MODE, bool OBSTACLES, int CHAIN, int STEPPING>
__global__ void __launch_bounds__(PNR_DYN_THREADS, STEPPING == PNR_STEPPING_BULLET ? 4 : PNR_DYN_MIN_CTAS)
pnr_step_dynamic_kernel(const __grid_constant__ PnrParams p, float4* __restrict__ state, const float* __restrict__ actions,
                        float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ done,
                        PnrStats* __restrict__ stats, uint32_t tick, uint32_t domain, const float* __restrict__ f_applied,
                        double* __restrict__ f_delta, float f_clip, const PnrMulti multi) {
    extern __shared__ __align__(128) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int hl = lane & 15;                                  // row of the half tile this lane packs
    const bool upper = lane >= 16;
    float* tile = smem + warp * PNR_HALF_FLOATS;
    float* row = tile + hl * PNR_OBS_DIM;
    const int64_t N = p.n_envs;
    const int64_t n_tiles = (N + PNR_TILE_ENVS - 1) / PNR_TILE_ENVS;
    bool tile_busy = false;
    pnr_pdl_trigger();                                         // see pnr_step_kernel: the next step's set-up runs under this tail
    // obs[18:54] never change: written once per warp; the lane pair of a row shares them (r_lo block / r_hi block)
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) {
        if (!upper) { row[18 + i] = p.r_lo[i]; row[24 + i] = p.cos_r_lo[i]; row[30 + i] = p.sin_r_lo[i]; }
        else { row[36 + i] = p.r_hi[i]; row[42 + i] = p.cos_r_hi[i]; row[48 + i] = p.sin_r_hi[i]; }
    }
    // fused observation normaliser (pnr_filter_fuse; warp-uniform run-time switch): after a half tile is packed the warp
    // runs the column pass of pnr_filter_kernel on its 101 changing columns (lane = column, four passes) and pushes the
    // float64 column sums to accumulator copy blockIdx % SLOTS.  The 36 constant columns are normalised here, once, and
    // their statistics added analytically by one thread of the grid.
    const bool filt = f_applied != nullptr;
    if (filt) {
        __syncwarp();
        const int c0 = upper ? 36 : 18;
#pragma unroll
        for (int c = 0; c < 18; ++c)
            row[c0 + c] = pnr_normalise(row[c0 + c], f_applied[c0 + c], f_applied[PNR_OBS_DIM + c0 + c], f_clip);
    }
    pnr_pdl_wait();                                            // the previous step's state planes are complete and visible
    for (int64_t t_idx = (int64_t)blockIdx.x * PNR_DYN_WARPS + warp; t_idx < n_tiles;
         t_idx += (int64_t)gridDim.x * PNR_DYN_WARPS) {
        const int64_t env_raw = t_idx * PNR_TILE_ENVS + lane;
        const bool active = env_raw < N;
        const int64_t env = active ? env_raw : N - 1;

        PnrEnv s;
        pnr_load_env_cg(state, N, env, s);
        // a rollout fragment in ONE launch (PnrMulti, pnr_step_many): the warp keeps its tile and runs n_steps consecutive
        // steps on it with the env state in registers -- tiles never depend on each other (1 for an ordinary pnr_step)
#pragma unroll 1
        for (int32_t step = 0; step < multi.n_steps; ++step) {
        const float2* a2 = reinterpret_cast<const float2*>(actions + (int64_t)step * multi.act_stride + env * PNR_DOF);
        const float2 act01 = pnr_ld_stream(a2), act23 = pnr_ld_stream(a2 + 1), act45 = pnr_ld_stream(a2 + 2);
        // the action drives THIS step's substeps (a motor target, not the kinematic env's delayed acceleration)
        s.a[0] = act01.x; s.a[1] = act01.y; s.a[2] = act23.x; s.a[3] = act23.y; s.a[4] = act45.x; s.a[5] = act45.y;
        pnr_dynamic_substeps<CHAIN, STEPPING>(p, s.r, s.v, s.a);
        // this step's output buffers (launch-uniform; formed after the substep loop so that nothing but `step` lives across it)
        float* __restrict__ const obs_s = obs + (int64_t)step * multi.obs_stride;
        float* __restrict__ const reward_s = reward + (int64_t)step * N;
        uint8_t* __restrict__ const done_s = done + (int64_t)step * N;
        const uint32_t tick_s = tick + (uint32_t)step;

        PnrPose o;
        const bool reached = pnr_pose_reached<true>(p, s, o);   // q is inside the joint limits
        const float pot_new = pnr_potential(p, o.dist);
        float rew = pnr_reward(p, s.pot, pot_new, reached);
        if (OBSTACLES) {
            PnrSinCos sc;
#pragma unroll
            for (int i = 0; i < PNR_DOF; ++i) { sc.sn[i] = o.sn[i]; sc.cs[i] = o.cs[i]; }
            rew = pnr_contact_penalty(p, rew, pnr_contact_depth(p, sc, pnr_load_box(p, env), 0, 1));
        }
        s.pot = pot_new;
        s.t += 1;
        s.ep_ret = __fadd_rn(s.ep_ret, rew);
        bool is_done;
        const uint8_t flags = pnr_step_flags(p, reached, s.t, is_done);
        if (active) {
            reward_s[env] = rew;
            done_s[env] = flags;
        }
        pnr_episode_stats(stats, is_done && active, reached && active, s.ep_ret, s.t, lane);

        float vmax_abs = 0.f;                                  // joint rates are not bounded by construction here
#pragma unroll
        for (int i = 0; i < PNR_DOF; ++i) vmax_abs = fmaxf(vmax_abs, fmaxf(fabsf(s.v[i]), fabsf(s.a[i])));
        bool fast = !p.trig_slow && vmax_abs <= PNR_TRIG_FAST_LIMIT;
        const bool do_reset = is_done && (p.auto_reset != 0);
        // what the observation shows: the post-substep state (terminal mode), or the fresh episode for finished envs
        PnrEnv so = s;
        if (do_reset) {
            float q[PNR_DOF], tg[3], box[5];
            pnr_reset_draws(p, p.env_id_base + env, pnr_reset_key(p, pnr_tickdom(tick_s, domain)), q, tg, box);
            pnr_reset_env(s, q, tg);
            if (active) pnr_store_box(p, env, box);
        }
        if (OBS_MODE == PNR_OBS_AUTORESET) {
            if (__any_sync(PNR_FULL_MASK, do_reset)) {
                PnrPose o2;
                pnr_pose<true>(p, s, o2);
                if (do_reset) { o = o2; so = s; fast = true; }
            }
        }
        if (step + 1 == multi.n_steps) {                        // the state goes back to memory after the tile's last step
            if (active) pnr_store_env(state, N, env, s);
        }

        // ---- observation: two half tiles of 16 rows; in round h the lane pair (l, l + 16) packs env 16 h + l
        // the partner lane receives joints 3..5 of its pair's env (one exchange serves both rounds)
        float pr[3], psn[3], pcs[3], pv[3], pa[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            pr[k] = __shfl_xor_sync(PNR_FULL_MASK, so.r[3 + k], 16);
            psn[k] = __shfl_xor_sync(PNR_FULL_MASK, o.sn[3 + k], 16);
            pcs[k] = __shfl_xor_sync(PNR_FULL_MASK, o.cs[3 + k], 16);
            pv[k] = __shfl_xor_sync(PNR_FULL_MASK, so.v[3 + k], 16);
            pa[k] = __shfl_xor_sync(PNR_FULL_MASK, so.a[3 + k], 16);
        }
        const bool pfast = __shfl_xor_sync(PNR_FULL_MASK, fast ? 1 : 0, 16) != 0;
        const int64_t rows_left = N - t_idx * PNR_TILE_ENVS;
        const int rows_valid = rows_left < PNR_TILE_ENVS ? (int)rows_left : PNR_TILE_ENVS;
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
            const int rows_half = min(max(rows_valid - h * PNR_HALF_ROWS, 0), PNR_HALF_ROWS);
            if (rows_half == 0) break;                         // warp-uniform
            if (tile_busy) pnr_tile_wait(lane);
            const bool owner = upper == (h == 1);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int j = owner ? k : 3 + k;
                float* rowj = row + j;
                const float r = owner ? so.r[k] : pr[k];
                pnr_pack_joint_head(rowj, r, owner ? o.sn[k] : psn[k], owner ? o.cs[k] : pcs[k]);
                pnr_pack_joint_rest(rowj, owner ? p.r_lo[k] : p.r_lo[3 + k], owner ? p.r_hi[k] : p.r_hi[3 + k], r,
                                    owner ? so.v[k] : pv[k], owner ? so.a[k] : pa[k], owner ? fast : pfast);
            }
            if (owner) {
                row[126] = o.ptr[0]; row[127] = o.ptr[1]; row[128] = o.ptr[2];
                row[129] = so.tgt[0]; row[130] = so.tgt[1]; row[131] = so.tgt[2];
                row[132] = so.tgt[0] - o.ptr[0]; row[133] = so.tgt[1] - o.ptr[1]; row[134] = so.tgt[2] - o.ptr[2];
                row[135] = o.dist;
                row[136] = so.pot;
            }
            if (filt) {
                __syncwarp();
                double* f_slot = f_delta ? pnr_filter_slot(f_delta, blockIdx.x) : nullptr;
#pragma unroll 1
                for (int pass = 0; pass < 4; ++pass) {
                    const int cc = pass * 32 + lane;                   // index among the 101 changing columns
                    if (cc < PNR_OBS_DIM - 36) {
                        const int c = cc < 18 ? cc : cc + 36;
                        // pnr_filter_column written out: as a call it costs 4 to 16 bytes more spill in three instantiations
                        const float mean = f_applied[c], inv = f_applied[PNR_OBS_DIM + c];
                        float* colp = tile + c;
                        double s0 = 0.0, q0 = 0.0, s1 = 0.0, q1 = 0.0;
                        int r = 0;
#pragma unroll 4
                        for (; r + 1 < rows_half; r += 2) {
                            const float d0 = colp[r * PNR_OBS_DIM] - mean, d1 = colp[(r + 1) * PNR_OBS_DIM] - mean;
                            const double e0 = (double)d0, e1 = (double)d1;
                            s0 += e0; q0 = fma(e0, e0, q0);
                            s1 += e1; q1 = fma(e1, e1, q1);
                            colp[r * PNR_OBS_DIM] = fminf(fmaxf(d0 * inv, -f_clip), f_clip);
                            colp[(r + 1) * PNR_OBS_DIM] = fminf(fmaxf(d1 * inv, -f_clip), f_clip);
                        }
                        if (r < rows_half) {
                            const float d0 = colp[r * PNR_OBS_DIM] - mean;
                            const double e0 = (double)d0;
                            s0 += e0; q0 = fma(e0, e0, q0);
                            colp[r * PNR_OBS_DIM] = fminf(fmaxf(d0 * inv, -f_clip), f_clip);
                        }
                        if (f_slot) {
                            atomicAdd(&f_slot[1 + c], s0 + s1);
                            atomicAdd(&f_slot[1 + PNR_OBS_DIM + c], q0 + q1);
                        }
                    }
                }
            }
            pnr_emit_tile(tile, obs_s + t_idx * (int64_t)PNR_TILE_FLOATS + (int64_t)h * PNR_HALF_FLOATS, rows_half, lane);
            tile_busy = true;
        }
        }                                                       // steps of the fragment
    }
    if (filt && f_delta && blockIdx.x == 0 && warp == 0) {         // rows pushed + the constant columns of all N rows
        if (lane == 0) atomicAdd(&f_delta[0], (double)N * multi.n_steps);
        for (int c = 18 + lane; c < 54; c += 32) pnr_filter_const_column(p, f_applied, f_delta, c, (double)N * multi.n_steps);
    }
    if (blockIdx.x == 0 && warp == 0 && lane == 0) atomicAdd(&stats->env_steps, (double)N * multi.n_steps);   // one writer per launch
    if (lane == 0) pnr_bulk_wait_read<0>();
}

