// Kernels of the kinematic reach env (Tier A): fused step, reset, observe, state get/set, stats.
// sm_100a; launched from pnr_api.cu.
#include "pnr_kernels.cuh"
#include "pnr_launch.h"

// ---------------------------------------------------------------------------------------------
// K1: the fused env step.  One CTA of 4 warps owns a tile of 32 envs (lane = env); the work of ONE env is
// split across the 4 warps so that its dependent instruction chain is ~4x shorter and 4x more warps are
// resident per byte of shared memory than with one thread per env:
//   warps 0..2 ("joint warps") : joints 2k, 2k+1 -- act() integrator (pioneer_knm_env.py:111-146), their
//                                21 + 21 observation columns incl. 10 (sin, cos) pairs, state planes RV_k, A_k
//   warp 3     ("task warp")   : forward kinematics of the pointer from the joint warps' sin/cos (read back
//                                from the tile), reward / done / TimeLimit (:151-165), episode statistics,
//                                auto-reset (reset_world, :76-105), observation tail, planes X0, X1,
//                                reward / done outputs, and the TMA bulk store of the finished tile
// A rollout fragment (PnrMulti, n_steps steps in one launch) runs TILE-OUTER, STEP-INNER: a CTA takes a tile, runs all
// n_steps steps on it, then takes its next tile.  Every warp reads its state planes once when a tile starts, keeps the env
// state in registers across the steps -- in the layout of its planes: r, v | a of its two joints for a joint warp, target,
// t | potential, return for the task warp -- and writes it back once after the tile's last step.
// The CTA's work items, (tile, step) in that order, alternate between TWO tile buffers and run as a producer / consumer
// pipeline coupled only by named barriers:
//   HEAD[b]  joint warps arrive once r, cos r, sin r of their joints are in buffer b; the task warp waits on it
//   DONE[b]  joint warps arrive once all their columns (and, after a tile's last step, planes) are written; the task warp
//            waits, then stores
//   FREE[b]  the task warp arrives once the bulk store of the item before this one has been read AND this item's resets
//            are published (below); joint warps wait before they write the head of the next item into buffer b
//   JOINT    (OBSTACLES only) the three joint warps among themselves, once their heads are in the tile: each then sums the
//            penetration depths of its share of the capsule table into shared memory; the task warp adds the three partials
//            behind DONE and only then writes reward, return and episode statistics
// Step s + 1 of an env depends on step s only through an auto-reset, and only the task warp decides it.  Before it arrives
// at FREE it publishes the item's reset mask and, for the reset lanes, the new joint angles (and box) in shared memory.  The
// joint warps integrate the next step of the tile from their registers before they wait on FREE and redo it from the
// reset state for the (rare) masked lanes after it.  So no barrier spans the whole CTA: the joint warps work on item i+1
// while the task warp finishes item i, across step and tile boundaries alike.  A ragged last tile (a byte count that is
// no multiple of 16, so no bulk store) is streamed out by the task warp alone, under the same protocol.
// Grid = min(tiles, resident CTAs of the whole GPU); grid-stride over tiles.
// ---------------------------------------------------------------------------------------------
// In-kernel auto-reset of ONE env by the task warp once its step is decided: new joint angles, target and box from the Philox
// stream (a = v = 0, potential = 0, elapsed = 0).  The joint angles, and the box of the random-box variant, go to the lane's
// column of `pub` (stride 32) for the joint warps' next step of the tile, the box also to its plane; after the tile's LAST
// step the env's eight state planes are written too.  In PNR_OBS_AUTORESET mode the env's observation row is replaced by the
// first observation of the new episode.  Returns the new target.
// Rare (once per episode), so deliberately not inlined: keeps registers and code out of the hot loop.
// (Tried and dropped: drawing the next episode as soon as the TimeLimit hit is known, before the task warp waits for the
// joint warps -- the divergent Philox lane delays the whole task warp, which IS the critical path there: 11.8 -> 12.9 us
// per 65,536-env step.)
template <int OBS_MODE, bool OBSTACLES>
__device__ __noinline__ float4 pnr_auto_reset(const PnrParams& p, float4* __restrict__ state, int64_t env, uint64_t tickdom,
                                              float* __restrict__ row, float* __restrict__ pub, bool last) {
    PnrEnv s;
    float q[PNR_DOF], tg[3], box[5];
    pnr_reset_draws(p, p.env_id_base + env, pnr_reset_key(p, tickdom), q, tg, box);
    pnr_reset_env(s, q, tg);
    pnr_store_box(p, env, box);
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) pub[i * 32] = q[i];
    if (OBSTACLES && p.random_box >= 0) {
#pragma unroll
        for (int i = 0; i < 5; ++i) pub[(PNR_DOF + i) * 32] = box[i];
    }
    if (last) pnr_store_env(state, p.n_envs, env, s);
    if (OBS_MODE == PNR_OBS_AUTORESET) {
        PnrPose o;
        pnr_pose<true>(p, s, o);                              // fresh joint angles lie inside the limits
        pnr_pack_obs_dyn<true>(p, row, s, o, s.pot);
    }
    return make_float4(tg[0], tg[1], tg[2], 0.f);
}

// FILTER = true fuses the observation normaliser (pnr_filter.cu, 'ConcurrentMeanStdFilter') into the step: what leaves the
// kernel is clip((x - mean) * inv_std), and the column statistics of the raw values go to the same float64 accumulator
// pnr_filter_apply feeds, so the 548 B/env observation is never re-read.  Every warp normalises the columns it owns
// while the tile is still in shared memory: a joint warp runs one column pass (lane = one of its 30 changing
// columns, 32 rows, float64 sum / sum of squares of x - mean), the task warp normalises its 11 tail values in
// registers and adds them, per lane and per step, to float64 sums in shared memory; the 36 constant columns are normalised
// once per CTA and their statistics are added analytically by block 0.  The raw r / cos r / sin r the task warp needs for
// the forward kinematics travel through a small scratch area next to the tile buffers (the tile copy gets normalised).
template <int ARITH, int OBS_MODE, bool OBSTACLES, bool FILTER>
__global__ void __launch_bounds__(PNR_STEP_THREADS, FILTER ? PNR_STEP_MIN_CTAS_FILTER : PNR_STEP_MIN_CTAS)
pnr_step_kernel(const __grid_constant__ PnrParams p, float4* __restrict__ state, const float* __restrict__ actions,
                float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ done,
                PnrStats* __restrict__ stats, uint32_t tick, uint32_t domain, const float* __restrict__ f_applied,
                double* __restrict__ f_delta, float f_clip, const PnrMulti multi) {
    extern __shared__ __align__(128) float tiles[];           // PNR_STEP_BUFS tiles: the bulk store of one drains
    // the task warp's resets of its current item, for the joint warps' next step of the tile: lane mask, joint angles of
    // env `lane` at s_pub[j * 32 + lane]; OBSTACLES: rows 6..10 hold the tile's current per-env box (centre x y, half
    // extents x y z), written by joint warp 0 when a tile starts and by the task warp at a reset
    __shared__ uint32_t s_reset;
    __shared__ float s_pub[(OBSTACLES ? PNR_DOF + 5 : PNR_DOF) * 32];
    const int lane = threadIdx.x & 31;                        // while the next is being filled
    const int part = threadIdx.x >> 5;                        // warp-uniform role
    float* tile = tiles;
    float* row = tile + lane * PNR_OBS_DIM;
    float* scratch = tiles + PNR_STEP_BUFS * PNR_TILE_FLOATS; // FILTER only: raw r, cos r, sin r per env, per buffer
    float* srow = scratch + lane * PNR_FSCRATCH_STRIDE;
    // OBSTACLES only: partial contact depths of the three joint warps, per buffer [joint warp][env]
    float* const pen = scratch + (FILTER ? PNR_STEP_BUFS * PNR_FSCRATCH_FLOATS : 0);
    const int64_t N = p.n_envs;
    const int64_t n_tiles = (N + PNR_TILE_ENVS - 1) / PNR_TILE_ENVS;
    const int64_t stride = gridDim.x;
    int64_t t_idx = blockIdx.x;
    if (t_idx >= n_tiles) return;                             // CTA-uniform
    // back-to-back steps (pnr_step_many, CUDA graphs): the next step's CTAs may take the SM slots this grid's CTAs free one
    // by one and run their set-up (constant columns, barriers) under this grid's tail; they stop at pnr_pdl_wait()
    pnr_pdl_trigger();

    const int j0 = part < 3 ? 2 * part : 0;                   // first joint of a joint warp
    float* rowj = row + j0;
    // loop-invariant limits of this warp's two joints, read once from the constant bank
    const float vmax0 = p.v_max[j0], vmax1 = p.v_max[j0 + 1];
    const float rlo0 = p.r_lo[j0], rlo1 = p.r_lo[j0 + 1], rhi0 = p.r_hi[j0], rhi1 = p.r_hi[j0 + 1];
    float4* const rv_plane = pnr_plane_rv(state, N, part < 3 ? part : 0);
    float2* const a_plane = pnr_plane_a(state, N, part < 3 ? part : 0);
    float4* const x0_plane = pnr_plane_x0(state, N);
    float2* const x1_plane = pnr_plane_x1(state, N);

    // obs[18:54] never change: written once per CTA (into every tile buffer)
    if (part < 3) {
#pragma unroll
        for (int b = 0; b < PNR_STEP_BUFS; ++b) {
            pnr_pack_joint_const(p, row + b * PNR_TILE_FLOATS, j0);
            pnr_pack_joint_const(p, row + b * PNR_TILE_FLOATS, j0 + 1);
        }
    }
    // fused normaliser: the column this lane owns in the column pass, its applied statistics and accumulators
    int f_col = 0;
    float f_mean = 0.f, f_inv = 0.f;
    double f_sum = 0.0, f_sq = 0.0;
    __shared__ double f_tacc[FILTER ? 22 * 32 : 1];               // task warp: float64 sum / sum of squares per lane, per tail column
    if (FILTER) {
        if (part < 3) {
            // lanes 0..5 -> column blocks 0..2 (r, cos r, sin r), lanes 6..29 -> blocks 9..20; blocks 3..8 are constant
            const int kk = lane < 6 ? (lane >> 1) : (lane >> 1) + 6;
            f_col = 6 * kk + j0 + (lane & 1);
            if (lane < 30) { f_mean = f_applied[f_col]; f_inv = f_applied[PNR_OBS_DIM + f_col]; }
#pragma unroll
            for (int g = 0; g < 6; ++g) {                      // normalise the constant columns in place
#pragma unroll
                for (int jj = 0; jj < 2; ++jj) {
                    const int c = 18 + 6 * g + j0 + jj;
                    const float y = pnr_normalise(row[c], f_applied[c], f_applied[PNR_OBS_DIM + c], f_clip);
#pragma unroll
                    for (int b = 0; b < PNR_STEP_BUFS; ++b) row[b * PNR_TILE_FLOATS + c] = y;
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < 22; ++i) f_tacc[i * 32 + lane] = 0.0;   // each lane owns its column of f_tacc
        }
    }

    // the env state of the current tile in registers, in plane layout (joint warp: r r v v | a a; task warp: target t | potential
    // return); software pipeline: the next tile's planes and the next item's action are loaded while this item is worked on.
    // (State planes through L2 only: with programmatic dependent launch this CTA may have started on an SM before the previous
    // step finished elsewhere; nothing is re-read, so L1 would buy nothing.)
    float4 st4, ld4;
    float2 st2, ld2, ld_act = make_float2(0.f, 0.f);
    auto load_planes = [&](int64_t tile_idx) {
        const int64_t e_raw = tile_idx * PNR_TILE_ENVS + lane;
        const int64_t e = e_raw < N ? e_raw : N - 1;
        if (part < 3) {
            ld4 = __ldcg(rv_plane + e);
            ld2 = __ldcg(a_plane + e);
        } else {
            ld4 = __ldcg(x0_plane + e);
            ld2 = __ldcg(x1_plane + e);
        }
    };
    auto load_act = [&](int64_t tile_idx, int32_t s) {
        if (part < 3) {
            const int64_t e_raw = tile_idx * PNR_TILE_ENVS + lane;
            const int64_t e = e_raw < N ? e_raw : N - 1;
            ld_act = pnr_ld_stream(reinterpret_cast<const float2*>(actions + (int64_t)s * multi.act_stride + e * PNR_DOF) + part);
        }
    };
    pnr_pdl_wait();                                           // the previous step's state planes are complete and visible
    load_planes(t_idx);
    load_act(t_idx, 0);
    int buf = 0;
    int64_t iter = 0;                                         // work items this CTA has started
    int32_t step = 0;                                         // step of the fragment (PnrMulti; 1 step for pnr_step)

    for (;;) {
        const bool last = step + 1 == multi.n_steps;          // the tile's last step: its state goes back to the planes
        const int64_t next_tile = last ? t_idx + stride : t_idx;
        const bool more = next_tile < n_tiles;                // CTA-uniform: another item follows on this CTA
        // this step's buffers (launch-uniform bases)
        float* __restrict__ const obs_s = obs + (int64_t)step * multi.obs_stride;
        float* __restrict__ const reward_s = reward + (int64_t)step * N;
        uint8_t* __restrict__ const done_s = done + (int64_t)step * N;
        const uint32_t tick_s = tick + (uint32_t)step;
        const int64_t env_raw = t_idx * PNR_TILE_ENVS + lane;
        const bool active = env_raw < N;
        const int64_t env = active ? env_raw : N - 1;         // tail lanes shadow the last env, stores masked
        const int64_t rows_left = N - t_idx * PNR_TILE_ENVS;
        const int rows_valid = rows_left < PNR_TILE_ENVS ? (int)rows_left : PNR_TILE_ENVS;
        if (step == 0) { st4 = ld4; st2 = ld2; }              // a new tile: its state, read once
        const float2 c_act = ld_act;
        float4 box_a = make_float4(0.f, 0.f, 0.f, 0.f);       // OBSTACLES, joint warp 0: the new tile's boxes
        float box_z = 0.f;
        if (OBSTACLES && part == 0 && step == 0 && p.random_box >= 0) { box_a = p.box_a[env]; box_z = p.box_z[env]; }
        if (more) {
            if (last) load_planes(next_tile);
            load_act(next_tile, last ? 0 : step + 1);
        }

        float r1[2], v1[2], sn[2], cs[2];
        if (part < 3) {
            // --- act(): integrate with the PREVIOUS action (one-step actuation delay); registers only
            auto advance = [&]() {
                pnr_integrate_joint<ARITH>(p, vmax0, rlo0, rhi0, st2.x, st4.z, st4.x, v1[0], r1[0]);
                pnr_integrate_joint<ARITH>(p, vmax1, rlo1, rhi1, st2.y, st4.w, st4.y, v1[1], r1[1]);
                pnr_sincos_fast(r1[0], sn[0], cs[0]);         // r is inside the joint limits: fast path
                pnr_sincos_fast(r1[1], sn[1], cs[1]);
            };
            advance();
            if (iter >= 1) pnr_bar_sync2<PNR_BAR_FREE, PNR_STEP_THREADS>(buf);   // buffer reusable, resets published
            if (step > 0 && ((s_reset >> lane) & 1u)) {       // the task warp reset this env after the previous step
                st4 = make_float4(s_pub[j0 * 32 + lane], s_pub[(j0 + 1) * 32 + lane], 0.f, 0.f);
                st2 = make_float2(0.f, 0.f);
                advance();
            }
            pnr_pack_joint_head(rowj, r1[0], sn[0], cs[0]);
            pnr_pack_joint_head(rowj + 1, r1[1], sn[1], cs[1]);
            if (FILTER) {                                      // the raw values for the task warp's forward kinematics
                pnr_pack_joint_head(srow + j0, r1[0], sn[0], cs[0]);
                pnr_pack_joint_head(srow + j0 + 1, r1[1], sn[1], cs[1]);
            }
            pnr_bar_arrive2<PNR_BAR_HEAD, PNR_STEP_THREADS>(buf);
        } else {
            pnr_bar_sync2<PNR_BAR_HEAD, PNR_STEP_THREADS>(buf);   // r, cos r, sin r of all six joints are in the tile
        }

        bool do_reset = false;
        // OBSTACLES: what the task warp carries across the DONE barrier (the penalty is summed from the joint warps' partials)
        float d_rew = 0.f;
        int32_t d_t = 0;
        bool d_done = false, d_reached = false;
        if (part < 3) {
            // --- the other 15 dynamic columns of each joint; latch the new action (stored unclipped, :144)
            const bool fast = !p.trig_slow && fmaxf(fabsf(c_act.x), fabsf(c_act.y)) <= PNR_TRIG_FAST_LIMIT;
            pnr_pack_joint_rest(rowj, rlo0, rhi0, r1[0], v1[0], c_act.x, fast);
            pnr_pack_joint_rest(rowj + 1, rlo1, rhi1, r1[1], v1[1], c_act.y, fast);
            st4 = make_float4(r1[0], r1[1], v1[0], v1[1]);
            st2 = c_act;
            if (last && active) {
                rv_plane[env] = st4;
                a_plane[env] = st2;
            }
            if (OBSTACLES) {
                // capsule penetration depths, the capsule table split over the three joint warps (on the task warp alone
                // they were the CTA's critical path: 59 % of the stall samples were joint warps parked at DONE).  Every
                // joint's sin/cos is needed: the joint warps meet once their heads are in the tile.
                if (part == 0 && step == 0) {
                    s_pub[6 * 32 + lane] = box_a.x; s_pub[7 * 32 + lane] = box_a.y;
                    s_pub[8 * 32 + lane] = box_a.z; s_pub[9 * 32 + lane] = box_a.w; s_pub[10 * 32 + lane] = box_z;
                }
                pnr_bar_sync<PNR_BAR_JOINT, 3 * 32>();
                const float* head = FILTER ? srow : row;
                PnrSinCos sc;
#pragma unroll
                for (int i = 0; i < PNR_DOF; ++i) { sc.cs[i] = head[6 + i]; sc.sn[i] = head[12 + i]; }
                const float bz = s_pub[10 * 32 + lane];
                const PnrBox rb = {s_pub[6 * 32 + lane], s_pub[7 * 32 + lane], bz, s_pub[8 * 32 + lane], s_pub[9 * 32 + lane], bz};
                pen[(buf * 3 + part) * 32 + lane] = pnr_contact_depth(p, sc, rb, part, 3);
            }
            if (FILTER) {                                      // column pass over this warp's 30 changing columns
                __syncwarp();
                if (lane < 30) pnr_filter_column(tile + f_col, rows_valid, f_mean, f_inv, f_clip, f_sum, f_sq);
            }
        } else {
            // --- pose from the joint warps' sin/cos, distance, reward, done
            PnrPose o;
            const float* head = FILTER ? srow : row;           // raw r | cos r | sin r of this env
#pragma unroll
            for (int i = 0; i < PNR_DOF; ++i) { o.cs[i] = head[6 + i]; o.sn[i] = head[12 + i]; }
            const float tgt[3] = {st4.x, st4.y, st4.z};
            int32_t t = __float_as_int(st4.w);
            const float pot_old = st2.x;
            float ep_ret = st2.y;
            pnr_fk_tip(p, o.sn, o.cs, o.ptr);
            const float dx = tgt[0] - o.ptr[0], dy = tgt[1] - o.ptr[1], dz = tgt[2] - o.ptr[2];
            o.dist = sqrtf(fmaf(dx, dx, fmaf(dy, dy, dz * dz)));
            bool reached = o.dist < p.done_distance;
            if (fabsf(o.dist - p.done_distance) < p.done_band) {   // decide in float64 where float32 could flip it
                PnrBandIn in;
#pragma unroll
                for (int i = 0; i < PNR_DOF; ++i) in.r[i] = head[i];
                in.tgt[0] = tgt[0]; in.tgt[1] = tgt[1]; in.tgt[2] = tgt[2];
                const PnrBandOut bo = pnr_fk_band_f64(p, in);
                o.ptr[0] = bo.ptr[0]; o.ptr[1] = bo.ptr[1]; o.ptr[2] = bo.ptr[2];
                o.dist = bo.dist;
                reached = bo.within != 0;
            }
            const float pot_new = pnr_potential(p, o.dist);
            const float rew = pnr_reward(p, pot_old, pot_new, reached);
            t += 1;
            bool is_done;
            const uint8_t flags = pnr_step_flags(p, reached, t, is_done);
            if (active) done_s[env] = flags;
            if (OBSTACLES) {                                   // the penalty arrives with DONE: reward, return and statistics wait
                d_rew = rew; d_t = t; d_done = is_done; d_reached = reached;
            } else {
                ep_ret = __fadd_rn(ep_ret, rew);
                if (active) reward_s[env] = rew;
                pnr_episode_stats(stats, is_done && active, reached && active, ep_ret, t, lane);
            }

            // observation tail: pointer, target, difference, distance, potential (terminal values)
            float tail[11] = {o.ptr[0], o.ptr[1], o.ptr[2], tgt[0], tgt[1], tgt[2],
                              tgt[0] - o.ptr[0], tgt[1] - o.ptr[1], tgt[2] - o.ptr[2], o.dist, pot_new};
            if (FILTER) {                                      // normalise in registers, float64 statistics per lane
#pragma unroll
                for (int i = 0; i < 11; ++i) {
                    const float d = tail[i] - f_applied[126 + i];
                    if (active) {
                        const double e = (double)d;
                        f_tacc[i * 32 + lane] += e;
                        f_tacc[(11 + i) * 32 + lane] = fma(e, e, f_tacc[(11 + i) * 32 + lane]);
                    }
                    tail[i] = fminf(fmaxf(d * f_applied[PNR_OBS_DIM + 126 + i], -f_clip), f_clip);
                }
            }
#pragma unroll
            for (int i = 0; i < 11; ++i) row[126 + i] = tail[i];

            st4.w = __int_as_float(t);
            st2 = make_float2(pot_new, ep_ret);                // OBSTACLES: the return is completed behind DONE
            if (last && active) {
                x0_plane[env] = st4;
                if (!OBSTACLES) x1_plane[env] = st2;
            }
            do_reset = is_done && active && (p.auto_reset != 0);   // handled after DONE (rare)
        }
        pnr_fence_async_smem();                               // generic-proxy tile writes -> async proxy
        if (part < 3) pnr_bar_arrive2<PNR_BAR_DONE, PNR_STEP_THREADS>(buf);
        else pnr_bar_sync2<PNR_BAR_DONE, PNR_STEP_THREADS>(buf);   // tile complete (joint planes stored after a last step)

        if (part == 3) {
            if (OBSTACLES) {                                  // capsule penetration penalty, then the deferred writes
                const float* pb = pen + buf * PNR_PEN_FLOATS + lane;
                const float depth = (pb[0] + pb[32]) + pb[64];
                const float rew = pnr_contact_penalty(p, d_rew, depth);
                st2.y = __fadd_rn(st2.y, rew);
                if (active) {
                    reward_s[env] = rew;
                    if (last) x1_plane[env] = st2;
                }
                pnr_episode_stats(stats, d_done && active, d_reached && active, st2.y, d_t, lane);
            }
            // rare: auto-reset (reset_world, :76-105).  Only the auto-reset observation mode rewrites the row, so only there
            // does the reset have to precede the tile's store; terminal mode resets AFTER handing the tile to the copy engine.
            // Either way before FREE: that is where the joint warps pick the new episode up.
            const unsigned reset_mask = __ballot_sync(PNR_FULL_MASK, do_reset);
            float* const pub = s_pub + lane;
            const uint64_t tickdom = pnr_tickdom(tick_s, domain);
            if (OBS_MODE == PNR_OBS_AUTORESET && reset_mask) {
                if (do_reset) {
                    const float4 tg = pnr_auto_reset<OBS_MODE, OBSTACLES>(p, state, env, tickdom, row, pub, last);
                    st4 = make_float4(tg.x, tg.y, tg.z, __int_as_float(0));
                    st2 = make_float2(0.f, 0.f);
                }
                pnr_fence_async_smem();
            }
            __syncwarp();
            if (pnr_tile_is_bulk(rows_valid)) {
                if (lane == 0) {
                    pnr_bulk_store(obs_s + t_idx * (int64_t)PNR_TILE_FLOATS, tile,
                                   (uint32_t)(rows_valid * PNR_OBS_DIM * sizeof(float)));
                    pnr_bulk_commit();
                    // every store but the one just committed has finished READING its buffer: the previous item's
                    // buffer is free again
                    pnr_bulk_wait_read<1>();
                }
            } else {                                          // ragged last tile of the grid: the task warp streams it out
                pnr_emit_tile_manual(tile, obs_s + t_idx * (int64_t)PNR_TILE_FLOATS, rows_valid, lane, 32);
                if (lane == 0) pnr_bulk_wait_read<0>();
            }
            if (OBS_MODE != PNR_OBS_AUTORESET && do_reset) {
                const float4 tg = pnr_auto_reset<OBS_MODE, OBSTACLES>(p, state, env, tickdom, row, pub, last);
                st4 = make_float4(tg.x, tg.y, tg.z, __int_as_float(0));
                st2 = make_float2(0.f, 0.f);
            }
            if (lane == 0) s_reset = reset_mask;
            __syncwarp();
            if (more) pnr_bar_arrive2<PNR_BAR_FREE, PNR_STEP_THREADS>(buf ^ 1);
        }
        if (!more) break;
        t_idx = next_tile;
        step = last ? 0 : step + 1;
        buf ^= 1;                                             // next item goes into the other buffer
        ++iter;
        tile = tiles + buf * PNR_TILE_FLOATS;
        row = tile + lane * PNR_OBS_DIM;
        rowj = row + j0;
        if (FILTER) srow = scratch + buf * PNR_FSCRATCH_FLOATS + lane * PNR_FSCRATCH_STRIDE;
    }
    if (FILTER && f_delta != nullptr) {                       // column statistics of this CTA's rows, into copy blockIdx % SLOTS
        double* f_slot = pnr_filter_slot(f_delta, blockIdx.x);
        if (part < 3) {
            if (lane < 30) {
                atomicAdd(&f_slot[1 + f_col], f_sum);
                atomicAdd(&f_slot[1 + PNR_OBS_DIM + f_col], f_sq);
            }
            if (blockIdx.x == 0 && lane < 12)                  // the constant columns of all N rows, analytically
                pnr_filter_const_column(p, f_applied, f_delta, 18 + 6 * (lane >> 1) + j0 + (lane & 1), (double)N * multi.n_steps);
        } else {
#pragma unroll
            for (int i = 0; i < 11; ++i) {
                double a = f_tacc[i * 32 + lane], b = f_tacc[(11 + i) * 32 + lane];
#pragma unroll
                for (int ofs = 16; ofs > 0; ofs >>= 1) {
                    a += __shfl_xor_sync(PNR_FULL_MASK, a, ofs);
                    b += __shfl_xor_sync(PNR_FULL_MASK, b, ofs);
                }
                if (lane == 0) {
                    atomicAdd(&f_slot[1 + 126 + i], a);
                    atomicAdd(&f_slot[1 + PNR_OBS_DIM + 126 + i], b);
                }
            }
            if (blockIdx.x == 0 && lane == 0) atomicAdd(&f_delta[0], (double)N * multi.n_steps);
        }
    }
    if (part == 3 && lane == 0 && blockIdx.x == 0) atomicAdd(&stats->env_steps, (double)N * multi.n_steps);   // one writer per launch
    if (part == 3 && lane == 0) pnr_bulk_wait_read<0>();      // smem must outlive the copy engine's reads
}

// ---------------------------------------------------------------------------------------------
// K0: reset / observe on a list of envs (idx == nullptr: env k = k).  MODE 0 = reset, 1 = observe.
// ---------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(PNR_STEP_THREADS)
pnr_reset_observe_kernel(const __grid_constant__ PnrParams p, float4* __restrict__ state,
                         const int64_t* __restrict__ idx, int64_t n, const float* __restrict__ q0,
                         const float* __restrict__ target, float* __restrict__ obs_out, uint32_t tick) {
    extern __shared__ __align__(128) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* tile = smem + warp * PNR_TILE_FLOATS;
    const int64_t N = p.n_envs;
    const int64_t n_tiles = (n + PNR_TILE_ENVS - 1) / PNR_TILE_ENVS;
    bool tile_busy = false;
    for (int64_t t_idx = (int64_t)blockIdx.x * PNR_STEP_WARPS + warp; t_idx < n_tiles;
         t_idx += (int64_t)gridDim.x * PNR_STEP_WARPS) {
        const int64_t k_raw = t_idx * PNR_TILE_ENVS + lane;
        const bool active = k_raw < n;
        const int64_t k = active ? k_raw : n - 1;
        const int64_t env = idx ? idx[k] : k;
        PnrEnv s;
        if (MODE == 0) {
            float q[PNR_DOF], tg[3], box[5];
            pnr_reset_draws(p, p.env_id_base + env, pnr_reset_key(p, pnr_tickdom(tick, 0u)), q, tg, box);
            if (q0) {
#pragma unroll
                for (int i = 0; i < PNR_DOF; ++i) q[i] = q0[k * PNR_DOF + i];
            }
            if (target) { tg[0] = target[k * 3 + 0]; tg[1] = target[k * 3 + 1]; tg[2] = target[k * 3 + 2]; }
            pnr_reset_env(s, q, tg);
            if (active) { pnr_store_env(state, N, env, s); pnr_store_box(p, env, box); }
        } else {
            pnr_load_env(state, N, env, s);
        }
        if (obs_out) {
            // injected joint angles may lie anywhere: library sincos for every column here (not the hot path)
            PnrPose o;
            pnr_pose_reached<false>(p, s, o);
            if (tile_busy) pnr_tile_wait(lane);
            pnr_pack_obs_const(p, tile + lane * PNR_OBS_DIM);
            pnr_pack_obs_dyn<false>(p, tile + lane * PNR_OBS_DIM, s, o, s.pot);
            const int64_t rows_left = n - t_idx * PNR_TILE_ENVS;
            pnr_emit_tile(tile, obs_out + t_idx * (int64_t)PNR_TILE_FLOATS,
                          rows_left < PNR_TILE_ENVS ? (int)rows_left : PNR_TILE_ENVS, lane);
            tile_busy = true;
        }
    }
    if (lane == 0) pnr_bulk_wait_read<0>();
}

// ---------------------------------------------------------------------------------------------
// RLlib's reset_at(i) after a done (the sampler feeds the policy the RESET observation, bullet_env.py:187-190): for every
// env whose done flag is set -- pnr_step has already reset it -- optionally save the terminal row, then overwrite the row with
// the first observation of the new episode, normalised / pushed into the statistics like the step kernel's output when the
// filter is fused.  Rare rows, thread per env, scalar global stores; fixed launch shape, so it can live in a CUDA graph.
// ---------------------------------------------------------------------------------------------
__global__ void pnr_observe_done_kernel(const __grid_constant__ PnrParams p, float4* __restrict__ state,
                                        const uint8_t* __restrict__ done, float* __restrict__ obs,
                                        float* __restrict__ terminal_out, const float* __restrict__ f_applied,
                                        double* __restrict__ f_delta, float f_clip) {
    const int64_t N = p.n_envs;
    for (int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; env < N; env += (int64_t)gridDim.x * blockDim.x) {
        if (!(done[env] & PNR_DONE)) continue;
        float* row = obs + env * PNR_OBS_DIM;
        if (terminal_out) {
            float* dst = terminal_out + env * PNR_OBS_DIM;
            for (int c = 0; c < PNR_OBS_DIM; ++c) dst[c] = row[c];
        }
        PnrEnv s;
        pnr_load_env(state, N, env, s);
        PnrPose o;
        pnr_pose_reached<false>(p, s, o);
        pnr_pack_obs_const(p, row);
        pnr_pack_obs_dyn<false>(p, row, s, o, s.pot);
        if (f_applied) {
            double* slot = f_delta ? pnr_filter_slot(f_delta, (uint32_t)env) : nullptr;
            for (int c = 0; c < PNR_OBS_DIM; ++c) {
                if (slot) {
                    const double d = (double)(row[c] - f_applied[c]);
                    atomicAdd(&slot[1 + c], d);
                    atomicAdd(&slot[1 + PNR_OBS_DIM + c], d * d);
                }
                row[c] = pnr_normalise(row[c], f_applied[c], f_applied[PNR_OBS_DIM + c], f_clip);
            }
            if (slot) atomicAdd(&slot[0], 1.0);
        }
    }
}

cudaError_t pnr_launch_observe_done(const PnrParams& p, int device, float4* state, const uint8_t* done, float* obs,
                                    float* terminal_out, const float* f_applied, double* f_delta, float f_clip,
                                    cudaStream_t stream) {
    const int64_t cap = (int64_t)pnr_sm_count(device) * 8;
    int64_t grid = (p.n_envs + 127) / 128;
    if (grid > cap) grid = cap;
    pnr_observe_done_kernel<<<(unsigned)grid, 128, 0, stream>>>(p, state, done, obs, terminal_out, f_applied, f_delta, f_clip);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// state planes <-> row-major arrays (Joint.position()/velocity(), env.a/v/r/potential); utility path
// ---------------------------------------------------------------------------------------------
template <bool SET>
__global__ void pnr_state_io_kernel(float4* __restrict__ state, int64_t N, float* r, float* v, float* a,
                                    float* potential, float* target, int32_t* t, float* ep_return) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    PnrEnv s;
    pnr_load_env(state, N, e, s);
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) {
        if (r) { if (SET) s.r[i] = r[e * PNR_DOF + i]; else r[e * PNR_DOF + i] = s.r[i]; }
        if (v) { if (SET) s.v[i] = v[e * PNR_DOF + i]; else v[e * PNR_DOF + i] = s.v[i]; }
        if (a) { if (SET) s.a[i] = a[e * PNR_DOF + i]; else a[e * PNR_DOF + i] = s.a[i]; }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
        if (target) { if (SET) s.tgt[i] = target[e * 3 + i]; else target[e * 3 + i] = s.tgt[i]; }
    if (potential) { if (SET) s.pot = potential[e]; else potential[e] = s.pot; }
    if (t) { if (SET) s.t = t[e]; else t[e] = s.t; }
    if (ep_return) { if (SET) s.ep_ret = ep_return[e]; else ep_return[e] = s.ep_ret; }
    if (SET) pnr_store_env(state, N, e, s);
}

// per-env random box <-> row-major float[N,6] (centre xyz, half extents xyz); utility path
template <bool SET>
__global__ void pnr_box_io_kernel(float4* __restrict__ box_a, float* __restrict__ box_z, int64_t N, float* __restrict__ box) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    if (SET) {
        box_a[e] = make_float4(box[e * 6 + 0], box[e * 6 + 1], box[e * 6 + 3], box[e * 6 + 4]);
        box_z[e] = box[e * 6 + 5];                              // the box stands on z = 0: centre z = half height
    } else {
        const float4 a = box_a[e];
        const float z = box_z[e];
        box[e * 6 + 0] = a.x; box[e * 6 + 1] = a.y; box[e * 6 + 2] = z;
        box[e * 6 + 3] = a.z; box[e * 6 + 4] = a.w; box[e * 6 + 5] = z;
    }
}

// PNR_HOST_COMPACT: gather the 101 changing columns (0:18 and 54:137) of every row for the D2H copy; thread = output float
__global__ void pnr_compact_obs_kernel(const float* __restrict__ full, float* __restrict__ compact, int64_t n_out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = i / PNR_OBS_COMPACT_DIM;
        const int c = (int)(i - row * PNR_OBS_COMPACT_DIM);
        const int col = c < PNR_OBS_CONST_BEGIN ? c : c + (PNR_OBS_CONST_END - PNR_OBS_CONST_BEGIN);
        pnr_st_stream(compact + i, full[row * PNR_OBS_DIM + col]);
    }
}

__global__ void pnr_stats_snapshot_kernel(PnrStats* stats, double* out, int clear) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        for (int i = 0; i < PNR_STATS_LEN; ++i) out[i] = pnr_stats_read(stats, i);
        if (clear) pnr_stats_clear(stats);
    }
}

// The reduction half of the path's one collective: `gathered` = the packed statistics vectors of all ranks (what one
// all-gather delivered), combined in rank order by pnr_stats_combine; `extra` doubles per rank behind the eight (the
// observation filter's delta) are summed.  One small kernel instead of half a dozen indexing / reduction launches.
__global__ void pnr_stats_merge_kernel(const double* __restrict__ gathered, int world, int len, double* __restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= len) return;
    double acc = gathered[c];
    for (int r = 1; r < world; ++r) {
        acc = pnr_stats_combine(c, acc, gathered[(size_t)r * len + c]);
    }
    out[c] = acc;
}

cudaError_t pnr_launch_stats_merge(const double* gathered, int world, int len, double* out, cudaStream_t stream) {
    pnr_stats_merge_kernel<<<(len + 127) / 128, 128, 0, stream>>>(gathered, world, len, out);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// host-callable launchers (declared in pnr_launch.h)
// ---------------------------------------------------------------------------------------------
int pnr_sm_count(int device) {
    static int sms_of[PNR_MAX_DEVICES] = {};
    int& sms = sms_of[device % PNR_MAX_DEVICES];
    if (sms == 0) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    return sms;
}

cudaError_t pnr_prepare(const void* kernel, int device, int threads, size_t smem, int* resident) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
    *resident = pnr_sm_count(device) * (per_sm < 1 ? 1 : per_sm);
    return cudaSuccess;
}

// Resident CTAs per SM of the kinematic step kernel, measured on B200 (profiles/r03_step_65536.md): with the steps of a
// fragment pipelined per tile, 4 CTAs per SM stream best from 2,048 tiles on (131,072 envs: 14.2 us per step against 15.1
// with 5 or 6; 65,536 envs: 7.9 against 8.2 with 6); smaller grids keep 6 per SM so that up to 888 tiles run at once.
static int pnr_step_ctas_per_sm(int64_t n_tiles) { return n_tiles >= 2048 ? 4 : 6; }

// grid = min(CTAs needed, CTAs resident on the whole GPU): a multiple of the SM count once the batch is large
static int64_t pnr_grid_for(int64_t n_envs, int envs_per_cta, int resident) {
    const int64_t blocks = (n_envs + envs_per_cta - 1) / envs_per_cta;
    return blocks < resident ? (blocks > 0 ? blocks : 1) : resident;
}

cudaError_t pnr_launch_step(const PnrParams& p, int device, int arith, int obs_mode, float4* state, const float* actions, float* obs,
                            float* reward, uint8_t* done, PnrStats* stats, uint32_t tick, uint32_t domain, const float* f_applied,
                            double* f_delta, float f_clip, PnrMulti multi, cudaStream_t stream) {
    typedef void (*Kern)(const PnrParams, float4*, const float*, float*, float*, uint8_t*, PnrStats*, uint32_t, uint32_t,
                         const float*, double*, float, const PnrMulti);
    // the obstacle variant and the fused normaliser are separate instantiations: the plain kernel carries no trace of
    // them (a call site alone cost 40 % at 1M envs through caller-saved register spills)
    static Kern kernels[2][2][2] = {
        {{pnr_step_kernel<PNR_ARITH_F32, PNR_OBS_TERMINAL, false, false>, pnr_step_kernel<PNR_ARITH_F32, PNR_OBS_TERMINAL, true, false>},
         {pnr_step_kernel<PNR_ARITH_F32, PNR_OBS_AUTORESET, false, false>, pnr_step_kernel<PNR_ARITH_F32, PNR_OBS_AUTORESET, true, false>}},
        {{pnr_step_kernel<PNR_ARITH_LEGACY64, PNR_OBS_TERMINAL, false, false>, pnr_step_kernel<PNR_ARITH_LEGACY64, PNR_OBS_TERMINAL, true, false>},
         {pnr_step_kernel<PNR_ARITH_LEGACY64, PNR_OBS_AUTORESET, false, false>, pnr_step_kernel<PNR_ARITH_LEGACY64, PNR_OBS_AUTORESET, true, false>}}};
    static Kern fused[2] = {pnr_step_kernel<PNR_ARITH_F32, PNR_OBS_TERMINAL, false, true>,
                            pnr_step_kernel<PNR_ARITH_F32, PNR_OBS_TERMINAL, true, true>};
    static int grids[PNR_MAX_DEVICES][2][2][2][2] = {};  // cudaFuncSetAttribute is per device
    const int obst = p.n_obstacles > 0 ? 1 : 0;
    const int filt = f_applied != nullptr ? 1 : 0;
    if (filt && (arith != PNR_ARITH_F32 || obs_mode != PNR_OBS_TERMINAL)) return cudaErrorInvalidValue;
    Kern k = filt ? fused[obst] : kernels[arith][obs_mode][obst];
    const size_t smem = (filt ? PNR_STEP_SMEM_FILTER : PNR_STEP_SMEM) + (obst ? PNR_STEP_SMEM_OBST : 0);
    int& resident = grids[device % PNR_MAX_DEVICES][arith][obs_mode][obst][filt];
    if (resident == 0) {
        cudaError_t e = pnr_prepare((const void*)k, device, PNR_STEP_THREADS, smem, &resident);
        if (e != cudaSuccess) return e;
    }
    const int64_t n_tiles = (p.n_envs + PNR_TILE_ENVS - 1) / PNR_TILE_ENVS;
    const int cap = pnr_step_ctas_per_sm(n_tiles) * pnr_sm_count(device);
    const int64_t grid = pnr_grid_for(p.n_envs, PNR_TILE_ENVS, cap < resident ? cap : resident);
    // programmatic dependent launch pays where the launch tail is a visible share of the step (65,536 envs: 13.2 -> 11.8 us);
    // on long grids the early-resident successor only takes SM slots from this grid (1,048,576 envs: 146 -> 151 us).
    // One launch per fragment: fragments are timed the same with and without it (profiles/r03_step_65536.md)
    return pnr_launch_pdl(k, n_tiles <= 8192, grid, PNR_STEP_THREADS, smem, stream, p, state, actions, obs, reward, done,
                          stats, tick, domain, f_applied, f_delta, f_clip, multi);
}

cudaError_t pnr_launch_reset_observe(const PnrParams& p, int device, int mode, float4* state, const int64_t* idx, int64_t n,
                                     const float* q0, const float* target, float* obs_out, uint32_t tick,
                                     cudaStream_t stream) {
    typedef void (*Kern)(const PnrParams, float4*, const int64_t*, int64_t, const float*, const float*, float*, uint32_t);
    static Kern kernels[2] = {pnr_reset_observe_kernel<0>, pnr_reset_observe_kernel<1>};
    static int grids[PNR_MAX_DEVICES][2] = {};
    int& resident = grids[device % PNR_MAX_DEVICES][mode];
    if (resident == 0) {
        cudaError_t e = pnr_prepare((const void*)kernels[mode], device, PNR_STEP_THREADS, PNR_RO_SMEM, &resident);
        if (e != cudaSuccess) return e;
    }
    if (n <= 0) return cudaSuccess;
    const int64_t grid = pnr_grid_for(n, PNR_TILE_ENVS * PNR_STEP_WARPS, resident);
    kernels[mode]<<<(unsigned)grid, PNR_STEP_THREADS, PNR_RO_SMEM, stream>>>(p, state, idx, n, q0, target, obs_out, tick);
    return cudaGetLastError();
}

cudaError_t pnr_launch_state_io(bool set, float4* state, int64_t N, float* r, float* v, float* a, float* potential,
                                float* target, int32_t* t, float* ep_return, cudaStream_t stream) {
    const int threads = 256;
    const unsigned grid = (unsigned)((N + threads - 1) / threads);
    if (set) pnr_state_io_kernel<true><<<grid, threads, 0, stream>>>(state, N, r, v, a, potential, target, t, ep_return);
    else pnr_state_io_kernel<false><<<grid, threads, 0, stream>>>(state, N, r, v, a, potential, target, t, ep_return);
    return cudaGetLastError();
}

cudaError_t pnr_launch_box_io(bool set, float4* box_a, float* box_z, int64_t N, float* box, cudaStream_t stream) {
    const int threads = 256;
    const unsigned grid = (unsigned)((N + threads - 1) / threads);
    if (set) pnr_box_io_kernel<true><<<grid, threads, 0, stream>>>(box_a, box_z, N, box);
    else pnr_box_io_kernel<false><<<grid, threads, 0, stream>>>(box_a, box_z, N, box);
    return cudaGetLastError();
}

cudaError_t pnr_launch_compact_obs(int device, const float* full, float* compact, int64_t n_rows, cudaStream_t stream) {
    const int64_t n_out = n_rows * PNR_OBS_COMPACT_DIM;
    if (n_out <= 0) return cudaSuccess;
    const int64_t cap = (int64_t)pnr_sm_count(device) * 8;           // 8 CTAs of 256 threads per SM, grid-stride
    int64_t grid = (n_out + 255) / 256;
    if (grid > cap) grid = cap;
    pnr_compact_obs_kernel<<<(unsigned)grid, 256, 0, stream>>>(full, compact, n_out);
    return cudaGetLastError();
}

__global__ void pnr_tick_advance_kernel(PnrStats* stats, uint32_t n, int absolute) {
    if (threadIdx.x == 0 && blockIdx.x == 0) stats->tick_offset = absolute ? n : stats->tick_offset + n;
}
__global__ void pnr_env_steps_set_kernel(PnrStats* stats, double env_steps) {
    if (threadIdx.x == 0 && blockIdx.x == 0) stats->env_steps = env_steps;
}
cudaError_t pnr_launch_env_steps_set(PnrStats* stats, double env_steps, cudaStream_t stream) {
    pnr_env_steps_set_kernel<<<1, 32, 0, stream>>>(stats, env_steps);
    return cudaGetLastError();
}

cudaError_t pnr_launch_tick_advance(PnrStats* stats, uint32_t n, int absolute, cudaStream_t stream) {
    pnr_tick_advance_kernel<<<1, 32, 0, stream>>>(stats, n, absolute);
    return cudaGetLastError();
}

cudaError_t pnr_launch_stats_snapshot(PnrStats* stats, double* out, int clear, cudaStream_t stream) {
    pnr_stats_snapshot_kernel<<<1, 32, 0, stream>>>(stats, out, clear);
    return cudaGetLastError();
}
