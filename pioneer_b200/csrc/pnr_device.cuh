// Device-side parameter block, Philox reset generator and small math helpers shared by the kernels.
// sm_100a only (compiled with -gencode arch=compute_100a,code=sm_100a).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/pioneer_b200.h"

#define PNR_AXIS_X 0
#define PNR_AXIS_Y 1
#define PNR_AXIS_Z 2
#define PNR_AXIS_GENERAL 3

// Everything the kernels need besides per-env state.  Passed BY VALUE as a __grid_constant__ kernel
// parameter: it lands in the constant bank, reads are warp-uniform, and several handles with different
// configurations can coexist in one process (a __constant__ symbol could not).
struct PnrParams {
    // flattened chain, float32 copies for the hot path (pioneer_b200/urdf.py)
    float axis[PNR_DOF][3];
    float origin_xyz[PNR_DOF][3];
    float origin_rot[PNR_DOF][9];
    float tip_xyz[3];
    int32_t axis_code[PNR_DOF];     // PNR_AXIS_*: axis-aligned joints rotate with 4 FMA instead of Rodrigues
    float axis_sign[PNR_DOF];       // +1 / -1 for axis-aligned joints
    int32_t origin_has_rot[PNR_DOF];
    // float64 copies for the done-band re-evaluation (matches the reference's double-precision FK)
    double axis64[PNR_DOF][3];
    double origin_xyz64[PNR_DOF][3];
    double origin_rot64[PNR_DOF][9];
    double tip_xyz64[3];
    // bounds (pioneer_knm_env.py:56-58), all float32 like the reference
    float r_lo[PNR_DOF], r_hi[PNR_DOF], v_max[PNR_DOF];
    // the constant third of the observation: cos/sin of r_lo and r_hi (pioneer_knm_env.py:196-197)
    float cos_r_lo[PNR_DOF], sin_r_lo[PNR_DOF], cos_r_hi[PNR_DOF], sin_r_hi[PNR_DOF];
    float dt32, eps32;
    double dt64, eps64;
    float done_distance, done_band;
    float pot_max, pot_slope;       // (award_max - award_done), award_potential_slope
    float penalty_step, award_done;
    double done_distance64;
    float target_lo[3], target_hi[3];
    int32_t max_episode_steps;
    int32_t auto_reset;
    int32_t trig_slow;              // v_max beyond the fast sincos range: joint-rate columns take the library path
    // dynamic (Tier-B) mode: composite rigid body of each moving frame about the frame origin, control, stepping
    float dyn_io[PNR_DOF][6];       // rotational inertia about the frame origin: xx xy xz yy yz zz
    float dyn_mc[PNR_DOF][3];       // mass * centre of mass
    float dyn_mass[PNR_DOF];
    float dyn_tau_max[PNR_DOF];     // effort * torque_scale
    float dyn_damping[PNR_DOF];
    // the tip body's articulated inertia after its own rank-1 update (I^a = I^A - U U^T / d): constants of the robot,
    // float64 on the host (pnr_build_params).  I, M symmetric (xx xy xz yy yz zz), H row-major, U = (ua; ul), 1 / d
    float dyn_tip_I[6], dyn_tip_H[9], dyn_tip_M[6], dyn_tip_ua[3], dyn_tip_ul[3], dyn_tip_dinv;
    float dyn_kp, dyn_kd, dyn_dt, dyn_gravity;
    int32_t dyn_frame_skip, dyn_use_pd;
    // opt-in Bullet-like substep (PNR_STEPPING_BULLET; oracle/dynamics_oracle.c::dyn_substep_bullet)
    int32_t dyn_stepping;
    float dyn_com[PNR_DOF][3];      // centre of mass of each composite body, moving-frame coordinates
    float dyn_icom[PNR_DOF][6];     // rotational inertia about the centre of mass: xx xy xz yy yz zz
    float dyn_link_damping, dyn_max_velocity, dyn_motor_kp, dyn_motor_kd, dyn_motor_impulse;   // impulse = force * dt
    int32_t chain_kind;             // 1: axes Z Y Y X Y X, positive, identity origin rotations (the shipped robot)
    int32_t dyn_iso_links;          // 1: every link but the tip has its centre of mass on the frame origin and an isotropic inertia
    // obstacle variant: link capsules (moving-frame coordinates) against static plane / box / sphere obstacles
    int32_t n_capsules, n_obstacles;
    int32_t capsule_body[PNR_MAX_CAPSULES];
    float capsule_radius[PNR_MAX_CAPSULES];
    float capsule_p0[PNR_MAX_CAPSULES][3], capsule_p1[PNR_MAX_CAPSULES][3];
    int32_t obstacle_type[PNR_MAX_OBSTACLES];
    float obstacle_p[PNR_MAX_OBSTACLES][3], obstacle_e[PNR_MAX_OBSTACLES][3];
    float contact_penalty;
    // per-env random box (pioneer/temp/pioneer_env.py:169-192): obstacle `random_box` (-1: none) is redrawn at every reset;
    // centre x y | half extents x y live in box_a[env], the half height (= centre z: the box stands on z = 0) in box_z[env]
    int32_t random_box;
    float box_pos_lo[2], box_pos_hi[2], box_size_lo[3], box_size_hi[3];
    float4* box_a;
    float* box_z;
    const struct PnrStats* stats_ro;   // the handle's PnrStats (reset key of graph-captured launches: seed, device-side tick advance)
    uint32_t seed_lo, seed_hi;         // the reset key of eager launches (the host keeps it current; no global load on that path)
    int64_t env_id_base;
    int64_t n_envs;
};

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11), bit-identical to oracle/reach_oracle.py::philox4x32_10
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 pnr_philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ float pnr_u01(uint32_t x) { return __fmul_rn((float)(x >> 8), 5.9604644775390625e-08f); }

// lo + (hi - lo) * u with separately rounded multiply and add (no FMA) so the CPU oracle reproduces it
__device__ __forceinline__ float pnr_uniform(float lo, float hi, float u) {
    return __fadd_rn(lo, __fmul_rn(__fsub_rn(hi, lo), u));
}

// Reset key.  The Philox key is the seed, which lives in DEVICE memory (PnrStats::seed_*; pnr_seed reaches kernels that are
// already captured in a CUDA graph); the counter is (global env id lo, hi, tick, block | domain << 8).  `tick` is the host's
// call counter for eager launches (domain 0); launches captured into CUDA graph number g (domain g >= 1) add the device-side
// offset that pnr_tick_advance bumps once per replay, so no (domain, tick) pair is ever used twice.
struct PnrResetKey { uint32_t seed_lo, seed_hi, tick, domain; };

// 6 joint positions then 3 target coordinates (reference draw order, pioneer_knm_env.py:80-90), then the per-env box of the
// obstacle variant: 3 half extents, 2 centre coordinates (draw order of pioneer/temp/pioneer_env.py:173-174)
__device__ __forceinline__ void pnr_reset_draws(const PnrParams& p, int64_t global_env, PnrResetKey k,
                                                float (&q)[PNR_DOF], float (&tgt)[3], float (&box)[5]) {
    const uint32_t g0 = (uint32_t)global_env, g1 = (uint32_t)((uint64_t)global_env >> 32), dom = k.domain << 8;
    const uint4 b0 = pnr_philox4x32_10(make_uint4(g0, g1, k.tick, dom | 0u), k.seed_lo, k.seed_hi);
    const uint4 b1 = pnr_philox4x32_10(make_uint4(g0, g1, k.tick, dom | 1u), k.seed_lo, k.seed_hi);
    const uint4 b2 = pnr_philox4x32_10(make_uint4(g0, g1, k.tick, dom | 2u), k.seed_lo, k.seed_hi);
    q[0] = pnr_uniform(p.r_lo[0], p.r_hi[0], pnr_u01(b0.x));
    q[1] = pnr_uniform(p.r_lo[1], p.r_hi[1], pnr_u01(b0.y));
    q[2] = pnr_uniform(p.r_lo[2], p.r_hi[2], pnr_u01(b0.z));
    q[3] = pnr_uniform(p.r_lo[3], p.r_hi[3], pnr_u01(b0.w));
    q[4] = pnr_uniform(p.r_lo[4], p.r_hi[4], pnr_u01(b1.x));
    q[5] = pnr_uniform(p.r_lo[5], p.r_hi[5], pnr_u01(b1.y));
    tgt[0] = pnr_uniform(p.target_lo[0], p.target_hi[0], pnr_u01(b1.z));
    tgt[1] = pnr_uniform(p.target_lo[1], p.target_hi[1], pnr_u01(b1.w));
    tgt[2] = pnr_uniform(p.target_lo[2], p.target_hi[2], pnr_u01(b2.x));
    if (p.random_box >= 0) {                                  // warp-uniform (constant bank)
        const uint4 b3 = pnr_philox4x32_10(make_uint4(g0, g1, k.tick, dom | 3u), k.seed_lo, k.seed_hi);
        box[2] = pnr_uniform(p.box_size_lo[0], p.box_size_hi[0], pnr_u01(b2.y));     // half extents x y z
        box[3] = pnr_uniform(p.box_size_lo[1], p.box_size_hi[1], pnr_u01(b2.z));
        box[4] = pnr_uniform(p.box_size_lo[2], p.box_size_hi[2], pnr_u01(b2.w));
        box[0] = pnr_uniform(p.box_pos_lo[0], p.box_pos_hi[0], pnr_u01(b3.x));       // centre x y (z = half height)
        box[1] = pnr_uniform(p.box_pos_lo[1], p.box_pos_hi[1], pnr_u01(b3.y));
    }
}
__device__ __forceinline__ void pnr_store_box(const PnrParams& p, int64_t env, const float (&box)[5]) {
    if (p.random_box >= 0) {
        p.box_a[env] = make_float4(box[0], box[1], box[2], box[3]);
        p.box_z[env] = box[4];
    }
}

// np.clip for scalars: NaN propagates (comparisons are false)
template <typename T>
__device__ __forceinline__ T pnr_clip(T x, T lo, T hi) { return x < lo ? lo : (x > hi ? hi : x); }

// ---------------------------------------------------------------------------------------------
// streaming global accesses: state planes are re-read next step (keep in L2), observations are
// written once and consumed by someone else (evict-first so they do not push the state out of L2)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pnr_st_stream(float4* ptr, const float4& v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(ptr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void pnr_st_stream(float* ptr, float v) {
    asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(ptr), "f"(v) : "memory");
}
__device__ __forceinline__ float2 pnr_ld_stream(const float2* ptr) {
    float2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(ptr));
    return v;
}

// ---------------------------------------------------------------------------------------------
// TMA bulk store shared -> global (cp.async.bulk, sm_90+/sm_100a): one elected lane hands a whole
// contiguous observation tile to the copy engine instead of 35 LDS.128 + STG.128 round trips per lane.
// Protocol: every writer executes fence.proxy.async (generic-proxy smem writes -> async proxy), the warp
// syncs, one lane issues + commits; before the tile is overwritten that lane waits for the READ of smem.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pnr_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void pnr_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void pnr_bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(gdst), "r"(pnr_smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pnr_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void pnr_bulk_wait_read() {      // returns once at most PENDING groups still read smem
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(PENDING) : "memory");
}

// Programmatic dependent launch (sm_90+): a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may
// start while its predecessor in the stream is still draining; pnr_pdl_wait() blocks until the predecessor has completed
// and its memory is visible (everything that touches env state comes after it), pnr_pdl_trigger() lets the successor's
// CTAs be scheduled as soon as this grid's CTAs free their SM slots.  Both are no-ops for ordinary launches.
__device__ __forceinline__ void pnr_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pnr_pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// A rollout fragment in ONE launch of the kinematic step kernel (pnr_step_many): the CTA runs the n_steps consecutive steps
// of each of its tiles before it takes the next tile -- tiles never depend on each other, so no grid-wide synchronisation is
// needed between the steps.  Step s reads actions + s * act_stride and writes obs + s * obs_stride (floats), reward / done
// + s * N.  n_steps = 1 for an ordinary pnr_step.
struct PnrMulti { int32_t n_steps; int64_t act_stride, obs_stride; };

// named CTA barriers (ids 1..15; id 0 is __syncthreads): producer warps ARRIVE without waiting, the consumer SYNCs.
// `count` = all participating threads (arrivers + waiters).  Both order prior shared / global accesses of the CTA.
// The ids are immediates: with register ids ptxas reserves all 16 barriers per CTA, which caps the SM at 4 CTAs.
template <int ID, int COUNT>
__device__ __forceinline__ void pnr_bar_sync() { asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(COUNT) : "memory"); }
template <int ID, int COUNT>
__device__ __forceinline__ void pnr_bar_arrive() { asm volatile("bar.arrive %0, %1;" ::"n"(ID), "n"(COUNT) : "memory"); }
// barrier pair selected by the (CTA-uniform) tile buffer index
template <int ID, int COUNT>
__device__ __forceinline__ void pnr_bar_sync2(int buf) { if (buf) pnr_bar_sync<ID + 1, COUNT>(); else pnr_bar_sync<ID, COUNT>(); }
template <int ID, int COUNT>
__device__ __forceinline__ void pnr_bar_arrive2(int buf) { if (buf) pnr_bar_arrive<ID + 1, COUNT>(); else pnr_bar_arrive<ID, COUNT>(); }

// orderable unsigned encoding of a float (for atomicMax/atomicMin on episode returns)
__device__ __host__ __forceinline__ uint32_t pnr_float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
    const uint32_t u = __float_as_uint(f);
#else
    uint32_t u; memcpy(&u, &f, 4);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __host__ __forceinline__ float pnr_ordered_to_float(uint32_t o) {
    const uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}

// device-side episode statistics (one per handle)
struct PnrStats {
    double episodes, sum_return, sum_length, sum_return_sq, reached;
    double env_steps;               // env-steps since the last clear: counted by the step kernels, so graph replays count too
    uint32_t max_return_ord, min_return_ord;
    // added to the host's call counter where a kernel keys the reset generator (in-kernel auto-reset).  The host counter
    // is a kernel argument and therefore FROZEN into a captured CUDA graph; pnr_tick_advance bumps this one from inside
    // the graph, so every replay draws fresh reset states.  0 unless pnr_tick_advance is used.
    uint32_t tick_offset;
    uint32_t seed_lo, seed_hi;      // the reset generator's key (pnr_create / pnr_seed)
};
// The statistics window as the host reads it, PNR_STATS_LEN doubles: episodes, sum of returns, sum of lengths, sum of squared
// returns, max return, min return, env-steps, reached.
__device__ __forceinline__ double pnr_stats_read(const PnrStats* stats, int i) {
    switch (i) {
        case 0: return stats->episodes;
        case 1: return stats->sum_return;
        case 2: return stats->sum_length;
        case 3: return stats->sum_return_sq;
        case 4: return (double)pnr_ordered_to_float(stats->max_return_ord);
        case 5: return (double)pnr_ordered_to_float(stats->min_return_ord);
        case 6: return stats->env_steps;
        default: return stats->reached;
    }
}
__device__ __forceinline__ void pnr_stats_clear(PnrStats* stats) {
    stats->episodes = stats->sum_return = stats->sum_length = stats->sum_return_sq = stats->reached = 0.0;
    stats->env_steps = 0.0;
    stats->max_return_ord = pnr_float_to_ordered(-INFINITY);
    stats->min_return_ord = pnr_float_to_ordered(INFINITY);
}
// how ranks combine field i of their windows, in rank order: MAX of the max returns, MIN of the min returns, SUM of the rest
// (and of whatever follows the window in a packed vector, the observation filter's sums)
__device__ __forceinline__ double pnr_stats_combine(int i, double acc, double x) {
    return i == 4 ? fmax(acc, x) : (i == 5 ? fmin(acc, x) : acc + x);
}
// tickdom = domain << 32 | host call counter: ONE 64-bit argument for the rare, non-inlined reset paths
__device__ __forceinline__ PnrResetKey pnr_reset_key(const PnrParams& p, uint64_t tickdom) {
    PnrResetKey k;
    k.domain = (uint32_t)(tickdom >> 32);
    if (k.domain) {                 // captured in a CUDA graph: the parameter block is frozen, seed and advance live in memory
        const PnrStats* __restrict__ stats = p.stats_ro;
        k.seed_lo = stats->seed_lo; k.seed_hi = stats->seed_hi;
        k.tick = (uint32_t)tickdom + stats->tick_offset;
    } else {
        k.seed_lo = p.seed_lo; k.seed_hi = p.seed_hi;
        k.tick = (uint32_t)tickdom;
    }
    return k;
}
__device__ __forceinline__ uint64_t pnr_tickdom(uint32_t tick, uint32_t domain) { return ((uint64_t)domain << 32) | tick; }
