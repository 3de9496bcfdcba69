// C-ABI of pioneer_b200 (include/pioneer_b200.h): handle lifetime, parameter block, launches.
// No torch types, no exceptions across the boundary, no CPU fallback.
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <new>
#include <string>

#include "pnr_launch.h"

static thread_local std::string g_last_error;

static int pnr_fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

#define PNR_CUDA(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess)                                                                  \
            return pnr_fail(PNR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

struct pnr_handle {
    int device = 0;
    int64_t n_envs = 0;
    PnrParams params;
    pnr_config cfg;
    pnr_model model;
    float4* state = nullptr;        // 6 planes of float4[n_envs]
    PnrStats* stats = nullptr;
    double* stats_out = nullptr;    // device double[8] snapshot
    double* stats_host = nullptr;   // pinned
    uint32_t tick = 0;              // keys the reset generator: one tick per reset/step call
    uint64_t seed = 0;              // host copy of the key in PnrStats::seed_*
    uint32_t n_graphs = 0;          // CUDA graphs this handle's steps were captured into: each gets its own reset-key domain
    unsigned long long capture_id = 0;
    float4* box_a = nullptr;        // per-env random box (cfg.random_box): centre x y | half extents x y
    float* box_z = nullptr;         //                                      half height = centre z
    int64_t launches = 0;
    float a_max[PNR_DOF];
    // observation normaliser (pnr_filter_*): device accumulator, applied statistics, host-side running statistics
    double* filt_delta = nullptr;        // device double[PNR_FILTER_SLOTS][PNR_FILTER_DELTA_LEN]; copy 0 is what is read
    float* filt_applied = nullptr;       // device float[2 * PNR_OBS_DIM]: mean, 1 / (std + 1e-8)
    double* filt_state = nullptr;        // device double[PNR_FILTER_DELTA_LEN]: running count, mean[137], M2[137]
    double* filt_merged = nullptr;       // device staging for a merged delta handed in from the host
    double filt_clip = 10.0;
    int filt_demean = 1, filt_destd = 1;
    int filt_fused = 0, filt_fused_update = 1;   // pnr_filter_fuse: the step kernel normalises and pushes statistics
    // host-buffer path (pnr_step_host, pnr_step_host_begin / _end): two device staging sets, so that the D2H of step k
    // (copy streams) overlaps H2D + kernel of step k + 1 (compute stream)
    struct HostSlot {
        float *actions = nullptr, *obs = nullptr, *reward = nullptr, *compact = nullptr;
        uint8_t* done = nullptr;
        cudaEvent_t kernel_done = nullptr, copy1_done = nullptr, copy2_done = nullptr;
        bool busy = false;
    } slot[2];
    bool host_ready = false;
    int host_next = 0, host_inflight = 0;
    cudaStream_t host_stream = nullptr, copy_stream1 = nullptr, copy_stream2 = nullptr;
    cudaEvent_t host_order_event = nullptr;
    // pnr_iteration_sync: this rank's window and the peers' windows as mapped into this process
    unsigned char* sync_window = nullptr;
    PnrSyncPeers sync_peers = {};
    bool sync_ipc_opened[PNR_SYNC_MAX_PEERS] = {};
};

struct PnrDeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit PnrDeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~PnrDeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// Build stamp: the content hash of the sources this library was built from (pioneer_b200/build.py looks for the marker
// in the file to decide whether the library is stale -- file times do not survive a snapshot copy to another box).
#ifndef PNR_SRC_HASH
#define PNR_SRC_HASH "unknown"
#endif
extern "C" const char* pnr_source_hash(void) { return "PNR_SRC_HASH:" PNR_SRC_HASH; }

extern "C" int pnr_abi_version(void) { return PNR_ABI_VERSION; }
extern "C" const char* pnr_last_error(void) { return g_last_error.c_str(); }

extern "C" void pnr_default_config(pnr_config* c) {
    if (!c) return;
    std::memset(c, 0, sizeof(*c));
    c->max_v_to_r = 2.0; c->max_a_to_v = 10.0;                  // pioneer_knm_env.py:21-22
    c->done_distance = 0.1;                                      // :24
    c->award_max = 100.0; c->award_done = 5.0;                   // :26-27
    c->award_potential_slope = 10.0; c->penalty_step = 1.0 / 100; // :28-29
    c->target_lo[0] = 15; c->target_lo[1] = -10; c->target_lo[2] = 2;   // :31
    c->target_hi[0] = 25; c->target_hi[1] = 10; c->target_hi[2] = 6;    // :32
    c->timestep = 1.0 / 240; c->frame_skip = 10; c->gravity = 0.0;      // bullet_env.py:38-41
    c->max_episode_steps = 500;                                  // pioneer_knm_train.py:27
    c->arith = PNR_ARITH_F32;
    c->obs_mode = PNR_OBS_TERMINAL;
    c->auto_reset = 1;
    c->mode = PNR_MODE_KINEMATIC;
    c->kp = 0.0; c->kd = 0.0; c->torque_scale = 1.0;
    c->n_obstacles = 0;
    c->contact_penalty = 0.0;
    // per-env random box, off; ranges around the demo box (half extents (0.5, 0.5, 5) at (10, 5, 0), pioneer_knm_env.py:249-255)
    c->random_box = 0;
    c->box_pos_lo[0] = 8; c->box_pos_lo[1] = -6; c->box_pos_hi[0] = 14; c->box_pos_hi[1] = 6;
    c->box_size_lo[0] = 0.3; c->box_size_lo[1] = 0.3; c->box_size_lo[2] = 3.0;
    c->box_size_hi[0] = 0.7; c->box_size_hi[1] = 0.7; c->box_size_hi[2] = 7.0;
    // Bullet-like substep, off; Bullet's defaults [UPSTREAM-MEMORY]
    c->stepping = PNR_STEPPING_EXPLICIT;
    c->link_damping = 0.04; c->max_velocity = 100.0;
    c->motor_kp = 0.1; c->motor_kd = 1.0; c->motor_max_force = 0.0;
}

static int pnr_build_params(const pnr_model& m, const pnr_config& c, int64_t n_envs, int64_t env_id_base,
                            uint64_t seed, PnrParams& p, float (&a_max)[PNR_DOF]) {
    std::memset(&p, 0, sizeof(p));
    if (m.dof != PNR_DOF) return pnr_fail(PNR_ERR_UNSUPPORTED, "pnr_model.dof must be 6 (PNR_DOF)");
    for (int j = 0; j < PNR_DOF; ++j) {
        double n2 = 0;
        for (int k = 0; k < 3; ++k) n2 += m.axis[j][k] * m.axis[j][k];
        if (std::fabs(n2 - 1.0) > 1e-9) return pnr_fail(PNR_ERR_INVALID, "pnr_model.axis must be unit vectors");
        int code = PNR_AXIS_GENERAL;
        float sign = 1.f;
        for (int k = 0; k < 3; ++k)
            if (std::fabs(std::fabs(m.axis[j][k]) - 1.0) < 1e-12) { code = k; sign = m.axis[j][k] > 0 ? 1.f : -1.f; }
        p.axis_code[j] = code;
        p.axis_sign[j] = sign;
        bool has_rot = false;
        for (int k = 0; k < 9; ++k) {
            const double ident = (k % 4 == 0) ? 1.0 : 0.0;
            if (std::fabs(m.origin_rot[j][k] - ident) > 1e-15) has_rot = true;
            p.origin_rot[j][k] = (float)m.origin_rot[j][k];
            p.origin_rot64[j][k] = m.origin_rot[j][k];
        }
        p.origin_has_rot[j] = has_rot ? 1 : 0;
        for (int k = 0; k < 3; ++k) {
            p.axis[j][k] = (float)m.axis[j][k];
            p.axis64[j][k] = m.axis[j][k];
            p.origin_xyz[j][k] = (float)m.origin_xyz[j][k];
            p.origin_xyz64[j][k] = m.origin_xyz[j][k];
        }
        // bounds exactly as the reference derives them (pioneer_knm_env.py:56-58, 217-220):
        // float32 limits; python scalar * float32 array stays float32
        p.r_lo[j] = (float)m.lower[j];
        p.r_hi[j] = (float)m.upper[j];
        p.v_max[j] = (float)c.max_v_to_r * (p.r_hi[j] - p.r_lo[j]);
        a_max[j] = (float)c.max_a_to_v * p.v_max[j];
        if (!(p.v_max[j] <= 1.0e5f)) p.trig_slow = 1;      // joint rates beyond the fast sincos range (pnr_trig.cuh)
        // the step kernel evaluates sin/cos of angles inside [r_lo, r_hi] and of limit distances with the fast path
        if (!(std::fabs(m.lower[j]) <= 1.0e4 && std::fabs(m.upper[j]) <= 1.0e4 && m.lower[j] <= m.upper[j]))
            return pnr_fail(PNR_ERR_UNSUPPORTED, "pnr_model joint limits must satisfy -1e4 <= lower <= upper <= 1e4 rad");
        // float32 cos/sin of float32 limits (np.cos on a float32 array); computed in double and rounded once
        p.cos_r_lo[j] = (float)std::cos((double)p.r_lo[j]); p.sin_r_lo[j] = (float)std::sin((double)p.r_lo[j]);
        p.cos_r_hi[j] = (float)std::cos((double)p.r_hi[j]); p.sin_r_hi[j] = (float)std::sin((double)p.r_hi[j]);
    }
    for (int k = 0; k < 3; ++k) {
        p.tip_xyz[k] = (float)m.tip_xyz[k];
        p.tip_xyz64[k] = m.tip_xyz[k];
        p.target_lo[k] = (float)c.target_lo[k];
        p.target_hi[k] = (float)c.target_hi[k];
    }
    if (!(c.timestep > 0) || c.frame_skip < 1) return pnr_fail(PNR_ERR_INVALID, "timestep/frame_skip must be positive");
    // dynamic mode: composite bodies about their frame origins (parallel-axis shift of the URDF inertials)
    for (int j = 0; j < PNR_DOF; ++j) {
        const double m_ = m.body_mass[j];
        const double* c_ = m.body_com[j];
        const double* I_ = m.body_inertia[j];
        const double cc = c_[0] * c_[0] + c_[1] * c_[1] + c_[2] * c_[2];
        const int idx[6][2] = {{0, 0}, {0, 1}, {0, 2}, {1, 1}, {1, 2}, {2, 2}};
        for (int k = 0; k < 6; ++k) {
            const int a = idx[k][0], b = idx[k][1];
            p.dyn_io[j][k] = (float)(I_[3 * a + b] + m_ * ((a == b ? cc : 0.0) - c_[a] * c_[b]));
        }
        for (int k = 0; k < 3; ++k) p.dyn_mc[j][k] = (float)(m_ * c_[k]);
        p.dyn_mass[j] = (float)m_;
        p.dyn_tau_max[j] = (float)(m.effort[j] * c.torque_scale);
        p.dyn_damping[j] = (float)m.damping[j];
        for (int k = 0; k < 3; ++k) p.dyn_com[j][k] = (float)c_[k];
        for (int k = 0; k < 6; ++k) p.dyn_icom[j][k] = (float)I_[3 * idx[k][0] + idx[k][1]];
        if (c.mode == PNR_MODE_DYNAMIC && !(m_ > 0.0))
            return pnr_fail(PNR_ERR_INVALID, "dynamic mode needs a positive composite mass on every moving frame");
    }
    {   // tip joint: I^A = own body only, so U = I^A S, d = S^T U and I^a = I^A - U U^T / d do not depend on the state
        const int j = PNR_DOF - 1;
        const double m_ = m.body_mass[j];
        const double* c_ = m.body_com[j];
        const double* I_ = m.body_inertia[j];
        const double cc = c_[0] * c_[0] + c_[1] * c_[1] + c_[2] * c_[2];
        double I3[3][3], H3[3][3], M3[3][3];
        const double mc[3] = {m_ * c_[0], m_ * c_[1], m_ * c_[2]};
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) {
                I3[a][b] = I_[3 * a + b] + m_ * ((a == b ? cc : 0.0) - c_[a] * c_[b]);
                M3[a][b] = a == b ? m_ : 0.0;
            }
        H3[0][0] = 0; H3[0][1] = -mc[2]; H3[0][2] = mc[1];
        H3[1][0] = mc[2]; H3[1][1] = 0; H3[1][2] = -mc[0];
        H3[2][0] = -mc[1]; H3[2][1] = mc[0]; H3[2][2] = 0;
        double ua[3], ul[3], d = 0;
        for (int a = 0; a < 3; ++a) {
            ua[a] = ul[a] = 0;
            for (int b = 0; b < 3; ++b) { ua[a] += I3[a][b] * m.axis[j][b]; ul[a] += H3[b][a] * m.axis[j][b]; }
        }
        for (int a = 0; a < 3; ++a) d += m.axis[j][a] * ua[a];
        const double dinv = d != 0.0 ? 1.0 / d : 0.0;
        const int idx[6][2] = {{0, 0}, {0, 1}, {0, 2}, {1, 1}, {1, 2}, {2, 2}};
        for (int k = 0; k < 6; ++k) {
            const int a = idx[k][0], b = idx[k][1];
            p.dyn_tip_I[k] = (float)(I3[a][b] - ua[a] * ua[b] * dinv);
            p.dyn_tip_M[k] = (float)(M3[a][b] - ul[a] * ul[b] * dinv);
        }
        for (int a = 0; a < 3; ++a) {
            for (int b = 0; b < 3; ++b) p.dyn_tip_H[3 * a + b] = (float)(H3[a][b] - ua[a] * ul[b] * dinv);
            p.dyn_tip_ua[a] = (float)ua[a];
            p.dyn_tip_ul[a] = (float)ul[a];
        }
        p.dyn_tip_dinv = (float)dinv;
        // I^a S = 0: for an axis-aligned tip joint (code k) column / row k of I^a and row k of H^a are exact zeros;
        // the specialised kernel relies on it (pnr_rotk_sym_z), so the rounding residue is cleared
        const int kt = p.axis_code[j];
        if (kt != PNR_AXIS_GENERAL)
            for (int a = 0; a < 3; ++a) {
                const int lo = a < kt ? a : kt, hi = a < kt ? kt : a;
                const int sym_index[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
                p.dyn_tip_I[sym_index[lo][hi]] = 0.f;
                p.dyn_tip_H[3 * kt + a] = 0.f;
            }
    }
    // obstacle variant; without a penalty weight there is nothing to compute
    p.contact_penalty = (float)c.contact_penalty;
    p.n_obstacles = (c.contact_penalty != 0.0) ? c.n_obstacles : 0;
    p.n_capsules = m.n_capsules;
    for (int i = 0; i < m.n_capsules; ++i)
        if (m.capsule_body[i] < 0 || m.capsule_body[i] >= PNR_DOF)
            return pnr_fail(PNR_ERR_INVALID, "pnr_model.capsule_body out of range");
    // the kernels walk the chain base-to-tip ONCE and visit the capsules of a body when its frame is current: the device table
    // is ordered by body (stable, so capsules of one body keep the caller's order)
    int order[PNR_MAX_CAPSULES];
    for (int i = 0; i < m.n_capsules; ++i) order[i] = i;
    std::stable_sort(order, order + m.n_capsules, [&](int a, int b) { return m.capsule_body[a] < m.capsule_body[b]; });
    for (int slot = 0; slot < m.n_capsules; ++slot) {
        const int i = slot, src = order[slot];
        p.capsule_body[i] = m.capsule_body[src];
        p.capsule_radius[i] = (float)m.capsule_radius[src];
        for (int k = 0; k < 3; ++k) { p.capsule_p0[i][k] = (float)m.capsule_p0[src][k]; p.capsule_p1[i][k] = (float)m.capsule_p1[src][k]; }
    }
    for (int i = 0; i < c.n_obstacles; ++i) {
        const int t = c.obstacle_type[i];
        if (t != PNR_OBSTACLE_PLANE && t != PNR_OBSTACLE_BOX && t != PNR_OBSTACLE_SPHERE)
            return pnr_fail(PNR_ERR_INVALID, "pnr_config.obstacle_type must be plane, box or sphere");
        p.obstacle_type[i] = t;
        for (int k = 0; k < 3; ++k) { p.obstacle_p[i][k] = (float)c.obstacle_p[i][k]; p.obstacle_e[i][k] = (float)c.obstacle_e[i][k]; }
    }
    {   // the shipped robot's axis pattern gets the specialised dynamics kernel (pnr_dynamics.cuh, PNR_CHAIN_PIONEER)
        const int pattern[PNR_DOF] = {PNR_AXIS_Z, PNR_AXIS_Y, PNR_AXIS_Y, PNR_AXIS_X, PNR_AXIS_Y, PNR_AXIS_X};
        bool match = true;
        const int origin_axis[PNR_DOF] = {-1, 2, 2, 1, 0, -1};       // the only non-zero origin component (-1: none)
        for (int j = 0; j < PNR_DOF; ++j) {
            match = match && p.axis_code[j] == pattern[j] && p.axis_sign[j] > 0.f && !p.origin_has_rot[j];
            match = match && std::fabs(m.lower[j]) <= 64.0 && std::fabs(m.upper[j]) <= 64.0;   // pnr_sincos_bounded in the ABA
            for (int k = 0; k < 3; ++k) match = match && (k == origin_axis[j] || m.origin_xyz[j][k] == 0.0);
        }
        p.chain_kind = match ? 1 : 0;
        // the stub inertials of the shipped URDF (pioneer_knm_6dof.urdf: mass, identity-like inertia, no <origin>):
        // composite bodies 0..4 have their centre of mass on the frame origin and an isotropic inertia (PNR_CHAIN_PIONEER_ISO)
        bool iso = true;
        for (int j = 0; j + 1 < PNR_DOF; ++j) {
            const double* c_ = m.body_com[j];
            const double* I_ = m.body_inertia[j];
            iso = iso && c_[0] == 0.0 && c_[1] == 0.0 && c_[2] == 0.0 && I_[1] == 0.0 && I_[2] == 0.0 && I_[3] == 0.0 &&
                  I_[5] == 0.0 && I_[6] == 0.0 && I_[7] == 0.0 && I_[0] == I_[4] && I_[4] == I_[8];
        }
        p.dyn_iso_links = iso ? 1 : 0;
    }
    if (c.stepping != PNR_STEPPING_EXPLICIT && c.stepping != PNR_STEPPING_BULLET)
        return pnr_fail(PNR_ERR_INVALID, "pnr_config.stepping must be PNR_STEPPING_EXPLICIT or PNR_STEPPING_BULLET");
    p.dyn_stepping = c.stepping;
    p.dyn_link_damping = (float)c.link_damping;
    p.dyn_max_velocity = (float)c.max_velocity;
    p.dyn_motor_kp = (float)c.motor_kp; p.dyn_motor_kd = (float)c.motor_kd;
    p.dyn_motor_impulse = (float)(c.motor_max_force * c.timestep);
    p.dyn_kp = (float)c.kp; p.dyn_kd = (float)c.kd;
    p.dyn_use_pd = (c.kp != 0.0 || c.kd != 0.0) ? 1 : 0;
    p.dyn_dt = (float)c.timestep;
    p.dyn_gravity = (float)c.gravity;
    p.dyn_frame_skip = c.frame_skip;
    p.dt64 = c.timestep * c.frame_skip;          // World.step_time, bullet_scene.py:277-279
    p.eps64 = 1e-5;                              // pioneer_knm_env.py:61
    p.dt32 = (float)p.dt64;
    p.eps32 = (float)p.eps64;
    p.done_distance = (float)c.done_distance;
    p.done_distance64 = c.done_distance;
    p.done_band = 1e-3f;                         // >> float32 FK error (~1e-5 at 30-unit reach)
    p.pot_max = (float)(c.award_max - c.award_done);
    p.pot_slope = (float)c.award_potential_slope;
    p.penalty_step = (float)c.penalty_step;
    p.award_done = (float)c.award_done;
    p.max_episode_steps = c.max_episode_steps;
    p.auto_reset = c.auto_reset;
    p.seed_lo = (uint32_t)seed;                  // eager launches; graph-captured ones read PnrStats::seed_*
    p.seed_hi = (uint32_t)(seed >> 32);
    p.random_box = -1;
    if (c.random_box) {
        for (int i = 0; i < c.n_obstacles && p.random_box < 0; ++i)
            if (c.obstacle_type[i] == PNR_OBSTACLE_BOX) p.random_box = i;
        if (p.random_box < 0) return pnr_fail(PNR_ERR_INVALID, "pnr_config.random_box needs a box among the obstacles");
        for (int k = 0; k < 2; ++k) { p.box_pos_lo[k] = (float)c.box_pos_lo[k]; p.box_pos_hi[k] = (float)c.box_pos_hi[k]; }
        for (int k = 0; k < 3; ++k) {
            p.box_size_lo[k] = (float)c.box_size_lo[k]; p.box_size_hi[k] = (float)c.box_size_hi[k];
            if (!(c.box_size_lo[k] > 0.0) || !(c.box_size_hi[k] >= c.box_size_lo[k]))
                return pnr_fail(PNR_ERR_INVALID, "pnr_config.box_size_lo / box_size_hi must be positive and ordered");
        }
        if (p.n_obstacles == 0) p.random_box = -1;           // no penalty weight: nothing reads the box
    }
    p.env_id_base = env_id_base;
    p.n_envs = n_envs;
    return PNR_OK;
}

// Developer / test hook (not part of include/pioneer_b200.h): the parameter block the kernels would receive for this
// model and configuration, built on the host without touching CUDA.  tests/csrc/aba_check.cu feeds it to the
// host-compiled dynamics header.  Returns sizeof(PnrParams), or a negative status.
extern "C" int64_t pnr_debug_build_params(const pnr_model* model, const pnr_config* cfg, int64_t n_envs, void* out,
                                          int64_t capacity) {
    if (!model || !cfg) return pnr_fail(PNR_ERR_INVALID, "pnr_debug_build_params: null argument");
    if (out && capacity >= (int64_t)sizeof(PnrParams)) {
        float a_max[PNR_DOF];
        int rc = pnr_build_params(*model, *cfg, n_envs, 0, 0, *static_cast<PnrParams*>(out), a_max);
        if (rc != PNR_OK) return rc;
    }
    return (int64_t)sizeof(PnrParams);
}

extern "C" int pnr_create(const pnr_model* model, const pnr_config* cfg, int64_t n_envs, int64_t env_id_base,
                          int device, uint64_t seed, pnr_handle** out) {
    if (!model || !cfg || !out) return pnr_fail(PNR_ERR_INVALID, "pnr_create: null argument");
    if (n_envs < 1) return pnr_fail(PNR_ERR_INVALID, "pnr_create: n_envs must be >= 1");
    if (cfg->arith != PNR_ARITH_F32 && cfg->arith != PNR_ARITH_LEGACY64)
        return pnr_fail(PNR_ERR_INVALID, "pnr_create: unknown arith");
    if (cfg->obs_mode != PNR_OBS_TERMINAL && cfg->obs_mode != PNR_OBS_AUTORESET)
        return pnr_fail(PNR_ERR_INVALID, "pnr_create: unknown obs_mode");
    if (cfg->mode != PNR_MODE_KINEMATIC && cfg->mode != PNR_MODE_DYNAMIC)
        return pnr_fail(PNR_ERR_INVALID, "pnr_create: unknown mode");
    if (cfg->mode == PNR_MODE_DYNAMIC && cfg->arith != PNR_ARITH_F32)
        return pnr_fail(PNR_ERR_UNSUPPORTED, "pnr_create: the dynamic mode computes in float32 (arith must be PNR_ARITH_F32)");
    if (cfg->n_obstacles < 0 || cfg->n_obstacles > PNR_MAX_OBSTACLES || model->n_capsules < 0 ||
        model->n_capsules > PNR_MAX_CAPSULES)
        return pnr_fail(PNR_ERR_INVALID, "pnr_create: too many obstacles / capsules");
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0)
        return pnr_fail(PNR_ERR_CUDA, std::string("pnr_create: no CUDA device (there is no CPU fallback): ") +
                                          cudaGetErrorString(ce));
    if (device < 0 || device >= count || device >= PNR_MAX_DEVICES)
        return pnr_fail(PNR_ERR_INVALID, "pnr_create: bad device index");
    pnr_handle* h = new (std::nothrow) pnr_handle();
    if (!h) return pnr_fail(PNR_ERR_ALLOC, "pnr_create: out of host memory");
    h->device = device;
    h->n_envs = n_envs;
    h->cfg = *cfg;
    h->model = *model;
    int rc = pnr_build_params(*model, *cfg, n_envs, env_id_base, seed, h->params, h->a_max);
    if (rc != PNR_OK) { delete h; return rc; }
    PnrDeviceGuard guard(device);
    if (!guard.ok) { delete h; return pnr_fail(PNR_ERR_CUDA, "pnr_create: cudaSetDevice failed"); }
    auto bail = [&](cudaError_t e, const char* what) {
        std::string msg = std::string(what) + ": " + cudaGetErrorString(e);
        pnr_destroy(h);
        return pnr_fail(e == cudaErrorMemoryAllocation ? PNR_ERR_ALLOC : PNR_ERR_CUDA, msg);
    };
    cudaError_t e;
    if ((e = cudaMalloc(&h->state, sizeof(float4) * 6 * (size_t)n_envs)) != cudaSuccess) return bail(e, "cudaMalloc(state)");
    if ((e = cudaMalloc(&h->stats, sizeof(PnrStats))) != cudaSuccess) return bail(e, "cudaMalloc(stats)");
    if ((e = cudaMemset(h->stats, 0, sizeof(PnrStats))) != cudaSuccess) return bail(e, "cudaMemset(stats)");
    h->params.stats_ro = h->stats;
    h->seed = seed;
    {
        const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
        if ((e = cudaMemcpy(reinterpret_cast<char*>(h->stats) + offsetof(PnrStats, seed_lo), key, sizeof(key),
                            cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "cudaMemcpy(seed)");
    }
    if (h->params.random_box >= 0) {
        if ((e = cudaMalloc(&h->box_a, sizeof(float4) * (size_t)n_envs)) != cudaSuccess) return bail(e, "cudaMalloc(box)");
        if ((e = cudaMalloc(&h->box_z, sizeof(float) * (size_t)n_envs)) != cudaSuccess) return bail(e, "cudaMalloc(box)");
        h->params.box_a = h->box_a;
        h->params.box_z = h->box_z;
    }
    if ((e = cudaMalloc(&h->stats_out, sizeof(double) * PNR_STATS_LEN)) != cudaSuccess) return bail(e, "cudaMalloc(stats_out)");
    if ((e = cudaMallocHost(&h->stats_host, sizeof(double) * PNR_STATS_LEN)) != cudaSuccess) return bail(e, "cudaMallocHost");
    // clear statistics, then reset every env (reset_world) with tick 0
    if ((e = pnr_launch_stats_snapshot(h->stats, h->stats_out, 1, nullptr)) != cudaSuccess) return bail(e, "stats init");
    if ((e = pnr_launch_reset_observe(h->params, device, 0, h->state, nullptr, n_envs, nullptr, nullptr, nullptr,
                                      h->tick, nullptr)) != cudaSuccess) return bail(e, "initial reset");
    h->launches += 2;
    h->tick += 1;
    if ((e = cudaStreamSynchronize(nullptr)) != cudaSuccess) return bail(e, "pnr_create sync");
    *out = h;
    return PNR_OK;
}

extern "C" void pnr_destroy(pnr_handle* h) {
    if (!h) return;
    PnrDeviceGuard guard(h->device);
    for (cudaStream_t st : {h->host_stream, h->copy_stream1, h->copy_stream2})
        if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    if (h->host_order_event) cudaEventDestroy(h->host_order_event);
    for (auto& sl : h->slot) {
        for (cudaEvent_t ev : {sl.kernel_done, sl.copy1_done, sl.copy2_done}) if (ev) cudaEventDestroy(ev);
        cudaFree(sl.actions); cudaFree(sl.obs); cudaFree(sl.reward); cudaFree(sl.compact); cudaFree(sl.done);
    }
    for (int r = 0; r < PNR_SYNC_MAX_PEERS; ++r)
        if (h->sync_ipc_opened[r]) cudaIpcCloseMemHandle(h->sync_peers.window[r]);
    cudaFree(h->sync_window);
    cudaFree(h->state); cudaFree(h->stats); cudaFree(h->stats_out); cudaFree(h->box_a); cudaFree(h->box_z);
    cudaFree(h->filt_delta); cudaFree(h->filt_applied); cudaFree(h->filt_state); cudaFree(h->filt_merged);
    if (h->stats_host) cudaFreeHost(h->stats_host);
    delete h;
}

extern "C" int64_t pnr_num_envs(const pnr_handle* h) { return h ? h->n_envs : 0; }
extern "C" int64_t pnr_launch_count(const pnr_handle* h) { return h ? h->launches : 0; }

extern "C" int pnr_get_bounds(const pnr_handle* h, float* r_lo, float* r_hi, float* v_max, float* a_max) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_get_bounds: null handle");
    for (int j = 0; j < PNR_DOF; ++j) {
        if (r_lo) r_lo[j] = h->params.r_lo[j];
        if (r_hi) r_hi[j] = h->params.r_hi[j];
        if (v_max) v_max[j] = h->params.v_max[j];
        if (a_max) a_max[j] = h->a_max[j];
    }
    return PNR_OK;
}

extern "C" int pnr_tick_advance(pnr_handle* h, uint32_t n, void* stream) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_tick_advance: null handle");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(pnr_launch_tick_advance(h->stats, n, 0, (cudaStream_t)stream));
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_get_counters(const pnr_handle* h, uint32_t* tick, double* env_steps, uint64_t* seed) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_get_counters: null handle");
    if (tick || env_steps) {                      // the steps may have run on any stream
        PnrDeviceGuard guard(h->device);
        PNR_CUDA(cudaDeviceSynchronize());
    }
    if (tick) {                                   // host call counter + what graph replays added on the device
        PnrDeviceGuard guard(h->device);
        uint32_t off = 0;
        PNR_CUDA(cudaMemcpy(&off, reinterpret_cast<const char*>(h->stats) + offsetof(PnrStats, tick_offset), sizeof(off),
                            cudaMemcpyDeviceToHost));
        *tick = h->tick + off;
    }
    if (env_steps) {                              // counted on the device by the step kernels
        PnrDeviceGuard guard(h->device);
        PNR_CUDA(cudaMemcpy(env_steps, reinterpret_cast<const char*>(h->stats) + offsetof(PnrStats, env_steps),
                            sizeof(double), cudaMemcpyDeviceToHost));
    }
    if (seed) *seed = h->seed;
    return PNR_OK;
}

extern "C" int pnr_set_counters(pnr_handle* h, uint32_t tick, double env_steps) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_set_counters: null handle");
    {
        PnrDeviceGuard guard(h->device);
        PNR_CUDA(pnr_launch_tick_advance(h->stats, 0, 1, nullptr));       // the device-side offset is folded into `tick`
        PNR_CUDA(pnr_launch_env_steps_set(h->stats, env_steps, nullptr));
        PNR_CUDA(cudaStreamSynchronize(nullptr));
    }
    h->tick = tick;
    return PNR_OK;
}

extern "C" int pnr_seed(pnr_handle* h, uint64_t seed) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_seed: null handle");
    PnrDeviceGuard guard(h->device);
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    PNR_CUDA(cudaDeviceSynchronize());            // steps in flight keep the old key
    PNR_CUDA(cudaMemcpy(reinterpret_cast<char*>(h->stats) + offsetof(PnrStats, seed_lo), key, sizeof(key), cudaMemcpyHostToDevice));
    h->seed = seed;
    h->params.seed_lo = key[0];
    h->params.seed_hi = key[1];
    return PNR_OK;
}

extern "C" int pnr_reset(pnr_handle* h, const int64_t* idx, int64_t n, const float* q0, const float* target,
                         float* obs_out, void* stream) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_reset: null handle");
    if (n < 0 || (!idx && n != h->n_envs)) return pnr_fail(PNR_ERR_INVALID, "pnr_reset: idx == NULL requires n == n_envs");
    if (reinterpret_cast<uintptr_t>(obs_out) & 15)            // the tile leaves through cp.async.bulk / 16-byte stores
        return pnr_fail(PNR_ERR_INVALID, "pnr_reset: obs_out must be 16-byte aligned");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(pnr_launch_reset_observe(h->params, h->device, 0, h->state, idx, n, q0, target, obs_out, h->tick,
                                      (cudaStream_t)stream));
    h->tick += 1;
    h->launches += (n > 0);
    return PNR_OK;
}

extern "C" int pnr_observe(pnr_handle* h, const int64_t* idx, int64_t n, float* obs_out, void* stream) {
    if (!h || !obs_out) return pnr_fail(PNR_ERR_INVALID, "pnr_observe: null argument");
    if (n < 0 || (!idx && n != h->n_envs)) return pnr_fail(PNR_ERR_INVALID, "pnr_observe: idx == NULL requires n == n_envs");
    if (reinterpret_cast<uintptr_t>(obs_out) & 15)
        return pnr_fail(PNR_ERR_INVALID, "pnr_observe: obs_out must be 16-byte aligned");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(pnr_launch_reset_observe(h->params, h->device, 1, h->state, idx, n, nullptr, nullptr, obs_out, h->tick,
                                      (cudaStream_t)stream));
    h->launches += (n > 0);
    return PNR_OK;
}

static int pnr_step_impl(pnr_handle* h, const float* actions, float* obs, float* reward, uint8_t* done, void* stream,
                         PnrMulti multi = PnrMulti{1, 0, 0}) {
    if (!h || !actions || !obs || !reward || !done) return pnr_fail(PNR_ERR_INVALID, "pnr_step: null argument");
    if ((reinterpret_cast<uintptr_t>(obs) & 15) || (reinterpret_cast<uintptr_t>(actions) & 7))
        return pnr_fail(PNR_ERR_INVALID, "pnr_step: obs must be 16-byte and actions 8-byte aligned");
    PnrDeviceGuard guard(h->device);
    // a launch that is being captured into a CUDA graph draws its reset keys from that graph's own domain (see the header)
    uint32_t domain = 0;
    {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        unsigned long long id = 0;
        if (stream && cudaStreamGetCaptureInfo((cudaStream_t)stream, &cs, &id) == cudaSuccess && cs == cudaStreamCaptureStatusActive) {
            if (h->n_graphs == 0 || id != h->capture_id) { h->n_graphs += 1; h->capture_id = id; }
            domain = h->n_graphs;
        }
    }
    if (h->cfg.mode == PNR_MODE_DYNAMIC)
        PNR_CUDA(pnr_launch_step_dynamic(h->params, h->device, h->cfg.obs_mode, h->state, actions, obs, reward, done,
                                         h->stats, h->tick, domain, h->filt_fused ? h->filt_applied : nullptr,
                                         (h->filt_fused && h->filt_fused_update) ? h->filt_delta : nullptr,
                                         (float)h->filt_clip, multi, (cudaStream_t)stream));
    else
        PNR_CUDA(pnr_launch_step(h->params, h->device, h->cfg.arith, h->cfg.obs_mode, h->state, actions, obs, reward, done,
                                 h->stats, h->tick, domain, h->filt_fused ? h->filt_applied : nullptr,
                                 (h->filt_fused && h->filt_fused_update) ? h->filt_delta : nullptr, (float)h->filt_clip,
                                 multi, (cudaStream_t)stream));
    h->tick += (uint32_t)multi.n_steps;
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_step(pnr_handle* h, const float* actions, float* obs, float* reward, uint8_t* done, void* stream) {
    return pnr_step_impl(h, actions, obs, reward, done, stream);
}

extern "C" int pnr_step_many(pnr_handle* h, int32_t n_steps, const float* actions, int64_t action_stride, float* obs,
                             int64_t obs_stride, float* reward, uint8_t* done, void* stream) {
    if (!h || n_steps < 0) return pnr_fail(PNR_ERR_INVALID, "pnr_step_many: bad argument");
    if (n_steps == 0) return PNR_OK;
    // The whole fragment is ONE launch (PnrMulti): every CTA (kinematic kernel; each tile's steps back to back) or warp
    // (dynamic kernel; the env state stays in registers) runs the n_steps steps on its own tiles -- tiles never depend on each
    // other, so there is no launch gap and no grid-wide wait between the steps.  A single step reads no stride.
    if (n_steps > 1) {
        if ((reinterpret_cast<uintptr_t>(obs) & 15) || ((obs_stride * sizeof(float)) & 15))
            return pnr_fail(PNR_ERR_INVALID, "pnr_step_many: obs and obs_stride * 4 must be multiples of 16 bytes");
        if ((action_stride * sizeof(float)) & 7)
            return pnr_fail(PNR_ERR_INVALID, "pnr_step_many: action_stride * 4 must be a multiple of 8 bytes");
    }
    return pnr_step_impl(h, actions, obs, reward, done, stream, PnrMulti{n_steps, action_stride, obs_stride});
}

extern "C" int pnr_observe_done(pnr_handle* h, const uint8_t* done, float* obs, float* terminal_obs, void* stream) {
    if (!h || !done || !obs) return pnr_fail(PNR_ERR_INVALID, "pnr_observe_done: null argument");
    PnrDeviceGuard guard(h->device);
    const bool fused = h->filt_fused != 0;
    PNR_CUDA(pnr_launch_observe_done(h->params, h->device, h->state, done, obs, terminal_obs, fused ? h->filt_applied : nullptr,
                                     (fused && h->filt_fused_update) ? h->filt_delta : nullptr, (float)h->filt_clip,
                                     (cudaStream_t)stream));
    h->launches += 1;
    return PNR_OK;
}

static int pnr_host_setup(pnr_handle* h) {
    if (h->host_ready) return PNR_OK;
    const size_t n = (size_t)h->n_envs;
    auto setup = [&]() -> cudaError_t {                           // all or nothing; what was allocated is kept for the retry
        cudaError_t e;
        if (!h->host_stream && (e = cudaStreamCreateWithFlags(&h->host_stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if (!h->copy_stream1 && (e = cudaStreamCreateWithFlags(&h->copy_stream1, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if (!h->copy_stream2 && (e = cudaStreamCreateWithFlags(&h->copy_stream2, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if (!h->host_order_event && (e = cudaEventCreateWithFlags(&h->host_order_event, cudaEventDisableTiming)) != cudaSuccess) return e;
        for (auto& sl : h->slot) {
            for (cudaEvent_t* ev : {&sl.kernel_done, &sl.copy1_done, &sl.copy2_done})
                if (!*ev && (e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming)) != cudaSuccess) return e;
            if (!sl.actions && (e = cudaMalloc(&sl.actions, n * PNR_DOF * sizeof(float))) != cudaSuccess) return e;
            if (!sl.obs && (e = cudaMalloc(&sl.obs, n * PNR_OBS_DIM * sizeof(float))) != cudaSuccess) return e;
            if (!sl.reward && (e = cudaMalloc(&sl.reward, n * sizeof(float))) != cudaSuccess) return e;
            if (!sl.done && (e = cudaMalloc(&sl.done, n)) != cudaSuccess) return e;
        }
        return cudaSuccess;
    };
    const cudaError_t e = setup();
    if (e != cudaSuccess)
        return pnr_fail(e == cudaErrorMemoryAllocation ? PNR_ERR_ALLOC : PNR_ERR_CUDA,
                        std::string("pnr_step_host: staging set-up: ") + cudaGetErrorString(e));
    h->host_ready = true;
    return PNR_OK;
}

extern "C" int pnr_step_host_begin(pnr_handle* h, const float* actions, float* obs, float* reward, uint8_t* done, int layout) {
    if (!h || !actions || !obs || !reward || !done) return pnr_fail(PNR_ERR_INVALID, "pnr_step_host_begin: null argument");
    if (layout != PNR_HOST_FULL && layout != PNR_HOST_COMPACT) return pnr_fail(PNR_ERR_INVALID, "pnr_step_host_begin: unknown layout");
    PnrDeviceGuard guard(h->device);
    int rc = pnr_host_setup(h);
    if (rc != PNR_OK) return rc;
    pnr_handle::HostSlot& sl = h->slot[h->host_next];
    if (sl.busy) return pnr_fail(PNR_ERR_INVALID, "pnr_step_host_begin: two steps are already in flight; call pnr_step_host_end");
    const size_t n = (size_t)h->n_envs;
    const int width = layout == PNR_HOST_COMPACT ? PNR_OBS_COMPACT_DIM : PNR_OBS_DIM;
    if (layout == PNR_HOST_COMPACT && !sl.compact) {
        cudaError_t e = cudaMalloc(&sl.compact, n * PNR_OBS_COMPACT_DIM * sizeof(float));
        if (e != cudaSuccess) return pnr_fail(PNR_ERR_ALLOC, std::string("pnr_step_host_begin: ") + cudaGetErrorString(e));
    }
    cudaStream_t s = h->host_stream;
    // the library's own (non-blocking) streams: order them after whatever the caller queued on the default stream (a reset,
    // a set_state, a previous pnr_step); work on other non-blocking streams is the caller's to synchronise
    if (h->host_inflight == 0) {
        PNR_CUDA(cudaEventRecord(h->host_order_event, nullptr));
        PNR_CUDA(cudaStreamWaitEvent(s, h->host_order_event, 0));
    }
    PNR_CUDA(cudaMemcpyAsync(sl.actions, actions, n * PNR_DOF * sizeof(float), cudaMemcpyHostToDevice, s));
    rc = pnr_step(h, sl.actions, sl.obs, sl.reward, sl.done, s);
    if (rc != PNR_OK) return rc;
    const float* src = sl.obs;
    if (layout == PNR_HOST_COMPACT) {
        PNR_CUDA(pnr_launch_compact_obs(h->device, sl.obs, sl.compact, h->n_envs, s));
        h->launches += 1;
        src = sl.compact;
    }
    PNR_CUDA(cudaEventRecord(sl.kernel_done, s));
    // The observation copy is what bounds this call (PCIe).  Two copy engines working on the two halves keep the link
    // fuller than one; reward / done ride on the first stream.
    const size_t total = n * (size_t)width;
    const size_t half = (n / 2) * (size_t)width;
    PNR_CUDA(cudaStreamWaitEvent(h->copy_stream1, sl.kernel_done, 0));
    PNR_CUDA(cudaStreamWaitEvent(h->copy_stream2, sl.kernel_done, 0));
    PNR_CUDA(cudaMemcpyAsync(obs + half, src + half, (total - half) * sizeof(float), cudaMemcpyDeviceToHost, h->copy_stream2));
    PNR_CUDA(cudaEventRecord(sl.copy2_done, h->copy_stream2));
    if (half > 0) PNR_CUDA(cudaMemcpyAsync(obs, src, half * sizeof(float), cudaMemcpyDeviceToHost, h->copy_stream1));
    PNR_CUDA(cudaMemcpyAsync(reward, sl.reward, n * sizeof(float), cudaMemcpyDeviceToHost, h->copy_stream1));
    PNR_CUDA(cudaMemcpyAsync(done, sl.done, n, cudaMemcpyDeviceToHost, h->copy_stream1));
    PNR_CUDA(cudaEventRecord(sl.copy1_done, h->copy_stream1));
    sl.busy = true;
    h->host_next ^= 1;
    h->host_inflight += 1;
    return PNR_OK;
}

extern "C" int pnr_step_host_end(pnr_handle* h) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_step_host_end: null handle");
    if (h->host_inflight == 0) return pnr_fail(PNR_ERR_INVALID, "pnr_step_host_end: no step in flight");
    PnrDeviceGuard guard(h->device);
    pnr_handle::HostSlot& sl = h->slot[h->host_inflight == 2 ? h->host_next : (h->host_next ^ 1)];   // the oldest one
    PNR_CUDA(cudaEventSynchronize(sl.copy1_done));
    PNR_CUDA(cudaEventSynchronize(sl.copy2_done));
    sl.busy = false;
    h->host_inflight -= 1;
    return PNR_OK;
}

extern "C" int pnr_step_host(pnr_handle* h, const float* actions, float* obs, float* reward, uint8_t* done) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_step_host: null argument");
    while (h->host_inflight > 0) {                                  // results of asynchronous steps land first
        int rc = pnr_step_host_end(h);
        if (rc != PNR_OK) return rc;
    }
    int rc = pnr_step_host_begin(h, actions, obs, reward, done, PNR_HOST_FULL);
    return rc != PNR_OK ? rc : pnr_step_host_end(h);
}

extern "C" int pnr_get_obs_constants(const pnr_handle* h, float* out36) {
    if (!h || !out36) return pnr_fail(PNR_ERR_INVALID, "pnr_get_obs_constants: null argument");
    const PnrParams& p = h->params;
    for (int j = 0; j < PNR_DOF; ++j) {                             // pnr_pack_obs_const
        out36[j] = p.r_lo[j];       out36[6 + j] = p.cos_r_lo[j];   out36[12 + j] = p.sin_r_lo[j];
        out36[18 + j] = p.r_hi[j];  out36[24 + j] = p.cos_r_hi[j];  out36[30 + j] = p.sin_r_hi[j];
    }
    return PNR_OK;
}

extern "C" int pnr_expand_obs_host(const pnr_handle* h, const float* compact, float* full, int64_t n_rows) {
    if (!h || !compact || !full || n_rows < 0) return pnr_fail(PNR_ERR_INVALID, "pnr_expand_obs_host: bad argument");
    float c36[PNR_OBS_CONST_END - PNR_OBS_CONST_BEGIN];
    pnr_get_obs_constants(h, c36);
    for (int64_t r = 0; r < n_rows; ++r) {
        const float* src = compact + r * PNR_OBS_COMPACT_DIM;
        float* dst = full + r * PNR_OBS_DIM;
        std::memcpy(dst, src, PNR_OBS_CONST_BEGIN * sizeof(float));
        std::memcpy(dst + PNR_OBS_CONST_BEGIN, c36, sizeof(c36));
        std::memcpy(dst + PNR_OBS_CONST_END, src + PNR_OBS_CONST_BEGIN, (PNR_OBS_DIM - PNR_OBS_CONST_END) * sizeof(float));
    }
    return PNR_OK;
}

extern "C" int pnr_get_state(pnr_handle* h, float* r, float* v, float* a, float* potential, float* target,
                             int32_t* t, float* ep_return, void* stream) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_get_state: null handle");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(pnr_launch_state_io(false, h->state, h->n_envs, r, v, a, potential, target, t, ep_return, (cudaStream_t)stream));
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_set_state(pnr_handle* h, const float* r, const float* v, const float* a, const float* potential,
                             const float* target, const int32_t* t, const float* ep_return, void* stream) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_set_state: null handle");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(pnr_launch_state_io(true, h->state, h->n_envs, const_cast<float*>(r), const_cast<float*>(v),
                                 const_cast<float*>(a), const_cast<float*>(potential), const_cast<float*>(target),
                                 const_cast<int32_t*>(t), const_cast<float*>(ep_return), (cudaStream_t)stream));
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_get_boxes(pnr_handle* h, float* box, void* stream) {
    if (!h || !box) return pnr_fail(PNR_ERR_INVALID, "pnr_get_boxes: null argument");
    if (!h->box_a) return pnr_fail(PNR_ERR_UNSUPPORTED, "pnr_get_boxes: the handle was created without cfg.random_box");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(pnr_launch_box_io(false, h->box_a, h->box_z, h->n_envs, box, (cudaStream_t)stream));
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_set_boxes(pnr_handle* h, const float* box, void* stream) {
    if (!h || !box) return pnr_fail(PNR_ERR_INVALID, "pnr_set_boxes: null argument");
    if (!h->box_a) return pnr_fail(PNR_ERR_UNSUPPORTED, "pnr_set_boxes: the handle was created without cfg.random_box");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(pnr_launch_box_io(true, h->box_a, h->box_z, h->n_envs, const_cast<float*>(box), (cudaStream_t)stream));
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_set_stats(pnr_handle* h, const double* in8) {
    if (!h || !in8) return pnr_fail(PNR_ERR_INVALID, "pnr_set_stats: null argument");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(cudaDeviceSynchronize());
    PnrStats st;
    PNR_CUDA(cudaMemcpy(&st, h->stats, sizeof(st), cudaMemcpyDeviceToHost));
    st.episodes = in8[0]; st.sum_return = in8[1]; st.sum_length = in8[2]; st.sum_return_sq = in8[3];
    st.max_return_ord = pnr_float_to_ordered((float)in8[4]);
    st.min_return_ord = pnr_float_to_ordered((float)in8[5]);
    st.env_steps = in8[6]; st.reached = in8[7];
    PNR_CUDA(cudaMemcpy(h->stats, &st, sizeof(st), cudaMemcpyHostToDevice));
    return PNR_OK;
}

extern "C" int pnr_stats_device(pnr_handle* h, double* out_device, int clear, void* stream) {
    if (!h || !out_device) return pnr_fail(PNR_ERR_INVALID, "pnr_stats_device: null argument");
    PnrDeviceGuard guard(h->device);
    PNR_CUDA(pnr_launch_stats_snapshot(h->stats, out_device, clear, (cudaStream_t)stream));
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_stats_merge_device(const double* gathered, int world, int len, double* out, void* stream) {
    if (!gathered || !out || world < 1 || len < PNR_STATS_LEN) return pnr_fail(PNR_ERR_INVALID, "pnr_stats_merge_device: bad argument");
    PNR_CUDA(pnr_launch_stats_merge(gathered, world, len, out, (cudaStream_t)stream));
    return PNR_OK;
}

static int pnr_filter_ensure(pnr_handle* h, cudaStream_t stream);

static int pnr_sync_window_ensure(pnr_handle* h) {
    if (h->sync_window) return PNR_OK;
    PNR_CUDA(cudaMalloc(&h->sync_window, PNR_SYNC_WINDOW_BYTES));
    PNR_CUDA(cudaMemset(h->sync_window, 0, PNR_SYNC_WINDOW_BYTES));
    PNR_CUDA(cudaDeviceSynchronize());
    return PNR_OK;
}

extern "C" int pnr_sync_window_create(pnr_handle* h, unsigned char* ipc_handle_out) {
    if (!h || !ipc_handle_out) return pnr_fail(PNR_ERR_INVALID, "pnr_sync_window_create: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == PNR_SYNC_IPC_BYTES, "PNR_SYNC_IPC_BYTES is the size of a CUDA IPC handle");
    PnrDeviceGuard guard(h->device);
    int rc = pnr_sync_window_ensure(h);
    if (rc != PNR_OK) return rc;
    cudaIpcMemHandle_t ipc;
    PNR_CUDA(cudaIpcGetMemHandle(&ipc, h->sync_window));
    std::memcpy(ipc_handle_out, &ipc, sizeof(ipc));
    return PNR_OK;
}

extern "C" int pnr_sync_window_ptr(pnr_handle* h, void** window_out) {
    if (!h || !window_out) return pnr_fail(PNR_ERR_INVALID, "pnr_sync_window_ptr: null argument");
    PnrDeviceGuard guard(h->device);
    int rc = pnr_sync_window_ensure(h);
    if (rc != PNR_OK) return rc;
    *window_out = h->sync_window;
    return PNR_OK;
}

static int pnr_sync_disconnect(pnr_handle* h) {
    for (int r = 0; r < PNR_SYNC_MAX_PEERS; ++r) {
        if (h->sync_ipc_opened[r]) cudaIpcCloseMemHandle(h->sync_peers.window[r]);
        h->sync_ipc_opened[r] = false;
        h->sync_peers.window[r] = nullptr;
    }
    h->sync_peers.world = 0;
    return PNR_OK;
}

extern "C" int pnr_sync_window_connect_ptrs(pnr_handle* h, void* const* windows, int world, int rank) {
    if (!h || !windows) return pnr_fail(PNR_ERR_INVALID, "pnr_sync_window_connect_ptrs: null argument");
    if (world < 1 || world > PNR_SYNC_MAX_PEERS || rank < 0 || rank >= world)
        return pnr_fail(PNR_ERR_INVALID, "pnr_sync_window_connect_ptrs: need 1 <= world <= PNR_SYNC_MAX_PEERS and 0 <= rank < world");
    PnrDeviceGuard guard(h->device);
    int rc = pnr_sync_window_ensure(h);
    if (rc != PNR_OK) return rc;
    PNR_CUDA(cudaDeviceSynchronize());                         // no exchange of the old connection is still running
    pnr_sync_disconnect(h);
    PNR_CUDA(cudaMemset(h->sync_window, 0, PNR_SYNC_WINDOW_BYTES));   // sequence numbers and flags restart with the connection
    PNR_CUDA(cudaDeviceSynchronize());
    for (int r = 0; r < world; ++r) {
        if (r != rank && !windows[r]) return pnr_fail(PNR_ERR_INVALID, "pnr_sync_window_connect_ptrs: null window");
        h->sync_peers.window[r] = r == rank ? h->sync_window : static_cast<unsigned char*>(windows[r]);
    }
    h->sync_peers.world = world;
    h->sync_peers.rank = rank;
    return PNR_OK;
}

extern "C" int pnr_sync_window_connect(pnr_handle* h, const unsigned char* ipc_handles, int world, int rank) {
    if (!h || !ipc_handles) return pnr_fail(PNR_ERR_INVALID, "pnr_sync_window_connect: null argument");
    if (world < 1 || world > PNR_SYNC_MAX_PEERS || rank < 0 || rank >= world)
        return pnr_fail(PNR_ERR_INVALID, "pnr_sync_window_connect: need 1 <= world <= PNR_SYNC_MAX_PEERS and 0 <= rank < world");
    PnrDeviceGuard guard(h->device);
    int rc = pnr_sync_window_ensure(h);
    if (rc != PNR_OK) return rc;
    PNR_CUDA(cudaDeviceSynchronize());
    pnr_sync_disconnect(h);
    void* mapped[PNR_SYNC_MAX_PEERS] = {};
    bool opened[PNR_SYNC_MAX_PEERS] = {};
    for (int r = 0; r < world; ++r) {
        if (r == rank) continue;
        cudaIpcMemHandle_t ipc;
        std::memcpy(&ipc, ipc_handles + (size_t)r * PNR_SYNC_IPC_BYTES, sizeof(ipc));
        cudaError_t e = cudaIpcOpenMemHandle(&mapped[r], ipc, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            for (int q = 0; q < r; ++q) if (opened[q]) cudaIpcCloseMemHandle(mapped[q]);
            cudaGetLastError();
            return pnr_fail(PNR_ERR_CUDA, std::string("pnr_sync_window_connect: cudaIpcOpenMemHandle(rank ") + std::to_string(r) +
                                              "): " + cudaGetErrorString(e));
        }
        opened[r] = true;
    }
    rc = pnr_sync_window_connect_ptrs(h, mapped, world, rank);
    if (rc != PNR_OK) {
        for (int r = 0; r < world; ++r) if (opened[r]) cudaIpcCloseMemHandle(mapped[r]);
        return rc;
    }
    for (int r = 0; r < world; ++r) h->sync_ipc_opened[r] = opened[r];
    return PNR_OK;
}

extern "C" int pnr_iteration_sync(pnr_handle* h, int with_filter, int clear, double* out_device, int timeout_ms, void* stream) {
    if (!h || !out_device) return pnr_fail(PNR_ERR_INVALID, "pnr_iteration_sync: null argument");
    if (reinterpret_cast<uintptr_t>(out_device) & 7)
        return pnr_fail(PNR_ERR_INVALID, "pnr_iteration_sync: out_device must be 8-byte aligned");
    if (timeout_ms < 0) return pnr_fail(PNR_ERR_INVALID, "pnr_iteration_sync: timeout_ms < 0");
    PnrDeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    if (with_filter) {
        int rc = pnr_filter_ensure(h, s);
        if (rc != PNR_OK) return rc;
    }
    PnrSyncPeers peers = h->sync_peers;
    if (peers.world < 1) { peers.world = 1; peers.rank = 0; }
    PNR_CUDA(pnr_launch_iteration_sync(h->stats, clear, with_filter ? h->filt_delta : nullptr, h->filt_state, h->filt_applied,
                                       h->filt_demean, h->filt_destd, peers, (unsigned long long)timeout_ms * 1000000ull,
                                       out_device, s));
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_sync_status(pnr_handle* h, int* timed_out) {
    if (!h || !timed_out) return pnr_fail(PNR_ERR_INVALID, "pnr_sync_status: null argument");
    *timed_out = 0;
    if (!h->sync_window) return PNR_OK;
    PnrDeviceGuard guard(h->device);
    uint32_t st = 0;
    PNR_CUDA(cudaMemcpy(&st, h->sync_window + PNR_SYNC_STATUS_OFF, sizeof(st), cudaMemcpyDeviceToHost));   // synchronises
    *timed_out = st ? 1 : 0;
    return PNR_OK;
}

extern "C" int pnr_stats(pnr_handle* h, double* out, int clear, void* stream) {
    if (!h || !out) return pnr_fail(PNR_ERR_INVALID, "pnr_stats: null argument");
    PnrDeviceGuard guard(h->device);
    int rc = pnr_stats_device(h, h->stats_out, clear, stream);
    if (rc != PNR_OK) return rc;
    PNR_CUDA(cudaMemcpyAsync(h->stats_host, h->stats_out, sizeof(double) * PNR_STATS_LEN, cudaMemcpyDeviceToHost,
                             (cudaStream_t)stream));
    PNR_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    std::memcpy(out, h->stats_host, sizeof(double) * PNR_STATS_LEN);
    return PNR_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// observation normaliser
// ---------------------------------------------------------------------------------------------------------------
// The running statistics live on the device (filt_state); the applied statistics (what the kernels subtract / scale by)
// are derived from them by a kernel, so a synchronisation never leaves the stream.
static int pnr_filter_refresh(pnr_handle* h, cudaStream_t stream) {
    PNR_CUDA(pnr_launch_filter_refresh(h->filt_state, h->filt_applied, h->filt_demean, h->filt_destd, stream));
    return PNR_OK;
}

static int pnr_filter_ensure(pnr_handle* h, cudaStream_t stream) {
    if (h->filt_delta) return PNR_OK;
    PNR_CUDA(cudaMalloc(&h->filt_delta, sizeof(double) * PNR_FILTER_SLOTS * PNR_FILTER_DELTA_LEN));
    PNR_CUDA(cudaMalloc(&h->filt_applied, sizeof(float) * 2 * PNR_OBS_DIM));
    PNR_CUDA(cudaMalloc(&h->filt_state, sizeof(double) * PNR_FILTER_DELTA_LEN));
    PNR_CUDA(cudaMalloc(&h->filt_merged, sizeof(double) * PNR_FILTER_DELTA_LEN));
    PNR_CUDA(cudaMemsetAsync(h->filt_delta, 0, sizeof(double) * PNR_FILTER_SLOTS * PNR_FILTER_DELTA_LEN, stream));
    PNR_CUDA(cudaMemsetAsync(h->filt_state, 0, sizeof(double) * PNR_FILTER_DELTA_LEN, stream));
    return pnr_filter_refresh(h, stream);
}

extern "C" int pnr_filter_configure(pnr_handle* h, double clip, int demean, int destd) {
    if (!h || !(clip > 0.0)) return pnr_fail(PNR_ERR_INVALID, "pnr_filter_configure: bad argument");
    PnrDeviceGuard guard(h->device);
    h->filt_clip = clip; h->filt_demean = demean ? 1 : 0; h->filt_destd = destd ? 1 : 0;
    int rc = pnr_filter_ensure(h, nullptr);
    if (rc != PNR_OK) return rc;
    // the accumulator is relative to the applied mean: rows pushed under the old setting are dropped
    PNR_CUDA(cudaMemsetAsync(h->filt_delta, 0, sizeof(double) * PNR_FILTER_SLOTS * PNR_FILTER_DELTA_LEN, nullptr));
    return pnr_filter_refresh(h, nullptr);
}

extern "C" int pnr_filter_fuse(pnr_handle* h, int on, int update) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_filter_fuse: null handle");
    if (on && h->cfg.mode == PNR_MODE_KINEMATIC && (h->cfg.arith != PNR_ARITH_F32 || h->cfg.obs_mode != PNR_OBS_TERMINAL))
        return pnr_fail(PNR_ERR_UNSUPPORTED, "pnr_filter_fuse: in the kinematic mode the fused normaliser is built for float32 "
                                             "arithmetic and terminal observations; use pnr_filter_apply otherwise");
    PnrDeviceGuard guard(h->device);
    if (on) {
        int rc = pnr_filter_ensure(h, nullptr);
        if (rc != PNR_OK) return rc;
    }
    h->filt_fused = on ? 1 : 0;
    h->filt_fused_update = update ? 1 : 0;
    return PNR_OK;
}

extern "C" int pnr_filter_apply(pnr_handle* h, const float* obs_in, float* obs_out, int64_t n_rows, int update,
                                int normalize, void* stream) {
    if (!h || !obs_in || !obs_out || n_rows < 0) return pnr_fail(PNR_ERR_INVALID, "pnr_filter_apply: bad argument");
    if ((reinterpret_cast<uintptr_t>(obs_in) & 15) || (reinterpret_cast<uintptr_t>(obs_out) & 15))
        return pnr_fail(PNR_ERR_INVALID, "pnr_filter_apply: observation buffers must be 16-byte aligned");
    PnrDeviceGuard guard(h->device);
    int rc = pnr_filter_ensure(h, (cudaStream_t)stream);
    if (rc != PNR_OK) return rc;
    PNR_CUDA(pnr_launch_filter(h->device, obs_in, obs_out, n_rows, h->filt_applied, h->filt_delta, (float)h->filt_clip,
                               update, normalize, (cudaStream_t)stream));
    h->launches += (n_rows > 0);
    return PNR_OK;
}

extern "C" int pnr_filter_delta_device(pnr_handle* h, double* out_device, void* stream) {
    if (!h || !out_device) return pnr_fail(PNR_ERR_INVALID, "pnr_filter_delta_device: null argument");
    if (reinterpret_cast<uintptr_t>(out_device) & 7)
        return pnr_fail(PNR_ERR_INVALID, "pnr_filter_delta_device: out_device must be 8-byte aligned");
    PnrDeviceGuard guard(h->device);
    int rc = pnr_filter_ensure(h, (cudaStream_t)stream);
    if (rc != PNR_OK) return rc;
    PNR_CUDA(pnr_launch_filter_fold(h->filt_delta, (cudaStream_t)stream));
    PNR_CUDA(cudaMemcpyAsync(out_device, h->filt_delta, sizeof(double) * PNR_FILTER_DELTA_LEN, cudaMemcpyDeviceToDevice,
                             (cudaStream_t)stream));
    return PNR_OK;
}

extern "C" int pnr_filter_sync_device(pnr_handle* h, const double* merged_device, void* stream) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_filter_sync_device: null handle");
    PnrDeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = pnr_filter_ensure(h, s);
    if (rc != PNR_OK) return rc;
    PNR_CUDA(pnr_launch_filter_sync(h->filt_delta, merged_device, h->filt_state, h->filt_applied, h->filt_demean,
                                    h->filt_destd, s));
    h->launches += 1;
    return PNR_OK;
}

extern "C" int pnr_filter_sync(pnr_handle* h, const double* merged, void* stream) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_filter_sync: null handle");
    PnrDeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = pnr_filter_ensure(h, s);
    if (rc != PNR_OK) return rc;
    if (merged) {                                 // pageable source: the copy is staged before the call returns
        PNR_CUDA(cudaMemcpyAsync(h->filt_merged, merged, sizeof(double) * PNR_FILTER_DELTA_LEN, cudaMemcpyHostToDevice, s));
        return pnr_filter_sync_device(h, h->filt_merged, stream);
    }
    return pnr_filter_sync_device(h, nullptr, stream);
}

extern "C" int pnr_filter_get(pnr_handle* h, double* count, double* mean, double* var) {
    if (!h) return pnr_fail(PNR_ERR_INVALID, "pnr_filter_get: null handle");
    PnrDeviceGuard guard(h->device);
    double st[PNR_FILTER_DELTA_LEN] = {};
    if (h->filt_state) {
        PNR_CUDA(cudaDeviceSynchronize());        // whatever stream the last synchronisation ran on
        PNR_CUDA(cudaMemcpy(st, h->filt_state, sizeof(st), cudaMemcpyDeviceToHost));
    }
    if (count) *count = st[0];
    for (int c = 0; c < PNR_OBS_DIM; ++c) {
        if (mean) mean[c] = st[1 + c];
        if (var) var[c] = st[0] > 1.0 ? st[1 + PNR_OBS_DIM + c] / (st[0] - 1.0) : st[1 + c] * st[1 + c];
    }
    return PNR_OK;
}

extern "C" int pnr_filter_set(pnr_handle* h, double count, const double* mean, const double* var, void* stream) {
    if (!h || !mean || !var || count < 0.0) return pnr_fail(PNR_ERR_INVALID, "pnr_filter_set: bad argument");
    PnrDeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = pnr_filter_ensure(h, s);
    if (rc != PNR_OK) return rc;
    double st[PNR_FILTER_DELTA_LEN];
    st[0] = count;
    for (int c = 0; c < PNR_OBS_DIM; ++c) {
        st[1 + c] = mean[c];
        st[1 + PNR_OBS_DIM + c] = count > 1.0 ? var[c] * (count - 1.0) : 0.0;
    }
    PNR_CUDA(cudaMemcpyAsync(h->filt_state, st, sizeof(st), cudaMemcpyHostToDevice, s));
    PNR_CUDA(cudaStreamSynchronize(s));           // `st` is a stack buffer
    PNR_CUDA(cudaMemsetAsync(h->filt_delta, 0, sizeof(double) * PNR_FILTER_SLOTS * PNR_FILTER_DELTA_LEN, s));
    return pnr_filter_refresh(h, s);
}
