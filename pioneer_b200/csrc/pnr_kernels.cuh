// Device functions of the fused reach-env step: state planes, joint integrator, forward kinematics,
// reward/done, reset, observation tile.  A tile is 32 envs whose 32 x 137 observation rows form ONE
// contiguous 17,536-byte span of the output, staged in shared memory (row stride 137 words is odd =>
// bank-conflict free) and handed to the TMA copy engine as one bulk store (cp.async.bulk shared -> global);
// ragged tail tiles fall back to coalesced float4 stores.
#pragma once
#include "pnr_device.cuh"
#include "pnr_trig.cuh"

#define PNR_TILE_ENVS 32
#define PNR_TILE_FLOATS (PNR_TILE_ENVS * PNR_OBS_DIM)      // 4384 floats = 17,536 B = 1096 float4
#define PNR_FULL_MASK 0xffffffffu

// per-env state.  HBM layout (96 B / env, plane-major so every warp access is one coalesced span), cut along
// the work split of the step kernel: warp k of a CTA owns joints 2k and 2k+1, the fourth warp owns the task.
//   RV_k  float4[N], k = 0..2 : r[2k] r[2k+1] v[2k] v[2k+1]          at S + k N
//   X0    float4[N]           : target x y z, t (int bits)            at S + 3 N
//   A_k   float2[N], k = 0..2 : a[2k] a[2k+1] (last action applied)   at (float2*)(S + 4 N) + k N
//   X1    float2[N]           : potential, episode return             at (float2*)(S + 4 N) + 3 N
struct PnrEnv {
    float r[PNR_DOF], v[PNR_DOF], a[PNR_DOF];
    float pot, ep_ret;
    float tgt[3];
    int32_t t;
};

__device__ __forceinline__ float4* pnr_plane_rv(float4* S, int64_t N, int k) { return S + (int64_t)k * N; }
__device__ __forceinline__ float4* pnr_plane_x0(float4* S, int64_t N) { return S + 3 * N; }
__device__ __forceinline__ float2* pnr_plane_a(float4* S, int64_t N, int k) {
    return reinterpret_cast<float2*>(S + 4 * N) + (int64_t)k * N;
}
__device__ __forceinline__ float2* pnr_plane_x1(float4* S, int64_t N) { return reinterpret_cast<float2*>(S + 4 * N) + 3 * N; }

__device__ __forceinline__ void pnr_load_env(float4* __restrict__ S, int64_t N, int64_t e, PnrEnv& s) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float4 rv = pnr_plane_rv(S, N, k)[e];
        const float2 a = pnr_plane_a(S, N, k)[e];
        s.r[2 * k] = rv.x; s.r[2 * k + 1] = rv.y; s.v[2 * k] = rv.z; s.v[2 * k + 1] = rv.w;
        s.a[2 * k] = a.x; s.a[2 * k + 1] = a.y;
    }
    const float4 x0 = pnr_plane_x0(S, N)[e];
    const float2 x1 = pnr_plane_x1(S, N)[e];
    s.tgt[0] = x0.x; s.tgt[1] = x0.y; s.tgt[2] = x0.z; s.t = __float_as_int(x0.w);
    s.pot = x1.x; s.ep_ret = x1.y;
}

// the same through L2 only (ld.global.cg): the planes are read once per launch, and a step launched with programmatic
// dependent launch may sit on its SM before the previous step has finished elsewhere
__device__ __forceinline__ void pnr_load_env_cg(float4* __restrict__ S, int64_t N, int64_t e, PnrEnv& s) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float4 rv = __ldcg(pnr_plane_rv(S, N, k) + e);
        const float2 a = __ldcg(pnr_plane_a(S, N, k) + e);
        s.r[2 * k] = rv.x; s.r[2 * k + 1] = rv.y; s.v[2 * k] = rv.z; s.v[2 * k + 1] = rv.w;
        s.a[2 * k] = a.x; s.a[2 * k + 1] = a.y;
    }
    const float4 x0 = __ldcg(pnr_plane_x0(S, N) + e);
    const float2 x1 = __ldcg(pnr_plane_x1(S, N) + e);
    s.tgt[0] = x0.x; s.tgt[1] = x0.y; s.tgt[2] = x0.z; s.t = __float_as_int(x0.w);
    s.pot = x1.x; s.ep_ret = x1.y;
}

__device__ __forceinline__ void pnr_store_env(float4* __restrict__ S, int64_t N, int64_t e, const PnrEnv& s) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        pnr_plane_rv(S, N, k)[e] = make_float4(s.r[2 * k], s.r[2 * k + 1], s.v[2 * k], s.v[2 * k + 1]);
        pnr_plane_a(S, N, k)[e] = make_float2(s.a[2 * k], s.a[2 * k + 1]);
    }
    pnr_plane_x0(S, N)[e] = make_float4(s.tgt[0], s.tgt[1], s.tgt[2], __int_as_float(s.t));
    pnr_plane_x1(S, N)[e] = make_float2(s.pot, s.ep_ret);
}

// reset_world (pioneer_knm_env.py:92-105): a = v = 0, potential = 0; TimeLimit.reset: elapsed = 0
__device__ __forceinline__ void pnr_reset_env(PnrEnv& s, const float (&q)[PNR_DOF], const float (&tgt)[3]) {
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) { s.r[i] = q[i]; s.v[i] = 0.f; s.a[i] = 0.f; }
    s.tgt[0] = tgt[0]; s.tgt[1] = tgt[1]; s.tgt[2] = tgt[2];
    s.pot = 0.f; s.ep_ret = 0.f; s.t = 0;
}

// ---------------------------------------------------------------------------------------------
// act() integrator for one joint (pioneer_knm_env.py:120-141).  Every operation is an explicitly
// rounded intrinsic: no FMA contraction, so r and v are BIT-EXACT against the oracle.
//   PNR_ARITH_F32      : the reference source under NumPy >= 2 (all float32)
//   PNR_ARITH_LEGACY64 : NumPy 1.x promotion (float64 intermediates, float32 stores; SURVEY.md row A4)
// ---------------------------------------------------------------------------------------------
// exact float32 quotient num / den.  A velocity that is ALREADY saturated gives num == +0 on every following
// step; the hardware's fast division path rejects zero numerators and falls into a ~40-instruction subroutine,
// so that (very common) case is answered directly with the IEEE result: +-0, or NaN for a zero / NaN divisor.
__device__ __forceinline__ float pnr_div_exact(float num, float den) {
    const bool zero = num == 0.f;
    const float q = __fdiv_rn(zero ? 1.f : num, den);
    const float q0 = (den != 0.f && den == den) ? copysignf(0.f, den) : __int_as_float(0x7fc00000);
    return zero ? q0 : q;
}

template <int ARITH>
__device__ __forceinline__ void pnr_integrate_joint(const PnrParams& p, float vmax, float r_lo, float r_hi, float a0,
                                                    float v0, float r0, float& v1_out, float& r1_out) {
    float v1, r1;
    if (ARITH == PNR_ARITH_F32) {
        const float dt = p.dt32;
        v1 = __fadd_rn(v0, __fmul_rn(a0, dt));                                   // :121
        float dt_p1 = dt, dt_p2 = 0.f;
        const bool hi = v1 > vmax, lo = v1 < -vmax;                              // :125, :129
        if (hi || lo) {
            const float vsat = hi ? vmax : -vmax;
            const float q = pnr_div_exact(__fsub_rn(vsat, v0), __fadd_rn(a0, p.eps32));  // :126, :130
            dt_p1 = pnr_clip(q, 0.f, dt);
            dt_p2 = __fsub_rn(dt, dt_p1);
            v1 = vsat;
        }
        const float half = __fmul_rn(0.5f, __fadd_rn(v0, v1));                   // :134
        r1 = __fadd_rn(__fadd_rn(r0, __fmul_rn(half, dt_p1)), __fmul_rn(v1, dt_p2));
    } else {
        const double dt = p.dt64;
        v1 = (float)__dadd_rn((double)v0, __dmul_rn((double)a0, dt));
        double dt_p1 = dt, dt_p2 = 0.0;
        const bool hi = v1 > vmax, lo = v1 < -vmax;
        if (hi || lo) {
            const float vsat = hi ? vmax : -vmax;
            const double q = __ddiv_rn((double)__fsub_rn(vsat, v0), __dadd_rn((double)a0, p.eps64));
            dt_p1 = pnr_clip(q, 0.0, dt);
            dt_p2 = __dsub_rn(dt, dt_p1);
            v1 = vsat;
        }
        const double half = __dmul_rn(0.5, (double)__fadd_rn(v0, v1));
        r1 = (float)__dadd_rn(__dadd_rn((double)r0, __dmul_rn(half, dt_p1)), __dmul_rn((double)v1, dt_p2));
    }
    if (r1 >= r_hi) { r1 = r_hi; v1 = 0.f; }                                     // :135-137
    if (r1 <= r_lo) { r1 = r_lo; v1 = 0.f; }                                     // :139-141
    v1_out = v1; r1_out = r1;
}

// library sine/cosine, any argument (reset / observe kernels and the out-of-range fallback of the step kernel)
__device__ __forceinline__ void pnr_sincos(float x, float& s, float& c) { sincosf(x, &s, &c); }

// FAST: straight-line Cody-Waite + polynomial (pnr_trig.cuh), valid for |x| <= PNR_TRIG_FAST_LIMIT.
// The step kernel uses it for r, r - r_lo, r_hi - r (clamped to the joint limits by the integrator) and,
// under a per-env guard, for v and a.
template <bool FAST>
__device__ __forceinline__ void pnr_sincos_sel(float x, float& s, float& c) {
    if (FAST) pnr_sincos_fast(x, s, c);
    else sincosf(x, &s, &c);
}

// ---------------------------------------------------------------------------------------------
// Forward kinematics of the tracked tip ('robot:pointer'), evaluated tip-to-base:
//   p <- origin_j + R_origin_j * Rot(axis_j, q_j) * p          (URDF: child = parent*T(origin)*Rot(axis,q))
// replaces resetJointState x6 + getLinkState (pioneer_knm_env.py:148-151, bullet_scene.py:58).
// ---------------------------------------------------------------------------------------------
// one stage of the chain: v <- origin_j + R_origin_j * Rot(axis_j, q_j) * v
__device__ __forceinline__ void pnr_fk_stage(const PnrParams& p, int j, float sn, float c, float& x, float& y, float& z) {
    const float s = sn * p.axis_sign[j];
    const int code = p.axis_code[j];            // warp-uniform (constant bank)
    if (code == PNR_AXIS_X) {
        const float ny = fmaf(c, y, -s * z), nz = fmaf(s, y, c * z);
        y = ny; z = nz;
    } else if (code == PNR_AXIS_Y) {
        const float nx = fmaf(c, x, s * z), nz = fmaf(-s, x, c * z);
        x = nx; z = nz;
    } else if (code == PNR_AXIS_Z) {
        const float nx = fmaf(c, x, -s * y), ny = fmaf(s, x, c * y);
        x = nx; y = ny;
    } else {                                     // Rodrigues: p c + (k x p) s + k (k.p)(1-c)
        const float kx = p.axis[j][0], ky = p.axis[j][1], kz = p.axis[j][2];
        const float kp = (kx * x + ky * y + kz * z) * (1.f - c);
        const float nx = fmaf(x, c, fmaf(ky * z - kz * y, s, kx * kp));
        const float ny = fmaf(y, c, fmaf(kz * x - kx * z, s, ky * kp));
        const float nz = fmaf(z, c, fmaf(kx * y - ky * x, s, kz * kp));
        x = nx; y = ny; z = nz;
    }
    if (p.origin_has_rot[j]) {
        const float* R = p.origin_rot[j];
        const float nx = R[0] * x + R[1] * y + R[2] * z;
        const float ny = R[3] * x + R[4] * y + R[5] * z;
        const float nz = R[6] * x + R[7] * y + R[8] * z;
        x = nx; y = ny; z = nz;
    }
    x += p.origin_xyz[j][0]; y += p.origin_xyz[j][1]; z += p.origin_xyz[j][2];
}

// rotation of (x, y, z) about a coordinate axis known at compile time, then the joint origin translation
template <int CODE>
__device__ __forceinline__ void pnr_fk_stage_fixed(const PnrParams& p, int j, float s, float c, float& x, float& y, float& z) {
    if (CODE == PNR_AXIS_X) { const float ny = fmaf(c, y, -s * z), nz = fmaf(s, y, c * z); y = ny; z = nz; }
    else if (CODE == PNR_AXIS_Y) { const float nx = fmaf(c, x, s * z), nz = fmaf(-s, x, c * z); x = nx; z = nz; }
    else { const float nx = fmaf(c, x, -s * y), ny = fmaf(s, x, c * y); x = nx; y = ny; }
    x += p.origin_xyz[j][0]; y += p.origin_xyz[j][1]; z += p.origin_xyz[j][2];
}

__device__ __forceinline__ void pnr_fk_tip(const PnrParams& p, const float (&sn)[PNR_DOF], const float (&cs)[PNR_DOF],
                                           float (&out)[3]) {
    float x = p.tip_xyz[0], y = p.tip_xyz[1], z = p.tip_xyz[2];
    if (p.chain_kind == 1) {
        // the shipped robot (axes Z Y Y X Y X, positive, no origin rotations; detected by pnr_create): one uniform
        // branch instead of three per joint on the task warp's critical path.  Same operations, same results.
        pnr_fk_stage_fixed<PNR_AXIS_X>(p, 5, sn[5], cs[5], x, y, z);
        pnr_fk_stage_fixed<PNR_AXIS_Y>(p, 4, sn[4], cs[4], x, y, z);
        pnr_fk_stage_fixed<PNR_AXIS_X>(p, 3, sn[3], cs[3], x, y, z);
        pnr_fk_stage_fixed<PNR_AXIS_Y>(p, 2, sn[2], cs[2], x, y, z);
        pnr_fk_stage_fixed<PNR_AXIS_Y>(p, 1, sn[1], cs[1], x, y, z);
        pnr_fk_stage_fixed<PNR_AXIS_Z>(p, 0, sn[0], cs[0], x, y, z);
    } else {
#pragma unroll
        for (int j = PNR_DOF - 1; j >= 0; --j) pnr_fk_stage(p, j, sn[j], cs[j], x, y, z);
    }
    out[0] = x; out[1] = y; out[2] = z;
}

// ---------------------------------------------------------------------------------------------
// Obstacle variant (this repo's extension; the reference instantiates a box and a plane only in its GUI demo,
// pioneer_knm_env.py:249-261, and a per-episode random box only in its legacy path, pioneer/temp/pioneer_env.py:169-192):
// sum over (link capsule, obstacle) pairs of max(0, radius - d), d = the minimum of the obstacle's signed-distance function
// over the capsule's axis segment -- exact for every kind: plane (linear: the nearer end point), sphere (closest point of the
// segment), axis-aligned box (below: breakpoint enumeration, as oracle/contact.h and oracle/reach_oracle.py::contact_depth
// do in float64).
// INLINED into the obstacle instantiations: as a separate function it received the kernel parameters by reference, and every
// table entry (capsule end points, axis codes, joint origins, obstacle geometry) became a generic LD.E through that pointer
// instead of a constant-bank operand -- 144 dependent loads on the task warp's critical path; the variant ran 5x slower
// than the plain kernel (49 us vs 9 us per step at 65,536 envs) for ~4 k instructions of arithmetic.
// ---------------------------------------------------------------------------------------------
struct PnrSinCos { float sn[PNR_DOF], cs[PNR_DOF]; };
struct PnrBox { float px, py, pz, ex, ey, ez; };

// The signed distance to the box (coordinates relative to its centre) is |max(q, 0)| + min(max_i q_i, 0), q_i = |x_i| - e_i.
// Inside the box the signed distance is max_i(|x_i| - e_i): along the segment a convex, piecewise LINEAR function of t whose
// minimum lies at an end point, at a kink of one term (x_i = 0) or where two terms cross -- 2 + 3 + 12 candidates, each
// evaluated exactly (a candidate that is no breakpoint of the maximum, or lies outside the box, only yields a larger value).
__device__ __forceinline__ float pnr_box_face_term(float t, float ax, float ay, float az, float dx, float dy, float dz,
                                                   float ex, float ey, float ez) {
    t = fminf(fmaxf(t, 0.f), 1.f);                             // fmaxf drops a NaN candidate (0 / 0): it becomes t = 0
    return fmaxf(fabsf(fmaf(t, dx, ax)) - ex, fmaxf(fabsf(fmaf(t, dy, ay)) - ey, fabsf(fmaf(t, dz, az)) - ez));
}
__device__ __forceinline__ float pnr_segment_box_inside(float ax, float ay, float az, float dx, float dy, float dz,
                                                        float ex, float ey, float ez) {
    const float a3[3] = {ax, ay, az}, d3[3] = {dx, dy, dz}, e3[3] = {ex, ey, ez};
    float best = fminf(pnr_box_face_term(0.f, ax, ay, az, dx, dy, dz, ex, ey, ez),
                       pnr_box_face_term(1.f, ax, ay, az, dx, dy, dz, ex, ey, ez));
#pragma unroll
    for (int i = 0; i < 3; ++i)
        best = fminf(best, pnr_box_face_term(__fdividef(-a3[i], d3[i]), ax, ay, az, dx, dy, dz, ex, ey, ez));
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
        for (int j = i + 1; j < 3; ++j) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {                      // s_i (a_i + t d_i) - e_i = s_j (a_j + t d_j) - e_j, s = +-1
                const float si = (k & 1) ? -1.f : 1.f, sj = (k & 2) ? -1.f : 1.f;
                const float num = (sj * a3[j] - e3[j]) - (si * a3[i] - e3[i]);
                const float den = si * d3[i] - sj * d3[j];
                best = fminf(best, pnr_box_face_term(__fdividef(num, den), ax, ay, az, dx, dy, dz, ex, ey, ez));
            }
        }
    }
    return best;
}

// Outside the box the squared distance F(t) = sum_i max(|x_i(t)| - e_i, 0)^2 along the segment is convex and piecewise
// quadratic with at most six breakpoints (x_i = +-e_i), so g = F'/2 is piecewise LINEAR and non-decreasing: evaluate g at
// the breakpoints that fall inside the current bracket (no sorting: each one either raises the lower end or lowers the
// upper end), then solve the remaining linear piece -- the exact minimiser in 8 evaluations of g instead of 24 halvings.
// F ~ 0 there means the axis grazes or enters the box; only then the signed (negative) distance needs the candidates above.
__device__ __forceinline__ float pnr_box_gap_slope(float t, float ax, float ay, float az, float dx, float dy, float dz,
                                                   float ex, float ey, float ez) {
    const float x = fmaf(t, dx, ax), y = fmaf(t, dy, ay), z = fmaf(t, dz, az);
    const float qx = fmaxf(fabsf(x) - ex, 0.f), qy = fmaxf(fabsf(y) - ey, 0.f), qz = fmaxf(fabsf(z) - ez, 0.f);
    return fmaf(copysignf(qx, x), dx, fmaf(copysignf(qy, y), dy, copysignf(qz, z) * dz));
}
__device__ __forceinline__ float pnr_segment_box_exact(float ax, float ay, float az, float dx, float dy, float dz,
                                                       float ex, float ey, float ez) {
    float lo = 0.f, hi = 1.f;
    float glo = pnr_box_gap_slope(0.f, ax, ay, az, dx, dy, dz, ex, ey, ez);
    float ghi = pnr_box_gap_slope(1.f, ax, ay, az, dx, dy, dz, ex, ey, ez);
    float t;
    if (glo >= 0.f) t = 0.f;                                   // F does not decrease from the first end point
    else if (ghi <= 0.f) t = 1.f;                              // ... or still decreases at the second
    else {
        const float a3[3] = {ax, ay, az}, d3[3] = {dx, dy, dz}, e3[3] = {ex, ey, ez};
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float inv = __fdividef(1.f, d3[i]);          // d_i = 0: the candidates are inf / NaN and fail both tests
#pragma unroll
            for (int sgn = 0; sgn < 2; ++sgn) {
                const float tb = ((sgn ? -e3[i] : e3[i]) - a3[i]) * inv;
                if (tb > lo && tb < hi) {
                    const float gb = pnr_box_gap_slope(tb, ax, ay, az, dx, dy, dz, ex, ey, ez);
                    if (gb < 0.f) { lo = tb; glo = gb; } else { hi = tb; ghi = gb; }
                }
            }
        }
        const float w = ghi - glo;                             // glo < 0 <= ghi
        t = w > 0.f ? fmaf(hi - lo, -glo / w, lo) : lo;
        t = fminf(fmaxf(t, lo), hi);
    }
    const float x = fmaf(t, dx, ax), y = fmaf(t, dy, ay), z = fmaf(t, dz, az);
    const float qx = fmaxf(fabsf(x) - ex, 0.f), qy = fmaxf(fabsf(y) - ey, 0.f), qz = fmaxf(fabsf(z) - ez, 0.f);
    const float f2 = qx * qx + qy * qy + qz * qz;
    if (f2 > 1e-8f) return sqrtf(f2);                          // clear of the box by more than 1e-4
    const float in = pnr_segment_box_inside(ax, ay, az, dx, dy, dz, ex, ey, ez);   // grazing or inside: rounding cannot tell which
    return in < 0.f ? in : sqrtf(f2);
}

// world frame of body j from that of body j - 1 (x_world = o + R x_body, R row-major):
//   o += R origin_j;   R <- R R_origin_j Rot(axis_j, q_j)         (URDF: child = parent * T(origin) * Rot(axis, q))
__device__ __forceinline__ void pnr_frame_advance(const PnrParams& p, int j, float sn, float c, float (&R)[9], float (&o)[3]) {
    const float tx = p.origin_xyz[j][0], ty = p.origin_xyz[j][1], tz = p.origin_xyz[j][2];
#pragma unroll
    for (int r = 0; r < 3; ++r) o[r] = fmaf(R[3 * r], tx, fmaf(R[3 * r + 1], ty, fmaf(R[3 * r + 2], tz, o[r])));
    if (p.origin_has_rot[j]) {
        const float* Q = p.origin_rot[j];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float a = R[3 * r], b = R[3 * r + 1], d = R[3 * r + 2];
            R[3 * r] = a * Q[0] + b * Q[3] + d * Q[6];
            R[3 * r + 1] = a * Q[1] + b * Q[4] + d * Q[7];
            R[3 * r + 2] = a * Q[2] + b * Q[5] + d * Q[8];
        }
    }
    const float s = sn * p.axis_sign[j];
    const int code = p.axis_code[j];             // warp-uniform (constant bank)
    // a rotation about a coordinate axis mixes two columns (u, w) of R: u' = c u + s w, w' = -s u + c w with
    // (u, w) = columns (1, 2) for X, (2, 0) for Y, (0, 1) for Z
    if (code == PNR_AXIS_X) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float cu = R[3 * r + 1], cw = R[3 * r + 2];
            R[3 * r + 1] = fmaf(c, cu, s * cw); R[3 * r + 2] = fmaf(c, cw, -s * cu);
        }
    } else if (code == PNR_AXIS_Y) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float cu = R[3 * r + 2], cw = R[3 * r];
            R[3 * r + 2] = fmaf(c, cu, s * cw); R[3 * r] = fmaf(c, cw, -s * cu);
        }
    } else if (code == PNR_AXIS_Z) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float cu = R[3 * r], cw = R[3 * r + 1];
            R[3 * r] = fmaf(c, cu, s * cw); R[3 * r + 1] = fmaf(c, cw, -s * cu);
        }
    } else {                                     // Rodrigues: Rot = c I + s [k]x + (1 - c) k k^T
        const float kx = p.axis[j][0], ky = p.axis[j][1], kz = p.axis[j][2], v = 1.f - c;
        const float M[9] = {fmaf(v, kx * kx, c), fmaf(v, kx * ky, -s * kz), fmaf(v, kx * kz, s * ky),
                            fmaf(v, ky * kx, s * kz), fmaf(v, ky * ky, c), fmaf(v, ky * kz, -s * kx),
                            fmaf(v, kz * kx, -s * ky), fmaf(v, kz * ky, s * kx), fmaf(v, kz * kz, c)};
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float a = R[3 * r], b = R[3 * r + 1], d = R[3 * r + 2];
            R[3 * r] = a * M[0] + b * M[3] + d * M[6];
            R[3 * r + 1] = a * M[1] + b * M[4] + d * M[7];
            R[3 * r + 2] = a * M[2] + b * M[5] + d * M[8];
        }
    }
}

// `rb`: this env's random box (used for obstacle p.random_box when that is >= 0).  The chain is walked base-to-tip ONCE: the
// capsule table is ordered by body (pnr_create), so a capsule's end points are two matrix-vector products in the frame
// that is current when its body is reached (before: every end point was carried through every joint stage up to its body,
// 12 stages per capsule).
// Capsules c_first, c_first + c_step, ... are summed (K1 splits the table over its three joint warps; K2 passes 0, 1).
__device__ __forceinline__ float pnr_contact_depth(const PnrParams& p, const PnrSinCos& sc, const PnrBox& rb, int c_first,
                                                   int c_step) {
    float sn[PNR_DOF], cs[PNR_DOF];              // indexed by the running joint counter: lives in local memory
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) { sn[i] = sc.sn[i]; cs[i] = sc.cs[i]; }
    float R[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f}, org[3] = {0.f, 0.f, 0.f};
    int joint = 0;
    float total = 0.f;
#pragma unroll 1
    for (int c = c_first; c < p.n_capsules; c += c_step) {
        const int body = p.capsule_body[c];
#pragma unroll 1
        for (; joint <= body; ++joint) pnr_frame_advance(p, joint, sn[joint], cs[joint], R, org);
        const float u0 = p.capsule_p0[c][0], u1 = p.capsule_p0[c][1], u2 = p.capsule_p0[c][2];
        const float w0 = p.capsule_p1[c][0], w1 = p.capsule_p1[c][1], w2 = p.capsule_p1[c][2];
        const float ax = fmaf(R[0], u0, fmaf(R[1], u1, fmaf(R[2], u2, org[0])));
        const float ay = fmaf(R[3], u0, fmaf(R[4], u1, fmaf(R[5], u2, org[1])));
        const float az = fmaf(R[6], u0, fmaf(R[7], u1, fmaf(R[8], u2, org[2])));
        const float bx = fmaf(R[0], w0, fmaf(R[1], w1, fmaf(R[2], w2, org[0])));
        const float by = fmaf(R[3], w0, fmaf(R[4], w1, fmaf(R[5], w2, org[1])));
        const float bz = fmaf(R[6], w0, fmaf(R[7], w1, fmaf(R[8], w2, org[2])));
        const float radius = p.capsule_radius[c];
        const float dx = bx - ax, dy = by - ay, dz = bz - az;
#pragma unroll 1
        for (int o = 0; o < p.n_obstacles; ++o) {
            float px = p.obstacle_p[o][0], py = p.obstacle_p[o][1], pz = p.obstacle_p[o][2];
            float ex = p.obstacle_e[o][0], ey = p.obstacle_e[o][1], ez = p.obstacle_e[o][2];
            if (o == p.random_box) { px = rb.px; py = rb.py; pz = rb.pz; ex = rb.ex; ey = rb.ey; ez = rb.ez; }
            float d;
            if (p.obstacle_type[o] == PNR_OBSTACLE_PLANE) {
                const float da = (ax - px) * ex + (ay - py) * ey + (az - pz) * ez;
                const float db = (bx - px) * ex + (by - py) * ey + (bz - pz) * ez;
                d = fminf(da, db);
            } else if (p.obstacle_type[o] == PNR_OBSTACLE_SPHERE) {
                const float len2 = fmaxf(dx * dx + dy * dy + dz * dz, 1e-30f);
                float t = ((px - ax) * dx + (py - ay) * dy + (pz - az) * dz) / len2;
                t = fminf(fmaxf(t, 0.f), 1.f);
                const float cx = fmaf(t, dx, ax) - px, cy = fmaf(t, dy, ay) - py, cz = fmaf(t, dz, az) - pz;
                d = sqrtf(cx * cx + cy * cy + cz * cz) - ex;
            } else {
                d = pnr_segment_box_exact(ax - px, ay - py, az - pz, dx, dy, dz, ex, ey, ez);
            }
            total += fmaxf(0.f, radius - d);
        }
    }
    return total;
}
// the env's random box (zeros when the variant is off)
__device__ __forceinline__ PnrBox pnr_load_box(const PnrParams& p, int64_t env) {
    PnrBox b = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (p.random_box >= 0) {
        const float4 a = p.box_a[env];
        const float z = p.box_z[env];
        b.px = a.x; b.py = a.y; b.pz = z; b.ex = a.z; b.ey = a.w; b.ez = z;
    }
    return b;
}

// float64 twin, only for envs whose float32 distance falls inside the done band: the reference
// evaluates `distance < done_distance` in double (pioneer_knm_env.py:155-160), so the done mask is
// decided in double exactly where float32 could flip it.  Rare => deliberately not inlined.
// Arguments and results travel BY VALUE: arrays passed by reference to a non-inlined function would have to live
// in local memory on every step, taken or not (18 local stores per tile in the task warp before this).
struct PnrBandIn { float r[PNR_DOF]; float tgt[3]; };
struct PnrBandOut { float ptr[3]; float dist; int within; };

static __device__ __noinline__ PnrBandOut pnr_fk_band_f64(const PnrParams& p, PnrBandIn in) {
    double x = p.tip_xyz64[0], y = p.tip_xyz64[1], z = p.tip_xyz64[2];
    for (int j = PNR_DOF - 1; j >= 0; --j) {
        double s, c;
        sincos((double)in.r[j], &s, &c);
        const double kx = p.axis64[j][0], ky = p.axis64[j][1], kz = p.axis64[j][2];
        const double kp = (kx * x + ky * y + kz * z) * (1.0 - c);
        const double nx = x * c + (ky * z - kz * y) * s + kx * kp;
        const double ny = y * c + (kz * x - kx * z) * s + ky * kp;
        const double nz = z * c + (kx * y - ky * x) * s + kz * kp;
        const double* R = p.origin_rot64[j];
        x = R[0] * nx + R[1] * ny + R[2] * nz + p.origin_xyz64[j][0];
        y = R[3] * nx + R[4] * ny + R[5] * nz + p.origin_xyz64[j][1];
        z = R[6] * nx + R[7] * ny + R[8] * nz + p.origin_xyz64[j][2];
    }
    const double dx = (double)in.tgt[0] - x, dy = (double)in.tgt[1] - y, dz = (double)in.tgt[2] - z;
    const double d = sqrt(dx * dx + dy * dy + dz * dz);
    PnrBandOut o;
    o.ptr[0] = (float)x; o.ptr[1] = (float)y; o.ptr[2] = (float)z;
    o.dist = (float)d;
    o.within = d < p.done_distance64 ? 1 : 0;
    return o;
}

// convenience wrapper for the thread-per-env kernels (not the step kernel's task warp)
__device__ __forceinline__ void pnr_fk_tip_f64(const PnrParams& p, const float (&r)[PNR_DOF], const float (&tgt)[3],
                                               float (&ptr_out)[3], float& dist_out, bool& within) {
    PnrBandIn in;
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) in.r[i] = r[i];
    in.tgt[0] = tgt[0]; in.tgt[1] = tgt[1]; in.tgt[2] = tgt[2];
    const PnrBandOut o = pnr_fk_band_f64(p, in);
    ptr_out[0] = o.ptr[0]; ptr_out[1] = o.ptr[1]; ptr_out[2] = o.ptr[2];
    dist_out = o.dist;
    within = o.within != 0;
}

// sincos of the joint angles + tip position + distance to the target for the current r
struct PnrPose {
    float sn[PNR_DOF], cs[PNR_DOF];
    float ptr[3];
    float dist;
};

template <bool FAST>
__device__ __forceinline__ void pnr_pose(const PnrParams& p, const PnrEnv& s, PnrPose& o) {
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) pnr_sincos_sel<FAST>(s.r[i], o.sn[i], o.cs[i]);
    pnr_fk_tip(p, o.sn, o.cs, o.ptr);
    const float dx = s.tgt[0] - o.ptr[0], dy = s.tgt[1] - o.ptr[1], dz = s.tgt[2] - o.ptr[2];
    o.dist = sqrtf(fmaf(dx, dx, fmaf(dy, dy, dz * dz)));
}

// compute_potential (pioneer_knm_env.py:232-236)
__device__ __forceinline__ float pnr_potential(const PnrParams& p, float dist) {
    return __fdiv_rn(p.pot_max, __fadd_rn(__fdiv_rn(dist, p.pot_slope), 1.f));
}

// The step kernels' task code, written once so that every mode rounds alike.
// Reward (pioneer_knm_env.py:162-165, in this rounding order): (potential - old_potential) + (-penalty_step) + (award_done | 0)
__device__ __forceinline__ float pnr_reward(const PnrParams& p, float pot_old, float pot_new, bool reached) {
    return __fadd_rn(__fadd_rn(__fsub_rn(pot_new, pot_old), -p.penalty_step), reached ? p.award_done : 0.f);
}
// done / TimeLimit flags after the episode's t-th step: TRUNCATED marks a timeout that did not also reach the target
__device__ __forceinline__ uint8_t pnr_step_flags(const PnrParams& p, bool reached, int32_t t, bool& is_done) {
    const bool timeout = p.max_episode_steps > 0 && t >= p.max_episode_steps;
    is_done = reached || timeout;
    return (is_done ? PNR_DONE : 0) | ((timeout && !reached) ? PNR_TRUNCATED : 0);
}
// obstacle variant: the reward less the capsule penetration penalty
__device__ __forceinline__ float pnr_contact_penalty(const PnrParams& p, float rew, float depth) {
    return __fsub_rn(rew, __fmul_rn(p.contact_penalty, depth));
}

// pose of the env's current r and whether it reached its target, decided in float64 where float32 could flip it
// (thread-per-env kernels; the step kernel's task warp takes the sin / cos of its joint warps from shared memory)
template <bool FAST>
__device__ __forceinline__ bool pnr_pose_reached(const PnrParams& p, const PnrEnv& s, PnrPose& o) {
    pnr_pose<FAST>(p, s, o);
    bool reached = o.dist < p.done_distance;
    if (fabsf(o.dist - p.done_distance) < p.done_band) pnr_fk_tip_f64(p, s.r, s.tgt, o.ptr, o.dist, reached);
    return reached;
}

// ---------------------------------------------------------------------------------------------
// observe() (pioneer_knm_env.py:184-211): the 137-float row of one env, written into the warp's
// shared-memory tile at row `lane`.  The 36 columns that never change (r_lo, r_hi and their cos / sin,
// obs[18:54]) are written once per warp per kernel; every step rewrites the other 101.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pnr_pack_obs_const(const PnrParams& p, float* __restrict__ row) {
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) {
        row[18 + i] = p.r_lo[i];   row[24 + i] = p.cos_r_lo[i];  row[30 + i] = p.sin_r_lo[i];
        row[36 + i] = p.r_hi[i];   row[42 + i] = p.cos_r_hi[i];  row[48 + i] = p.sin_r_hi[i];
    }
}

template <bool FAST>
__device__ __forceinline__ void pnr_pack_obs_dyn(const PnrParams& p, float* __restrict__ row, const PnrEnv& s,
                                                 const PnrPose& o, float pot, bool force_slow = false) {
    float sn, cs;
#pragma unroll
    for (int i = 0; i < PNR_DOF; ++i) {
        const float r = s.r[i];
        row[0 + i] = r;            row[6 + i] = o.cs[i];         row[12 + i] = o.sn[i];
        const float dlo = __fsub_rn(r, p.r_lo[i]);
        pnr_sincos_sel<FAST>(dlo, sn, cs);
        row[54 + i] = dlo;         row[60 + i] = cs;             row[66 + i] = sn;
        const float dhi = __fsub_rn(p.r_hi[i], r);
        pnr_sincos_sel<FAST>(dhi, sn, cs);
        row[72 + i] = dhi;         row[78 + i] = cs;             row[84 + i] = sn;
        row[90 + i] = s.v[i];
        row[108 + i] = s.a[i];
    }
    row[126] = o.ptr[0]; row[127] = o.ptr[1]; row[128] = o.ptr[2];
    row[129] = s.tgt[0]; row[130] = s.tgt[1]; row[131] = s.tgt[2];
    row[132] = s.tgt[0] - o.ptr[0]; row[133] = s.tgt[1] - o.ptr[1]; row[134] = s.tgt[2] - o.ptr[2];
    row[135] = o.dist;
    row[136] = pot;
    // cos / sin of the joint rates and of the stored (unclipped) action: straight-line code unless this env
    // holds an argument outside the fast range, which a policy bounded by the action space never produces
    bool fast = FAST && !p.trig_slow && !force_slow;
    if (FAST) {
        float m = 0.f;
#pragma unroll
        for (int i = 0; i < PNR_DOF; ++i) m = fmaxf(m, fabsf(s.a[i]));
        fast = fast && (m <= PNR_TRIG_FAST_LIMIT);       // fmaxf drops NaN: a NaN action yields NaN on both paths
    }
    if (fast) {
#pragma unroll
        for (int i = 0; i < PNR_DOF; ++i) {
            pnr_sincos_fast(s.v[i], sn, cs);
            row[96 + i] = cs;      row[102 + i] = sn;
            pnr_sincos_fast(s.a[i], sn, cs);
            row[114 + i] = cs;     row[120 + i] = sn;
        }
    } else {
#pragma unroll 1
        for (int i = 0; i < PNR_DOF; ++i) {
            pnr_sincos(s.v[i], sn, cs);
            row[96 + i] = cs;      row[102 + i] = sn;
            pnr_sincos(s.a[i], sn, cs);
            row[114 + i] = cs;     row[120 + i] = sn;
        }
    }
}

// the observation normaliser's element map: clip((x - mean) * inv_std, +-clip)   (pnr_filter.cu, fused step kernel)
__device__ __forceinline__ float pnr_normalise(float x, float mean, float inv_std, float clip) {
    return fminf(fmaxf((x - mean) * inv_std, -clip), clip);
}

// The fused normaliser's column pass: one column of a shared-memory tile (`rows` rows) is normalised in place, and the
// float64 sum and sum of squares of x - mean are ADDED to s and q.  Two independent chains; the statistics depend on the
// order of these additions.
__device__ __forceinline__ void pnr_filter_column(float* colp, int rows, float mean, float inv, float clip, double& s,
                                                  double& q) {
    double s1 = 0.0, q1 = 0.0;
    int r = 0;
#pragma unroll 4
    for (; r + 1 < rows; r += 2) {
        const float d0 = colp[r * PNR_OBS_DIM] - mean, d1 = colp[(r + 1) * PNR_OBS_DIM] - mean;
        const double e0 = (double)d0, e1 = (double)d1;
        s += e0; q = fma(e0, e0, q);
        s1 += e1; q1 = fma(e1, e1, q1);
        colp[r * PNR_OBS_DIM] = fminf(fmaxf(d0 * inv, -clip), clip);
        colp[(r + 1) * PNR_OBS_DIM] = fminf(fmaxf(d1 * inv, -clip), clip);
    }
    if (r < rows) {
        const float d0 = colp[r * PNR_OBS_DIM] - mean;
        const double e0 = (double)d0;
        s += e0; q = fma(e0, e0, q);
        colp[r * PNR_OBS_DIM] = fminf(fmaxf(d0 * inv, -clip), clip);
    }
    s += s1; q += q1;
}

// the statistics of constant column c (18 <= c < 54) over `rows` rows, added analytically to the accumulator
__device__ __forceinline__ void pnr_filter_const_column(const PnrParams& p, const float* __restrict__ f_applied,
                                                        double* __restrict__ f_delta, int c, double rows) {
    const int g = (c - 18) / PNR_DOF, j = (c - 18) % PNR_DOF;
    const float x = g == 0 ? p.r_lo[j] : g == 1 ? p.cos_r_lo[j] : g == 2 ? p.sin_r_lo[j]
                  : g == 3 ? p.r_hi[j] : g == 4 ? p.cos_r_hi[j] : p.sin_r_hi[j];
    const double d = (double)(x - f_applied[c]);
    atomicAdd(&f_delta[1 + c], rows * d);
    atomicAdd(&f_delta[1 + PNR_OBS_DIM + c], rows * d * d);
}

// ---- per-joint column groups for the step kernel's joint warps (joint j owns columns j, 6+j, ..., 120+j) ----
__device__ __forceinline__ void pnr_pack_joint_const(const PnrParams& p, float* __restrict__ row, int j) {
    row[18 + j] = p.r_lo[j];   row[24 + j] = p.cos_r_lo[j];  row[30 + j] = p.sin_r_lo[j];
    row[36 + j] = p.r_hi[j];   row[42 + j] = p.cos_r_hi[j];  row[48 + j] = p.sin_r_hi[j];
}

// `rowj` = row + j: every store below has an immediate offset from one base register
__device__ __forceinline__ void pnr_pack_joint_head(float* __restrict__ rowj, float r, float sn, float cs) {
    rowj[0] = r;               rowj[6] = cs;                 rowj[12] = sn;
}

// r - r_lo, r_hi - r, v, a and their cos / sin.  `fast_va`: v and a are inside the fast sincos range
__device__ __forceinline__ void pnr_pack_joint_rest(float* __restrict__ rowj, float r_lo, float r_hi, float r,
                                                    float v, float a, bool fast_va) {
    float sn, cs;
    const float dlo = __fsub_rn(r, r_lo);
    pnr_sincos_fast(dlo, sn, cs);
    rowj[54] = dlo;            rowj[60] = cs;                rowj[66] = sn;
    const float dhi = __fsub_rn(r_hi, r);
    pnr_sincos_fast(dhi, sn, cs);
    rowj[72] = dhi;            rowj[78] = cs;                rowj[84] = sn;
    rowj[90] = v;
    rowj[108] = a;
    if (fast_va) {
        pnr_sincos_fast(v, sn, cs);
        rowj[96] = cs;         rowj[102] = sn;
        pnr_sincos_fast(a, sn, cs);
        rowj[114] = cs;        rowj[120] = sn;
    } else {
        pnr_sincos(v, sn, cs);
        rowj[96] = cs;         rowj[102] = sn;
        pnr_sincos(a, sn, cs);
        rowj[114] = cs;        rowj[120] = sn;
    }
}

// episode statistics of one warp (= one tile): one set of atomics per warp that saw an episode end
__device__ __forceinline__ void pnr_episode_stats(PnrStats* __restrict__ stats, bool ended, bool reached, float ep_ret,
                                                  int32_t t, int lane) {
    const unsigned done_mask = __ballot_sync(PNR_FULL_MASK, ended);
    if (done_mask) {
        const bool mine = (done_mask >> lane) & 1u;
        float ret = mine ? ep_ret : 0.f, ret2 = ret * ret, len = mine ? (float)t : 0.f;
        float mx = mine ? ep_ret : -INFINITY, mn = mine ? ep_ret : INFINITY;
#pragma unroll
        for (int ofs = 16; ofs > 0; ofs >>= 1) {
            ret += __shfl_xor_sync(PNR_FULL_MASK, ret, ofs);
            ret2 += __shfl_xor_sync(PNR_FULL_MASK, ret2, ofs);
            len += __shfl_xor_sync(PNR_FULL_MASK, len, ofs);
            mx = fmaxf(mx, __shfl_xor_sync(PNR_FULL_MASK, mx, ofs));
            mn = fminf(mn, __shfl_xor_sync(PNR_FULL_MASK, mn, ofs));
        }
        const unsigned reach_mask = __ballot_sync(PNR_FULL_MASK, reached);
        if (lane == 0) {
            atomicAdd(&stats->episodes, (double)__popc(done_mask));
            atomicAdd(&stats->sum_return, (double)ret);
            atomicAdd(&stats->sum_length, (double)len);
            atomicAdd(&stats->sum_return_sq, (double)ret2);
            atomicAdd(&stats->reached, (double)__popc(reach_mask));
            atomicMax(&stats->max_return_ord, pnr_float_to_ordered(mx));
            atomicMin(&stats->min_return_ord, pnr_float_to_ordered(mn));
        }
    }
}

// hand the warp's tile (rows_valid x 137 floats, contiguous in `out`) to global memory.  Full tiles (and any
// tile whose byte count is a multiple of 16) go out as ONE TMA bulk store issued by lane 0; other ragged tails
// use coalesced 16-byte stores.  Call pnr_tile_wait() before writing the tile again.
__device__ __forceinline__ bool pnr_tile_is_bulk(int rows_valid) { return (rows_valid & 3) == 0; }

// ragged tail: `n_threads` threads (tid = 0 .. n_threads-1) stream the tile with coalesced 16-byte stores
__device__ __forceinline__ void pnr_emit_tile_manual(const float* __restrict__ tile, float* __restrict__ out,
                                                     int rows_valid, int tid, int n_threads) {
    const int total = rows_valid * PNR_OBS_DIM;
    const int n4 = total >> 2;
    const float4* t4 = reinterpret_cast<const float4*>(tile);
    float4* o4 = reinterpret_cast<float4*>(out);
#pragma unroll 4
    for (int i = tid; i < n4; i += n_threads) pnr_st_stream(o4 + i, t4[i]);
    for (int i = (n4 << 2) + tid; i < total; i += n_threads) pnr_st_stream(out + i, tile[i]);
}

// one warp owns the tile (reset / observe kernels)
__device__ __forceinline__ void pnr_emit_tile(const float* __restrict__ tile, float* __restrict__ out,
                                              int rows_valid, int lane) {
    pnr_fence_async_smem();
    __syncwarp();
    if (pnr_tile_is_bulk(rows_valid)) {
        if (lane == 0) {
            pnr_bulk_store(out, tile, (uint32_t)(rows_valid * PNR_OBS_DIM * sizeof(float)));
            pnr_bulk_commit();
        }
    } else {
        pnr_emit_tile_manual(tile, out, rows_valid, lane, 32);
    }
}

// the tile may be overwritten once the copy engine has finished READING it
__device__ __forceinline__ void pnr_tile_wait(int lane) {
    if (lane == 0) pnr_bulk_wait_read<0>();
    __syncwarp();
}
