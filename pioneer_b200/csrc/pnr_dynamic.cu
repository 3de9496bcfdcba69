// K2: the fused env step of the dynamic (Tier-B) mode.  One thread per env: frame_skip substeps of
// [PD / torque control -> Featherstone ABA -> semi-implicit Euler -> limit stops] with the joint state in
// registers, then the same task code as the kinematic env (pioneer_knm_env.py:151-211): forward kinematics of
// the pointer, reward, done, TimeLimit, statistics, auto-reset, 137-float observation staged per warp in shared
// memory and stored with one TMA bulk copy.  Bound: FP32 pipe (10 x ~1.45 kflop per env-step against 761 B).
#include "pnr_dynamic_kernel.cuh"

cudaError_t pnr_launch_step_dynamic(const PnrParams& p, int device, int obs_mode, float4* state, const float* actions,
                                    float* obs, float* reward, uint8_t* done, PnrStats* stats, uint32_t tick, uint32_t domain,
                                    const float* f_applied, double* f_delta, float f_clip, PnrMulti multi, cudaStream_t stream) {
    typedef PnrDynKernel Kern;
#define PNR_DYN_ROW(CH, ST) \
    {{pnr_step_dynamic_kernel<PNR_OBS_TERMINAL, false, CH, ST>, pnr_step_dynamic_kernel<PNR_OBS_TERMINAL, true, CH, ST>}, \
     {pnr_step_dynamic_kernel<PNR_OBS_AUTORESET, false, CH, ST>, pnr_step_dynamic_kernel<PNR_OBS_AUTORESET, true, CH, ST>}}
    static Kern explicit_kernels[3][2][2] = {PNR_DYN_ROW(PNR_CHAIN_GENERIC, PNR_STEPPING_EXPLICIT),
                                             PNR_DYN_ROW(PNR_CHAIN_PIONEER, PNR_STEPPING_EXPLICIT),
                                             PNR_DYN_ROW(PNR_CHAIN_PIONEER_ISO, PNR_STEPPING_EXPLICIT)};
    static int grids[PNR_MAX_DEVICES][2][3][2][2] = {};
    const int obst = p.n_obstacles > 0 ? 1 : 0;
    const int stepping = p.dyn_stepping == PNR_STEPPING_BULLET ? 1 : 0;
    const int chain = p.chain_kind == 1 ? (p.dyn_iso_links ? PNR_CHAIN_PIONEER_ISO : PNR_CHAIN_PIONEER) : PNR_CHAIN_GENERIC;
    Kern kern = stepping ? pnr_dynamic_bullet_kernel(chain, obs_mode, obst) : explicit_kernels[chain][obs_mode][obst];
    int& resident = grids[device % PNR_MAX_DEVICES][stepping][chain][obs_mode][obst];
    if (resident == 0) {
        cudaError_t e = pnr_prepare((const void*)kern, device, PNR_DYN_THREADS, PNR_DYN_SMEM, &resident);
        if (e != cudaSuccess) return e;
    }
    const int64_t per_cta = PNR_TILE_ENVS * PNR_DYN_WARPS;
    int64_t grid = (p.n_envs + per_cta - 1) / per_cta;
    if (grid > resident) grid = resident;
    if (grid < 1) grid = 1;
    return pnr_launch_pdl(kern, true, grid, PNR_DYN_THREADS, PNR_DYN_SMEM, stream, p, state, actions, obs, reward, done, stats,
                          tick, domain, f_applied, f_delta, f_clip, multi);
}
