// Internal interfaces between the translation units of libbanet_sm100.so.
#pragma once
#include "common.cuh"

namespace banet {

struct BuildParams {
    int nb, N, C, K, h, w, c2;
    const float *conv1, *conv2, *intr, *p, *D, *B, *R, *T, *W;
    float* partials;
    int slot_floats, max_span, tiles_per_pair;
    long long total_tiles;
    int grid_w, grid_h, tiles_x, tiles_y;   // dense-grid 8x8 tiling (tensor-core path); grid_w == 0 -> linear 64-pixel tiles
    int kq_i, kq_j;                   // fp32 SIMT path, K > 128: the 128 x 128 block of H_dd this launch computes
    int band_rows;                    // dense-grid tensor-core kernels: tiles are walked in bands of this many tile rows, column by column inside a band
    int tap_prefetch;                 // generation 6: 0 off, 1 the geometry warps prefetch the tap footprint into L2 (halo from the tile's border pixels), 2 = every pixel also fetches its lower row
    int l2_hints;                     // generation 6: 0 none, 1 read-once streams evict-first, 2 = 1 + taps evict-last
    int hdd_transposed;               // tensor-core path stores the H_dd block of a slot column-major (coalesced TMEM drains)
    int force_direct;                 // generation 7, testing: take the global-tap fallback for every tile
};

struct BuildPlan {
    int KP, grid, max_span, slot_floats, tiles_per_pair;
    long long total_tiles;
    size_t ws_bytes;
};

int num_sms();

// fp32 SIMT path (lm_build.cu)
int build_plan(const banet_level_t* lv, int num_sms, BuildPlan* plan);
int lm_build_simt(const banet_level_t* lv, const BuildPlan& plan, const float* R, const float* T, const float* W,
                  float* H, float* g, float* rbar_sum, float* nvalid, void* ws, cudaStream_t st);

int launch_lm_reduce(const BuildParams& prm, int grid_build, float* H, float* g, float* rbar_sum, float* nvalid, cudaStream_t st);

// tensor-core path (lm_build_tc_host.cu + lm_build_tc6.cu / lm_build_tc7.cu on lm_build_tc_roles.cuh): K in {32,64,128}, C in {64,128}
void set_tuning(const banet_tuning_t& t);
const banet_tuning_t& tuning();
void lm_build_tc7_window(int* wx, int* wy);
bool tc_supported(const banet_level_t* lv);
int build_plan_tc(const banet_level_t* lv, int num_sms, BuildPlan* plan);
int lm_build_tc(const banet_level_t* lv, const BuildPlan& plan, int mode, const float* R, const float* T, const float* W,
                float* H, float* g, float* rbar_sum, float* nvalid, void* ws, cudaStream_t st);

// precision resolution + dispatch (abi.cu)
int resolve_precision(const banet_level_t* lv, int precision);      // -> BANET_PREC_* actually used, or <0 (error set)
int plan_for(const banet_level_t* lv, int resolved, BuildPlan* plan);
int build_dispatch(const banet_level_t* lv, int resolved, const BuildPlan& plan, const float* R, const float* T, const float* W,
                   float* H, float* g, float* rbar_sum, float* nvalid, void* ws, cudaStream_t st);

// lambda MLP / solve / update (lm_solve.cu)
int lm_lambda(const float* rbar_sum, int nb, int N, int C, const float* mlp, float base, float* lambda_out, cudaStream_t st);
int lm_solve_update(const float* H, const float* g, const float* lambda, int nb, int K, const banet_solve_opts_t& opts,
                    const float* R, const float* T, const float* W, float* R_out, float* T_out, float* W_out,
                    float* delta, int32_t* status, int status_accumulate, cudaStream_t st);

// fused lambda-MLP + damping + blocked Cholesky + update, one launch (lm_step.cu); mlp == nullptr: lambda_in is used as is
struct StepMode { float lambda_exp0; int rbar_per_valid, use_vmatrix, clamp_theta; };
constexpr StepMode kStepBundleNet = {2.0f, 0, 1, 1};          // bundlenet.py:241-276
bool lm_step_supported(int P, int C);
int lm_step(const float* H, const float* g, const float* rbar_sum, int nb, int N, int C, int K, const float* mlp, float base, const float* lambda_in,
            const StepMode& mode, const float* nvalid, const banet_solve_opts_t& opts, const float* R, const float* T, const float* W, float* R_out, float* T_out, float* W_out,
            float* delta, float* lambda_out, int32_t* status, int status_accumulate, cudaStream_t st);

int launch_pose_update(const float* delta, int nb, int P, const float* R, const float* T, float* R_out, float* T_out, cudaStream_t st);

// joint step of a keyframe window: nf pairs sharing one W (lm_window.cu); ws: lm_window_step_workspace_floats floats
bool lm_window_supported(int nf, int K, int C);
size_t lm_window_step_workspace_floats(int nf, int K, int C);
int lm_window_broadcast_w(float* W, int nf, int K, cudaStream_t st);
int lm_window_step(const float* H, const float* g, const float* rbar_sum, int nf, int N, int C, int K, const float* mlp, float base,
                   const float* lambda_in, const banet_solve_opts_t& opts, float* R, float* T, float* W, float* ws, float* lambda_out,
                   int32_t* status, cudaStream_t st);

// legacy pose-only tracker loop with device-side accept / reject and early termination (lm_legacy.cu)
size_t lm_track_legacy_workspace_bytes(const banet_level_t* levels, int nlevels);
int lm_track_legacy(const banet_level_t* levels, int nlevels, const int* level_iters, const float* const* mlp_weights, const banet_legacy_opts_t& o,
                    float* R, float* T, int32_t* iters_done, float* valid_ratio, int32_t* status, void* ws, size_t ws_bytes, cudaStream_t st);

// backward of one iteration (lm_bwd.cu)
int lm_build_bwd(const banet_level_t* lv, const float* R, const float* T, const float* W, const float* dH, const float* dg, const float* drbar,
                 int exact_sym, float* dconv1, float* dconv2, float* dD, float* dB, float* dR, float* dT, float* dW, cudaStream_t st);
int lm_solve_update_bwd(const float* H, const float* g, const float* lambda, const float* delta, int nb, int K, const banet_solve_opts_t& opts,
                        const float* R, const float* T, const float* gRn, const float* gTn, const float* gWn,
                        float* dH, float* dg, float* dlambda, float* dR, float* dT, float* dW, cudaStream_t st);

}  // namespace banet
