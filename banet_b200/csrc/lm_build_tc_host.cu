// Host side of the tensor-core build path (sm_100a: TMA + tcgen05 + TMEM): support check, launch plan, tensor maps, dispatch to
// the kernel generations.
//
// Maths and partial-slot contract are those of lm_build.cu (reference bundlenet.py:206-263 + utils.cu:219-417); the basis contraction
// runs on the 5th-gen tensor cores:
//
//     D[128 x 160] += Bt^T R          per 64-pixel tile, kind::tf32, fp32 accumulate in TMEM
//        Bt [64 px x 128]  the basis tile exactly as it lies in HBM (TMA, 128B/32B-atom swizzle) = MN-major "A"
//        R  [64 px x 160]  row n = [ s_n * b_n (128) | v_n (6) | t_n | 0 ... ]  built by the algebra warps = MN-major "B"
//     => D[i][j<128] = H_dd[i][j],  D[i][128+r] = H_cd[r][i] (r<6),  D[i][134] = g_d[i]
//
// Precision modes (tf32 keeps 10 mantissa bits; products are exact, accumulation is fp32):
//   MODE 1  one pass:   A and R both rounded by us (A stochastically, in place; R to nearest)
//   MODE 2  two passes: + A_lo = b - trunc(b)                       (only R's unbiased rounding remains)
//   MODE 3  three passes: + R_lo = s*b - rna(s*b)                   (fp32-grade: the dropped term is ~2^-22)
//
// Tiles: 64 points.  With the dense-grid hint (banet_level_t::grid_w/h) a tile is an 8x8 pixel patch fetched by ONE 3-D TMA box;
// without the hint a tile is 64 consecutive points (2-D TMA box).
//
// Kernel generations:
//   7 (lm_build_tc7.cu)  F2-only conv2 + dense grid: the tile's F2 footprint is staged into shared memory by TMA (channel chunks),
//                        the 12 gradient/bilinear taps of every pixel come from LDS; per-tile fallback to global taps when the
//                        footprint of a tile does not fit the staged window.  MODE 1 (where it is the default) and 2.
//   6 (lm_build_tc6.cu)  everything else (the reference's [F2|gx|gy] layout, unstructured point lists, MODE 3): taps by ld.global.
#include "common.cuh"
#include "lm_build.h"
#include "tc_utils.cuh"
#include "tmap.h"

namespace banet {

constexpr int TC_TILE = 64;

int lm_build_tc6_launch(int mode, bool fly, int nch, int kblk, const CUtensorMap& tm, const BuildParams& prm, int grid, cudaStream_t st);
int lm_build_tc7_launch(int mode, int nch, int kblk, const CUtensorMap& tmB, const CUtensorMap& tmF, const CUtensorMap& tmC, const BuildParams& prm, int grid,
                        cudaStream_t st);
bool lm_build_tc7_supported(int mode, int nch, int kblk);

constexpr int kTc6DefaultBandRows = 1, kTc6DefaultL2Hints = 0, kTc6DefaultTapPrefetch = 0;
static banet_tuning_t g_tuning = {0, 0, 4, 0, 0, 0};
void set_tuning(const banet_tuning_t& t) { g_tuning = t; }
const banet_tuning_t& tuning() { return g_tuning; }

bool tc_supported(const banet_level_t* lv)
{
    const bool k_ok = lv->K == 128 || lv->K == 64 || lv->K == 32;
    return k_ok && (lv->C == 64 || lv->C == 128) && (lv->conv2_channels == lv->C || lv->conv2_channels == 3 * lv->C) &&
           ((reinterpret_cast<uintptr_t>(lv->conv1) | reinterpret_cast<uintptr_t>(lv->conv2) | reinterpret_cast<uintptr_t>(lv->B)) % 16 == 0) &&
           (long long)lv->nb * lv->N < (1LL << 31) && (long long)lv->nb * ((lv->N + 63) / 64 + 80) < (1LL << 31) &&
           (long long)lv->h * lv->w * lv->conv2_channels < (1LL << 31);
}

// Generation 7 applies to the F2-only layout on a dense grid (tap coordinates are packed in 16 bits).  Default choice (tc_generation = 0),
// from interleaved A/B runs at the board's steady power state (profiles/r02d_gen6_vs_gen7_f2layout.txt): in the single-pass mode (TF32X1)
// generation 7 is 9 % (640x480) to 15 % (320x240) faster than generation 6 on this layout; in the two- and three-pass modes its gather
// warps also carry the operand splitting and generation 6 is faster.  banet_set_tuning forces either (6 / 7).
static bool use_gen7(const banet_level_t* lv, int mode, int kblk)
{
    const bool wanted = g_tuning.tc_generation == 7 || (g_tuning.tc_generation == 0 && mode == 1);
    return wanted && lv->conv2_channels == lv->C && lv->grid_w > 0 && lv->h < 65536 && lv->w < 65536 &&
           lm_build_tc7_supported(mode, lv->C / 64, kblk);
}

int build_plan_tc(const banet_level_t* lv, int num_sms, BuildPlan* plan)
{
    plan->KP = 128;
    if (lv->grid_w > 0) plan->tiles_per_pair = ((lv->grid_w + 7) / 8) * ((lv->grid_h + 7) / 8);
    else plan->tiles_per_pair = (lv->N + TC_TILE - 1) / TC_TILE;
    plan->total_tiles = (long long)lv->nb * plan->tiles_per_pair;
    long long grid = num_sms;
    if (grid > plan->total_tiles) grid = plan->total_tiles;
    if (grid < 1) grid = 1;
    plan->grid = (int)grid;
    const long long tiles_per_cta = (plan->total_tiles + grid - 1) / grid;
    plan->max_span = (int)((tiles_per_cta + plan->tiles_per_pair - 2) / plan->tiles_per_pair) + 1;
    SlotLayout L{lv->K, lv->C};
    plan->slot_floats = L.floats();
    plan->ws_bytes = align_up((size_t)plan->grid * plan->max_span * plan->slot_floats * sizeof(float), 256);
    return BANET_OK;
}

int lm_build_tc(const banet_level_t* lv, const BuildPlan& plan, int mode, const float* R, const float* T, const float* W,
                float* H, float* g, float* rbar_sum, float* nvalid, void* ws, cudaStream_t st)
{
    BANET_REQUIRE(tc_supported(lv), BANET_ERR_UNSUPPORTED,
                  "lm_build (tensor-core path) needs K in {32,64,128}, C in {64,128}, 16-B aligned tensors; got K=%d C=%d", lv->K, lv->C);
    const int kblk = lv->K / 32;
    if (kblk != 4 && mode == 1) mode = 2;          // K = 64 / 32: the single-pass mode is not instantiated
    CUtensorMap tm;
    int rc;
    if (lv->grid_w > 0) rc = make_tmap_f32_3d_sw128_32b(&tm, lv->B, (uint64_t)lv->nb * lv->grid_h, lv->grid_w, lv->K, 8, 8, 32);
    else rc = make_tmap_f32_2d_sw128_32b(&tm, lv->B, (uint64_t)lv->nb * lv->N, lv->K, TC_TILE, 32);
    if (rc) return rc;
    const bool fly = lv->conv2_channels == lv->C;
    BuildParams prm;
    prm.nb = lv->nb; prm.N = lv->N; prm.C = lv->C; prm.K = lv->K; prm.h = lv->h; prm.w = lv->w; prm.c2 = lv->conv2_channels;
    prm.conv1 = lv->conv1; prm.conv2 = lv->conv2; prm.intr = lv->intr; prm.p = lv->p; prm.D = lv->D; prm.B = lv->B;
    prm.R = R; prm.T = T; prm.W = W;
    prm.partials = reinterpret_cast<float*>(ws);
    prm.slot_floats = plan.slot_floats; prm.max_span = plan.max_span;
    prm.tiles_per_pair = plan.tiles_per_pair; prm.total_tiles = plan.total_tiles;
    prm.grid_w = lv->grid_w; prm.grid_h = lv->grid_h;
    prm.tiles_x = lv->grid_w > 0 ? (lv->grid_w + 7) / 8 : 0; prm.tiles_y = lv->grid_h > 0 ? (lv->grid_h + 7) / 8 : 0;
    prm.band_rows = 1; prm.l2_hints = 0; prm.tap_prefetch = 0; prm.kq_i = 0; prm.kq_j = 0;
    prm.hdd_transposed = 1;
    prm.force_direct = g_tuning.tc7_force_direct;
    const int nch = lv->C / 64;
    if (use_gen7(lv, mode, kblk)) {
        int band = g_tuning.tc7_band_rows; if (band < 1) band = 1; if (band > prm.tiles_y) band = prm.tiles_y;
        prm.band_rows = band;
        CUtensorMap tmF;        // staged F2 windows: 32 channels x WX x WY texels
        int wx = 0, wy = 0; lm_build_tc7_window(&wx, &wy);
        rc = make_tmap_f32_nhwc(&tmF, lv->conv2, lv->nb, lv->h, lv->w, lv->conv2_channels, 32, wx, wy);
        if (rc) return rc;
        CUtensorMap tmC;        // conv1 chunk of an 8x8 tile: 32 channels x 8 x 8 pixels of [nb, grid_h, grid_w, C]
        rc = make_tmap_f32_nhwc(&tmC, lv->conv1, lv->nb, lv->grid_h, lv->grid_w, lv->C, 32, 8, 8);
        if (rc) return rc;
        rc = lm_build_tc7_launch(mode, nch, kblk, tm, tmF, tmC, prm, plan.grid, st);
    } else {
        // dense grid: band walk + L2 policy (defaults picked from the B200 measurements in profiles/r02c_*)
        int band = g_tuning.tc6_band_rows > 0 ? g_tuning.tc6_band_rows : kTc6DefaultBandRows;
        if (band > prm.tiles_y) band = prm.tiles_y;
        prm.band_rows = lv->grid_w > 0 && band > 1 ? band : 1;
        prm.l2_hints = g_tuning.tc6_l2_hints > 0 ? g_tuning.tc6_l2_hints - 1 : kTc6DefaultL2Hints;
        prm.tap_prefetch = g_tuning.tc6_tap_prefetch > 0 ? g_tuning.tc6_tap_prefetch - 1 : kTc6DefaultTapPrefetch;
        rc = lm_build_tc6_launch(mode, fly, nch, kblk, tm, prm, plan.grid, st);
    }
    if (rc) return rc;
    return launch_lm_reduce(prm, plan.grid, H, g, rbar_sum, nvalid, st);
}

}  // namespace banet
