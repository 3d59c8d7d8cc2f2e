// lm_build_tc6.cu — tensor-core build kernel, generation 6: every phase has its own warpgroup, phases of different tiles overlap.
//
// Roles, barriers and the pipeline code both generations share: lm_build_tc_roles.cuh.  What generation 6 does in them (register budgets by
// setmaxnreg, 48 / 88 / 72 / 32 = 64 512 of the SM's 65 536 registers):
//
//   geometry warps (48 regs)  b.W; in MODE 1 they also round the basis tile to tf32 in place; tap offsets -> pixel records
//   gather warps   (88 regs)  13 tap loads per (pixel, 4 channels) by ld.global -> blend / accumulate -> M, q
//   algebra warps  (72 regs)  besides the shared algebra: the R rows s_n * b_n (A_lo, R_lo) into smem; L2-hinted basis TMA
//   drainer warps  (32 regs)
#include "lm_build_tc_roles.cuh"
#include "tmap.h"
#include <stdlib.h>

namespace banet { namespace v6 {
using namespace tcb;

__device__ __forceinline__ float hsum16(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 8); v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2); v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

template <int MODE, bool FLY> struct Smem {
    // basis-tile stages (TMA ring) and pixel-record buffers.  Deeper rings decouple the roles, but whatever smem the CTA takes is lost
    // to the L1 that catches the tap overlap of neighbouring pixels: measured best per mode / layout (640x480, 32 pairs):
    //   TF32X2 + [F2|gx|gy] layout: 3 stages (192 KB -> 196 KB carve-out, 60 KB L1) 7.4 ms vs 4 stages (228 KB) 8.6 ms
    //   TF32X2 + F2-only layout   : 4 stages 7.2 ms vs 3 stages 8.8 ms;  TF32X1: 4 stages 5.6 ms vs 3 stages 6.1 ms
    static constexpr int NST = MODE == 3 ? 3 : (MODE == 2 && !FLY) ? 3 : 4;
    static constexpr int NREC = MODE == 3 ? 2 : 3;
    static constexpr int off_A = 0;
    static constexpr int off_R = NST * STAGE_A;
    static constexpr int off_Alo = off_R + STAGE_R;
    static constexpr int off_Rlo = off_Alo + (MODE >= 2 ? STAGE_A : 0);
    static constexpr int off_misc = off_Rlo + (MODE == 3 ? STAGE_R : 0);
    static constexpr int off_bar = off_misc;                           // NBARS mbarriers
    static constexpr int off_tmem = off_bar + NBARS * 8;
    static constexpr int off_tile = off_misc + 192;                    // [NREC][4] ints: pair index of the tile in record buffer s
    static constexpr int off_pose = off_tile + 64;                     // [W0][16] floats (private to each geometry warp)
    static constexpr int off_w = off_pose + W0 * 16 * 4;               // [W0][128] floats: W of the pair (private to each geometry warp)
    static constexpr int off_rec = off_w + W0 * 128 * 4;               // [NREC][TILE][REC] floats
    static constexpr int off_rbs = off_rec + NREC * TILE * REC * 4;    // [GW][128] floats: rbar hand-over gather -> algebra
    static constexpr int off_ccs = off_rbs + GW * 128 * 4;             // [AW][28] floats: H_cc / g_c / nvalid partials per algebra warp
    static constexpr int total = off_ccs + AW * 28 * 4;
    static constexpr int slack = MODE == 3 ? 0 : 512;                  // MODE 3 fills the SM: the (512-B) base alignment is checked, not padded
    static constexpr int bytes = total + slack;
};

template <int NCH, bool FLY, int MODE, int KBLK = 4>
__global__ void __launch_bounds__(THREADS, 1)
lm_build_tc6_kernel(const __grid_constant__ CUtensorMap tmapB, const BuildParams prm)
{
    using SM = Smem<MODE, FLY>;
    constexpr int NST = SM::NST, NREC = SM::NREC;
    // KBLK = K / 32 basis blocks actually present (K = 128, 64 or 32).  The smem / TMEM geometry stays that of K = 128 (M = 128 rows of D,
    // 32-KB stages); blocks >= KBLK are never loaded, read by the SIMT loops or drained, and the [v | t] block of R follows the last one.
    constexpr int KR = 32 * KBLK, NMMA = KBLK == 4 ? NN : KR + 16;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // align through the 32-bit shared address so that the compiler keeps every access in the shared state space (LDS/STS, not generic LD/ST)
    unsigned char* base = smem_raw + (SM::slack ? ((512u - (smem_u32(smem_raw) & 511u)) & 511u) : 0u);
    if (SM::slack == 0 && (smem_u32(smem_raw) & 511u)) __trap();      // fail loudly: swizzle atoms need 512-B aligned stage bases
    const Barriers bar(reinterpret_cast<uint64_t*>(base + SM::off_bar));
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(base + SM::off_tmem);
    int* sTile = reinterpret_cast<int*>(base + SM::off_tile);
    float* sPose = reinterpret_cast<float*>(base + SM::off_pose);
    float* sW = reinterpret_cast<float*>(base + SM::off_w);
    float* sRec = reinterpret_cast<float*>(base + SM::off_rec);
    float* sRbs = reinterpret_cast<float*>(base + SM::off_rbs);
    float* sCcs = reinterpret_cast<float*>(base + SM::off_ccs);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int N = prm.N, h = prm.h, w = prm.w, c2 = prm.c2;
    const bool grid2d = prm.grid_w > 0;
    constexpr int C = 64 * NCH;
    const long long t_begin = part_begin(prm.total_tiles, gridDim.x, blockIdx.x);
    const long long t_end   = part_begin(prm.total_tiles, gridDim.x, blockIdx.x + 1);
    const int ntiles = (int)(t_end - t_begin);

    if (tid == 0) {
        init_barriers<NST, NREC>(bar);
        prefetch_tmap(&tmapB);
    }
    const uint32_t tmem = setup_tmem<MODE, KBLK>(base + SM::off_R, base + SM::off_Rlo, s_tmem, tid, warp);

    // lane -> (row r of the warp's 16, half hf of the 128 basis columns); 16-B chunk walk rotated by the row so that every
    // quarter-warp touches 8 distinct bank groups of the swizzled tile (used by the b.W and the R-row loops)
    const int r16 = lane & 15, hf = lane >> 4;

    if (warp < W0) {
        // ===================================================================== geometry warps: b.W, warp, mask, tap offsets -> records
        setmaxnreg_dec<48>();
        const int gwi = warp, nlr = gwi * 16 + r16;
        float* myPose = sPose + gwi * 16;
        float* myW = sW + gwi * 128;
        int geom_b = -1;
        uint32_t dseed = 0;                                  // MODE 1: dither seed of the current pair
        TileCoord nxt = tile_coord(prm, t_begin);
        int nxt_r = (int)((unsigned)t_begin - (unsigned)nxt.b * (unsigned)prm.tiles_per_pair);
        for (int j = 0; j < ntiles; ++j) {
            const TileCoord tc = nxt;
            if (++nxt_r == prm.tiles_per_pair) { nxt_r = 0; ++nxt.b; nxt.tx0 = 0; nxt.ty0 = 0; nxt.n0 = 0; nxt.cnt = grid2d ? TILE : min(TILE, N); }
            else if (grid2d && prm.band_rows > 1) nxt = tile_coord(prm, t_begin + j + 1);
            else if (grid2d) { nxt.tx0 += 8; if (nxt.tx0 >= prm.tiles_x * 8) { nxt.tx0 = 0; nxt.ty0 += 8; } }
            else { nxt.n0 += TILE; nxt.cnt = min(TILE, N - nxt.n0); }
            const int b = tc.b;
            if (gwi == 1 && j + 2 < ntiles) prefetch_inputs<C>(prm, tile_coord(prm, t_begin + j + 2), grid2d, N, lane);
            if (b != geom_b) {
                geom_b = b;
                __syncwarp();
                if (lane < 9) myPose[lane] = prm.R[b * 9 + lane];
                else if (lane < 12) myPose[lane] = prm.T[b * 3 + lane - 9];
                else if (lane < 16) myPose[lane] = prm.intr[b * 4 + lane - 12];
                if (KBLK == 4 || 4 * lane < KR)
                    *reinterpret_cast<float4*>(myW + 4 * lane) = __ldg(reinterpret_cast<const float4*>(prm.W + (size_t)b * KR + 4 * lane));
                if constexpr (MODE == 1)     // a pure function of the inputs that changes whenever the iterate changes (see tf32_stochastic4)
                    dseed = (__float_as_uint(__ldg(prm.W + (size_t)b * KR)) * 0x9E3779B1u) ^ (__float_as_uint(__ldg(prm.W + (size_t)b * KR + 1)) * 0x85EBCA77u)
                          ^ (__float_as_uint(__ldg(prm.W + (size_t)b * KR + 2)) * 0xC2B2AE3Du) ^ __float_as_uint(__ldg(prm.T + b * 3)) ^ (uint32_t)b;
                __syncwarp();
            }
            const int s = j % NST, sr = j % NREC;
            const unsigned char* As = base + SM::off_A + s * STAGE_A;
            // global inputs of this lane's pixel first (their latency hides behind the waits and the dot product)
            float p0 = 0.f, p1 = 0.f, p2 = 0.f, D0 = 0.f;
            int n = 0; bool valid = false;
            if (grid2d) { const int gx = tc.tx0 + (nlr & 7), gy = tc.ty0 + (nlr >> 3); valid = gx < prm.grid_w && gy < prm.grid_h; n = gy * prm.grid_w + gx; }
            else { valid = nlr < tc.cnt; n = tc.n0 + nlr; }
            if (lane < 16 && valid) {
                const float* pp = prm.p + (size_t)b * 3 * N + n;
                p0 = __ldg(pp); p1 = __ldg(pp + N); p2 = __ldg(pp + 2 * (size_t)N);
                D0 = __ldg(prm.D + (size_t)b * N + n);
            }
            mbar_wait_parked(&bar.recfree[sr], ((j / NREC) & 1) ^ 1);
            mbar_wait_parked(&bar.fullB[s], (j / NST) & 1);
            float mydot;
            {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int blk = 2 * hf + (i >> 3), c = ((i & 7) + r16) & 7;
                    if (KBLK != 4 && blk >= KBLK) continue;
                    const float4 bv = *reinterpret_cast<const float4*>(As + blk * 8192 + sw128_32b_off(nlr, c));
                    const float4 w4 = *reinterpret_cast<const float4*>(myW + blk * 32 + c * 4);
                    acc.x = fmaf(bv.x, w4.x, acc.x); acc.y = fmaf(bv.y, w4.y, acc.y); acc.z = fmaf(bv.z, w4.z, acc.z); acc.w = fmaf(bv.w, w4.w, acc.w);
                    if constexpr (MODE == 1)     // single-pass mode: round the basis tile to tf32 IN PLACE (the tensor core would truncate it)
                        *reinterpret_cast<float4*>(const_cast<unsigned char*>(As) + blk * 8192 + sw128_32b_off(nlr, c)) =
                            tf32_stochastic4(bv, dseed ^ ((uint32_t)n * 0x9E3779B1u) ^ ((uint32_t)(blk * 8 + c) * 0x85EBCA77u));
                }
                if constexpr (MODE == 1) fence_proxy_async_smem();      // the MMA reads this stage through the async proxy
                mydot = (acc.x + acc.y) + (acc.z + acc.w);
                mydot += __shfl_xor_sync(0xffffffffu, mydot, 16);
            }
            if (lane < 16) {                                 // thread per pixel
                const auto [mask, x, y, iZ, rx, ry, rz, dx, dy, x0, y0] = project_pixel(myPose, p0, p1, p2, D0, mydot, valid, w, h);
                uint32_t o[4], cx[2] = {0u, 0u};
                if constexpr (FLY) {                             // rows y0-1 .. y0+2 as float offsets, columns x0-1 .. x0+2 as packed pixel indices
                    o[0] = (uint32_t)(reflect_i(y0 - 1, h) * w * c2); o[1] = (uint32_t)(y0 * w * c2);
                    o[2] = (uint32_t)(reflect_i(y0 + 1, h) * w * c2); o[3] = (uint32_t)(reflect_i(y0 + 2, h) * w * c2);
                    cx[0] = (uint32_t)reflect_i(x0 - 1, w) | ((uint32_t)x0 << 16);
                    cx[1] = (uint32_t)reflect_i(x0 + 1, w) | ((uint32_t)reflect_i(x0 + 2, w) << 16);
                }
                if constexpr (!FLY) {
                    const int x1 = min(x0 + 1, w - 1), y1 = min(y0 + 1, h - 1);
                    o[0] = (uint32_t)((y0 * w + x0) * c2); o[1] = (uint32_t)((y0 * w + x1) * c2);
                    o[2] = (uint32_t)((y1 * w + x0) * c2); o[3] = (uint32_t)((y1 * w + x1) * c2);
                }
                if (prm.tap_prefetch && mask != 0.f) {
                    // pull this pixel's share of the tile's tap footprint into L2 one to two tiles before the gather warps load it: the gather is
                    // bound by the latency of its 13 dependent-free loads, not by their count.  Interior pixels fetch their (x0, y0) texel only;
                    // the tile's border pixels add the halo, so that under a near-unit warp every texel is requested about once.
                    const float* imgp = prm.conv2 + (size_t)b * h * w * c2;
                    const int px = nlr & 7, py = nlr >> 3;
                    const bool edge_x = !grid2d || px == 7, edge_y = !grid2d || py == 7 || prm.tap_prefetch == 2;
                    if constexpr (!FLY) {
                        const uint32_t by = (uint32_t)c2 * 4u;
                        prefetch_l2_bulk(imgp + o[0], by);
                        if (edge_x && o[1] != o[0]) prefetch_l2_bulk(imgp + o[1], by);
                        if (edge_y && o[2] != o[0]) {
                            prefetch_l2_bulk(imgp + o[2], by);
                            if (edge_x && o[3] != o[2]) prefetch_l2_bulk(imgp + o[3], by);
                        }
                    } else {
                        const bool first_x = !grid2d || px == 0, first_y = !grid2d || py == 0;
                        const int xs = max(x0 - (first_x ? 1 : 0), 0), xe = min(x0 + (edge_x ? 2 : 0), w - 1);
                        const uint32_t by = (uint32_t)(xe - xs + 1) * (uint32_t)c2 * 4u;
                        prefetch_l2_bulk(imgp + ((size_t)y0 * w + xs) * c2, by);
                        if (first_y && y0 > 0) prefetch_l2_bulk(imgp + ((size_t)(y0 - 1) * w + xs) * c2, by);
                        if (edge_y) {
                            if (y0 + 1 < h) prefetch_l2_bulk(imgp + ((size_t)(y0 + 1) * w + xs) * c2, by);
                            if (y0 + 2 < h) prefetch_l2_bulk(imgp + ((size_t)(y0 + 2) * w + xs) * c2, by);
                        }
                    }
                }
                float* rec = sRec + (sr * TILE + nlr) * REC;
                *reinterpret_cast<uint4*>(rec) = make_uint4(o[0], o[1], o[2], o[3]);
                *reinterpret_cast<float4*>(rec + 4) = make_float4(mask, x, y, iZ);
                *reinterpret_cast<float4*>(rec + 8) = make_float4(rx, ry, rz, __int_as_float(valid ? n : 0));
                *reinterpret_cast<float4*>(rec + 12) = make_float4(dx, dy, __uint_as_float(cx[0]), __uint_as_float(cx[1]));
            }
            if (gwi == 0 && lane == 0) sTile[sr * 4] = b;
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar.recs[sr]);
        }
    } else if (warp < W0 + GW) {
        // ===================================================================== gather warps: records -> taps -> M, q
        setmaxnreg_inc<88>();
        const int g = warp - W0, hw = lane >> 4, hl = lane & 15;
        constexpr int PXW = TILE / GW;                       // 4 pixels per warp and tile
        constexpr int NUNIT = (PXW / 2) * NCH;
        float rb[NCH * 4];
#pragma unroll
        for (int u = 0; u < NCH * 4; ++u) rb[u] = 0.f;
        float4 tb[13];
        float m11 = 0.f, m12 = 0.f, m22 = 0.f, q1 = 0.f, q2 = 0.f;
        int cur_b = -1, ndump = 0;
        // L2 policy: conv1 is read exactly once (evict-first), the taps are what neighbouring tiles re-read
        const uint64_t pol_stream = prm.l2_hints >= 1 ? l2_policy_evict_first() : l2_policy_evict_normal();
        const uint64_t pol_tap = prm.l2_hints >= 2 ? l2_policy_evict_last() : l2_policy_evict_normal();

        auto dump_rb = [&]() {
            if (ndump > 0) mbar_wait_parked(bar.rbfree, (ndump - 1) & 1);       // the algebra warps consumed the previous hand-over
#pragma unroll
            for (int u = 0; u < NCH * 4; ++u) rb[u] += __shfl_xor_sync(0xffffffffu, rb[u], 16);
            if (hw == 0) {
#pragma unroll
                for (int j = 0; j < NCH; ++j)
                    *reinterpret_cast<float4*>(sRbs + g * 128 + 64 * j + 4 * hl) = make_float4(rb[4 * j], rb[4 * j + 1], rb[4 * j + 2], rb[4 * j + 3]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar.rbdump);
#pragma unroll
            for (int u = 0; u < NCH * 4; ++u) rb[u] = 0.f;
            ++ndump;
        };

        for (int j = 0; j < ntiles; ++j) {
            const int s = j % NREC;
            mbar_wait_parked(&bar.recs[s], (j / NREC) & 1);
            const int b = sTile[s * 4];
            if (b != cur_b) { if (cur_b >= 0) dump_rb(); cur_b = b; }
            float* rec = sRec + (s * TILE + g * PXW) * REC;
            const float* c1b = prm.conv1 + (size_t)b * N * C + 4 * hl;
            const float* imgb = prm.conv2 + (size_t)b * h * w * c2 + 4 * hl;
#pragma unroll
            for (int u = 0; u < NUNIT; ++u) {
                const int pl = 2 * (u / NCH) + hw, co = 64 * (u % NCH), jc = u % NCH;
                const float mask = rec[pl * REC + 4];
                if (mask != 0.f) {
                    const uint4 o = *reinterpret_cast<const uint4*>(rec + pl * REC);
                    const int n = __float_as_int(rec[pl * REC + 11]);
                    const float* img = imgb + co;
                    auto ldt = [&](const float* q) { return ldg4_hint(q, pol_tap); };
                    tb[0] = ld_stream_f4_hint(c1b + (size_t)n * C + co, pol_stream);
                    if constexpr (!FLY) {
                        const float* t00 = img + o.x; const float* t01 = img + o.y; const float* t10 = img + o.z; const float* t11 = img + o.w;
                        tb[1] = ldt(t00); tb[2] = ldt(t01); tb[3] = ldt(t10); tb[4] = ldt(t11);
                        tb[5] = ldt(t00 + C); tb[6] = ldt(t01 + C); tb[7] = ldt(t10 + C); tb[8] = ldt(t11 + C);
                        tb[9] = ldt(t00 + 2 * C); tb[10] = ldt(t01 + 2 * C); tb[11] = ldt(t10 + 2 * C); tb[12] = ldt(t11 + 2 * C);
                    } else {
                        const uint2 cxy = *reinterpret_cast<const uint2*>(rec + pl * REC + 14);
                        const float* rm = img + o.x; const float* r0 = img + o.y; const float* r1 = img + o.z; const float* rp = img + o.w;
                        const uint32_t oM = (cxy.x & 0xffffu) * c2, o0 = (cxy.x >> 16) * c2, o1 = (cxy.y & 0xffffu) * c2, oP = (cxy.y >> 16) * c2;
                        tb[1] = ldt(r0 + oM); tb[2] = ldt(r0 + o0); tb[3] = ldt(r0 + o1); tb[4] = ldt(r0 + oP);      // aM0 a00 a10 aP0
                        tb[5] = ldt(r1 + oM); tb[6] = ldt(r1 + o0); tb[7] = ldt(r1 + o1); tb[8] = ldt(r1 + oP);      // aM1 a01 a11 aP1
                        tb[9] = ldt(rm + o0); tb[10] = ldt(rm + o1); tb[11] = ldt(rp + o0); tb[12] = ldt(rp + o1);   // a0m a1m a0p a1p
                    }
                }
                if (jc == 0) { m11 = m12 = m22 = q1 = q2 = 0.f; }
                if (mask != 0.f) {
                    const float2 dxy = *reinterpret_cast<const float2*>(rec + pl * REC + 12);
                    const float dx = dxy.x, dy = dxy.y;
                    const float w00 = (1.f - dx) * (1.f - dy), w01 = dx * (1.f - dy), w10 = (1.f - dx) * dy, w11 = dx * dy;
                    const float4* t = tb;
                    if constexpr (!FLY) {
#define BANET_CH(F, CI)                                                                                              \
                        {                                                                                            \
                            const float f2 = w00 * t[1].F + w01 * t[2].F + w10 * t[3].F + w11 * t[4].F;              \
                            const float gx = w00 * t[5].F + w01 * t[6].F + w10 * t[7].F + w11 * t[8].F;              \
                            const float gy = w00 * t[9].F + w01 * t[10].F + w10 * t[11].F + w11 * t[12].F;           \
                            const float d = t[0].F - f2;                                                             \
                            m11 = fmaf(gx, gx, m11); m12 = fmaf(gx, gy, m12); m22 = fmaf(gy, gy, m22);               \
                            q1 = fmaf(gx, d, q1); q2 = fmaf(gy, d, q2);                                              \
                            rb[4 * jc + CI] += fabsf(d);                                                             \
                        }
                        BANET_CH(x, 0) BANET_CH(y, 1) BANET_CH(z, 2) BANET_CH(w, 3)
#undef BANET_CH
                    } else {
                        const float h00 = 0.5f * w00, h01 = 0.5f * w01, h10 = 0.5f * w10, h11 = 0.5f * w11;
#define BANET_CH(F, CI)                                                                                              \
                        {                                                                                            \
                            const float f2 = w00 * t[2].F + w01 * t[3].F + w10 * t[6].F + w11 * t[7].F;              \
                            const float gx = h00 * (t[3].F - t[1].F) + h01 * (t[4].F - t[2].F)                       \
                                           + h10 * (t[7].F - t[5].F) + h11 * (t[8].F - t[6].F);                      \
                            const float gy = h00 * (t[6].F - t[9].F) + h10 * (t[11].F - t[2].F)                      \
                                           + h01 * (t[7].F - t[10].F) + h11 * (t[12].F - t[3].F);                    \
                            const float d = t[0].F - f2;                                                             \
                            m11 = fmaf(gx, gx, m11); m12 = fmaf(gx, gy, m12); m22 = fmaf(gy, gy, m22);               \
                            q1 = fmaf(gx, d, q1); q2 = fmaf(gy, d, q2);                                              \
                            rb[4 * jc + CI] += fabsf(d);                                                             \
                        }
                        BANET_CH(x, 0) BANET_CH(y, 1) BANET_CH(z, 2) BANET_CH(w, 3)
#undef BANET_CH
                    }
                }
                if (jc == NCH - 1) {
                    m11 = hsum16(m11); m12 = hsum16(m12); m22 = hsum16(m22); q1 = hsum16(q1); q2 = hsum16(q2);
                    if (hl == 0) {           // totals overwrite dx,dy / n of this pixel's record (no longer needed; the tap offsets stay for the prefetcher)
                        *reinterpret_cast<float4*>(rec + pl * REC + 12) = make_float4(m11, m12, m22, q1);
                        rec[pl * REC + 11] = q2;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar.gath[s]);
        }
        if (cur_b >= 0) dump_rb();
    } else if (warp < W0 + GW + AW) {
        // ===================================================================== algebra warps: 2x7 algebra, R rows, MMA + TMA issue
        setmaxnreg_dec<72>();
        const int awi = warp - (W0 + GW);                    // 0..3: pixels / rows 16*awi .. 16*awi+15
        const int atid = tid - (W0 + GW) * 32;
        const int nlr = awi * 16 + r16;
        unsigned char* Rs = base + SM::off_R;
        float cc[28];
#pragma unroll
        for (int q = 0; q < 28; ++q) cc[q] = 0.f;
        int scale_b = -1, sspan = -1;
        float fx = 0.f, fy = 0.f;
        int rr = (ntiles > 0) ? (int)((unsigned)t_begin % (unsigned)prm.tiles_per_pair) : 0;
        // issuer state (kept by every lane of warp 0, used by its lane 0)
        constexpr uint32_t idesc = make_idesc_tf32_mn_mn(128, NMMA);
        int chain = -1, tic = 0, set = 0, mspan = 0;
        bool new_span = true;
        uint32_t accH = 0, accL = 0;

        const uint64_t pol_basis = prm.l2_hints >= 1 ? l2_policy_evict_first() : l2_policy_evict_normal();     // the basis is read exactly once
        auto issue_tma = [&](int t) {                        // basis tile t -> stage t % NST (elected thread)
            const int st = t % NST;
            const TileCoord tc = tile_coord(prm, t_begin + t);
            mbar_arrive_expect_tx(&bar.fullB[st], KBLK * 8192);
            unsigned char* dst = base + SM::off_A + st * STAGE_A;
            if (grid2d) {
#pragma unroll
                for (int blk = 0; blk < KBLK; ++blk) tma_load_3d_hint(dst + blk * 8192, &tmapB, blk * 32, tc.tx0, tc.b * prm.grid_h + tc.ty0, &bar.fullB[st], pol_basis);
            } else {
                const int row = tc.b * N + tc.n0;
#pragma unroll
                for (int blk = 0; blk < KBLK; ++blk) tma_load_2d_hint(dst + blk * 8192, &tmapB, blk * 32, row, &bar.fullB[st], pol_basis);
            }
        };
        if (awi == 0 && lane == 0)
            for (int t = 0; t < NST && t < ntiles; ++t) issue_tma(t);      // every stage starts free

        for (int j = 0; j < ntiles; ++j) {
            const int s = j % NST, sr = j % NREC;
            const bool last_of_pair = (++rr == prm.tiles_per_pair) || (j == ntiles - 1);
            if (rr == prm.tiles_per_pair) rr = 0;
            const unsigned char* As = base + SM::off_A + s * STAGE_A;
            mbar_wait_parked(&bar.gath[sr], (j / NREC) & 1);
            const int b = sTile[sr * 4];
            if (b != scale_b) { scale_b = b; ++sspan; fx = __ldg(prm.intr + b * 4); fy = __ldg(prm.intr + b * 4 + 1); }
            float ext[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (lane < 16) pixel_algebra(sRec + (sr * TILE + nlr) * REC, fx, fy, cc, ext);
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar.recfree[sr]);        // the record buffer may be refilled (everything needed is in registers)
            const float sn = __shfl_sync(0xffffffffu, ext[7], r16);   // s_n of this lane's row
            mbar_wait_parked(&bar.fullB[s], (j / NST) & 1);  // long complete; orders the TMA writes before the reads below
            if (j > 0) {
                mbar_wait_parked(bar.rfree, (j - 1) & 1);    // MMAs of tile j-1 done: R / A_lo / R_lo and stage (j-1) % NST are free
                if (awi == 0 && lane == 0 && j - 1 + NST < ntiles) issue_tma(j - 1 + NST);
            }
            if (lane < 16) write_vt<MODE, KBLK>(Rs, base + SM::off_Rlo, nlr, ext);
            // R rows (and the split parts): elementwise on the lane's half row, so walk the PHYSICAL 16-B slots (rotated by the row: every
            // quarter-warp touches 8 distinct bank groups) and skip the swizzle arithmetic
            const uint32_t rowoff = hf * 16384 + nlr * 128;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                if (KBLK != 4 && 2 * hf + (i >> 3) >= KBLK) continue;
                const uint32_t off = rowoff + (i >> 3) * 8192 + (((i & 7) + r16) & 7) * 16;
                const float4 bv = *reinterpret_cast<const float4*>(As + off);
                const float4 pv = make_float4(sn * bv.x, sn * bv.y, sn * bv.z, sn * bv.w);
                float4 hv;
                if constexpr (MODE == 3) hv = make_float4(tf32_rna(pv.x), tf32_rna(pv.y), tf32_rna(pv.z), tf32_rna(pv.w));
                else hv = make_float4(tf32_rna_bits(pv.x), tf32_rna_bits(pv.y), tf32_rna_bits(pv.z), tf32_rna_bits(pv.w));   // MMA drops the low 13 bits
                *reinterpret_cast<float4*>(Rs + off) = hv;
                if constexpr (MODE >= 2)
                    *reinterpret_cast<float4*>(base + SM::off_Alo + off) = make_float4(bv.x - tf32_trunc(bv.x), bv.y - tf32_trunc(bv.y), bv.z - tf32_trunc(bv.z), bv.w - tf32_trunc(bv.w));
                if constexpr (MODE == 3)
                    *reinterpret_cast<float4*>(base + SM::off_Rlo + off) = make_float4(pv.x - hv.x, pv.y - hv.y, pv.z - hv.z, pv.w - hv.w);
            }
            fence_proxy_async_smem();
            team_bar<AW * 32>();                           // all 64 rows written
            if (awi == 0) {
                if (lane == 0) {                             // ---- tcgen05.mma issue for this tile
                    if (new_span) { mbar_wait_parked(bar.tmemfree, (mspan & 1) ^ 1); accL = 0; new_span = false; }
                    if (tic == 0) { ++chain; set = chain & 1; mbar_wait_parked(&bar.drained[set], ((chain >> 1) & 1) ^ 1); accH = 0; }
                    tc_fence_after_sync();
                    const uint32_t ahi = smem_u32(base + SM::off_A + s * STAGE_A);
                    const uint32_t rhi = smem_u32(base + SM::off_R), rlo = smem_u32(base + SM::off_Rlo), alo = smem_u32(base + SM::off_Alo);
#pragma unroll
                    for (int pass = 0; pass < MODE; ++pass) {
                        const uint32_t a0 = (pass == 1) ? alo : ahi;
                        const uint32_t r0 = (pass == 2) ? rlo : rhi;
                        const uint32_t dcol = tmem + (pass == 0 ? set * NN : ACCL);
#pragma unroll
                        for (int kk = 0; kk < TILE / 8; ++kk) {
                            mma_tf32_ss(dcol, make_desc_mn_sw128_32b(a0 + kk * 1024, 8192, 512),
                                        make_desc_mn_sw128_32b(r0 + kk * 1024, 8192, 512), idesc, pass == 0 ? accH : accL);
                            if (pass == 0) accH = 1; else accL = 1;
                        }
                    }
                    mma_commit(bar.rfree);
                    if (++tic == CHAIN) { mma_commit(&bar.chain_done[set]); tic = 0; }
                    if (last_of_pair) { if (tic > 0) mma_commit(&bar.chain_done[set]); mma_commit(bar.flushb); ++mspan; tic = 0; new_span = true; }
                }
                __syncwarp();
            }
            if (last_of_pair) flush<KBLK, C>(prm, bar, cc, sspan, sCcs, sRbs, awi, atid, lane);
        }
    } else {
        drainer_role<32, MODE, KBLK, C>(prm, bar, tmem, t_begin, ntiles, warp - (W0 + GW + AW), lane);
    }
    release_tmem(tmem, warp);
}

template <int NCH, bool FLY, int MODE, int KBLK = 4>
static int launch6(const CUtensorMap& tm, const BuildParams& prm, int grid, cudaStream_t st)
{
    auto kern = lm_build_tc6_kernel<NCH, FLY, MODE, KBLK>;
    const int smem = Smem<MODE, FLY>::bytes;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) { set_error("lm_build_tc6: smem attr (%d B): %s", smem, cudaGetErrorString(e)); return BANET_ERR_CUDA; }
    kern<<<grid, THREADS, smem, st>>>(tm, prm);
    BANET_CUDA_LAUNCH_CHECK("lm_build_tc6_kernel launch");
    return BANET_OK;
}
template <int NCH, bool FLY>
static int launch6_mode(int mode, int kblk, const CUtensorMap& tm, const BuildParams& prm, int grid, cudaStream_t st)
{
    if (kblk != 4) {             // K = 64 / 32 (opt-in, BANET_TC_SMALLK=1): instantiated for the two-pass and the fp32-grade mode only
        if (kblk == 2) return mode == 3 ? launch6<NCH, FLY, 3, 2>(tm, prm, grid, st) : launch6<NCH, FLY, 2, 2>(tm, prm, grid, st);
        return mode == 3 ? launch6<NCH, FLY, 3, 1>(tm, prm, grid, st) : launch6<NCH, FLY, 2, 1>(tm, prm, grid, st);
    }
    if (mode == 1) return launch6<NCH, FLY, 1>(tm, prm, grid, st);
    if (mode == 2) return launch6<NCH, FLY, 2>(tm, prm, grid, st);
    return launch6<NCH, FLY, 3>(tm, prm, grid, st);
}

}  // namespace v6

int lm_build_tc6_launch(int mode, bool fly, int nch, int kblk, const CUtensorMap& tm, const BuildParams& prm, int grid, cudaStream_t st)
{
    if (nch == 2) return fly ? v6::launch6_mode<2, true>(mode, kblk, tm, prm, grid, st) : v6::launch6_mode<2, false>(mode, kblk, tm, prm, grid, st);
    return fly ? v6::launch6_mode<1, true>(mode, kblk, tm, prm, grid, st) : v6::launch6_mode<1, false>(mode, kblk, tm, prm, grid, st);
}

}  // namespace banet
