// lm_build_tc_roles.cuh — the warp-specialised pipeline that both tensor-core build kernels share (lm_build_tc6.cu, lm_build_tc7.cu).
//
// Contract, slot layout and precision modes: see lm_build_tc_host.cu.  Roles (896 threads, 1 CTA / SM; each kernel sets its own register
// budgets by setmaxnreg):
//
//   warpgroup 0    4 geometry warps, 16 pixels each per tile, run ahead of everybody:
//                    b.W from the TMA-staged basis tile, warp / mask / tap coordinates -> pixel records (ring of NREC)
//   warpgroups 1-4 16 gather warps, 4 pixels each per tile: records -> taps -> blend / accumulate -> M, q
//   warpgroup 5    4 algebra warps, 16 pixels each per tile:
//                    2x7 per-pixel algebra (H_cc / g_c partials in registers), the [v | t] block of R into smem,
//                    then ONE elected thread issues the tile's tcgen05.mma and refills the freed basis stage by TMA
//   warpgroup 6    4 drainer warps (one TMEM lane quadrant each): TMEM chains -> partial slots (L2 evict-last), asynchronous
//   mbarriers (Barriers): fullB[NST] TMA landed | recs[NREC] geometry->gather | gath[NREC] gather->algebra | recfree[NREC] algebra->geometry |
//              rfree MMAs of the tile done (R, A_lo and the A stage reusable) | chain_done/drained[2], flushb, tmemfree issuer<->drainers |
//              rbdump/rbfree gather<->algebra hand-over of the |diff| sums at a pair change.
//
// What differs between the kernels stays in their files: the gather, who scales the R rows s_n * b_n, the order of the waits in the
// algebra loop, the shared-memory layout and the register budgets.  The tcgen05.mma issue and the per-pair load of pose / W / dither seed
// are also written out in each kernel: as shared functions they changed ptxas' register allocation (spills in the algebra role) or the
// instruction mix of the kernels.
#pragma once
#include "common.cuh"
#include "lm_build.h"
#include "tc_utils.cuh"

namespace banet { namespace tcb {
using namespace tc;

constexpr int TILE = 64, W0 = 4, GW = 16, AW = 4, DW = 4;      // geometry | gather | algebra | drainer warps
constexpr int THREADS = (W0 + GW + AW + DW) * 32;               // 896
constexpr int NN = 160;                                         // MMA N at K = 128: 128 basis columns + [v(6) | t] + pad
constexpr int STAGE_A = 4 * TILE * 128, STAGE_R = 5 * TILE * 128;
constexpr int REC = 16;                                         // floats per pixel record
constexpr int CHAIN = 8, TMEM_COLS = 512, ACCL = 320;           // tiles per hi-accumulator chain; TMEM: hi ping-pong at 0 / NN, lo at ACCL

// the mbarriers of the pipeline (NST <= 4 basis stages, NREC <= 3 record buffers); a kernel's own barriers follow at index NBARS
constexpr int NBARS = 22;
struct Barriers {
    uint64_t* fullB;        // [NST]  TMA landed
    uint64_t* rfree;        //        MMAs of the tile completed
    uint64_t* flushb;       //        every MMA of the span completed
    uint64_t* tmemfree;     //        lo accumulator drained
    uint64_t* chain_done;   // [2]
    uint64_t* drained;      // [2]
    uint64_t* recs;         // [NREC] records of the tile in buffer s written (count W0)
    uint64_t* gath;         // [NREC] M,q of the tile in buffer s written (count GW)
    uint64_t* recfree;      // [NREC] records of the tile in buffer s consumed by the algebra warps (count AW)
    uint64_t* rbdump;       //        gather warps parked their rbar partials (count GW)
    uint64_t* rbfree;       //        algebra warps consumed them (count AW)
    __device__ __forceinline__ explicit Barriers(uint64_t* b)
        : fullB(b), rfree(b + 4), flushb(b + 5), tmemfree(b + 6), chain_done(b + 7), drained(b + 9),
          recs(b + 11), gath(b + 14), recfree(b + 17), rbdump(b + 20), rbfree(b + 21) {}
};

template <int NT> __device__ __forceinline__ void team_bar() { asm volatile("bar.sync 2, %0;" :: "n"(NT) : "memory"); }
__device__ __forceinline__ int reflect_i(int i, int n) { i = i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); return i < 0 ? 0 : i; }

struct TileCoord { int b, n0, cnt, tx0, ty0; };
__device__ __forceinline__ TileCoord tile_coord(const BuildParams& prm, long long tl) {
    TileCoord tc;
    const unsigned t = (unsigned)tl, tpp = (unsigned)prm.tiles_per_pair;
    tc.b = (int)(t / tpp);
    const int r = (int)(t - (unsigned)tc.b * tpp);
    if (prm.grid_w > 0) {
        int tyi, txi;
        if (prm.band_rows > 1) {        // bands of band_rows tile rows, column by column inside a band: vertically adjacent tiles follow each other
            const int bsz = prm.tiles_x * prm.band_rows, band = r / bsz, rem = r - band * bsz;
            const int rows = min(prm.band_rows, prm.tiles_y - band * prm.band_rows);
            txi = rem / rows; tyi = band * prm.band_rows + (rem - txi * rows);
        } else { tyi = r / prm.tiles_x; txi = r - tyi * prm.tiles_x; }
        tc.ty0 = tyi * 8; tc.tx0 = txi * 8; tc.n0 = 0; tc.cnt = TILE;
    }
    else { tc.n0 = r * TILE; tc.cnt = min(TILE, prm.N - tc.n0); tc.tx0 = tc.ty0 = 0; }
    return tc;
}

// ===================================================================== prologue / epilogue
// thread 0: every barrier of the map, then the init fence (a kernel initialises its own barriers before calling this)
template <int NST, int NREC>
__device__ __forceinline__ void init_barriers(const Barriers& bar) {
    for (int i = 0; i < NST; ++i) mbar_init(&bar.fullB[i], 1);
    for (int i = 0; i < NREC; ++i) { mbar_init(&bar.recs[i], W0); mbar_init(&bar.gath[i], GW); mbar_init(&bar.recfree[i], AW); }
    mbar_init(bar.rfree, 1); mbar_init(bar.flushb, 1); mbar_init(bar.tmemfree, DW);
    mbar_init(&bar.chain_done[0], 1); mbar_init(&bar.chain_done[1], 1); mbar_init(&bar.drained[0], DW); mbar_init(&bar.drained[1], DW);
    mbar_init(bar.rbdump, GW); mbar_init(bar.rbfree, AW);
    fence_barrier_init();
}

// whole CTA: TMEM allocation (warp 0), the pad chunks of the [v | t] block of R (and of R_lo in MODE 3) zeroed once -- they stay zero --,
// fences so that the tensor core sees both; returns the TMEM base address
template <int MODE, int KBLK>
__device__ __forceinline__ uint32_t setup_tmem(unsigned char* Rs, unsigned char* Rlo, uint32_t* s_tmem, int tid, int warp) {
    if (warp == 0) tmem_alloc<TMEM_COLS>(s_tmem);
    for (int i = tid; i < TILE * 8; i += THREADS) {
        const int r = i >> 3, c = i & 7;
        *reinterpret_cast<float4*>(Rs + KBLK * 8192 + sw128_32b_off(r, c)) = make_float4(0.f, 0.f, 0.f, 0.f);
        if (MODE == 3) *reinterpret_cast<float4*>(Rlo + KBLK * 8192 + sw128_32b_off(r, c)) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    return *s_tmem;
}

__device__ __forceinline__ void release_tmem(uint32_t tmem, int warp) {
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc<TMEM_COLS>(tmem);
}

// ===================================================================== geometry warps
// L2 prefetch of the streaming inputs (conv1, p, D) of tile tn; one geometry warp runs it two tiles ahead
template <int C>
__device__ __forceinline__ void prefetch_inputs(const BuildParams& prm, const TileCoord& tn, bool grid2d, int N, int lane) {
    if (grid2d) {
        if (lane < 8) {
            const int gy = tn.ty0 + lane;
            if (gy < prm.grid_h && tn.tx0 < prm.grid_w) {
                const size_t n = (size_t)gy * prm.grid_w + tn.tx0;
                const int wpx = min(8, prm.grid_w - tn.tx0);
                prefetch_l2_bulk(prm.conv1 + ((size_t)tn.b * N + n) * C, (uint32_t)(wpx * C * 4));
                if ((n & 3) == 0 && (N & 3) == 0) {
                    const uint32_t by = (uint32_t)(((wpx * 4) + 15) & ~15);
                    prefetch_l2_bulk(prm.D + (size_t)tn.b * N + n, by);
#pragma unroll
                    for (int k = 0; k < 3; ++k) prefetch_l2_bulk(prm.p + ((size_t)tn.b * 3 + k) * N + n, by);
                }
            }
        }
    } else if (lane == 0) {
        prefetch_l2_bulk(prm.conv1 + ((size_t)tn.b * N + tn.n0) * C, (uint32_t)(tn.cnt * C * 4));
        if ((N & 3) == 0) {
            const uint32_t by = (uint32_t)(((tn.cnt * 4) + 15) & ~15);
            prefetch_l2_bulk(prm.D + (size_t)tn.b * N + tn.n0, by);
#pragma unroll
            for (int k = 0; k < 3; ++k) prefetch_l2_bulk(prm.p + ((size_t)tn.b * 3 + k) * N + tn.n0, by);
        }
    }
}

// one pixel warped by the pair's pose at depth D0 + b.W (bundlenet.py:208-224) and its mask (:231): camera ray r, projection (x, y),
// 1/Z, bilinear base texel (x0, y0) and weights (dx, dy); all zero outside the mask
struct Projection { float mask, x, y, iZ, rx, ry, rz, dx, dy; int x0, y0; };
__device__ __forceinline__ Projection project_pixel(const float* pose, float p0, float p1, float p2, float D0, float dot, bool valid, int w, int h) {
    Projection pj = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0, 0};
    if (valid) {
        const float Dt = D0 + dot;
        pj.rx = pose[0] * p0 + pose[1] * p1 + pose[2] * p2;
        pj.ry = pose[3] * p0 + pose[4] * p1 + pose[5] * p2;
        pj.rz = pose[6] * p0 + pose[7] * p1 + pose[8] * p2;
        const float X = pj.rx * Dt + pose[9], Y = pj.ry * Dt + pose[10], Z = pj.rz * Dt + pose[11];
        pj.x = X / Z; pj.y = Y / Z; pj.iZ = 1.0f / Z;
        const float u = pose[12] * pj.x + pose[14], v = pose[13] * pj.y + pose[15];
        if ((u >= 0.f) && (u <= (float)(w - 1)) && (v >= 0.f) && (v <= (float)(h - 1)) && isfinite(pj.iZ)) {
            pj.mask = 1.f;
            const float fu = floorf(u), fv = floorf(v);
            pj.x0 = (int)fu; pj.y0 = (int)fv; pj.dx = u - fu; pj.dy = v - fv;
        }
    }
    return pj;
}

// ===================================================================== algebra warps
// thread per pixel (bundlenet.py:49-74): adds the pixel's 2x7 algebra to the H_cc / g_c / nvalid partials cc and returns its row of the
// [v | t] block and s_n = jd^T M jd in ext[0..7]; rec is the pixel's record after the gather (M, q in place of dx, dy / n)
__device__ __forceinline__ void pixel_algebra(const float* rec, float fx, float fy, float (&cc)[28], float (&ext)[8]) {
    const float4 ra = *reinterpret_cast<const float4*>(rec + 12), rbq = *reinterpret_cast<const float4*>(rec + 4),
                 rc = *reinterpret_cast<const float4*>(rec + 8);
    if (rbq.x != 0.f) {
        const float m11 = ra.x, m12 = ra.y, m22 = ra.z, q1 = ra.w, q2 = rc.w, x = rbq.y, y = rbq.z, iZ = rbq.w;
        const float rx = rc.x, ry = rc.y, rz = rc.z;
        const float a0[6] = {-fx * (x * y), -fx * (-1.f - x * x), -fx * y, -fx * (-iZ), 0.f, -fx * (x * iZ)};
        const float a1[6] = {-fy * (1.f + y * y), -fy * (-(x * y)), -fy * (-x), 0.f, -fy * (-iZ), -fy * (y * iZ)};
        float ux[6], uy[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) { ux[i] = m11 * a0[i] + m12 * a1[i]; uy[i] = m12 * a0[i] + m22 * a1[i]; }
        int q = 0;
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int jj = i; jj < 6; ++jj) { cc[q] += a0[i] * ux[jj] + a1[i] * uy[jj]; ++q; }
#pragma unroll
        for (int i = 0; i < 6; ++i) cc[21 + i] += a0[i] * q1 + a1[i] * q2;
        cc[27] += 1.f;
        const float jd0 = fx * ((rx - rz * x) * iZ), jd1 = fy * ((ry - rz * y) * iZ);
        const float u0 = m11 * jd0 + m12 * jd1, u1 = m12 * jd0 + m22 * jd1;
#pragma unroll
        for (int i = 0; i < 6; ++i) ext[i] = a0[i] * u0 + a1[i] * u1;
        ext[6] = jd0 * q1 + jd1 * q2;
        ext[7] = jd0 * u0 + jd1 * u1;
    }
}

// R columns 128..134 of row nlr = [v(6) | t], column 135 stays zero; in MODE 3 their rounding remainders go to R_lo
template <int MODE, int KBLK>
__device__ __forceinline__ void write_vt(unsigned char* Rs, unsigned char* Rlo, int nlr, const float (&ext)[8]) {
    const float4 e0 = make_float4(tf32_rna(ext[0]), tf32_rna(ext[1]), tf32_rna(ext[2]), tf32_rna(ext[3]));
    const float4 e1 = make_float4(tf32_rna(ext[4]), tf32_rna(ext[5]), tf32_rna(ext[6]), 0.f);
    *reinterpret_cast<float4*>(Rs + KBLK * 8192 + sw128_32b_off(nlr, 0)) = e0;
    *reinterpret_cast<float4*>(Rs + KBLK * 8192 + sw128_32b_off(nlr, 1)) = e1;
    if constexpr (MODE == 3) {
        *reinterpret_cast<float4*>(Rlo + KBLK * 8192 + sw128_32b_off(nlr, 0)) = make_float4(ext[0] - e0.x, ext[1] - e0.y, ext[2] - e0.z, ext[3] - e0.w);
        *reinterpret_cast<float4*>(Rlo + KBLK * 8192 + sw128_32b_off(nlr, 1)) = make_float4(ext[4] - e1.x, ext[5] - e1.y, ext[6] - e1.z, 0.f);
    }
}

// last tile of a pair's span sp (all 4 algebra warps; atid = thread index inside the team): H_cc / g_c / nvalid and the |diff| sums that the
// gather warps parked in sRbs into the CTA's partial slot, in a fixed summation order
template <int KBLK, int C>
__device__ __forceinline__ void flush(const BuildParams& prm, const Barriers& bar, float (&cc)[28], int sp, float* sCcs, const float* sRbs,
                                      int awi, int atid, int lane) {
    const SlotLayout L{32 * KBLK, C};
    float* slot = prm.partials + ((size_t)blockIdx.x * prm.max_span + sp) * prm.slot_floats;
    // H_cc / g_c / nvalid: 16 pixel-lanes -> warp total (fixed shuffle tree) -> 4 warp partials summed in fixed order
#pragma unroll
    for (int q = 0; q < 28; ++q) {
        float v = cc[q];
        v += __shfl_xor_sync(0xffffffffu, v, 8); v += __shfl_xor_sync(0xffffffffu, v, 4);
        v += __shfl_xor_sync(0xffffffffu, v, 2); v += __shfl_xor_sync(0xffffffffu, v, 1);
        if (lane == 0) sCcs[awi * 28 + q] = v;
        cc[q] = 0.f;
    }
    mbar_wait_parked(bar.rbdump, sp & 1);                // the gather warps parked their |diff| sums for this pair
    team_bar<AW * 32>();
    if (atid < C) {
        float sum = 0.f;
#pragma unroll
        for (int wq = 0; wq < GW; ++wq) sum += sRbs[wq * 128 + atid];
        slot[L.off_rbar() + atid] = sum;
    }
    if (atid < 28) slot[L.off_cc() + atid] = (sCcs[atid] + sCcs[28 + atid]) + (sCcs[56 + atid] + sCcs[84 + atid]);
    team_bar<AW * 32>();
    if (lane == 0) mbar_arrive(bar.rbfree);
}

// ===================================================================== drainer warps: TMEM -> partial slots, fully asynchronous
// NREG: the role's register budget (setmaxnreg); dq: the warp's TMEM lane quadrant (= warp % 4)
template <int NREG, int MODE, int KBLK, int C>
__device__ __forceinline__ void drainer_role(const BuildParams& prm, const Barriers& bar, uint32_t tmem, long long t_begin, int ntiles, int dq, int lane) {
    setmaxnreg_dec<NREG>();
    constexpr int KR = 32 * KBLK;
    const SlotLayout L{KR, C};
    // The CTA's partial slot (<= 2 x 68 KB) is read-modify-written once per chain of CHAIN tiles.  Left to the default policy the streaming
    // inputs push it out of L2 between two chains: ncu showed 1.3 GB of DRAM writes per launch (and as many reads) for a kernel that writes
    // 20 MB of results.  evict-last keeps the 20 MB of slots of all CTAs resident.
    const uint64_t pol_slot = l2_policy_evict_last();
    auto drain_region = [&](float* slot, uint32_t col0, bool overwrite) {
        const int row = dq * 32 + lane;
        if (KBLK != 4 && dq * 32 >= KR) return;          // this lane quadrant holds no basis row (warp-uniform)
        const uint32_t tq = tmem + ((uint32_t)(dq * 32) << 16) + col0;
        float v[16];
#pragma unroll 1
        for (int cb = 0; cb < KR / 16; ++cb) {
            tmem_ld_32x16(tq + cb * 16, v);
            float* dst = slot + (size_t)(cb * 16) * KR + row;
            if (overwrite) {
#pragma unroll
                for (int j = 0; j < 16; ++j) st_f32_hint(dst + (size_t)j * KR, v[j], pol_slot);
            } else {
#pragma unroll
                for (int hb = 0; hb < 16; hb += 8) {     // 8 columns at a time: the drainers run on the smallest register budget
                    float o[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = ld_f32_hint(dst + (size_t)(hb + j) * KR, pol_slot);
#pragma unroll
                    for (int j = 0; j < 8; ++j) st_f32_hint(dst + (size_t)(hb + j) * KR, o[j] + v[hb + j], pol_slot);
                }
            }
        }
        tmem_ld_32x16(tq + KR, v);
        float* dst = slot + L.off_ext() + row;
#pragma unroll
        for (int r = 0; r < 7; ++r) {
            if (overwrite) st_f32_hint(dst + r * KR, v[r], pol_slot);
            else st_f32_hint(dst + r * KR, ld_f32_hint(dst + r * KR, pol_slot) + v[r], pol_slot);
        }
    };
    int chain = -1, tic = 0, span = 0, cur_b = -1;
    bool first = true;
    int b = (ntiles > 0) ? (int)((unsigned)t_begin / (unsigned)prm.tiles_per_pair) : 0;
    int rr = (ntiles > 0) ? (int)((unsigned)t_begin - (unsigned)b * (unsigned)prm.tiles_per_pair) : 0;
    auto drain_hi = [&]() {
        const int set = chain & 1;
        float* slot = prm.partials + ((size_t)blockIdx.x * prm.max_span + span) * prm.slot_floats;
        mbar_wait_parked(&bar.chain_done[set], (chain >> 1) & 1);
        tc_fence_after_sync();
        drain_region(slot, set * NN, first);
        first = false;
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar.drained[set]);
    };
    auto end_span = [&]() {
        if (tic > 0) drain_hi();
        if constexpr (MODE >= 2) {
            float* slot = prm.partials + ((size_t)blockIdx.x * prm.max_span + span) * prm.slot_floats;
            mbar_wait_parked(bar.flushb, span & 1);
            tc_fence_after_sync();
            drain_region(slot, ACCL, false);
            tc_fence_before_sync();
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar.tmemfree);
        ++span;
    };
    for (int it = 0; it < ntiles; ++it) {
        if (b != cur_b) { if (cur_b >= 0) end_span(); cur_b = b; tic = 0; first = true; }
        if (tic == 0) ++chain;
        if (++tic == CHAIN) { drain_hi(); tic = 0; }
        if (++rr == prm.tiles_per_pair) { rr = 0; ++b; }
    }
    if (cur_b >= 0) end_span();
}

}}  // namespace banet::tcb
