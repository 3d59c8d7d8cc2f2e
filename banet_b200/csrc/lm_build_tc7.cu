// lm_build_tc7.cu — tensor-core build kernel, generation 7: the F2 footprint of every 8x8 tile is staged into shared memory by TMA.
//
// Applies to the F2-only conv2 layout on a dense pixel grid (the BundleResize boundary: feature maps in, gradients derived on the fly,
// reference bundlenet.py:92-100, 385-389).  Same contract, slot layout, tensor-core contraction, precision modes and pipeline roles as generation 6
// (lm_build_tc_roles.cuh; lm_build_tc_host.cu has the overview); what changes is where the 12 taps per pixel and channel come from:
//
//   generation 6: 13 x ld.global.nc per (pixel, 4 channels), latency-bound (ncu r01b: long-scoreboard 65% of the issue interval, 0.75
//                 eligible warps per scheduler) and every texel fetched ~1.3x (L1) with 12 x the LSU traffic on the L1/L2 path;
//   generation 7: per tile the geometry warps publish the bounding box of the (reflected) tap coordinates; when it fits the staged
//                 window (WX x WY texels) gather warp 0 issues, per 32-channel chunk, ONE 4-D TMA box {32 ch, WX, WY, pair} into a ring
//                 of NWB window buffers (mbarrier complete_tx); the 16 gather warps then read their taps with LDS.128 (a quarter-warp
//                 per pixel reads one 128-B texel chunk = all 32 banks, conflict-free).  Loads in flight cost shared memory, not
//                 registers, and run NWB chunks ahead of the consumer.  conv1 (streaming, read once) stays on ld.global.nc with all
//                 C/32 chunk loads of a pixel in flight from the top of the tile.  Tiles whose footprint does not fit (strong local
//                 zoom / shear) take the generation-6 style global taps for that tile only (same arithmetic, same results).
//   tile order:   bands of `band_rows` tile rows walked column by column, so that the window halos of vertically AND horizontally
//                 adjacent tiles are re-read from L2 while they are still resident (generation 6 walks rows: vertical halo from HBM).
//
//   division of labour (measured, profiles/r02b_*: with the taps on LDS the kernel turned instruction-issue / role-latency bound, so work moved to
//                 where the warps are): the 16 gather warps also derive s_n = jd^T M jd and write the MMA operands of their pixel — the R row
//                 rna(s_n b_n) and the precision mode's side of the basis tile (stochastic tf32 rounding in place, or A_lo) — which the 4
//                 algebra warps did in generation 6; the geometry warps only form b.W and the warp; the per-channel arithmetic runs on packed
//                 fp32 pairs (FFMA2 / FMUL2 / FADD2); conv1 arrives with the window (one 4-D TMA box {32 ch, 8, 8, pair} per chunk).
//
// Register budgets 48 / 88 / 64 / 40 (geometry / gather / algebra / drainers); the window ring adds winfull[NWB] (TMA landed, count 1 + tx) /
// winfree[NWB] (count GW) to the barriers.
#include "lm_build_tc_roles.cuh"
#include "tmap.h"
#include <limits.h>

namespace banet { namespace v7 {
using namespace tcb;

constexpr int CHK = 32;                                         // channels per staged chunk: one texel chunk = 128 B = all 32 banks
constexpr int WX = 13, WY = 13;                                 // staged window (texels); an 8x8 tile needs >= 11..12 at unit zoom
constexpr int WIN_BYTES = WX * WY * CHK * 4;
constexpr int C1_BYTES = TILE * CHK * 4;                        // conv1 chunk of the tile: [8][8] pixels x 32 channels, pixel-major 128-B rows
constexpr int WBUF = WIN_BYTES + C1_BYTES;                      // one ring buffer = F2 window chunk + conv1 chunk

template <int MODE, int NCH> struct Smem {
    static_assert(MODE == 1 || MODE == 2, "generation 7 implements TF32X1 and TF32X2 (TF32X3 stays on generation 6: no room for the windows)");
    static constexpr int NST = MODE == 1 ? 3 : 2;
    static constexpr int NREC = 3;
    // window ring; never deeper than one tile's chunks (C/32 >= 2): the producer may look ahead into tile j+1 only (a wait on the records of
    // tile j+2 from inside tile j could close a cycle through the basis ring: rfree(j) <- gath[j] <- the producer itself)
    static constexpr int NWB = 2;
    static constexpr int off_A = 0;
    static constexpr int off_R = NST * STAGE_A;
    static constexpr int off_Alo = off_R + STAGE_R;
    static constexpr int off_win = off_Alo + (MODE >= 2 ? STAGE_A : 0);      // [NWB] x ([WY][WX][32] floats F2 window chunk | [64][32] floats conv1 chunk)
    static constexpr int off_misc = off_win + NWB * WBUF;
    static constexpr int off_bar = off_misc;                           // NBARS + 2*NWB mbarriers (<= 30)
    static constexpr int off_tmem = off_bar + (NBARS + 8) * 8;
    static constexpr int off_tile = off_misc + 256;                    // [NREC][8] ints: pair, tx0, ty0, fx, fy (float bits), dither seed of the tile in record buffer s
    static constexpr int off_box = off_tile + 128;                     // [NREC][W0][4] ints: tap bounding box (xmin,xmax,ymin,ymax) per geometry warp
    static constexpr int off_pose = off_box + NREC * W0 * 16;          // [W0][16] floats (private to each geometry warp)
    static constexpr int off_w = off_pose + W0 * 16 * 4;               // [W0][128] floats: W of the pair (private to each geometry warp)
    static constexpr int off_rec = off_w + W0 * 128 * 4;               // [NREC][TILE][REC] floats
    static constexpr int off_rbs = off_rec + NREC * TILE * REC * 4;    // [GW][128] floats: rbar hand-over gather -> algebra
    static constexpr int off_ccs = off_rbs + GW * 128 * 4;             // [AW][28] floats: H_cc / g_c / nvalid partials per algebra warp
    static constexpr int total = off_ccs + AW * 28 * 4;
    static constexpr int slack = 512;
    static constexpr int bytes = total + slack;
    static_assert(NWB >= 2 && NWB <= 4 && NST <= 4 && WIN_BYTES % 128 == 0, "ring sizes");
    static_assert(bytes <= 232448, "shared memory budget of one sm_100 CTA");
};

// packed fp32 pairs (sm_100: FFMA2 / FMUL2 / FADD2, one issue slot for two lanes' worth of channels; a (w, w) pair is encoded as a scalar broadcast)
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float a, float b) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float2 upk2(u64 v) { float2 r; asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v)); return r; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ ulonglong2 lds2x64(uint32_t saddr) {
    ulonglong2 r;
    asm volatile("ld.shared.v2.b64 {%0,%1}, [%2];" : "=l"(r.x), "=l"(r.y) : "r"(saddr));
    return r;
}
__device__ __forceinline__ ulonglong2 ldg2x64(const float* p) {
    ulonglong2 r;
    asm volatile("ld.global.nc.v2.b64 {%0,%1}, [%2];" : "=l"(r.x), "=l"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ float qsum8(float v) {               // sum over the 8 lanes of a quarter-warp
    v += __shfl_xor_sync(0xffffffffu, v, 4); v += __shfl_xor_sync(0xffffffffu, v, 2); v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}
// tile index -> (pair, 8x8 patch): bands of prm.band_rows tile rows, column by column inside a band (the dense-grid, banded case of tile_coord)
__device__ __forceinline__ TileCoord banded_tile_coord(const BuildParams& prm, long long tl) {
    TileCoord tc;
    const unsigned t = (unsigned)tl, tpp = (unsigned)prm.tiles_per_pair;
    tc.b = (int)(t / tpp);
    const int r = (int)(t - (unsigned)tc.b * tpp);
    const int bandsz = prm.tiles_x * prm.band_rows;
    const int band = r / bandsz, rem = r - band * bandsz;
    const int rows = min(prm.band_rows, prm.tiles_y - band * prm.band_rows);
    const int txi = rem / rows, tyi = band * prm.band_rows + (rem - txi * rows);
    tc.tx0 = txi * 8; tc.ty0 = tyi * 8; tc.n0 = 0; tc.cnt = TILE;
    return tc;
}

// incremental form of banded_tile_coord (no integer divisions per tile): walks the same band order
struct TileStepper {
    int b, r, band, txi, tyr, rows;              // pair, tile index inside the pair, band, tile column, row inside the band, rows of the band
    __device__ __forceinline__ void init(const BuildParams& prm, long long tl) {
        const unsigned t = (unsigned)tl, tpp = (unsigned)prm.tiles_per_pair;
        b = (int)(t / tpp); r = (int)(t - (unsigned)b * tpp);
        const int bandsz = prm.tiles_x * prm.band_rows;
        band = r / bandsz;
        const int rem = r - band * bandsz;
        rows = min(prm.band_rows, prm.tiles_y - band * prm.band_rows);
        txi = rem / rows; tyr = rem - txi * rows;
    }
    __device__ __forceinline__ int tx0() const { return txi * 8; }
    __device__ __forceinline__ int ty0(const BuildParams& prm) const { return (band * prm.band_rows + tyr) * 8; }
    __device__ __forceinline__ void next(const BuildParams& prm) {
        if (++r == prm.tiles_per_pair) { r = 0; ++b; band = 0; txi = 0; tyr = 0; rows = min(prm.band_rows, prm.tiles_y); return; }
        if (++tyr == rows) { tyr = 0; if (++txi == prm.tiles_x) { txi = 0; ++band; rows = min(prm.band_rows, prm.tiles_y - band * prm.band_rows); } }
    }
};

template <int NCH, int MODE, int KBLK = 4>
__global__ void __launch_bounds__(THREADS, 1)
lm_build_tc7_kernel(const __grid_constant__ CUtensorMap tmapB, const __grid_constant__ CUtensorMap tmapF, const __grid_constant__ CUtensorMap tmapC,
                    const BuildParams prm)
{
    using SM = Smem<MODE, NCH>;
    constexpr int NST = SM::NST, NREC = SM::NREC, NWB = SM::NWB;
    constexpr int KR = 32 * KBLK, NMMA = KBLK == 4 ? NN : KR + 16;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // align through the 32-bit shared address so that the compiler keeps every access in the shared state space (LDS/STS, not generic LD/ST)
    unsigned char* base = smem_raw + ((512u - (smem_u32(smem_raw) & 511u)) & 511u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(base + SM::off_bar);
    const Barriers bar(bars);
    uint64_t* winfull = bars + NBARS;        // [NWB]  window chunk landed (count 1 + tx bytes)
    uint64_t* winfree = bars + NBARS + 4;    // [NWB]  window chunk consumed by the gather warps (count GW)
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(base + SM::off_tmem);
    int* sTile = reinterpret_cast<int*>(base + SM::off_tile);
    int* sBox = reinterpret_cast<int*>(base + SM::off_box);
    float* sPose = reinterpret_cast<float*>(base + SM::off_pose);
    float* sW = reinterpret_cast<float*>(base + SM::off_w);
    float* sRec = reinterpret_cast<float*>(base + SM::off_rec);
    float* sRbs = reinterpret_cast<float*>(base + SM::off_rbs);
    float* sCcs = reinterpret_cast<float*>(base + SM::off_ccs);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int N = prm.N, h = prm.h, w = prm.w, c2 = prm.c2;
    constexpr int C = 64 * NCH;
    const long long t_begin = part_begin(prm.total_tiles, gridDim.x, blockIdx.x);
    const long long t_end   = part_begin(prm.total_tiles, gridDim.x, blockIdx.x + 1);
    const int ntiles = (int)(t_end - t_begin);

    if (tid == 0) {
        for (int i = 0; i < NWB; ++i) { mbar_init(&winfull[i], 1); mbar_init(&winfree[i], GW); }
        init_barriers<NST, NREC>(bar);
        prefetch_tmap(&tmapB); prefetch_tmap(&tmapF); prefetch_tmap(&tmapC);
    }
    const uint32_t tmem = setup_tmem<MODE, KBLK>(base + SM::off_R, nullptr, s_tmem, tid, warp);

    // lane -> (row r of the warp's 16, half hf of the 128 basis columns); 16-B chunk walk rotated by the row so that every
    // quarter-warp touches 8 distinct bank groups of the swizzled tile (used by the b.W and the R-row loops)
    const int r16 = lane & 15, hf = lane >> 4;

    if (warp < W0) {
        // ===================================================================== geometry warps: b.W, warp, mask, tap coordinates -> records
        setmaxnreg_dec<48>();
        const int gwi = warp, nlr = gwi * 16 + r16;
        float* myPose = sPose + gwi * 16;
        float* myW = sW + gwi * 128;
        int geom_b = -1;
        uint32_t dseed = 0;                                  // MODE 1: dither seed of the current pair
        TileStepper cur, ahead;
        cur.init(prm, t_begin);
        ahead.init(prm, t_begin); ahead.next(prm); ahead.next(prm);
        for (int j = 0; j < ntiles; ++j) {
            TileCoord tc; tc.b = cur.b; tc.tx0 = cur.tx0(); tc.ty0 = cur.ty0(prm); tc.n0 = 0; tc.cnt = TILE;
            cur.next(prm);
            const int b = tc.b;
            if (gwi == 1 && j + 2 < ntiles) prefetch_inputs<C>(prm, TileCoord{ahead.b, 0, TILE, ahead.tx0(), ahead.ty0(prm)}, true, N, lane);
            ahead.next(prm);
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
            const int gx = tc.tx0 + (nlr & 7), gy = tc.ty0 + (nlr >> 3);
            const bool valid = gx < prm.grid_w && gy < prm.grid_h;
            const int n = gy * prm.grid_w + gx;
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
                }
                mydot = (acc.x + acc.y) + (acc.z + acc.w);
                mydot += __shfl_xor_sync(0xffffffffu, mydot, 16);
            }
            int bxmin = INT_MAX, bxmax = INT_MIN, bymin = INT_MAX, bymax = INT_MIN;
            if (lane < 16) {                                 // thread per pixel
                const auto [mask, x, y, iZ, rx, ry, rz, dx, dy, x0, y0] = project_pixel(myPose, p0, p1, p2, D0, mydot, valid, w, h);
                // rows y0-1 .. y0+2 and columns x0-1 .. x0+2 with the REFLECT-by-one border of grad_fixed (bundlenet.py:97), 16 bits each
                const int ym = reflect_i(y0 - 1, h), y1 = reflect_i(y0 + 1, h), yp = reflect_i(y0 + 2, h);
                const int xm = reflect_i(x0 - 1, w), x1 = reflect_i(x0 + 1, w), xp = reflect_i(x0 + 2, w);
                if (mask != 0.f) {
                    bxmin = min(min(xm, x0), min(x1, xp)); bxmax = max(max(xm, x0), max(x1, xp));
                    bymin = min(min(ym, y0), min(y1, yp)); bymax = max(max(ym, y0), max(y1, yp));
                }
                float* rec = sRec + (sr * TILE + nlr) * REC;
                *reinterpret_cast<uint4*>(rec) = make_uint4((uint32_t)ym | ((uint32_t)y0 << 16), (uint32_t)y1 | ((uint32_t)yp << 16), 0u, 0u);
                *reinterpret_cast<float4*>(rec + 4) = make_float4(mask, x, y, iZ);
                *reinterpret_cast<float4*>(rec + 8) = make_float4(rx, ry, rz, __int_as_float(valid ? n : 0));
                *reinterpret_cast<float4*>(rec + 12) = make_float4(dx, dy, __uint_as_float((uint32_t)xm | ((uint32_t)x0 << 16)),
                                                                   __uint_as_float((uint32_t)x1 | ((uint32_t)xp << 16)));
            }
            bxmin = __reduce_min_sync(0xffffffffu, bxmin); bxmax = __reduce_max_sync(0xffffffffu, bxmax);
            bymin = __reduce_min_sync(0xffffffffu, bymin); bymax = __reduce_max_sync(0xffffffffu, bymax);
            if (lane == 0) {
                *reinterpret_cast<int4*>(sBox + (sr * W0 + gwi) * 4) = make_int4(bxmin, bxmax, bymin, bymax);
                if (gwi == 0) { sTile[sr * 8] = b; sTile[sr * 8 + 1] = tc.tx0; sTile[sr * 8 + 2] = tc.ty0;
                    sTile[sr * 8 + 3] = __float_as_int(myPose[12]); sTile[sr * 8 + 4] = __float_as_int(myPose[13]); sTile[sr * 8 + 5] = (int)dseed; }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar.recs[sr]);
        }
    } else if (warp < W0 + GW) {
        // ===================================================================== gather warps: records -> staged taps (LDS) -> M, q
        setmaxnreg_inc<88>();
        const int g = warp - W0, pq = lane >> 3, ql = lane & 7;          // quarter-warp pq handles pixel g*4+pq; lane ql its channels 4*ql..+3 of a chunk
        constexpr int NCHK = C / CHK;
        const int nchunks = ntiles * NCHK;
        float rb[NCHK * 4];                                                // |diff| sums of this lane's 4 channels of every chunk (its quarter's pixels)
#pragma unroll
        for (int u = 0; u < NCHK * 4; ++u) rb[u] = 0.f;
        int cur_b = -1, ndump = 0;
        const uint32_t win0 = smem_u32(base + SM::off_win);

        auto dump_rb = [&]() {
            if (ndump > 0) mbar_wait_parked(bar.rbfree, (ndump - 1) & 1);       // the algebra warps consumed the previous hand-over
#pragma unroll
            for (int u = 0; u < NCHK * 4; ++u) { rb[u] += __shfl_xor_sync(0xffffffffu, rb[u], 8); rb[u] += __shfl_xor_sync(0xffffffffu, rb[u], 16); }
            if (pq == 0) {
#pragma unroll
                for (int c = 0; c < NCHK; ++c)
                    *reinterpret_cast<float4*>(sRbs + g * 128 + CHK * c + 4 * ql) = make_float4(rb[4 * c], rb[4 * c + 1], rb[4 * c + 2], rb[4 * c + 3]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar.rbdump);
#pragma unroll
            for (int u = 0; u < NCHK * 4; ++u) rb[u] = 0.f;
            ++ndump;
        };
        // tile jt fits the staged window?  (every gather warp evaluates the same 16 ints: no hand-over needed)
        auto decide = [&](int jt, int& wx0, int& wy0) -> bool {
            const int4* bx = reinterpret_cast<const int4*>(sBox + (jt % NREC) * W0 * 4);
            const int4 b0 = bx[0], b1 = bx[1], b2 = bx[2], b3 = bx[3];
            const int xmn = min(min(b0.x, b1.x), min(b2.x, b3.x)), xmx = max(max(b0.y, b1.y), max(b2.y, b3.y));
            const int ymn = min(min(b0.z, b1.z), min(b2.z, b3.z)), ymx = max(max(b0.w, b1.w), max(b2.w, b3.w));
            wx0 = xmn; wy0 = ymn;
            return prm.force_direct == 0 && xmn <= xmx && (xmx - xmn) < WX && (ymx - ymn) < WY;
        };
        // producer duty of gather warp 0 (its lane 0): chunk q = (tile, 32-channel chunk) -> ring buffer q % NWB: the conv1 chunk of the tile
        // (always) and, when the tile's taps fit, the F2 window chunk.  Tile coordinates come from the geometry warps (sTile).
        auto issue_chunk = [&](int q) {
            const int jt = q / NCHK, c = q - jt * NCHK, buf = q % NWB;
            mbar_wait_parked(&bar.recs[jt % NREC], (jt / NREC) & 1);
            const int* ti = sTile + (jt % NREC) * 8;
            const int b = ti[0], tx0 = ti[1], ty0 = ti[2];
            int wx0, wy0;
            const bool staged = decide(jt, wx0, wy0);
            unsigned char* dst = base + SM::off_win + buf * WBUF;
            mbar_arrive_expect_tx(&winfull[buf], (staged ? WIN_BYTES : 0) + C1_BYTES);
            tma_load_4d(dst + WIN_BYTES, &tmapC, c * CHK, tx0, ty0, b, &winfull[buf]);
            if (staged) tma_load_4d(dst, &tmapF, c * CHK, wx0, wy0, b, &winfull[buf]);
        };
        if (g == 0) { if (lane == 0) { for (int q = 0; q < NWB && q < nchunks; ++q) issue_chunk(q); } __syncwarp(); }

        for (int j = 0; j < ntiles; ++j) {
            const int s = j % NREC;
            mbar_wait_parked(&bar.recs[s], (j / NREC) & 1);
            const int b = sTile[s * 8];
            if (b != cur_b) { if (cur_b >= 0) dump_rb(); cur_b = b; }
            int wx0, wy0;
            const bool staged = decide(j, wx0, wy0);
            const int pxi = g * 4 + pq;
            float* rec = sRec + (s * TILE + pxi) * REC;
            const float mask = rec[4];
            const uint2 ryp = *reinterpret_cast<const uint2*>(rec);
            const float4 r12 = *reinterpret_cast<const float4*>(rec + 12);
            const float4 rgeo = *reinterpret_cast<const float4*>(rec + 8);        // rx, ry, rz, n
            const float dx = r12.x, dy = r12.y;
            const uint32_t cxa = __float_as_uint(r12.z), cxb = __float_as_uint(r12.w);
            const int ym = ryp.x & 0xffffu, y0 = ryp.x >> 16, y1 = ryp.y & 0xffffu, yp = ryp.y >> 16;
            const int xm = cxa & 0xffffu, x0 = cxa >> 16, x1 = cxb & 0xffffu, xp = cxb >> 16;
            const float w00 = (1.f - dx) * (1.f - dy), w01 = dx * (1.f - dy), w10 = (1.f - dx) * dy, w11 = dx * dy;
            const u64 W00 = pk2(w00, w00), W01 = pk2(w01, w01), W10 = pk2(w10, w10), W11 = pk2(w11, w11);
            // tap addresses: staged = byte offsets inside a window buffer; direct = float offsets inside the pair's F2 map
            uint32_t rM, r0, r1, rP, oM, o0, o1, oP;
            if (staged) {
                rM = (uint32_t)((ym - wy0) * WX * 128); r0 = (uint32_t)((y0 - wy0) * WX * 128);
                r1 = (uint32_t)((y1 - wy0) * WX * 128); rP = (uint32_t)((yp - wy0) * WX * 128);
                oM = (uint32_t)((xm - wx0) * 128 + ql * 16); o0 = (uint32_t)((x0 - wx0) * 128 + ql * 16);
                o1 = (uint32_t)((x1 - wx0) * 128 + ql * 16); oP = (uint32_t)((xp - wx0) * 128 + ql * 16);
            } else {
                rM = (uint32_t)(ym * w * c2); r0 = (uint32_t)(y0 * w * c2); r1 = (uint32_t)(y1 * w * c2); rP = (uint32_t)(yp * w * c2);
                oM = (uint32_t)(xm * c2 + 4 * ql); o0 = (uint32_t)(x0 * c2 + 4 * ql); o1 = (uint32_t)(x1 * c2 + 4 * ql); oP = (uint32_t)(xp * c2 + 4 * ql);
            }
            const float* imgb = prm.conv2 + (size_t)b * h * w * c2;
            const uint32_t c1off = (uint32_t)(WIN_BYTES + pxi * 128 + ql * 16);
            u64 m11 = 0ull, m12 = 0ull, m22 = 0ull, q1 = 0ull, q2 = 0ull;        // packed (2 channels) sums of (2gx)^2, (2gx)(2gy), (2gy)^2, (2gx) d, (2gy) d
#pragma unroll
            for (int c = 0; c < NCHK; ++c) {
                const int q = j * NCHK + c, buf = q % NWB;
                mbar_wait_parked(&winfull[buf], (q / NWB) & 1);
                if (mask != 0.f) {
                    // grad_fixed on the fly (bundlenet.py:92-100): 2gx, 2gy = central differences at the 4 bilinear taps, as sums of positive minus sums of
                    // negative terms in packed fp32 pairs; the factors 1/2 are applied once per pixel.  Two load phases (the two middle rows, then the rows
                    // above / below) keep at most 8 of the 12 taps live; the empty asm ties phase B's address to a phase-A result so that ptxas cannot hoist it.
                    const uint32_t wb = win0 + buf * WBUF;
                    ulonglong2 aM0, a00, a10, aP0, aM1, a01, a11, aP1;
                    const float* img = imgb + c * CHK;
                    if (staged) {
                        aM0 = lds2x64(wb + r0 + oM); a00 = lds2x64(wb + r0 + o0); a10 = lds2x64(wb + r0 + o1); aP0 = lds2x64(wb + r0 + oP);
                        aM1 = lds2x64(wb + r1 + oM); a01 = lds2x64(wb + r1 + o0); a11 = lds2x64(wb + r1 + o1); aP1 = lds2x64(wb + r1 + oP);
                    } else {
                        aM0 = ldg2x64(img + r0 + oM); a00 = ldg2x64(img + r0 + o0); a10 = ldg2x64(img + r0 + o1); aP0 = ldg2x64(img + r0 + oP);
                        aM1 = ldg2x64(img + r1 + oM); a01 = ldg2x64(img + r1 + o0); a11 = ldg2x64(img + r1 + o1); aP1 = ldg2x64(img + r1 + oP);
                    }
                    const ulonglong2 f1 = lds2x64(wb + c1off);
                    u64 d[2], gx[2], gyP[2], gyN[2];
#define BANET_A(H, F)                                                                                               \
                    {                                                                                               \
                        u64 S = mul2(a00.F, W00); S = fma2(a10.F, W01, S); S = fma2(a01.F, W10, S); S = fma2(a11.F, W11, S);           \
                        d[H] = sub2(f1.F, S);                                                                       \
                        u64 P = mul2(a10.F, W00); P = fma2(aP0.F, W01, P); P = fma2(a11.F, W10, P); P = fma2(aP1.F, W11, P);           \
                        u64 Nn = mul2(aM0.F, W00); Nn = fma2(a00.F, W01, Nn); Nn = fma2(aM1.F, W10, Nn); Nn = fma2(a01.F, W11, Nn);    \
                        gx[H] = sub2(P, Nn);                                                                        \
                        gyP[H] = fma2(a11.F, W01, mul2(a01.F, W00));                                                \
                        gyN[H] = fma2(a10.F, W11, mul2(a00.F, W10));                                                \
                    }
                    BANET_A(0, x) BANET_A(1, y)
#undef BANET_A
                    uint32_t dep = (uint32_t)(d[0] & 0ull);
                    asm volatile("" : "+r"(dep) : "l"(gx[1]), "l"(gyP[0]));
                    ulonglong2 a0m, a1m, a0p, a1p;
                    if (staged) {
                        const uint32_t wb2 = wb + dep;
                        a0m = lds2x64(wb2 + rM + o0); a1m = lds2x64(wb2 + rM + o1); a0p = lds2x64(wb2 + rP + o0); a1p = lds2x64(wb2 + rP + o1);
                    } else {
                        const float* img2 = img + dep;
                        a0m = ldg2x64(img2 + rM + o0); a1m = ldg2x64(img2 + rM + o1); a0p = ldg2x64(img2 + rP + o0); a1p = ldg2x64(img2 + rP + o1);
                    }
#define BANET_B(H, F, K0)                                                                                           \
                    {                                                                                               \
                        const u64 P = fma2(a1p.F, W11, fma2(a0p.F, W10, gyP[H]));                                   \
                        const u64 Nn = fma2(a1m.F, W01, fma2(a0m.F, W00, gyN[H]));                                  \
                        const u64 gy = sub2(P, Nn);                                                                 \
                        m11 = fma2(gx[H], gx[H], m11); m12 = fma2(gx[H], gy, m12); m22 = fma2(gy, gy, m22);          \
                        q1 = fma2(gx[H], d[H], q1); q2 = fma2(gy, d[H], q2);                                         \
                        const float2 dd = upk2(d[H]);                                                               \
                        rb[4 * c + K0] += fabsf(dd.x); rb[4 * c + K0 + 1] += fabsf(dd.y);                             \
                    }
                    BANET_B(0, x, 0) BANET_B(1, y, 2)
#undef BANET_B
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&winfree[buf]);
                if (g == 0) {                                // refill the buffer just released with the chunk NWB ahead
                    if (lane == 0 && q + NWB < nchunks) { mbar_wait_parked(&winfree[buf], (q / NWB) & 1); issue_chunk(q + NWB); }
                    __syncwarp();
                }
            }
            float s11, s12, s22, sq1, sq2;
            { const float2 t = upk2(m11); s11 = 0.25f * (t.x + t.y); } { const float2 t = upk2(m12); s12 = 0.25f * (t.x + t.y); }
            { const float2 t = upk2(m22); s22 = 0.25f * (t.x + t.y); } { const float2 t = upk2(q1); sq1 = 0.5f * (t.x + t.y); }
            { const float2 t = upk2(q2); sq2 = 0.5f * (t.x + t.y); }
            s11 = qsum8(s11); s12 = qsum8(s12); s22 = qsum8(s22); sq1 = qsum8(sq1); sq2 = qsum8(sq2);
            // s_n = jd^T M jd of this quarter's pixel (DepthJacobianMatrix, bundlenet.py:63-74), every lane of the quarter
            float sn;
            {
                const float x = rec[5], y = rec[6], iZ = rec[7];
                const float fx = __int_as_float(sTile[s * 8 + 3]), fy = __int_as_float(sTile[s * 8 + 4]);
                const float jd0 = fx * ((rgeo.x - rgeo.z * x) * iZ), jd1 = fy * ((rgeo.y - rgeo.z * y) * iZ);
                const float u0 = s11 * jd0 + s12 * jd1, u1 = s12 * jd0 + s22 * jd1;
                sn = (mask != 0.f) ? jd0 * u0 + jd1 * u1 : 0.f;
            }
            __syncwarp();                                    // every lane has read its record before the totals overwrite part of it
            if (ql == 0) {               // totals overwrite dx,dy / tap columns / n of this pixel's record (no longer needed)
                *reinterpret_cast<float4*>(rec + 12) = make_float4(s11, s12, s22, sq1);
                rec[11] = sq2;
            }
            // ---- scaling pass: R row = rna(s_n * b_n) (the MMA's B operand), and the A-operand side of the precision mode, for this quarter's pixel:
            //      16 floats per lane = its 16-B chunk in each of the 4 basis blocks (a quarter reads / writes one whole 128-B row: conflict-free).
            //      Moved here from the 4 algebra warps: 16 warps share the work and the algebra -> MMA path of a tile becomes short.
            if (j > 0) mbar_wait_parked(bar.rfree, (j - 1) & 1);              // MMAs of tile j-1 done: R (and A_lo) are free
            {
                const int st = j % NST;
                mbar_wait_parked(&bar.fullB[st], (j / NST) & 1);              // long complete (the geometry warps needed it)
                unsigned char* As = base + SM::off_A + st * STAGE_A;
                unsigned char* Rs = base + SM::off_R;
                const uint32_t rowo = sw128_32b_off(pxi, ql);
                uint32_t hbase = 0;
                if constexpr (MODE == 1) hbase = (uint32_t)sTile[s * 8 + 5] ^ ((uint32_t)__float_as_int(rgeo.w) * 0x9E3779B1u);
#pragma unroll
                for (int blk = 0; blk < KBLK; ++blk) {
                    const uint32_t off = blk * 8192 + rowo;
                    const float4 bv = *reinterpret_cast<const float4*>(As + off);
                    *reinterpret_cast<float4*>(Rs + off) = make_float4(tf32_rna_bits(sn * bv.x), tf32_rna_bits(sn * bv.y), tf32_rna_bits(sn * bv.z), tf32_rna_bits(sn * bv.w));
                    if constexpr (MODE == 1)     // single-pass mode: the basis tile is rounded to tf32 IN PLACE
                        *reinterpret_cast<float4*>(As + off) = tf32_stochastic4(bv, hbase ^ ((uint32_t)(blk * 8 + ql) * 0x85EBCA77u));
                    if constexpr (MODE >= 2)
                        *reinterpret_cast<float4*>(base + SM::off_Alo + off) = make_float4(bv.x - tf32_trunc(bv.x), bv.y - tf32_trunc(bv.y), bv.z - tf32_trunc(bv.z), bv.w - tf32_trunc(bv.w));
                }
            }
            fence_proxy_async_smem();                        // the MMA reads R / A / A_lo through the async proxy
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar.gath[s]);
        }
        if (cur_b >= 0) dump_rb();
    } else if (warp < W0 + GW + AW) {
        // ===================================================================== algebra warps: 2x7 algebra (H_cc, g_c, [v | t]), MMA + TMA issue
        setmaxnreg_dec<64>();
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

        auto issue_tma = [&](int t) {                        // basis tile t -> stage t % NST (elected thread)
            const int st = t % NST;
            const TileCoord tc = banded_tile_coord(prm, t_begin + t);
            mbar_arrive_expect_tx(&bar.fullB[st], KBLK * 8192);
            unsigned char* dst = base + SM::off_A + st * STAGE_A;
#pragma unroll
            for (int blk = 0; blk < KBLK; ++blk) tma_load_3d(dst + blk * 8192, &tmapB, blk * 32, tc.tx0, tc.b * prm.grid_h + tc.ty0, &bar.fullB[st]);
        };
        if (awi == 0 && lane == 0)
            for (int t = 0; t < NST && t < ntiles; ++t) issue_tma(t);      // every stage starts free

        for (int j = 0; j < ntiles; ++j) {
            const int s = j % NST, sr = j % NREC;
            const bool last_of_pair = (++rr == prm.tiles_per_pair) || (j == ntiles - 1);
            if (rr == prm.tiles_per_pair) rr = 0;
            if (j > 0) {
                // MMAs of tile j-1 done: R / A_lo and stage (j-1) % NST are free.  Refill the stage BEFORE waiting for the gather of tile j: the
                // window producer (gather warp 0) looks ahead into tile j+1 and waits for its records, i.e. for the geometry warps, i.e. for
                // this very TMA when NST == 2 -- issued after gath[j] it would close a cycle through the gather warps themselves.
                mbar_wait_parked(bar.rfree, (j - 1) & 1);
                if (awi == 0 && lane == 0 && j - 1 + NST < ntiles) issue_tma(j - 1 + NST);
            }
            mbar_wait_parked(&bar.gath[sr], (j / NREC) & 1);
            const int b = sTile[sr * 8];
            if (b != scale_b) { scale_b = b; ++sspan; fx = __ldg(prm.intr + b * 4); fy = __ldg(prm.intr + b * 4 + 1); }
            float ext[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (lane < 16) pixel_algebra(sRec + (sr * TILE + nlr) * REC, fx, fy, cc, ext);
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar.recfree[sr]);    // the record buffer may be refilled (everything needed is in registers)
            mbar_wait_parked(&bar.fullB[s], (j / NST) & 1);  // long complete; orders the TMA writes before the reads below
            if (lane < 16) write_vt<MODE, KBLK>(Rs, nullptr, nlr, ext);
            // (the R rows s_n * b_n were written by the gather warps' scaling pass; this team only adds the [v | t] block)
            fence_proxy_async_smem();
            team_bar<AW * 32>();                           // all 64 rows written
            if (awi == 0) {
                if (lane == 0) {                             // ---- tcgen05.mma issue for this tile
                    if (new_span) { mbar_wait_parked(bar.tmemfree, (mspan & 1) ^ 1); accL = 0; new_span = false; }
                    if (tic == 0) { ++chain; set = chain & 1; mbar_wait_parked(&bar.drained[set], ((chain >> 1) & 1) ^ 1); accH = 0; }
                    tc_fence_after_sync();
                    const uint32_t ahi = smem_u32(base + SM::off_A + s * STAGE_A);
                    const uint32_t rhi = smem_u32(base + SM::off_R), alo = smem_u32(base + SM::off_Alo);
#pragma unroll
                    for (int pass = 0; pass < MODE; ++pass) {     // no R_lo pass: MODE <= 2
                        const uint32_t a0 = (pass == 1) ? alo : ahi;
                        const uint32_t r0 = rhi;
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
        drainer_role<40, MODE, KBLK, C>(prm, bar, tmem, t_begin, ntiles, warp - (W0 + GW + AW), lane);
    }
    release_tmem(tmem, warp);
}


template <int NCH, int MODE, int KBLK = 4>
static int launch7(const CUtensorMap& tmB, const CUtensorMap& tmF, const CUtensorMap& tmC, const BuildParams& prm, int grid, cudaStream_t st)
{
    auto kern = lm_build_tc7_kernel<NCH, MODE, KBLK>;
    const int smem = Smem<MODE, NCH>::bytes;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) { set_error("lm_build_tc7: smem attr (%d B): %s", smem, cudaGetErrorString(e)); return BANET_ERR_CUDA; }
    kern<<<grid, THREADS, smem, st>>>(tmB, tmF, tmC, prm);
    BANET_CUDA_LAUNCH_CHECK("lm_build_tc7_kernel launch");
    return BANET_OK;
}

}  // namespace v7

bool lm_build_tc7_supported(int mode, int nch, int kblk) { return (mode == 1 || mode == 2) && (nch == 1 || nch == 2) && kblk == 4; }
void lm_build_tc7_window(int* wx, int* wy) { *wx = v7::WX; *wy = v7::WY; }

int lm_build_tc7_launch(int mode, int nch, int kblk, const CUtensorMap& tmB, const CUtensorMap& tmF, const CUtensorMap& tmC, const BuildParams& prm, int grid,
                        cudaStream_t st)
{
    BANET_REQUIRE(lm_build_tc7_supported(mode, nch, kblk), BANET_ERR_UNSUPPORTED, "lm_build_tc7: mode %d / C=%d / K=%d not instantiated", mode, 64 * nch, 32 * kblk);
    if (nch == 2) return mode == 1 ? v7::launch7<2, 1>(tmB, tmF, tmC, prm, grid, st) : v7::launch7<2, 2>(tmB, tmF, tmC, prm, grid, st);
    return mode == 1 ? v7::launch7<1, 1>(tmB, tmF, tmC, prm, grid, st) : v7::launch7<1, 2>(tmB, tmF, tmC, prm, grid, st);
}

}  // namespace banet
