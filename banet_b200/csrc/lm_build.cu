// Fused normal-equation construction of one LM iteration (fp32 SIMT path).
//
// Replaces, in one streaming pass that never materialises J, G or d:
//   reference bundlenet.py:206-224 (depth update + warp), :226-239 (sample, mask, diff, grad),
//   :243 (sum_n |diff|), :259-261 (camera / depth Jacobians) and the native op
//   EquationConstruction utils.cu:219-417 (5 batched SGEMMs + 2 column reductions).
//
// Block decomposition used (SURVEY.md §7; proven exact by oracle.normal_equations_structured):
//   with M = G^T G (2x2), q = G^T d (2), J = [Jc (2x6) | jd b^T]:
//     H_cc = sum Jc^T M Jc           g_c = sum Jc^T q
//     H_cd = sum (Jc^T M jd) b^T     g_d = sum (jd^T q) b
//     H_dd = sum (jd^T M jd) b b^T
//
// Work decomposition: the nb*ceil(N/64) pixel tiles are split contiguously over a persistent grid
// (one CTA per SM); each CTA keeps its accumulators in registers across tiles and writes ONE partial
// slot per pair it touches; lm_reduce_kernel sums the slots in a fixed order (deterministic, no atomics).
#include "common.cuh"
#include "lm_build.h"

namespace banet {

constexpr int TILE_PX = 64;
constexpr int BUILD_THREADS = 256;
constexpr int BUILD_WARPS = BUILD_THREADS / 32;
constexpr int REC_ARRAYS = 16;          // per-pixel scalar record arrays

// per-pixel record array ids
enum { R_X0 = 0, R_Y0, R_DX, R_DY, R_MASK, R_X, R_Y, R_IZ, R_RX, R_RY, R_RZ, R_M11, R_M12, R_M22, R_Q1, R_Q2 };

template <int KP> struct BuildSmem {
    static constexpr int LDB = KP + 4;
    static constexpr int off_B = 0;
    static constexpr int off_W = off_B + (KP > 0 ? TILE_PX * LDB : 0);
    static constexpr int off_rec = off_W + (KP > 0 ? KP : 0);
    static constexpr int off_ext = off_rec + REC_ARRAYS * TILE_PX;      // [TILE_PX][8]: v0..v5, t, s
    static constexpr int off_pose = off_ext + TILE_PX * 8;              // R(9) T(3) intr(4)
    static constexpr int off_cc = off_pose + 16;                        // [2][32]
    static constexpr int off_rb = off_cc + 64;                          // [BUILD_WARPS][C]
    static size_t bytes(int C) { return (size_t)(off_rb + BUILD_WARPS * C) * sizeof(float); }
};

template <int G> __device__ __forceinline__ void lds_group(const float* p, float* out);
template <> __device__ __forceinline__ void lds_group<1>(const float* p, float* o) { o[0] = p[0]; }
template <> __device__ __forceinline__ void lds_group<2>(const float* p, float* o) {
    float2 v = *reinterpret_cast<const float2*>(p); o[0] = v.x; o[1] = v.y; }
template <> __device__ __forceinline__ void lds_group<4>(const float* p, float* o) {
    float4 v = *reinterpret_cast<const float4*>(p); o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }

__device__ __forceinline__ int reflect_idx(int i, int n) {      // tf.pad REFLECT by one (bundlenet.py:97)
    return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i);
}

// ---- S2 helper: accumulate one group of VEC channels of one pixel ------------------------------
template <int VEC> struct ChanVec;
template <> struct ChanVec<4> {
    float v[4];
    __device__ __forceinline__ void load(const float* p) { float4 t = __ldg(reinterpret_cast<const float4*>(p)); v[0]=t.x; v[1]=t.y; v[2]=t.z; v[3]=t.w; }
    __device__ __forceinline__ void load_stream(const float* p) { float4 t = ld_stream_f4(p); v[0]=t.x; v[1]=t.y; v[2]=t.z; v[3]=t.w; }
    __device__ __forceinline__ void load_smem(const float* p) { float4 t = *reinterpret_cast<const float4*>(p); v[0]=t.x; v[1]=t.y; v[2]=t.z; v[3]=t.w; }
    __device__ __forceinline__ void store_smem(float* p) const { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};
template <> struct ChanVec<1> {
    float v[1];
    __device__ __forceinline__ void load(const float* p) { v[0] = __ldg(p); }
    __device__ __forceinline__ void load_stream(const float* p) { v[0] = ld_stream_f1(p); }
    __device__ __forceinline__ void load_smem(const float* p) { v[0] = p[0]; }
    __device__ __forceinline__ void store_smem(float* p) const { p[0] = v[0]; }
};

template <int KP, int VEC>
__global__ void __launch_bounds__(BUILD_THREADS, (KP >= 128) ? 1 : 2)
lm_build_kernel(const BuildParams prm)
{
    using SM = BuildSmem<KP>;
    extern __shared__ __align__(16) float smem[];
    float* Bs   = smem + SM::off_B;
    float* sW   = smem + SM::off_W;
    float* rec  = smem + SM::off_rec;
    float* sExt = smem + SM::off_ext;
    float* sPose = smem + SM::off_pose;
    float* sCC  = smem + SM::off_cc;
    float* sRb  = smem + SM::off_rb;
    constexpr int LDB = SM::LDB;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = prm.N, C = prm.C, K = prm.K, h = prm.h, w = prm.w, c2 = prm.c2;
    const bool fly_grad = (c2 == C);

    // ---- accumulators (persist across the tiles of one pair) -----------------------------------
    // K > 128 (KP = 256): one launch per 128 x 128 block (prm.kq_i, prm.kq_j) of H_dd's lower triangle; the staged tile, the depth update and
    // the gather are those of the full basis, the register tile is that of K = 128 (a 16 x 16 tile would need 256 accumulators per thread)
    constexpr int KB = (KP > 128) ? 128 : KP;   // contraction block edge
    const int ki0 = (KP > 128) ? prm.kq_i * 128 : 0, kj0 = (KP > 128) ? prm.kq_j * 128 : 0;
    const bool first_block = (KP <= 128) || (prm.kq_i == 0 && prm.kq_j == 0), diag_block = (KP <= 128) || (prm.kq_i == prm.kq_j);
    constexpr int T  = KB / 16;                 // per-thread H_dd tile edge
    constexpr int G  = (T >= 4) ? 4 : (T > 0 ? T : 1);
    constexpr int NG = (T > 0) ? T / G : 0;
    constexpr int TT = (T > 0) ? T : 1;
    constexpr int NPART = (KP > 0) ? BUILD_THREADS / KB : 1;
    constexpr int EA = (KP > 0) ? (7 + NPART - 1) / NPART : 1;
    float acc[TT][TT];
    float accx[EA];
    float cc[28];                               // 21 H_cc (upper, row-major) + 6 g_c + nvalid
    const int ti = tid >> 4, tj = tid & 15;

    auto zero_acc = [&]() {
#pragma unroll
        for (int e = 0; e < TT; ++e)
#pragma unroll
            for (int f = 0; f < TT; ++f) acc[e][f] = 0.f;
#pragma unroll
        for (int q = 0; q < EA; ++q) accx[q] = 0.f;
#pragma unroll
        for (int q = 0; q < 28; ++q) cc[q] = 0.f;
        for (int c = tid; c < BUILD_WARPS * C; c += BUILD_THREADS) sRb[c] = 0.f;   // visible after the S0 barrier
    };

    const SlotLayout L{K, C};
    auto flush = [&](int span) {
        float* slot = prm.partials + ((size_t)blockIdx.x * prm.max_span + span) * prm.slot_floats;
        if constexpr (KP > 0) {
#pragma unroll
            for (int e = 0; e < TT; ++e) {
                const int row = ki0 + (e / G) * (16 * G) + G * ti + (e % G);
#pragma unroll
                for (int f = 0; f < TT; ++f) {
                    const int col = kj0 + (f / G) * (16 * G) + G * tj + (f % G);
                    if (row < K && col < K) slot[row * K + col] = acc[e][f];
                }
            }
            const int k = kj0 + tid % KB, part = tid / KB;
            if (diag_block) {
#pragma unroll
                for (int q = 0; q < EA; ++q) {
                    const int r = part * EA + q;
                    if (r < 7 && k < K) slot[L.off_ext() + r * K + k] = accx[q];
                }
            }
        }
        // cc: 28 values held by threads 0..63 -> warp reduce, combine the two warps through smem
        if (warp < 2) {
#pragma unroll
            for (int q = 0; q < 28; ++q) { float v = warp_sum(cc[q]); if (lane == 0) sCC[warp * 32 + q] = v; }
        }
        // rbar: sRb holds one row of per-channel |diff| sums per warp (accumulated in S2)
        __syncthreads();
        if (first_block) {
            if (tid < 28) slot[L.off_cc() + tid] = sCC[tid] + sCC[32 + tid];
            for (int c = tid; c < C; c += BUILD_THREADS) {
                float s = 0.f;
#pragma unroll
                for (int wq = 0; wq < BUILD_WARPS; ++wq) s += sRb[wq * C + c];
                slot[L.off_rbar() + c] = s;
            }
        }
        __syncthreads();
    };

    const long long t_begin = part_begin(prm.total_tiles, gridDim.x, blockIdx.x);
    const long long t_end   = part_begin(prm.total_tiles, gridDim.x, blockIdx.x + 1);
    int cur_b = -1, span = 0;

    for (long long t = t_begin; t < t_end; ++t) {
        const int b = (int)(t / prm.tiles_per_pair);
        const int n0 = (int)(t - (long long)b * prm.tiles_per_pair) * TILE_PX;
        const int cnt = min(TILE_PX, N - n0);

        if (b != cur_b) {
            if (cur_b >= 0) { flush(span); ++span; }
            zero_acc();
            if (tid < 9) sPose[tid] = prm.R[b * 9 + tid];
            else if (tid < 12) sPose[tid] = prm.T[b * 3 + tid - 9];
            else if (tid < 16) sPose[tid] = prm.intr[b * 4 + tid - 12];
            if constexpr (KP > 0) for (int k = tid; k < KP; k += BUILD_THREADS) sW[k] = (k < K) ? prm.W[b * K + k] : 0.f;
            cur_b = b;
        }

        // ---- S0: stage the basis tile (coalesced, read-once) ------------------------------------
        if constexpr (KP > 0) {
            const float* Bg = prm.B + ((size_t)b * N + n0) * K;
            if ((K & 3) == 0) {
                const int k4 = K >> 2, kp4 = KP >> 2;
                for (int i = tid; i < TILE_PX * kp4; i += BUILD_THREADS) {
                    const int n = i / kp4, q = i - n * kp4;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (n < cnt && q < k4) v = ld_stream_f4(Bg + (size_t)n * K + 4 * q);
                    *reinterpret_cast<float4*>(Bs + n * LDB + 4 * q) = v;
                }
            } else {
                for (int i = tid; i < TILE_PX * KP; i += BUILD_THREADS) {
                    const int n = i / KP, k = i - n * KP;
                    Bs[n * LDB + k] = (n < cnt && k < K) ? ld_stream_f1(Bg + (size_t)n * K + k) : 0.f;
                }
            }
        }
        __syncthreads();

        // ---- S1: per-pixel geometry, thread per pixel (bundlenet.py:208-224, mask :231) ----------
        if (tid < TILE_PX) {
            const int n = tid;
            float mask = 0.f, x = 0.f, y = 0.f, iZ = 0.f, rx = 0.f, ry = 0.f, rz = 0.f, dx = 0.f, dy = 0.f;
            int x0 = 0, y0 = 0;
            if (n < cnt) {
                const size_t gi = (size_t)b * N + n0 + n;
                const float* pp = prm.p + (size_t)b * 3 * N + n0 + n;
                const float p0 = pp[0], p1 = pp[N], p2 = pp[2 * (size_t)N];
                float Dt = prm.D[gi];
                if constexpr (KP > 0) {
                    float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll 4
                    for (int k = 0; k < KP; k += 4) {
                        const float4 bv = *reinterpret_cast<const float4*>(Bs + n * LDB + k);
                        const float4 wv = *reinterpret_cast<const float4*>(sW + k);
                        d0 = fmaf(bv.x, wv.x, d0); d1 = fmaf(bv.y, wv.y, d1);
                        d2 = fmaf(bv.z, wv.z, d2); d3 = fmaf(bv.w, wv.w, d3);
                    }
                    Dt += (d0 + d1) + (d2 + d3);
                }
                rx = sPose[0] * p0 + sPose[1] * p1 + sPose[2] * p2;
                ry = sPose[3] * p0 + sPose[4] * p1 + sPose[5] * p2;
                rz = sPose[6] * p0 + sPose[7] * p1 + sPose[8] * p2;
                const float X = rx * Dt + sPose[9], Y = ry * Dt + sPose[10], Z = rz * Dt + sPose[11];
                x = X / Z; y = Y / Z; iZ = 1.0f / Z;
                const float u = sPose[12] * x + sPose[14], v = sPose[13] * y + sPose[15];
                // reference mask: not(px<0 | px>w-1 | py<0 | py>h-1); non-finite projections are masked too
                const bool ok = (u >= 0.f) && (u <= (float)(w - 1)) && (v >= 0.f) && (v <= (float)(h - 1)) && isfinite(iZ);
                if (ok) {
                    mask = 1.f;
                    const float fu = floorf(u), fv = floorf(v);
                    x0 = (int)fu; y0 = (int)fv; dx = u - fu; dy = v - fv;
                }
            }
            rec[R_X0 * TILE_PX + n] = __int_as_float(x0); rec[R_Y0 * TILE_PX + n] = __int_as_float(y0);
            rec[R_DX * TILE_PX + n] = dx; rec[R_DY * TILE_PX + n] = dy; rec[R_MASK * TILE_PX + n] = mask;
            rec[R_X * TILE_PX + n] = x; rec[R_Y * TILE_PX + n] = y; rec[R_IZ * TILE_PX + n] = iZ;
            rec[R_RX * TILE_PX + n] = rx; rec[R_RY * TILE_PX + n] = ry; rec[R_RZ * TILE_PX + n] = rz;
        }
        __syncthreads();

        // ---- S2: feature gather, warp per pixel, lanes over channels (bundlenet.py:230-239) ------
        for (int i = 0; i < TILE_PX / BUILD_WARPS; ++i) {
            const int n = i * BUILD_WARPS + warp;
            float m11 = 0.f, m12 = 0.f, m22 = 0.f, q1 = 0.f, q2 = 0.f;
            if (rec[R_MASK * TILE_PX + n] != 0.f) {
                const int x0 = __float_as_int(rec[R_X0 * TILE_PX + n]), y0 = __float_as_int(rec[R_Y0 * TILE_PX + n]);
                const float dx = rec[R_DX * TILE_PX + n], dy = rec[R_DY * TILE_PX + n];
                const int x1 = min(x0 + 1, w - 1), y1 = min(y0 + 1, h - 1);
                const float w00 = (1.f - dx) * (1.f - dy), w01 = dx * (1.f - dy), w10 = (1.f - dx) * dy, w11 = dx * dy;
                const float* img = prm.conv2 + (size_t)b * h * w * c2;
                const float* t00 = img + ((size_t)y0 * w + x0) * c2;
                const float* t01 = img + ((size_t)y0 * w + x1) * c2;
                const float* t10 = img + ((size_t)y1 * w + x0) * c2;
                const float* t11 = img + ((size_t)y1 * w + x1) * c2;
                const float* c1 = prm.conv1 + ((size_t)b * N + n0 + n) * C;
                float* myRb = sRb + warp * C;
                for (int c = lane * VEC; c < C; c += 32 * VEC) {
                    ChanVec<VEC> f1, a00, a01, a10, a11, gx, gy;
                    f1.load_stream(c1 + c);
                    a00.load(t00 + c); a01.load(t01 + c); a10.load(t10 + c); a11.load(t11 + c);
                    if (!fly_grad) {
                        ChanVec<VEC> g00, g01, g10, g11;
                        g00.load(t00 + C + c); g01.load(t01 + C + c); g10.load(t10 + C + c); g11.load(t11 + C + c);
#pragma unroll
                        for (int u = 0; u < VEC; ++u) gx.v[u] = w00 * g00.v[u] + w01 * g01.v[u] + w10 * g10.v[u] + w11 * g11.v[u];
                        g00.load(t00 + 2 * C + c); g01.load(t01 + 2 * C + c); g10.load(t10 + 2 * C + c); g11.load(t11 + 2 * C + c);
#pragma unroll
                        for (int u = 0; u < VEC; ++u) gy.v[u] = w00 * g00.v[u] + w01 * g01.v[u] + w10 * g10.v[u] + w11 * g11.v[u];
                    } else {
                        // F2-only map: central differences with REFLECT-by-one borders (bundlenet.py:92-100) at each tap
#pragma unroll
                        for (int u = 0; u < VEC; ++u) { gx.v[u] = 0.f; gy.v[u] = 0.f; }
                        const int xs[2] = {x0, x1}, ys[2] = {y0, y1};
                        const float wt[4] = {w00, w01, w10, w11};
#pragma unroll
                        for (int tp = 0; tp < 4; ++tp) {
                            const int xx = xs[tp & 1], yy = ys[tp >> 1];
                            ChanVec<VEC> e, wv, s, nn;
                            e.load(img + ((size_t)yy * w + reflect_idx(xx + 1, w)) * c2 + c);
                            wv.load(img + ((size_t)yy * w + reflect_idx(xx - 1, w)) * c2 + c);
                            s.load(img + ((size_t)reflect_idx(yy + 1, h) * w + xx) * c2 + c);
                            nn.load(img + ((size_t)reflect_idx(yy - 1, h) * w + xx) * c2 + c);
#pragma unroll
                            for (int u = 0; u < VEC; ++u) {
                                gx.v[u] = fmaf(wt[tp], 0.5f * (e.v[u] - wv.v[u]), gx.v[u]);
                                gy.v[u] = fmaf(wt[tp], 0.5f * (s.v[u] - nn.v[u]), gy.v[u]);
                            }
                        }
                    }
                    ChanVec<VEC> ra;
                    ra.load_smem(myRb + c);
#pragma unroll
                    for (int u = 0; u < VEC; ++u) {
                        const float f2 = w00 * a00.v[u] + w01 * a01.v[u] + w10 * a10.v[u] + w11 * a11.v[u];
                        const float d = f1.v[u] - f2;
                        m11 = fmaf(gx.v[u], gx.v[u], m11); m12 = fmaf(gx.v[u], gy.v[u], m12); m22 = fmaf(gy.v[u], gy.v[u], m22);
                        q1 = fmaf(gx.v[u], d, q1); q2 = fmaf(gy.v[u], d, q2);
                        ra.v[u] += fabsf(d);
                    }
                    ra.store_smem(myRb + c);
                }
                m11 = warp_sum(m11); m12 = warp_sum(m12); m22 = warp_sum(m22); q1 = warp_sum(q1); q2 = warp_sum(q2);
            }
            if (lane == 0) {
                rec[R_M11 * TILE_PX + n] = m11; rec[R_M12 * TILE_PX + n] = m12; rec[R_M22 * TILE_PX + n] = m22;
                rec[R_Q1 * TILE_PX + n] = q1; rec[R_Q2 * TILE_PX + n] = q2;
            }
        }
        __syncthreads();

        // ---- S3: per-pixel 2x(6+1) algebra, thread per pixel (bundlenet.py:49-74) -----------------
        if (tid < TILE_PX) {
            const int n = tid;
            float ext[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (rec[R_MASK * TILE_PX + n] != 0.f) {
                const float x = rec[R_X * TILE_PX + n], y = rec[R_Y * TILE_PX + n], iZ = rec[R_IZ * TILE_PX + n];
                const float m11 = rec[R_M11 * TILE_PX + n], m12 = rec[R_M12 * TILE_PX + n], m22 = rec[R_M22 * TILE_PX + n];
                const float q1 = rec[R_Q1 * TILE_PX + n], q2 = rec[R_Q2 * TILE_PX + n];
                const float fx = sPose[12], fy = sPose[13];
                // CameraJacobianMatrix, negated (bundlenet.py:58-60)
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
                if constexpr (KP > 0) {
                    const float rx = rec[R_RX * TILE_PX + n], ry = rec[R_RY * TILE_PX + n], rz = rec[R_RZ * TILE_PX + n];
                    const float jd0 = fx * ((rx - rz * x) * iZ), jd1 = fy * ((ry - rz * y) * iZ);   // DepthJacobianMatrix :69-70
                    const float u0 = m11 * jd0 + m12 * jd1, u1 = m12 * jd0 + m22 * jd1;
#pragma unroll
                    for (int i = 0; i < 6; ++i) ext[i] = a0[i] * u0 + a1[i] * u1;
                    ext[6] = jd0 * q1 + jd1 * q2;
                    ext[7] = jd0 * u0 + jd1 * u1;
                }
            }
            if constexpr (KP > 0) {
                *reinterpret_cast<float4*>(sExt + n * 8) = make_float4(ext[0], ext[1], ext[2], ext[3]);
                *reinterpret_cast<float4*>(sExt + n * 8 + 4) = make_float4(ext[4], ext[5], ext[6], ext[7]);
            }
        }

        // ---- S4: basis contraction  H_dd += s b b^T,  [H_cd; g_d] += [v; t] b^T  (fp32 FFMA) ------
        if constexpr (KP > 0) {
            __syncthreads();
            const int k = kj0 + tid % KB, part = tid / KB;
#pragma unroll 2
            for (int n = 0; n < cnt; ++n) {
                if (rec[R_MASK * TILE_PX + n] == 0.f) continue;
                const float4 e0 = *reinterpret_cast<const float4*>(sExt + n * 8);
                const float4 e1 = *reinterpret_cast<const float4*>(sExt + n * 8 + 4);
                const float ev[8] = {e0.x, e0.y, e0.z, e0.w, e1.x, e1.y, e1.z, e1.w};
                const float s = ev[7];
                float a[TT], cvals[TT];
#pragma unroll
                for (int gq = 0; gq < NG; ++gq) {
                    lds_group<G>(Bs + n * LDB + ki0 + gq * 16 * G + G * ti, a + gq * G);
                    lds_group<G>(Bs + n * LDB + kj0 + gq * 16 * G + G * tj, cvals + gq * G);
                }
#pragma unroll
                for (int e = 0; e < TT; ++e) {
                    const float sa = s * a[e];
#pragma unroll
                    for (int f = 0; f < TT; ++f) acc[e][f] = fmaf(sa, cvals[f], acc[e][f]);
                }
                const float bk = Bs[n * LDB + k];
#pragma unroll
                for (int q = 0; q < EA; ++q) {
                    const int r = part * EA + q;
                    if (r < 7) accx[q] = fmaf(ev[r], bk, accx[q]);
                }
            }
        }
        __syncthreads();
    }
    if (cur_b >= 0) flush(span);
}

// ---- deterministic reduction of the partial slots -> H, g, rbar_sum, nvalid ----------------------
__global__ void __launch_bounds__(256)
lm_reduce_kernel(const BuildParams prm, int grid_build, float* __restrict__ H, float* __restrict__ g,
                 float* __restrict__ rbar_sum, float* __restrict__ nvalid)
{
    const int b = blockIdx.y, K = prm.K, C = prm.C, P = 6 + K;
    const SlotLayout L{K, C};
    const long long p0 = (long long)b * prm.tiles_per_pair, p1 = p0 + prm.tiles_per_pair;
    // slots that hold a partial of pair b: one per CTA whose tile range intersects [p0,p1) (a contiguous CTA range)
    __shared__ const float* s_slot[2 * kMaxSMs + 8];        // a pair can be spread over the whole grid (<= 2 CTAs per SM)
    __shared__ int s_n;
    if (threadIdx.x == 0) {
        int c0 = (int)((p0 * grid_build) / prm.total_tiles);
        while (c0 + 1 < grid_build && part_begin(prm.total_tiles, grid_build, c0 + 1) <= p0) ++c0;
        int n = 0;
        for (int c = c0; c < grid_build && n < 2 * kMaxSMs + 8; ++c) {
            const long long tb = part_begin(prm.total_tiles, grid_build, c), te = part_begin(prm.total_tiles, grid_build, c + 1);
            if (tb >= p1) break;
            if (tb >= te || te <= p0) continue;
            const int span = b - (int)(tb / prm.tiles_per_pair);
            s_slot[n++] = prm.partials + ((size_t)c * prm.max_span + span) * prm.slot_floats;
        }
        s_n = n;
    }
    __syncthreads();
    const int nslot = s_n;
    const int nel = L.off_rbar() + C;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nel; i += gridDim.x * blockDim.x) {
        int src = i;                                        // element (r, cI) of H_dd lives at cI*K + r in a transposed slot
        int r = 0, cI = 0;
        if (i < L.off_ext()) {
            r = i / K; cI = i - r * K;
            if (cI > r) continue;                           // only the lower triangle is used (and mirrored)
            if (prm.hdd_transposed) src = cI * K + r;
        }
        double s = 0.0;
        for (int q = 0; q < nslot; ++q) s += (double)s_slot[q][src];
        const float v = (float)s;
        if (i < L.off_ext()) {                              // H_dd: keep the lower triangle, mirror it
            H[((size_t)b * P + 6 + r) * P + 6 + cI] = v; H[((size_t)b * P + 6 + cI) * P + 6 + r] = v;
        } else if (i < L.off_cc()) {
            const int rr = (i - L.off_ext()) / K, k = (i - L.off_ext()) - rr * K;
            if (rr < 6) { H[((size_t)b * P + rr) * P + 6 + k] = v; H[((size_t)b * P + 6 + k) * P + rr] = v; }
            else g[(size_t)b * P + 6 + k] = v;
        } else if (i < L.off_rbar()) {
            const int q = i - L.off_cc();
            if (q < 21) {
                int rr = 0, rem = q;
                while (rem >= 6 - rr) { rem -= 6 - rr; ++rr; }
                const int cc = rr + rem;
                H[((size_t)b * P + rr) * P + cc] = v; H[((size_t)b * P + cc) * P + rr] = v;
            } else if (q < 27) g[(size_t)b * P + q - 21] = v;
            else if (q == 27) nvalid[b] = v;
        } else {
            rbar_sum[(size_t)b * C + i - L.off_rbar()] = v;
        }
    }
}

int launch_lm_reduce(const BuildParams& prm, int grid_build, float* H, float* g, float* rbar_sum, float* nvalid, cudaStream_t st)
{
    const int nel = prm.K * prm.K + 7 * prm.K + 32 + prm.C;
    int chunks = (nel + 2047) / 2048; if (chunks < 1) chunks = 1; if (chunks > 16) chunks = 16;
    lm_reduce_kernel<<<dim3(chunks, prm.nb), 256, 0, st>>>(prm, grid_build, H, g, rbar_sum, nvalid);
    BANET_CUDA_LAUNCH_CHECK("lm_reduce_kernel launch");
    return BANET_OK;
}

// ---- host side ------------------------------------------------------------------------------------
static int padded_K(int K) {
    if (K == 0) return 0;
    if (K <= 16) return 16;
    if (K <= 32) return 32;
    if (K <= 64) return 64;
    if (K <= 128) return 128;
    if (K <= 256) return 256;
    return -1;
}

int build_plan(const banet_level_t* lv, int num_sms, BuildPlan* plan)
{
    const int KP = padded_K(lv->K);
    BANET_REQUIRE(KP >= 0, BANET_ERR_UNSUPPORTED, "lm_build (fp32 SIMT): K=%d > 256 not supported", lv->K);
    BANET_REQUIRE(lv->C <= 2048, BANET_ERR_UNSUPPORTED, "lm_build: C=%d > 2048", lv->C);
    plan->KP = KP;
    plan->tiles_per_pair = (lv->N + TILE_PX - 1) / TILE_PX;
    plan->total_tiles = (long long)lv->nb * plan->tiles_per_pair;
    const int per_sm = (KP >= 128) ? 1 : 2;
    long long grid = (long long)num_sms * per_sm;
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

template <int KP, int VEC>
static int launch_build(const BuildParams& prm, int grid, cudaStream_t st)
{
    const size_t smem = BuildSmem<KP>::bytes(prm.C);
    auto kern = lm_build_kernel<KP, VEC>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("lm_build: smem attr (%zu B): %s", smem, cudaGetErrorString(e)); return BANET_ERR_CUDA; }
    kern<<<grid, BUILD_THREADS, smem, st>>>(prm);
    BANET_CUDA_LAUNCH_CHECK("lm_build_kernel launch");
    return BANET_OK;
}

int lm_build_simt(const banet_level_t* lv, const BuildPlan& plan, const float* R, const float* T, const float* W,
                  float* H, float* g, float* rbar_sum, float* nvalid, void* ws, cudaStream_t st)
{
    BuildParams prm;
    prm.nb = lv->nb; prm.N = lv->N; prm.C = lv->C; prm.K = lv->K; prm.h = lv->h; prm.w = lv->w; prm.c2 = lv->conv2_channels;
    prm.conv1 = lv->conv1; prm.conv2 = lv->conv2; prm.intr = lv->intr; prm.p = lv->p; prm.D = lv->D; prm.B = lv->B;
    prm.R = R; prm.T = T; prm.W = W;
    prm.partials = reinterpret_cast<float*>(ws);
    prm.slot_floats = plan.slot_floats; prm.max_span = plan.max_span;
    prm.tiles_per_pair = plan.tiles_per_pair; prm.total_tiles = plan.total_tiles;
    prm.kq_i = 0; prm.kq_j = 0;
    prm.grid_w = 0; prm.grid_h = 0; prm.tiles_x = 0; prm.tiles_y = 0; prm.band_rows = 1; prm.l2_hints = 0; prm.tap_prefetch = 0; prm.hdd_transposed = 0; prm.force_direct = 0;
    const bool vec4 = (lv->C % 4 == 0) && (lv->conv2_channels % 4 == 0) &&
                      ((reinterpret_cast<uintptr_t>(lv->conv1) | reinterpret_cast<uintptr_t>(lv->conv2)) % 16 == 0);
    int rc;
#define BANET_DISPATCH(KPV)                                                            \
    rc = vec4 ? launch_build<KPV, 4>(prm, plan.grid, st) : launch_build<KPV, 1>(prm, plan.grid, st)
    switch (plan.KP) {
        case 0:   BANET_DISPATCH(0); break;
        case 16:  BANET_DISPATCH(16); break;
        case 32:  BANET_DISPATCH(32); break;
        case 64:  BANET_DISPATCH(64); break;
        case 128: BANET_DISPATCH(128); break;
        case 256:                    // lower-triangle 128-blocks (0,0), (1,0), (1,1); lm_reduce mirrors
            rc = BANET_OK;
            for (int blk = 0; blk < 3 && rc == BANET_OK; ++blk) {
                prm.kq_i = blk == 0 ? 0 : 1; prm.kq_j = blk == 2 ? 1 : 0;
                BANET_DISPATCH(256);
            }
            break;
        default: set_error("lm_build: bad KP %d", plan.KP); return BANET_ERR_UNSUPPORTED;
    }
#undef BANET_DISPATCH
    if (rc != BANET_OK) return rc;
    return launch_lm_reduce(prm, plan.grid, H, g, rbar_sum, nvalid, st);
}

}  // namespace banet
