// sm_100a primitives used by the tensor-core build path: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (TMEM alloc / mma / commit / ld), shared-memory matrix descriptors and the 128B swizzle.
// Inline PTX only; no CUTLASS dependency.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace banet { namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) { }
}

// wait with a hardware suspend-time hint: the warp is parked by the barrier unit (no issue slots burnt on polling) and woken on completion
__device__ __forceinline__ void mbar_wait_parked(uint64_t* bar, uint32_t parity) {
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
                 :: "r"(smem_u32(bar)), "r"(parity), "r"(0x989680) : "memory");
}
template <int NREG> __device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" :: "n"(NREG)); }
template <int NREG> __device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" :: "n"(NREG)); }

// generic-proxy writes (st.shared) -> visible to the async proxy (TMA / tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load: box lands at `dst` (swizzled as the tensor map says), completes `bytes` on `bar`.
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// L2 eviction-priority policies (createpolicy) and the loads that carry one
__device__ __forceinline__ uint64_t l2_policy_evict_first()  { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t l2_policy_evict_last()   { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t l2_policy_evict_normal() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ void tma_load_2d_hint(void* dst, const CUtensorMap* m, int c0, int c1, uint64_t* bar, uint64_t pol) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
                 :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(pol) : "memory");
}
__device__ __forceinline__ void tma_load_3d_hint(void* dst, const CUtensorMap* m, int c0, int c1, int c2, uint64_t* bar, uint64_t pol) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
                 :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(pol) : "memory");
}
__device__ __forceinline__ float4 ld_stream_f4_hint(const float* p, uint64_t pol) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float ld_f32_hint(const float* p, uint64_t pol) {
    float r; asm volatile("ld.global.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol) : "memory"); return r;
}
__device__ __forceinline__ void st_f32_hint(float* p, float v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" :: "l"(p), "f"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ float4 ldg4_hint(const float* p, uint64_t pol) {
    float4 r;
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
    return r;
}

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, int c0, int c1, int c2, int c3, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

// L2 prefetch of a contiguous range (no destination, no completion)
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {      // bytes % 16 == 0, p 16-B aligned
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(p), "r"(bytes) : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
template <int COLS> __device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {      // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(dst_smem)), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS> __device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {        // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], kind::tf32, issued by ONE thread.
__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on `bar` once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 columns of 32-bit: thread i of the warp gets TMEM lane (lane_base + i), columns col..col+31
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float* out) {
    uint32_t r[32];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) out[i] = __uint_as_float(r[i]);
}

// 32 lanes x 16 columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, float* out) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) out[i] = __uint_as_float(r[i]);
}

// ---------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor for an MN-major 32-bit (tf32) operand.  The only canonical layout the
// tensor core accepts for MN-major tf32 is SWIZZLE_128B with 32-byte atomicity (LayoutType 1,
// "128B_BASE32B"; TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B):
//   Swizzle<2,5,2> o ((T,8,m),(4,k)) : ((1,T,LBO),(8T,SBO))   (T = 4 fp32)
// i.e. atoms of 4 k-rows x 128 B (32 MN-elements), row pitch 128 B, 32-byte chunk index ^= (row & 3);
// next 32 MN-elements at +LBO bytes, next 4 k-rows at +SBO bytes.  Atom bases 512-B aligned.
__device__ __forceinline__ uint64_t make_desc_mn_sw128_32b(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;                      // descriptor version 1 (sm_100)
    d |= (uint64_t)1 << 61;                      // LayoutType::SWIZZLE_128B_BASE32B
    return d;
}
// Instruction descriptor: kind::tf32, fp32 accumulate, A and B both MN-major, M x N.
__host__ __device__ constexpr uint32_t make_idesc_tf32_mn_mn(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// Byte offset of (row r, 16-byte chunk c in 0..7) inside one [rows][128 B] block in the 128B / 32B-atom swizzle
// (block base 512-B aligned): the 32-byte chunk index (c >> 1) is XORed with (r & 3).
__device__ __forceinline__ uint32_t sw128_32b_off(int r, int c) { return (uint32_t)(r * 128 + ((((c >> 1) ^ (r & 3)) << 5) | ((c & 1) << 4))); }

__device__ __forceinline__ float tf32_rna(float x) {          // round to nearest tf32 (10-bit mantissa), ties away
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}
// round-to-nearest (ties away) for an operand whose low 13 bits the tensor core ignores anyway: one integer add, no mask
__device__ __forceinline__ float tf32_rna_bits(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }
__device__ __forceinline__ float tf32_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
// Stochastic rounding of 4 values to tf32 with a dither hashed from `h` (the single-pass mode's basis tile: h mixes the iterate, the pixel
// and the column).  Truncation would bias the products (relH 1e-5); round-to-nearest is unbiased per launch (relH < 1e-6) but applies the
// SAME perturbation to the basis at every LM iteration, so its effect adds up coherently over a solve (W off by 1e-3 after 20 iterations).
// The dither is unbiased AND changes with the iterate, like the rounding of R does; it is a pure function of the inputs, so results stay
// bit-reproducible.
__device__ __forceinline__ float4 tf32_stochastic4(float4 v, uint32_t h) {
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15;
    uint32_t h2 = h * 0x846CA68Bu; h2 ^= h2 >> 16;
    return make_float4(__uint_as_float((__float_as_uint(v.x) + (h & 0x1fffu)) & 0xFFFFE000u),
                       __uint_as_float((__float_as_uint(v.y) + ((h >> 13) & 0x1fffu)) & 0xFFFFE000u),
                       __uint_as_float((__float_as_uint(v.z) + (h2 & 0x1fffu)) & 0xFFFFE000u),
                       __uint_as_float((__float_as_uint(v.w) + ((h2 >> 13) & 0x1fffu)) & 0xFFFFE000u));
}

}}  // namespace banet::tc
