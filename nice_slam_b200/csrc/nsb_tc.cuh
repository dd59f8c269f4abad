// nsb_tc.cuh -- tcgen05 primitives of the tensor-core tile kernels (nsb_tile.cuh): the 3xTF32 operand split, canonical-tile addressing,
// shared-memory descriptors and the kind::tf32 MMA, plus the optional phase-timing counters.
//
// Why 3xTF32: plain TF32 operands miss the 1e-4 parity bar by an order of magnitude (probe: 3e-4 relative on a single
// 32-wide GEMM); splitting every operand into hi = the 19 bits the tensor core reads, lo = x - hi (exact) and issuing
// lo*hi + hi*lo + hi*hi gives fp32-level results (probe_tcgen05.cu: 6e-6 abs on |ref| <= 20, same as an FP32 FMA chain).
//
// Operand tiles live in shared memory in the canonical K-major no-swizzle UMMA layout  [row/8][k/4][row%8][k%4]  (core matrix = 8 rows x 16 B).
#pragma once

namespace nsb {
namespace tc {

// Optional phase timing (make TIMING=1 -> libnsb_timing.so, tools/phase_timing.py): thread 0 of CTA 0 accumulates the cycles between
// consecutive marks per phase id; read back with nsb_debug_phases().  Compiled out of the product library.
#ifdef NSB_PHASE_TIMING
__device__ long long g_phase[64];
__device__ long long g_phase_last;
#define NSB_PH(id) do { if (blockIdx.x == 0 && threadIdx.x == 0) { const long long c_ = clock64(); ::nsb::tc::g_phase[id] += c_ - ::nsb::tc::g_phase_last; ::nsb::tc::g_phase_last = c_; } } while (0)
#define NSB_PH_RESET() do { if (blockIdx.x == 0 && threadIdx.x == 0) ::nsb::tc::g_phase_last = clock64(); } while (0)
#else
#define NSB_PH(id) do { } while (0)
#define NSB_PH_RESET() do { } while (0)
#endif

constexpr int TM = 128;                 // points per tile

// hi part of the 3xTF32 split: the top 19 bits (sign, exponent, 10 mantissa bits) -- exactly what the tensor core reads of
// an fp32 word.  Truncation instead of cvt.rna keeps x = hi + lo exact (lo has <= 13 significant bits, of which the MMA
// drops <= 3: 2^-21 |x|) and is one full-rate LOP instead of a quarter-rate conversion.
__device__ __forceinline__ float to_tf32(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

// element (row r, k) of a canonical tile of width K floats
__device__ __forceinline__ int canon_q(int r, int kq, int K) { return ((r >> 3) * (K >> 2) + kq) * 32 + (r & 7) * 4; }

__device__ __forceinline__ void put4(float* hi, float* lo, int r, int kq, int K, float4 v) {
  const int idx = canon_q(r, kq, K);
  float4 h, l;
  h.x = to_tf32(v.x); h.y = to_tf32(v.y); h.z = to_tf32(v.z); h.w = to_tf32(v.w);
  l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;   // exact; the MMA ignores the 13 low bits (<= 2^-21 |v|)
  *reinterpret_cast<float4*>(hi + idx) = h;
  *reinterpret_cast<float4*>(lo + idx) = l;
}

__device__ __forceinline__ uint64_t make_desc(const float* smem, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_u32(smem) >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;                         // descriptor version (Blackwell); layout_type 0 = no swizzle
  return d;
}
__device__ __forceinline__ uint32_t make_idesc(int M, int N) {      // D=F32, A=B=TF32, both K-major
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
// One lane of a CONVERGED warp (the MMA issue path runs in all lanes of warp 0: operands stay warp-uniform -> uniform registers, no per-MMA
// ELECT / R2UR.BROADCAST waterfall as when a single divergent thread issues; see nsb_tile.cuh).
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.b32 %0, 1, 0, q;\n\t}" : "=r"(p) :: "memory");
  return p;
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

}  // namespace tc
}  // namespace nsb
