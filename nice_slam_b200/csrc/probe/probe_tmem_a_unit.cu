// probe_tmem_a_unit.cu -- one real layer unit of the tile kernels (nsb_tile.cuh: mma_unit<4>): 3xTF32, M = 128, N = 32, K = 32, twelve
// tcgen05.mma (kind::tf32), B hi|lo from shared memory, with the A operand in three places:
//   form 0: A hi | lo in shared memory (K-major canonical tiles, as the kernels had it);
//   form 1: A hi and A lo in tensor memory (tcgen05.st.32x32b.x16, one row per thread, 8 columns per k-step);
//   form 2: A hi in tensor memory, A lo in shared memory.
// CTA = 256 threads (row = tid & 127, 16 columns per thread, the tile kernels' mapping), 256 TMEM columns.  Each form is timed (clock64) as
//   * round trip: write A -> publish (fence + one mbarrier arrival per warp) -> warp 0 issues the unit -> commit -> wait -> tcgen05.ld of D,
//   * throughput: warp 0 issues kUnits units back to back into the same D, one commit, wait,
// with one CTA per SM (160 KB of shared memory: nothing else fits) and with two co-resident CTAs per SM (110 KB, the forward tile kernel's footprint).
// The three forms must give bit-identical D (same products, same order, same accumulator); D is also checked against an fp64 reference.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o probe_tmem_a_unit probe_tmem_a_unit.cu
#include <cstdio>
#include <cstdint>
#include <cstring>
#include <cmath>
#include <vector>
#include <cuda_runtime.h>

constexpr int TM = 128, K = 32, N = 32, kReps = 64, kUnits = 64;
constexpr uint32_t kCols = 256, kAHi = 192, kALo = 224;           // TMEM: D = [0, 32), A hi = [192, 224), A lo = [224, 256)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t make_desc(const float* smem, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_u32(smem) >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
__device__ __forceinline__ int canon_q(int r, int kq) { return ((r >> 3) * (K >> 2) + kq) * 32 + (r & 7) * 4; }
__device__ __forceinline__ float to_tf32(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const long long t0 = clock64();
  for (;;) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (ok) return;
    if (clock64() - t0 > 4000000000ll) { printf("probe: mbarrier wait timed out (block %d)\n", blockIdx.x); __trap(); }
  }
}
__device__ __forceinline__ void mma_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d), "l"(a), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d), "r"(a), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
               ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]),
                 "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  for (int j = 0; j < 16; j++) v[j] = __uint_as_float(r[j]);
}

// the twelve MMAs of one unit: per k-step lo*hi, hi*lo, hi*hi (the kernels' order)
template <int FORM>
__device__ __forceinline__ void issue_unit(uint32_t d, uint64_t ah, uint64_t al, uint32_t th, uint32_t tl, uint64_t bh, uint64_t bl, uint32_t idesc, uint32_t acc) {
#pragma unroll
  for (int ks = 0; ks < K / 8; ks++) {
    const uint32_t a0 = ks == 0 ? acc : 1u;
    if (FORM == 0) { mma_ss(d, al + 16u * ks, bh + 16u * ks, idesc, a0); mma_ss(d, ah + 16u * ks, bl + 16u * ks, idesc, 1u); mma_ss(d, ah + 16u * ks, bh + 16u * ks, idesc, 1u); }
    if (FORM == 1) { mma_ts(d, tl + 8u * ks, bh + 16u * ks, idesc, a0); mma_ts(d, th + 8u * ks, bl + 16u * ks, idesc, 1u); mma_ts(d, th + 8u * ks, bh + 16u * ks, idesc, 1u); }
    if (FORM == 2) { mma_ss(d, al + 16u * ks, bh + 16u * ks, idesc, a0); mma_ts(d, th + 8u * ks, bl + 16u * ks, idesc, 1u); mma_ts(d, th + 8u * ks, bh + 16u * ks, idesc, 1u); }
  }
}

// cyc[block][form][0 = round trip, 1 = per unit back to back], smid[block]; D of block 0 per form
template <int FORM>
__device__ void run_form(float* a_s, float* b_s, uint64_t* bars, uint32_t tmem, const float (&av)[16], float* D, long long* cyc, uint32_t& par_ready, uint32_t& par_done) {
  const int tid = threadIdx.x, warp = tid >> 5, row = tid & (TM - 1), cg = tid >> 7;
  const uint32_t my = ((uint32_t)((warp & 3) * 32) << 16) + 16u * cg;
  const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
  const uint64_t ah = make_desc(a_s, 128u, 8u * 128u), al = ah + (uint64_t)((TM * K * 4) >> 4);
  const uint64_t bh = make_desc(b_s, 128u, 8u * 128u), bl = bh + (uint64_t)((N * K * 4) >> 4);
  float hi[16], lo[16];
  for (int j = 0; j < 16; j++) { hi[j] = to_tf32(av[j]); lo[j] = av[j] - hi[j]; }
  long long t_begin = 0;
  float dv[16];
  for (int rep = 0; rep <= kReps; rep++) {
    if (rep == 1) { __syncthreads(); t_begin = clock64(); }
    if (FORM == 0 || FORM == 2)
      for (int k = 0; k < 4; k++) {
        const int q = canon_q(row, 4 * cg + k);
        if (FORM == 0) *reinterpret_cast<float4*>(a_s + q) = make_float4(hi[4 * k], hi[4 * k + 1], hi[4 * k + 2], hi[4 * k + 3]);
        *reinterpret_cast<float4*>(a_s + TM * K + q) = make_float4(lo[4 * k], lo[4 * k + 1], lo[4 * k + 2], lo[4 * k + 3]);
      }
    if (FORM == 1 || FORM == 2) tmem_st16(tmem + kAHi + my, hi);
    if (FORM == 1) tmem_st16(tmem + kALo + my, lo);
    if (FORM == 0 || FORM == 2) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (FORM == 1 || FORM == 2) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if ((tid & 31) == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bars)) : "memory");
    if (warp == 0) {
      mbar_wait(bars, par_ready);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      uint32_t e;
      asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.b32 %0, 1, 0, q;\n\t}" : "=r"(e) :: "memory");
      if (e) {
        issue_unit<FORM>(tmem, ah, al, tmem + kAHi, tmem + kALo, bh, bl, idesc, 0u);
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bars + 1)) : "memory");
      }
      __syncwarp();
    }
    par_ready ^= 1u;
    mbar_wait(bars + 1, par_done); par_done ^= 1u;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    tmem_ld16(tmem + my, dv);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  const long long rt = (clock64() - t_begin) / kReps;
  if (blockIdx.x == 0) for (int j = 0; j < 16; j++) D[(FORM * TM + row) * N + 16 * cg + j] = dv[j];
  // throughput: the operands are in place (last round trip); warp 0 issues kUnits units into D
  long long tp = 0;
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const long long t0 = clock64();
    uint32_t e;
    asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.b32 %0, 1, 0, q;\n\t}" : "=r"(e) :: "memory");
    if (e) {
      for (int u = 0; u < kUnits; u++) issue_unit<FORM>(tmem, ah, al, tmem + kAHi, tmem + kALo, bh, bl, idesc, 0u);
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bars + 1)) : "memory");
    }
    __syncwarp();
    mbar_wait(bars + 1, par_done);
    tp = (clock64() - t0) / kUnits;
  }
  par_done ^= 1u;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (tid == 0) { cyc[(blockIdx.x * 3 + FORM) * 2] = rt; cyc[(blockIdx.x * 3 + FORM) * 2 + 1] = tp; }
}

__global__ void __launch_bounds__(256, 2) probe_kernel(const float* __restrict__ A, const float* __restrict__ W, float* __restrict__ D, long long* __restrict__ cyc, int* __restrict__ smid) {
  extern __shared__ __align__(1024) unsigned char smem[];
  float* a_s = reinterpret_cast<float*>(smem);            // A hi | lo  [128 x 32] canonical, 32 KB
  float* b_s = a_s + 2 * TM * K;                           // B hi | lo  [32 x 32] canonical, 8 KB
  __shared__ __align__(8) uint64_t bars[2];                // 0: A ready (8 warp arrivals), 1: MMAs done (commit)
  __shared__ uint32_t tmem_s;
  const int tid = threadIdx.x, warp = tid >> 5, row = tid & (TM - 1), cg = tid >> 7;
  for (int i = tid; i < N * K; i += blockDim.x) {
    const int n = i / K, k = i % K;
    const float w = W[i], h = to_tf32(w);
    const int q = canon_q(n, k >> 2) + (k & 3);
    b_s[q] = h; b_s[N * K + q] = w - h;
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_s)), "r"(kCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bars)), "r"(8u) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bars + 1)), "r"(1u) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    uint32_t s; asm volatile("mov.u32 %0, %%smid;" : "=r"(s)); smid[blockIdx.x] = (int)s;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_s;
  float av[16];
  for (int j = 0; j < 16; j++) av[j] = A[row * K + 16 * cg + j];
  uint32_t pr = 0, pd = 0;
  run_form<0>(a_s, b_s, bars, tmem, av, D, cyc, pr, pd);
  run_form<1>(a_s, b_s, bars, tmem, av, D, cyc, pr, pd);
  run_form<2>(a_s, b_s, bars, tmem, av, D, cyc, pr, pd);
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kCols) : "memory");
}

int main() {
  cudaDeviceProp prop; cudaGetDeviceProperties(&prop, 0);
  int clk = 0; cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, 0);
  printf("device: %s, %d SMs, max SM clock %d MHz\n", prop.name, prop.multiProcessorCount, clk / 1000);
  std::vector<float> hA(TM * K), hW(N * K), hD(3 * TM * N);
  uint32_t s = 4242u;
  auto rnd = [&]() { s = s * 1664525u + 1013904223u; return ((float)(s >> 8) / 16777216.0f - 0.5f) * 4.0f; };      // full fp32 mantissas
  for (auto& x : hA) x = rnd();
  for (auto& x : hW) x = rnd();
  const int nsm = prop.multiProcessorCount, maxb = 2 * nsm;
  float *dA, *dW, *dD; long long* dC; int* dS;
  cudaMalloc(&dA, hA.size() * 4); cudaMalloc(&dW, hW.size() * 4); cudaMalloc(&dD, hD.size() * 4);
  cudaMalloc(&dC, (size_t)maxb * 6 * 8); cudaMalloc(&dS, (size_t)maxb * 4);
  cudaMemcpy(dA, hA.data(), hA.size() * 4, cudaMemcpyHostToDevice); cudaMemcpy(dW, hW.data(), hW.size() * 4, cudaMemcpyHostToDevice);
  cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
  const char* fname[3] = {"A hi|lo in shared memory", "A hi and lo in TMEM", "A hi in TMEM, lo in shared"};
  for (int mode = 0; mode < 2; mode++) {
    const int blocks = mode == 0 ? nsm : 2 * nsm;
    const size_t sm = mode == 0 ? 160 * 1024 : 110 * 1024;
    probe_kernel<<<blocks, 256, sm>>>(dA, dW, dD, dC, dS);
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("kernel status: %s\n", cudaGetErrorString(e)); return 1; }
    std::vector<long long> c((size_t)blocks * 6); std::vector<int> sid(blocks);
    cudaMemcpy(c.data(), dC, c.size() * 8, cudaMemcpyDeviceToHost); cudaMemcpy(sid.data(), dS, sid.size() * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(hD.data(), dD, hD.size() * 4, cudaMemcpyDeviceToHost);
    std::vector<int> per(nsm, 0);
    for (int b = 0; b < blocks; b++) per[sid[b]]++;
    int shared_sms = 0; for (int x : per) shared_sms += x == 2;
    printf("\n%d CTA(s) per SM requested: %d CTAs, %zu KB shared memory each; SMs running two CTAs: %d of %d\n", mode + 1, blocks, sm / 1024, shared_sms, nsm);
    for (int f = 0; f < 3; f++) {
      double rt = 0, tp = 0; long long rmin = 1ll << 60, rmax = 0, tmin = 1ll << 60, tmax = 0;
      for (int b = 0; b < blocks; b++) {
        const long long r = c[(b * 3 + f) * 2], t = c[(b * 3 + f) * 2 + 1];
        rt += r; tp += t; rmin = r < rmin ? r : rmin; rmax = r > rmax ? r : rmax; tmin = t < tmin ? t : tmin; tmax = t > tmax ? t : tmax;
      }
      printf("  form %d %-28s  round trip %6.0f cycles (min %lld max %lld)   back-to-back %6.0f cycles per unit (min %lld max %lld)\n",
             f, fname[f], rt / blocks, rmin, rmax, tp / blocks, tmin, tmax);
    }
    double err = 0, mx = 0; int diff12 = 0;
    for (int r = 0; r < TM; r++) for (int n = 0; n < N; n++) {
      double ref = 0; for (int k = 0; k < K; k++) ref += (double)hA[r * K + k] * (double)hW[n * K + k];
      err = fmax(err, fabs(hD[r * N + n] - ref)); mx = fmax(mx, fabs(ref));
      for (int f = 1; f < 3; f++) diff12 += memcmp(&hD[r * N + n], &hD[(f * TM + r) * N + n], 4) != 0;
    }
    printf("  form 0 vs fp64: max abs err %.3e (max |ref| %.2f); elements of forms 1, 2 that differ bitwise from form 0: %d of %d\n", err, mx, diff12, 2 * TM * N);
  }
  return 0;
}
