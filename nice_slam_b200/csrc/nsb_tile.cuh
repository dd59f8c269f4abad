// nsb_tile.cuh -- tile-centric tensor-core kernels (round 2): two co-resident CTAs per SM, warp-specialised control warp.
//
// Work item = (128-point TILE of the batch's global (ray, sample) order, decoder).  A tile is independent of ray boundaries, so every
// tile is full (no padding rows for S = 48), small batches spread over all SMs (200 rays x 48 x 3 decoders = 225 items, all resident
// at once at two CTAs per SM) and the shared-memory footprint no longer grows with the number of samples per ray.  What needs whole
// rays -- compositing in the forward, the ray-gradient sums in the backward -- is done by the CTA that COMPLETES a ray: every item
// bumps the counters of the rays it touches after publishing its per-point results, the CTA that brings a counter to its target value
// composites / reduces that ray from global (L2) scratch in a fixed order (bit-reproducible), and resets the counter.
//
// CTA = 256 threads = two threads per tile row: thread tid owns row tid & 127 and the 16-column half tid >> 7 of every 32-wide epilogue
// (warp w touches TMEM lanes [32 (w & 3), +32) = its rows).  Thread 0 is also the TMA producer and the tcgen05.mma issuer (a ninth, dedicated
// control warp was measured first: registers are allocated per 4-warp granule, so 9 warps cost 12 warps' worth and only ONE CTA fitted per SM):
//   * weights stream through a 4-slot ring of operand UNITS (pre-split hi|lo canonical tiles, consumption order, nsb_common.cuh) with full
//     (TMA -> issuer) and empty (tcgen05.commit -> producer) mbarriers: three units of prefetch, no thread touches a weight;
//   * activations ping-pong between two 32 KB operand buffers; warps publish a tile by fence.proxy.async + one mbarrier.arrive per warp
//     (A_ready); thread 0 waits for the eight arrivals, issues the group's MMAs and commits to the buffer's `done` barrier -- there is no
//     __syncthreads in the chain, and the gather / embedding of tile n+1 overlaps the MMAs of tile n.  Operands that the epilogue threads
//     produce row by row (the forward's hidden-layer inputs, the hi parts of the backward's G / DU) go to TENSOR memory instead
//     (tcgen05.st, tcgen05.wait::st before the arrival): shared-memory operand reads are what bound the MMA groups.
// Shared memory: 64 KB activations + 40 KB ring + 6 KB headers + < 6 KB state <= 113 KB, TMEM 256 columns -> two CTAs per SM, i.e. two
// tiles in flight per SM with the hardware interleaving their (latency-bound) chains.
//
// Arithmetic is that of nsb_tc.cuh (3xTF32 split, same operand order), so results match the round-1 kernels to rounding of the output
// layer's partial sums.
#pragma once

namespace nsb {
namespace tl {

using tc::TM;
constexpr int kThreads = 256;                 // 8 warps: register allocation is per 4-warp granule, a ninth (control) warp would cost 12 warps' worth
constexpr int kEpiThreads = kThreads;
constexpr int kCG = 2, kCW = 16, kKQ = 4;      // column halves per row, columns per thread, 16-byte chunks per thread
constexpr uint32_t kTmemCols = 256;
constexpr int kSlots = 4;
constexpr int kSlotFloatsFwd = 2560;          // 10 KB: the largest forward unit (fc_c: [160 x 8] hi|lo)
constexpr int kSlotFloatsBwd = 2048;          //  8 KB: every backward unit is [32 x 32] hi|lo
constexpr int kABufFloats = 2 * TM * 32;      // one [128 x 32] operand tile, hi|lo = 32 KB
constexpr int kMaxTileRays = 18;              // rays one tile can touch (S >= 8)
constexpr int kMinSamples = 8;
constexpr long long kWaitCycles = 4000000000ll;      // ~2 s: a wait that long is a protocol bug -> trap instead of hanging the GPU

// barrier indices
enum { B_FULL = 0, B_EMPTY = 4, B_HDR = 8, B_AREADY = 10, B_DONE = 12, kNumBars = 14 };

__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// non-blocking poll (try_wait may suspend the thread for a hardware-defined time before it answers "not yet")
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// bounded wait: a protocol error traps (the launch fails with an error) instead of hanging the device
__device__ __forceinline__ void mbar_wait_b(uint64_t* bar, uint32_t parity) {
  if (mbar_try(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try(bar, parity)) {
    if (clock64() - t0 > kWaitCycles) { printf("nsb: mbarrier wait timed out (block %d thread %d bar %p parity %u)\n", blockIdx.x, threadIdx.x, (void*)bar, parity); __trap(); }
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void epi_sync() { __syncthreads(); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int j = 0; j < 16; j++) v[j] = __uint_as_float(r[j]);
}
// this thread's 16 columns of its lane (row); ordered before a tcgen05.mma of another thread by tcgen05.wait::st + publish_tmem
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
               ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]),
                 "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]) : "memory");
}

// ---- shared memory -------------------------------------------------------------------------------------------------------------
struct TileSmem {
  float* a[2];        // operand buffers
  float* ring;        // kSlots x slot_floats
  int slot_floats;
  float* hdr;         // 2 x kHdrFloats
  uint64_t* bars;
  uint32_t* tmem;
  unsigned char* extra;      // kernel-specific state behind the common part
};
__host__ __device__ constexpr size_t common_bytes(bool bwd) {     // + barriers (14 x 8) + TMEM slot
  return (2 * (size_t)kABufFloats + (size_t)kSlots * (bwd ? kSlotFloatsBwd : kSlotFloatsFwd) + 2 * kHdrFloats) * 4 + 128;
}
__device__ __forceinline__ void carve(unsigned char* base, TileSmem& t, bool bwd) {
  float* f = reinterpret_cast<float*>(base);
  t.a[0] = f; f += kABufFloats; t.a[1] = f; f += kABufFloats;
  t.slot_floats = bwd ? kSlotFloatsBwd : kSlotFloatsFwd;
  t.ring = f; f += kSlots * t.slot_floats;
  t.hdr = f; f += 2 * kHdrFloats;
  t.bars = reinterpret_cast<uint64_t*>(f);
  t.tmem = reinterpret_cast<uint32_t*>(f + 2 * kNumBars);
  t.extra = base + common_bytes(bwd);
}

// ---- unit sequences of the v2 operand images (nsb_common.cuh: op2_*) ---------------------------------------------------------------
__device__ __forceinline__ int fwd_units(int lv) { return op2_fwd_units(lv); }
__device__ __forceinline__ int bwd_units(int lv) { return op2_bwd_units(lv); }

// Producer cursor: walks the units of the decoders this CTA evaluates, in consumption order.
struct Loader {
  const KParams* P;
  int q, q1;          // current / end decoder slot
  int k;              // unit index inside decoder q
  uint32_t loaded;    // units issued so far (global sequence number of the next one)
  int mode;           // 0 = forward (3xTF32 units), 1 = backward, 2 = forward with FP16 hi|lo units (op3_*)
};
__device__ __forceinline__ bool loader_done(const Loader& L) { return L.q >= L.q1; }
__device__ __forceinline__ void loader_issue(Loader& L, const TileSmem& t) {
  const int lv = L.P->dec[L.q];
  const float* img = L.P->in.packed[lv] + (L.mode == 1 ? op2_bwd_offset(lv) : L.mode == 2 ? op3_fwd_offset(lv) : op2_fwd_offset(lv));
  int off, floats, n_units;
  if (L.mode == 1) { off = L.k * 2048; floats = 2048; n_units = bwd_units(lv); }
  else if (L.mode == 2) {
    const int nfc = op3_fc_units(lv), nl0 = op_nblk(lv);
    if (L.k < nfc) { off = L.k * 2560; floats = 2560; }
    else if (L.k < nfc + nl0) { off = nfc * 2560 + (L.k - nfc) * 2048; floats = 2048; }
    else { off = nfc * 2560 + nl0 * 2048 + (L.k - nfc - nl0) * 1024; floats = 1024; }
    n_units = op3_fwd_units(lv);
  } else {
    const int nfc = op2_fc_units(lv);
    if (L.k < nfc) { off = L.k * 2560; floats = 2560; } else { off = nfc * 2560 + (L.k - nfc) * 2048; floats = 2048; }
    n_units = fwd_units(lv);
  }
  const int slot = L.loaded & (kSlots - 1);
  uint64_t* bar = t.bars + B_FULL + slot;
  mbar_expect_tx(bar, (uint32_t)floats * 4u);
  tma_bulk_g2s(t.ring + slot * t.slot_floats, img + off, (uint32_t)floats * 4u, bar);
  L.loaded++;
  if (++L.k == n_units) { L.k = 0; L.q++; }
}
// refill one slot if a unit is pending and its slot's previous occupant has been issued (blocking on that unit's MMAs)
__device__ __forceinline__ bool loader_refill(Loader& L, const TileSmem& t, uint32_t issued) {
  if (loader_done(L) || L.loaded >= issued + kSlots) return false;
  if (L.loaded >= kSlots) { const uint32_t prev = L.loaded - kSlots; mbar_wait_b(t.bars + B_EMPTY + (prev & (kSlots - 1)), (prev >> 2) & 1u); }
  loader_issue(L, t);
  return true;
}
// request every unit whose slot is already free (non-blocking)
__device__ __forceinline__ void loader_top_up(Loader& L, const TileSmem& t, uint32_t issued) {
  while (!loader_done(L) && L.loaded < issued + kSlots) {
    if (L.loaded >= kSlots) { const uint32_t prev = L.loaded - kSlots; if (!mbar_test(t.bars + B_EMPTY + (prev & (kSlots - 1)), (prev >> 2) & 1u)) return; }
    loader_issue(L, t);
  }
}
__device__ __forceinline__ void load_header(const KParams& P, const TileSmem& t, int lv, int hb) {
  uint64_t* bar = t.bars + B_HDR + hb;
  mbar_expect_tx(bar, kHdrFloats * 4u);
  tma_bulk_g2s(t.hdr + hb * kHdrFloats, P.in.packed[lv] + op_fwd_offset(lv), kHdrFloats * 4u, bar);
}

// Issuer state (control thread)
struct Issuer {
  Loader L;
  uint32_t issued;    // units consumed so far
  uint32_t g;         // operand groups consumed so far (forward: buffer = g & 1)
};
// The issue path is executed by ALL lanes of warp 0, converged: everything that feeds a tcgen05.mma (descriptors, TMEM address, the
// counters `issued` / `g`) is computed identically in every lane from warp-uniform inputs, so ptxas keeps it in uniform registers and one
// elected lane issues the instruction.  (Issued from a single divergent thread, every MMA was wrapped in an ELECT / 5 x R2UR.BROADCAST /
// branch "waterfall": ~1 k cycles per 32 x 32 layer of twelve MMAs, 40 % of both kernels.)  Only the TMA producer bookkeeping (Loader) is
// lane 0's private, divergent state.
using tc::elect_one;
// wait for the operands of group `g` on A_ready[b]; while they are not there, lane 0 keeps the ring full
__device__ __forceinline__ void issuer_wait_operands(Issuer& I, const TileSmem& t, int b, uint32_t parity) {
  uint64_t* bar = t.bars + B_AREADY + b;
  const long long t0 = clock64();
  while (!mbar_test(bar, parity)) {                              // poll: the ring is topped up between polls
    if ((threadIdx.x & 31) == 0) loader_top_up(I.L, t, I.issued);
    if (clock64() - t0 > kWaitCycles) { printf("nsb: issuer timed out waiting for operands (block %d)\n", blockIdx.x); __trap(); }
  }
  tc::tc_fence_after();
}
// the unit the issuer is about to consume: make sure it was requested (lane 0), wait for it (all lanes), return its slot base
__device__ __forceinline__ const float* issuer_unit(Issuer& I, const TileSmem& t) {
  // (no __syncwarp anywhere in the issue path: elect.sync with the full member mask is itself the reconvergence point of the warp, and every
  // extra warp barrier / second elect per unit costs ~20-50 cycles on a path that handles up to six units per layer)
  if ((threadIdx.x & 31) == 0) {
    loader_top_up(I.L, t, I.issued);
    while (I.L.loaded <= I.issued) loader_refill(I.L, t, I.issued);
  }
  const int slot = I.issued & (kSlots - 1);
  mbar_wait_b(t.bars + B_FULL + slot, (I.issued >> 2) & 1u);
  return t.ring + slot * t.slot_floats;
}
__device__ __forceinline__ void issuer_group_done(const TileSmem& t, int bar) {
  if (elect_one()) tc::mma_commit(t.bars + bar);
}

// D[128 x N] (+)= A[:, ka0 .. ka0 + 8 ksteps) * B^T, 3xTF32.  A: [128 x 32] hi|lo tile; B: unit [N x KB] hi|lo, product starts at column kb0.
// The issuing thread is on the critical path of every layer step: descriptors are built once per unit and advanced by plain adds
// (one k-step of 8 floats = two 128-byte core matrices = +16 in the 16-byte-granular start-address field; shared memory < 256 KB, so the
// 14-bit field never carries).
// ... followed, in the same elected lane, by the commits that release the unit's ring slot (`empty`) and, for the last unit of a group, signal the
// group's completion (`done`, or nullptr)
template <int KSTEPS>
__device__ __forceinline__ void mma_unit(Issuer& I, const TileSmem& t, uint32_t d_tmem, const float* a, int ka0, const float* b, int N, int KB, int kb0, uint32_t& acc,
                                         uint64_t* done = nullptr) {
  const uint32_t idesc = tc::make_idesc(TM, N);
  const uint64_t ah = tc::make_desc(a + (ka0 >> 2) * 32, 128u, 8u * 128u);
  const uint64_t bh = tc::make_desc(b + (kb0 >> 2) * 32, 128u, (uint32_t)(KB >> 2) * 128u);
  const uint64_t al = ah + (uint64_t)((TM * 32 * 4) >> 4);
  const uint64_t bl = bh + (uint64_t)((N * KB * 4) >> 4);
  if (elect_one()) {
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ks++) {
      tc::mma_tf32(d_tmem, al + 16u * ks, bh + 16u * ks, idesc, ks == 0 ? acc : 1u);
      tc::mma_tf32(d_tmem, ah + 16u * ks, bl + 16u * ks, idesc, 1u);
      tc::mma_tf32(d_tmem, ah + 16u * ks, bh + 16u * ks, idesc, 1u);
    }
    tc::mma_commit(t.bars + B_EMPTY + (I.issued & (kSlots - 1)));
    if (done != nullptr) tc::mma_commit(done);
  }
  I.issued++;
  acc = 1u;
}
// The same unit (same three products, same order, same accumulator) with the A operand in TENSOR MEMORY: one row per lane, k-step ks at
// column +8 ks.  A hi is read from columns a_hi; A lo from columns a_lo, or -- a_lo_s != nullptr -- from the canonical shared-memory tile a_lo_s.
// Every N <= 64 MMA re-reads its whole [128 x 8] A slice, and the shared-memory operand reads are what bound the tensor pipe here
// (probe_tmem_a_unit.cu); tensor-memory A takes those bytes off shared memory.
__device__ __forceinline__ void mma_tf32_ta(uint32_t d_tmem, uint32_t a_tmem, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
               ::"r"(d_tmem), "r"(a_tmem), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
template <int KSTEPS>
__device__ __forceinline__ void mma_unit_ta(Issuer& I, const TileSmem& t, uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, const float* a_lo_s, const float* b, int N, int KB,
                                            uint32_t& acc, uint64_t* done = nullptr) {
  const uint32_t idesc = tc::make_idesc(TM, N);
  const uint64_t bh = tc::make_desc(b, 128u, (uint32_t)(KB >> 2) * 128u);
  const uint64_t bl = bh + (uint64_t)((N * KB * 4) >> 4);
  const uint64_t al = a_lo_s != nullptr ? tc::make_desc(a_lo_s, 128u, 8u * 128u) : 0ull;
  if (elect_one()) {
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ks++) {
      if (a_lo_s != nullptr) tc::mma_tf32(d_tmem, al + 16u * ks, bh + 16u * ks, idesc, ks == 0 ? acc : 1u);
      else mma_tf32_ta(d_tmem, a_lo + 8u * ks, bh + 16u * ks, idesc, ks == 0 ? acc : 1u);
      mma_tf32_ta(d_tmem, a_hi + 8u * ks, bl + 16u * ks, idesc, 1u);
      mma_tf32_ta(d_tmem, a_hi + 8u * ks, bh + 16u * ks, idesc, 1u);
    }
    tc::mma_commit(t.bars + B_EMPTY + (I.issued & (kSlots - 1)));
    if (done != nullptr) tc::mma_commit(done);
  }
  I.issued++;
  acc = 1u;
}

// ---- FP16 hi|lo forward (option fwd_f16) ------------------------------------------------------------------------------------------------------
// x = hi + lo with hi = fp16(x), lo = fp16(x - hi): 22 significant bits for |x| in [2^-3, 65504], an absolute error <= 2^-25 below (lo goes
// subnormal) -- the forward's operands (features, sin embedding, ReLU outputs, weights) are O(1) values, far inside the 1e-4 tolerance of the
// path.  kind::f16 contracts K = 16 per instruction: half the MMAs and half the shared-memory operand traffic of the 3xTF32 forward (which is
// what bounds the MMA phases: every N <= 64 MMA re-reads its [128 x K] A slice).  Conversions saturate (cvt.rn.satfinite): an operand beyond
// the fp16 range degrades instead of producing Inf/NaN.  The backward keeps 3xTF32 (gradients span far more than fp16's exponent range).
// 16-bit canonical K-major tile of width K halves: [row/8][k/8][row%8][k%8]; hi tile, then lo tile.
__device__ __forceinline__ uint32_t cvt_h2(float lo_elem, float hi_elem) {          // {fp16(lo_elem), fp16(hi_elem)} packed, saturating
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_elem), "f"(lo_elem));
  return r;
}
__device__ __forceinline__ void split_h2(float x, float y, uint32_t& h, uint32_t& l) {
  h = cvt_h2(x, y);
  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h));
  l = cvt_h2(x - f.x, y - f.y);
}
// four consecutive features (4-wide chunk kq of a 32-wide tile) of row r: 8 bytes in the hi tile, 8 in the lo tile
__device__ __forceinline__ void put4_h(float* tile, int r, int kq, const float4 v) {
  unsigned char* hi = reinterpret_cast<unsigned char*>(tile) + (((r >> 3) * 4 + (kq >> 1)) * 128 + (r & 7) * 16 + (kq & 1) * 8);
  uint2 h, l;
  split_h2(v.x, v.y, h.x, l.x); split_h2(v.z, v.w, h.y, l.y);
  *reinterpret_cast<uint2*>(hi) = h;
  *reinterpret_cast<uint2*>(hi + TM * 32 * 2) = l;
}
// this thread's 16 features (column group cg) of row r: two 16-byte chunks per tile
__device__ __forceinline__ void put16_h(float* tile, int r, int cg, const float (&v)[kCW]) {
#pragma unroll
  for (int c = 0; c < 2; c++) {
    unsigned char* hi = reinterpret_cast<unsigned char*>(tile) + (((r >> 3) * 4 + 2 * cg + c) * 128 + (r & 7) * 16);
    uint4 h, l;
    split_h2(v[8 * c], v[8 * c + 1], h.x, l.x); split_h2(v[8 * c + 2], v[8 * c + 3], h.y, l.y);
    split_h2(v[8 * c + 4], v[8 * c + 5], h.z, l.z); split_h2(v[8 * c + 6], v[8 * c + 7], h.w, l.w);
    *reinterpret_cast<uint4*>(hi) = h;
    *reinterpret_cast<uint4*>(hi + TM * 32 * 2) = l;
  }
}
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
// D[128 x N] (+)= A[:, ka0 .. ka0 + 16 KSTEPS) * B^T with the FP16 split.  A: [128 x 32] halves hi|lo; B: unit [N x KB] halves hi|lo.
// (one k-step = 16 halves = two 128-byte core matrices = +16 in the start-address field, as for tf32)
template <int KSTEPS>
__device__ __forceinline__ void mma_unit_h(Issuer& I, const TileSmem& t, uint32_t d_tmem, const float* a, int ka0, const float* b, int N, int KB, uint32_t& acc,
                                           uint64_t* done = nullptr) {
  const uint32_t idesc = (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);      // D = F32, A = B = F16, both K-major
  const uint64_t ah = tc::make_desc(a + (ka0 >> 3) * 32, 128u, 4u * 128u);
  const uint64_t bh = tc::make_desc(b, 128u, (uint32_t)(KB >> 3) * 128u);
  const uint64_t al = ah + (uint64_t)((TM * 32 * 2) >> 4);
  const uint64_t bl = bh + (uint64_t)((N * KB * 2) >> 4);
  if (elect_one()) {
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ks++) {
      mma_f16(d_tmem, al + 16u * ks, bh + 16u * ks, idesc, ks == 0 ? acc : 1u);
      mma_f16(d_tmem, ah + 16u * ks, bl + 16u * ks, idesc, 1u);
      mma_f16(d_tmem, ah + 16u * ks, bh + 16u * ks, idesc, 1u);
    }
    tc::mma_commit(t.bars + B_EMPTY + (I.issued & (kSlots - 1)));
    if (done != nullptr) tc::mma_commit(done);
  }
  I.issued++;
  acc = 1u;
}

// ---- epilogue-side helpers -------------------------------------------------------------------------------------------------------
// operands of this thread are written: make them visible to the async proxy, order earlier TMEM reads, arrive
__device__ __forceinline__ void publish(const TileSmem& t, int b) {
  fence_proxy_async(); tc::tc_fence_before();
  __syncwarp();                                                 // one arrival per warp (256 arrivals on one barrier word serialise)
  if ((threadIdx.x & 31) == 0) mbar_arrive(t.bars + B_AREADY + b);
}
// the same for operands of this thread written to tensor memory (and, SMEM, also to shared memory)
template <bool SMEM>
__device__ __forceinline__ void publish_tmem(const TileSmem& t, int b) {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  if (SMEM) fence_proxy_async();
  tc::tc_fence_before();
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(t.bars + B_AREADY + b);
}
// 3xTF32 split of this thread's 16 features (as tc::put4): hi = the bits the tensor core reads, lo = v - hi (exact)
__device__ __forceinline__ void split16(const float (&v)[kCW], float (&hi)[kCW], float (&lo)[kCW]) {
#pragma unroll
  for (int j = 0; j < kCW; j++) { hi[j] = tc::to_tf32(v[j]); lo[j] = v[j] - hi[j]; }
}
// 16 features (column half cg) of row r -> one canonical [128 x 32] tile
__device__ __forceinline__ void put16(float* tile, int r, int cg, const float (&v)[kCW]) {
#pragma unroll
  for (int k = 0; k < kKQ; k++) *reinterpret_cast<float4*>(tile + tc::canon_q(r, kKQ * cg + k, 32)) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
}
__device__ __forceinline__ void wait_group(const TileSmem& t, uint32_t m) {      // MMAs of operand group m (and all earlier ones) have completed
  mbar_wait_b(t.bars + B_DONE + (m & 1u), (m >> 1) & 1u);
  tc::tc_fence_after();
}

// 8 lanes per point, 4 points per pass: 32 channels of grid `g` -> [128 x 32] tile.  Warp w serves the rows of its lane quadrant (w & 3);
// the eight passes of a quadrant are split over the two warps that share it.  The loads of pass i+1 are issued before pass i is consumed
// (16 x 16-byte loads in flight per lane), corner offsets come from per-axis offsets (two adds per corner).
struct GatherPass {
  float4 v[8];
  float w[8];
  int src_lane;
};
template <bool FAST>
__device__ __forceinline__ void gather_issue(const nsb_grid& g, const float xn[3], int it, int lane, GatherPass& gp) {
  const int q = lane & 7;
  gp.src_lane = it * 4 + (lane >> 3);
  float x[3];
  x[0] = __shfl_sync(0xffffffffu, xn[0], gp.src_lane); x[1] = __shfl_sync(0xffffffffu, xn[1], gp.src_lane); x[2] = __shfl_sync(0xffffffffu, xn[2], gp.src_lane);
  const Tri t = make_tri(x, g.W, g.H, g.D);
  // branch-free clamped corners (tri_corner_clamped): the clamped upper corner carries weight exactly 0
  const long long ox[2] = {(long long)t.i0[0] * g.stride_w, (long long)min(t.i0[0] + 1, g.W - 1) * g.stride_w};
  const long long oy[2] = {(long long)t.i0[1] * g.stride_h, (long long)min(t.i0[1] + 1, g.H - 1) * g.stride_h};
  const long long oz[2] = {(long long)t.i0[2] * g.stride_d, (long long)min(t.i0[2] + 1, g.D - 1) * g.stride_d};
#pragma unroll
  for (int k = 0; k < 8; k++) gp.v[k] = grid_load4(g, oz[k >> 2] + oy[(k >> 1) & 1] + ox[k & 1], 4 * q, FAST);
  const float wxy[4] = {__fmul_rn(t.w0[0], t.w0[1]), __fmul_rn(t.w1[0], t.w0[1]), __fmul_rn(t.w0[0], t.w1[1]), __fmul_rn(t.w1[0], t.w1[1])};
#pragma unroll
  for (int k = 0; k < 8; k++) gp.w[k] = __fmul_rn(wxy[k & 3], (k & 4) ? t.w1[2] : t.w0[2]);      // == tri_weight(t, k)
}
template <bool H16 = false>
__device__ __forceinline__ void gather_consume(float* c_hi, float* c_lo, int qd, int lane, const GatherPass& gp) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const float w = gp.w[k];
    acc.x = fmaf(gp.v[k].x, w, acc.x); acc.y = fmaf(gp.v[k].y, w, acc.y); acc.z = fmaf(gp.v[k].z, w, acc.z); acc.w = fmaf(gp.v[k].w, w, acc.w);
  }
  if (H16) put4_h(c_hi, qd * 32 + gp.src_lane, lane & 7, acc);
  else tc::put4(c_hi, c_lo, qd * 32 + gp.src_lane, lane & 7, 32, acc);
}
// (the strided NCDHW form -- four scalar loads with 64-bit strides per corner -- is a separate, out-of-line copy: inlined next to the channels-last
// form at every unrolled corner it made up a third of the forward kernel's 19 k instructions, and instruction fetch shows up in the stall samples)
template <bool FAST, bool H16 = false>
__device__ __forceinline__ void gather_tile_t(const nsb_grid& g, float* c_hi, const float xn[3], int warp, int lane) {
  float* c_lo = c_hi + TM * 32;
  const int qd = warp & 3, it0 = (warp >> 2) * 4;
  if (FAST) {
    GatherPass A, B;
    gather_issue<true>(g, xn, it0, lane, A);
    gather_issue<true>(g, xn, it0 + 1, lane, B);
    gather_consume<H16>(c_hi, c_lo, qd, lane, A);
    gather_issue<true>(g, xn, it0 + 2, lane, A);
    gather_consume<H16>(c_hi, c_lo, qd, lane, B);
    gather_issue<true>(g, xn, it0 + 3, lane, B);
    gather_consume<H16>(c_hi, c_lo, qd, lane, A);
    gather_consume<H16>(c_hi, c_lo, qd, lane, B);
  } else {
#pragma unroll 1
    for (int it = it0; it < it0 + 4; it++) { GatherPass A; gather_issue<false>(g, xn, it, lane, A); gather_consume<H16>(c_hi, c_lo, qd, lane, A); }
  }
}
template <bool H16>
static __device__ __noinline__ void gather_tile_strided(const nsb_grid& g, float* c_hi, float x0, float x1, float x2, int warp, int lane) {
  const float xn[3] = {x0, x1, x2};
  gather_tile_t<false, H16>(g, c_hi, xn, warp, lane);
}
template <bool H16 = false>
__device__ __forceinline__ void gather_tile(const nsb_grid& g, float* c_hi, const float xn[3], int warp, int lane) {
  if (grid_fast(g)) gather_tile_t<true, H16>(g, c_hi, xn, warp, lane);
  else gather_tile_strided<H16>(g, c_hi, xn[0], xn[1], xn[2], warp, lane);
}
// this thread's 16 features of embedding block `blk` of its point -> [128 x 32] tile
template <bool H16 = false>
__device__ __forceinline__ void embed_tile(float* e_hi, const float* B, const float pf[3], int row, int cg, int blk) {
  float* e_lo = e_hi + TM * 32;
#pragma unroll
  for (int kq = kKQ * cg; kq < kKQ * cg + kKQ; kq++) {
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int f = 32 * blk + 4 * kq + j;
      float x = pf[0] * B[f]; x = fmaf(pf[1], B[kEmbPad + f], x); x = fmaf(pf[2], B[2 * kEmbPad + f], x);
      v[j] = f < kEmb ? __sinf(reduce_2pi(x)) : 0.0f;
    }
    if (H16) put4_h(e_hi, row, kq, make_float4(v[0], v[1], v[2], v[3]));
    else tc::put4(e_hi, e_lo, row, kq, 32, make_float4(v[0], v[1], v[2], v[3]));
  }
}

// ---- forward: what the issuing thread (thread 0) does after the CTA published operand group I.g --------------------------------------------
// TMEM: D1 = [0,32), D3 = [32,64) (layer 3; its skip part is accumulated while the embedding blocks are live), D2 = [64,224) (fc_c of the five layers),
// [224,256) = A lo of the hidden layers.  The A operand of layer i+1 (the ReLU output of layer i) never goes through shared memory (3xTF32 path):
// its hi part overwrites D2 slice i, whose last reader is epilogue i itself (the same lanes and columns, just before), its lo part goes to
// [224,256), whose last reader (layer i's MMAs) has completed when epilogue i starts.
constexpr uint32_t kFwdALo = 224u;
template <bool H16 = false>
__device__ __forceinline__ void issue_fc(Issuer& I, const TileSmem& t, uint32_t tmem, int half) {      // C tile `half` -> D2 += C * Wc^T (four K = 8 units)
  const int b = I.g & 1;
  issuer_wait_operands(I, t, b, (I.g >> 1) & 1u);
  if constexpr (H16) {                                           // two [160 x 16] FP16 units
    for (int u = 0; u < 2; u++) {
      const float* w = issuer_unit(I, t);
      uint32_t acc = (half == 0 && u == 0) ? 0u : 1u;
      mma_unit_h<1>(I, t, tmem + 64u, t.a[b], 16 * u, w, 160, 16, acc, u == 1 ? t.bars + B_DONE + b : nullptr);
    }
  } else {
    for (int u = 0; u < 4; u++) {
      const float* w = issuer_unit(I, t);
      uint32_t acc = (half == 0 && u == 0) ? 0u : 1u;
      mma_unit<1>(I, t, tmem + 64u, t.a[b], 8 * u, w, 160, 8, 0, acc, u == 3 ? t.bars + B_DONE + b : nullptr);
    }
  }
  I.g++;
}
template <bool H16 = false>
__device__ __forceinline__ void issue_l0(Issuer& I, const TileSmem& t, uint32_t tmem, int blk) {       // [D1 | D3] += E_blk * [W0_blk; W3E_blk]^T   (coarse: E = C)
  const int b = I.g & 1;
  issuer_wait_operands(I, t, b, (I.g >> 1) & 1u);
  if constexpr (H16) {                                           // one [64 x 32] FP16 unit
    const float* w = issuer_unit(I, t);
    uint32_t acc = blk == 0 ? 0u : 1u;
    mma_unit_h<2>(I, t, tmem, t.a[b], 0, w, 64, 32, acc, t.bars + B_DONE + b);
  } else {
    for (int h = 0; h < 2; h++) {
      const float* w = issuer_unit(I, t);
      uint32_t acc = (blk == 0 && h == 0) ? 0u : 1u;
      mma_unit<2>(I, t, tmem, t.a[b], 16 * h, w, 64, 16, 0, acc, h == 1 ? t.bars + B_DONE + b : nullptr);
    }
  }
  I.g++;
}
template <bool H16 = false>
__device__ __forceinline__ void issue_h(Issuer& I, const TileSmem& t, uint32_t tmem, int i) {          // layer i (1..4) from the H tile of layer i-1
  const int b = I.g & 1;
  issuer_wait_operands(I, t, b, (I.g >> 1) & 1u);
  const float* w = issuer_unit(I, t);
  uint32_t acc = i == 3 ? 1u : 0u;
  if (H16) mma_unit_h<2>(I, t, i == 3 ? tmem + 32u : tmem, t.a[b], 0, w, 32, 32, acc, t.bars + B_DONE + b);
  else mma_unit_ta<4>(I, t, i == 3 ? tmem + 32u : tmem, tmem + 64u + 32u * (i - 1), tmem + kFwdALo, nullptr, w, 32, 32, acc, t.bars + B_DONE + b);
  I.g++;
}

// ---- forward of one decoder: epilogue side.  n = operand-group counter (same sequence as the issuer's).  out[] = decoder outputs of this row.
template <bool H16 = false>
__device__ __forceinline__ void epi_forward(const KParams& P, const TileSmem& t, Issuer& I, int lv, const PointGeom& G, uint32_t tmem, uint32_t& n, int hb, uint32_t hdr_parity,
                                            float (&out)[4], uint32_t* __restrict__ gmask, float* acts = nullptr) {
  const int row = threadIdx.x & (TM - 1), cg = threadIdx.x >> 7, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool t0 = threadIdx.x < 32;                            // the issuing WARP (converged): after every publish it waits for the other warps and issues the group's MMAs
  const bool xyz = lv != 0;
  const int cd = op_cd(lv), no = lv == 3 ? 4 : 1;
  const uint32_t my = ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(kCW * cg);
  const uint32_t d1 = tmem + my, d3 = tmem + 32u + my, d2 = tmem + 64u + my;
  const float* hdr = t.hdr + hb * kHdrFloats;
  if (xyz) {
    for (int half = 0; half < cd / 32; half++) {
      if (n >= 2) wait_group(t, n - 2);
      if (threadIdx.x == 0) loader_top_up(I.L, t, I.issued);     // request whatever fits the ring before the long gather
      gather_tile<H16>(P.in.grid[half == 0 ? lv : 1], t.a[n & 1], G.xn, warp, lane);
      NSB_PH(1);
      publish(t, n & 1); n++;
      if (t0) issue_fc<H16>(I, t, tmem, half);
      NSB_PH(2);
    }
    mbar_wait_b(t.bars + B_HDR + hb, hdr_parity);
    for (int blk = 0; blk < 3; blk++) {
      if (n >= 2) wait_group(t, n - 2);
      if (threadIdx.x == 0) loader_top_up(I.L, t, I.issued);
      NSB_PH(6);
      embed_tile<H16>(t.a[n & 1], hdr + 464, G.pf, row, cg, blk);
      NSB_PH(3);
      publish(t, n & 1); n++;
      if (t0) issue_l0<H16>(I, t, tmem, blk);
      NSB_PH(4);
    }
  } else {
    if (n >= 2) wait_group(t, n - 2);
    gather_tile<H16>(P.in.grid[0], t.a[n & 1], G.xnc, warp, lane);
    publish(t, n & 1); n++;
    if (t0) issue_l0<H16>(I, t, tmem, 0);
    mbar_wait_b(t.bars + B_HDR + hb, hdr_parity);
  }
  float h[kCW];
#pragma unroll 1
  for (int i = 0; i < 5; i++) {
    wait_group(t, n - 1);                                        // pre-activation of layer i (and, in order, everything before it)
    if (threadIdx.x == 0) loader_top_up(I.L, t, I.issued);       // the layer's weight slots are free: request the next units now, under the epilogue
    NSB_PH(7);
    float v1[kCW];
    tmem_ld16(i == 3 ? d3 : d1, v1);
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < kCW; j++) { const float u = v1[j] + hdr[i * 32 + kCW * cg + j]; h[j] = u > 0.0f ? u : 0.0f; m |= u > 0.0f ? (1u << j) : 0u; }
    if (gmask != nullptr) reinterpret_cast<uint16_t*>(gmask)[i * 2 + cg] = (uint16_t)m;          // halfword cg of the 32-bit ReLU mask word
    if (xyz) {
      float v2[kCW];
      tmem_ld16(d2 + 32u * i, v2);
#pragma unroll
      for (int j = 0; j < kCW; j++) h[j] += v2[j] + hdr[160 + i * 32 + kCW * cg + j];
    }
    if (acts != nullptr) {                                       // layer outputs kept for the tensor-core weight gradients of the backward
#pragma unroll
      for (int k = 0; k < kKQ; k++) __stcg(reinterpret_cast<float4*>(acts + i * 32 + 4 * k), make_float4(h[4 * k], h[4 * k + 1], h[4 * k + 2], h[4 * k + 3]));
    }
    if (i == 4) break;
    if (H16) put16_h(t.a[n & 1], row, cg, h);
    else {
      float hi[kCW], lo[kCW];
      split16(h, hi, lo);
      tmem_st16(d2 + 32u * i, hi);
      tmem_st16(tmem + kFwdALo + my, lo);
    }
    NSB_PH(8);
    if (H16) publish(t, n & 1); else publish_tmem<false>(t, n & 1);
    n++;
    if (t0) issue_h<H16>(I, t, tmem, i + 1);
    NSB_PH(9);
  }
  NSB_PH(8);
  tc::tc_fence_before();
  // output layer: partial dot products over this thread's columns, summed over the two threads of the row through shared memory.
  // (buffer (n & 1) is free: its last reader was group n-2, complete.)
  float* part = t.a[n & 1];
  {
    float s[4];
#pragma unroll
    for (int o = 0; o < 4; o++) {
      s[o] = 0.0f;
      if (o < no) {
#pragma unroll
        for (int j = 0; j < kCW; j++) s[o] = fmaf(h[j], hdr[336 + o * 32 + kCW * cg + j], s[o]);
      }
    }
    *reinterpret_cast<float4*>(part + (cg * TM + row) * 4) = make_float4(s[0], s[1], s[2], s[3]);
  }
  epi_sync();
#pragma unroll
  for (int o = 0; o < 4; o++) out[o] = hdr[320 + o];
#pragma unroll
  for (int c = 0; c < kCG; c++) {
    const float4 v = *reinterpret_cast<const float4*>(part + (c * TM + row) * 4);
    out[0] += v.x; out[1] += v.y; out[2] += v.z; out[3] += v.w;
  }
  epi_sync();                                                    // partials consumed before the next decoder's gather reuses the buffer
  NSB_PH(12);
}

// ---- tensor-core weight gradients (the colour decoder in the mapper's colour stage, src/Mapper.py:339-341,503) --------------------------------
// dW_i = DU_i^T X_i, dWc_i = G_i^T C, dWo = g_out^T H_4, dB = P^T DX are contractions over the POINTS of a tile: both operands of the MMA have the
// points as K.  A row-major [128 points][32 features] tile is exactly an MN-major operand (M / N = feature contiguous, K = point strided), which
// kind::tf32 accepts in the SWIZZLE_128B_BASE32B shared-memory layout (descriptor layout type 1): 128-byte rows, the 32-byte chunk c of row p stored
// at chunk c ^ (p & 3).  Nothing is transposed: the epilogue threads write the same rows they own in the K-major chain tiles a second time in this
// layout (DU_i, G_i -> A operand, M = 128 = [DU | G | unused | unused] through the leading-dimension stride), the layer inputs X_i come back from the
// forward's `acts`, C and the embedding blocks are recomputed.  One MMA group = 16 k-steps x 3 (3xTF32) with N = 32 into TMEM columns [192, 224);
// rows 0..31 (DU part) or 32..63 (G part) are then reduced into the packed gradient image with 16-byte vector reductions.
constexpr int kMnTile = TM * 32;                               // floats of one tile (16 KB)
constexpr size_t kWgBytes = (size_t)6 * kMnTile * 4;           // A: DU hi|lo, G hi|lo (64 KB)  B: one tile hi|lo (32 KB)
constexpr uint32_t kWgCol = 192u;                              // TMEM columns [192, 224) of the weight-gradient accumulator
struct WgSmem { float* du; float* g; float* b; uint64_t* bar; uint32_t phase; float* dpk; };
__device__ __forceinline__ void split4(const float4 v, float4& h, float4& l) {
  h = make_float4(tc::to_tf32(v.x), tc::to_tf32(v.y), tc::to_tf32(v.z), tc::to_tf32(v.w));
  l = make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w);
}
// features [16 cg, 16 cg + 16) of row p -> hi | lo tiles
__device__ __forceinline__ void put_mn16(float* hi, int p, int cg, const float (&v)[kCW]) {
  float* lo = hi + kMnTile;
#pragma unroll
  for (int c = 0; c < 2; c++) {
    const int base = p * 32 + ((((2 * cg + c) ^ p) & 3) << 3);
#pragma unroll
    for (int h = 0; h < 2; h++) {
      float4 xh, xl; split4(make_float4(v[8 * c + 4 * h], v[8 * c + 4 * h + 1], v[8 * c + 4 * h + 2], v[8 * c + 4 * h + 3]), xh, xl);
      *reinterpret_cast<float4*>(hi + base + 4 * h) = xh; *reinterpret_cast<float4*>(lo + base + 4 * h) = xl;
    }
  }
}
__device__ __forceinline__ void get_mn16(const float* hi, int p, int cg, float (&v)[kCW]) {      // hi + lo = the value that was split
  const float* lo = hi + kMnTile;
#pragma unroll
  for (int c = 0; c < 2; c++) {
    const int base = p * 32 + ((((2 * cg + c) ^ p) & 3) << 3);
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const float4 a = *reinterpret_cast<const float4*>(hi + base + 4 * h), b = *reinterpret_cast<const float4*>(lo + base + 4 * h);
      v[8 * c + 4 * h] = a.x + b.x; v[8 * c + 4 * h + 1] = a.y + b.y; v[8 * c + 4 * h + 2] = a.z + b.z; v[8 * c + 4 * h + 3] = a.w + b.w;
    }
  }
}
// gather_tile with the MN-major destination (lane q of a point holds channels [4 q, 4 q + 4))
__device__ __forceinline__ void gather_tile_mn(const nsb_grid& g, float* c_hi, const float xn[3], int warp, int lane) {
  float* c_lo = c_hi + kMnTile;
  const bool fast = grid_fast(g);
  const int qd = warp & 3, it0 = (warp >> 2) * 4, q = lane & 7;
#pragma unroll 1
  for (int it = it0; it < it0 + 4; it++) {
    GatherPass A;
    if (fast) gather_issue<true>(g, xn, it, lane, A); else gather_issue<false>(g, xn, it, lane, A);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const float w = A.w[k];
      acc.x = fmaf(A.v[k].x, w, acc.x); acc.y = fmaf(A.v[k].y, w, acc.y); acc.z = fmaf(A.v[k].z, w, acc.z); acc.w = fmaf(A.v[k].w, w, acc.w);
    }
    const int p = qd * 32 + A.src_lane;
    float4 xh, xl; split4(acc, xh, xl);
    const int o = p * 32 + ((((q >> 1) ^ p) & 3) << 3) + 4 * (q & 1);
    *reinterpret_cast<float4*>(c_hi + o) = xh; *reinterpret_cast<float4*>(c_lo + o) = xl;
  }
}
__device__ __forceinline__ uint64_t make_desc_mn(const float* smem, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_u32(smem) >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;                                      // SWIZZLE_128B_BASE32B
  return d;
}
// warp 0, converged: D_w[128 x 32] = [DU | G | . | .]^T-contraction with the B tile over the 128 points; commits to w.bar
__device__ __forceinline__ void issue_wg_group(const WgSmem& w, uint32_t tmem) {
  tc::tc_fence_after();
  const uint32_t idesc = tc::make_idesc(TM, 32) | (1u << 15) | (1u << 16);          // A and B MN-major
  const uint64_t ah = make_desc_mn(w.du, 2u * kMnTile * 4u, 512u), al = ah + (uint64_t)((kMnTile * 4) >> 4);
  const uint64_t bh = make_desc_mn(w.b, 2u * kMnTile * 4u, 512u), bl = bh + (uint64_t)((kMnTile * 4) >> 4);
  if (elect_one()) {
#pragma unroll
    for (int ks = 0; ks < TM / 8; ks++) {                       // 8 points per MMA = 1024 bytes of rows
      tc::mma_tf32(tmem + kWgCol, al + 64u * ks, bh + 64u * ks, idesc, ks == 0 ? 0u : 1u);
      tc::mma_tf32(tmem + kWgCol, ah + 64u * ks, bl + 64u * ks, idesc, 1u);
      tc::mma_tf32(tmem + kWgCol, ah + 64u * ks, bh + 64u * ks, idesc, 1u);
    }
    tc::mma_commit(w.bar);
  }
  __syncwarp();
}
// One group: the B tile (and, the first time in a layer, the A tiles) have been written by all threads.  part 0 = rows of the DU block (D rows 0..31),
// part 1 = rows of the G block (32..63); dst = packed-image address of element (out 0, in 0), pitch in floats; n_rows <= 32 rows are reduced.
__device__ __forceinline__ void wg_group(WgSmem& w, uint32_t tmem, int part, float* dst, int pitch, int n_rows, bool transposed3 = false) {
  fence_proxy_async(); tc::tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) issue_wg_group(w, tmem);
  mbar_wait_b(w.bar, w.phase); w.phase ^= 1u;
  tc::tc_fence_after();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cg = threadIdx.x >> 7;
  if ((warp & 3) == part) {
    float v[kCW];
    tmem_ld16(tmem + kWgCol + ((uint32_t)(part * 32) << 16) + (uint32_t)(kCW * cg), v);
    if (transposed3) {                                           // dB[a][f] = D[f][a], a < 3 (the B tile held the three coordinates in columns 0..2)
      if (cg == 0 && lane < n_rows) { atomicAdd(dst + lane, v[0]); atomicAdd(dst + pitch + lane, v[1]); atomicAdd(dst + 2 * pitch + lane, v[2]); }
    } else if (lane < n_rows) {
      float* d = dst + (size_t)lane * pitch + kCW * cg;
#pragma unroll
      for (int k = 0; k < kKQ; k++) red_add_v4(d + 4 * k, v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
    }
  }
  tc::tc_fence_before();
}
// column sums of a [32 rows (lanes)][16] register tile: lane l returns the sum of column ((l >> 4) & 1) * 8 + ((l >> 3) & 1) * 4 + ((l >> 2) & 1) * 2 + ((l >> 1) & 1)
__device__ __forceinline__ float warp_colsum16(const float (&v)[kCW], int lane) {
  float a[8];
#pragma unroll
  for (int j = 0; j < 8; j++) { const float give = (lane & 16) ? v[j] : v[j + 8], keep = (lane & 16) ? v[j + 8] : v[j]; a[j] = keep + __shfl_xor_sync(0xffffffffu, give, 16); }
  float b[4];
#pragma unroll
  for (int j = 0; j < 4; j++) { const float give = (lane & 8) ? a[j] : a[j + 4], keep = (lane & 8) ? a[j + 4] : a[j]; b[j] = keep + __shfl_xor_sync(0xffffffffu, give, 8); }
  float c[2];
#pragma unroll
  for (int j = 0; j < 2; j++) { const float give = (lane & 4) ? b[j] : b[j + 2], keep = (lane & 4) ? b[j + 2] : b[j]; c[j] = keep + __shfl_xor_sync(0xffffffffu, give, 4); }
  const float give = (lane & 2) ? c[0] : c[1], keep = (lane & 2) ? c[1] : c[0];
  float d = keep + __shfl_xor_sync(0xffffffffu, give, 2);
  d += __shfl_xor_sync(0xffffffffu, d, 1);
  return d;
}
__device__ __forceinline__ int colsum_col(int lane) { return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1); }

// ---- backward (input gradients): what the issuing thread does after the CTA published layer i's operands (G in a[0], DU in a[1]) ---------------
// TMEM: D1 = [0,32) (g of the next layer), DC = [32,96) (dL/dc), DF = [96,192) (dL/d first input).  render_bwd_tile_kernel: G hi = [192,224),
// DU hi = [224,256) (their last readers, the previous layer's MMAs, have completed when the epilogue writes them); the lo parts stay in the lo
// halves of a[0] / a[1].  render_bwd_wg_tile_kernel accumulates its weight gradients in [192,224) and keeps both operands in shared memory.
constexpr uint32_t kBwdGHi = 192u, kBwdDuHi = 224u;
// one A operand of the layer's products: G (a[0]) or DU (a[1]); TA: hi in tensor memory at column a_hi, lo in shared memory
template <bool TA>
__device__ __forceinline__ void mma_unit_bwd(Issuer& I, const TileSmem& t, uint32_t d_tmem, const float* a, uint32_t a_hi, const float* w, uint32_t acc) {
  if (TA) mma_unit_ta<4>(I, t, d_tmem, a_hi, 0u, a + TM * 32, w, 32, 32, acc);
  else mma_unit<4>(I, t, d_tmem, a, 0, w, 32, 32, 0, acc);
}
template <bool TA>
__device__ __forceinline__ void issue_bwd_layer(Issuer& I, const TileSmem& t, uint32_t tmem, int lv, int i) {
  const bool xyz = lv != 0;
  const int cd = op_cd(lv), nfb = op_firstp(lv) / 32;
  issuer_wait_operands(I, t, 0, I.g & 1u);
  if (xyz) for (int c2 = 0; c2 < cd / 32; c2++)                 // DC += G * Wc_i
    mma_unit_bwd<TA>(I, t, tmem + 32u + 32u * c2, t.a[0], tmem + kBwdGHi, issuer_unit(I, t), i == 4 ? 0u : 1u);
  if (i >= 1)                                                   // D1 = DU * W_i[:, hidden]
    mma_unit_bwd<TA>(I, t, tmem, t.a[1], tmem + kBwdDuHi, issuer_unit(I, t), 0u);
  if (i == 3 || i == 0) {                                       // DF += DU * W_i[:, first input]
    for (int fb = 0; fb < nfb; fb++) mma_unit_bwd<TA>(I, t, tmem + 96u + 32u * fb, t.a[1], tmem + kBwdDuHi, issuer_unit(I, t), i == 3 ? 0u : 1u);
  }
  issuer_group_done(t, B_DONE);
  I.g++;
}

// ---- backward of one decoder: epilogue side.  Leaves dL/dc rows ([128][cd] fp32) in a[0] and the embedding-chain partials of dL/dp
// ([2][128][4] fp32) in a[1]; the caller scatters after an epi_sync().
template <bool WG>
__device__ __forceinline__ void epi_backward(const KParams& P, const TileSmem& t, Issuer& I, int lv, const PointGeom& G, uint32_t tmem, uint32_t& n, int hb, uint32_t hdr_parity,
                                             const float (&g_out)[4], const uint32_t* __restrict__ gmask, WgSmem* w = nullptr, const float* acts_row = nullptr) {
  const int row = threadIdx.x & (TM - 1), cg = threadIdx.x >> 7, warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  using DW = Dec<3>;                                             // packed gradient image of the colour decoder (the only WG decoder)
  float creg[kCW];                                               // WG: this thread's 16 grid features of its point
  const bool xyz = lv != 0;
  const int cd = op_cd(lv);
  const float* hdr = t.hdr + hb * kHdrFloats;
  const uint16_t* gm16 = reinterpret_cast<const uint16_t*>(gmask) + cg;      // halfword cg of the five 32-bit ReLU mask words
  const uint32_t m01 = (uint32_t)gm16[0] | ((uint32_t)gm16[2] << 16), m23 = (uint32_t)gm16[4] | ((uint32_t)gm16[6] << 16), m4 = gm16[8];
  mbar_wait_b(t.bars + B_HDR + hb, hdr_parity);
  const uint32_t my = ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(kCW * cg);
  const uint32_t dcc = tmem + 32u, dfc = tmem + 96u;
  float* g_hi = t.a[0]; float* du_hi = t.a[1];
  float g[kCW];
#pragma unroll
  for (int j = 0; j < kCW; j++) {
    float v = 0.0f;
#pragma unroll
    for (int o = 0; o < 4; o++) v = fmaf(hdr[336 + o * 32 + kCW * cg + j], g_out[o], v);       // rows >= NO are zero
    g[j] = v;
  }
  if constexpr (WG) {
    // grid features of this point -> registers (gathered once through the B tile)
    gather_tile_mn(P.in.grid[lv], w->b, G.xn, warp, lane);
    __syncthreads();
    get_mn16(w->b, row, cg, creg);
    __syncthreads();
    // output layer: dWo = g_out^T H_4 (A block 0 = g_out in columns 0..3), dbo = column sums of g_out
    float go[kCW];
#pragma unroll
    for (int j = 0; j < kCW; j++) go[j] = (cg == 0 && j < 4) ? g_out[j] : 0.0f;
    put_mn16(w->du, row, cg, go);
    float h4[kCW];
#pragma unroll
    for (int k = 0; k < kKQ; k++) {
      const float4 v = acts_row != nullptr ? __ldcg(reinterpret_cast<const float4*>(acts_row + 4 * 32 + 4 * k)) : make_float4(0.f, 0.f, 0.f, 0.f);
      h4[4 * k] = v.x; h4[4 * k + 1] = v.y; h4[4 * k + 2] = v.z; h4[4 * k + 3] = v.w;
    }
    put_mn16(w->b, row, cg, h4);
    wg_group(*w, tmem, 0, w->dpk + DW::o_WO, DW::PH, 4);
    if (cg == 0) {
      const float sb = warp_colsum16(go, lane);
      const int col = colsum_col(lane);
      if ((lane & 1) == 0 && col < 4) atomicAdd(w->dpk + DW::o_bo + col, sb);
    }
  }
#pragma unroll 1
  for (int i = 4; i >= 0; i--) {
    const uint32_t m = i == 4 ? m4 : (((i & 2) ? m23 : m01) >> (16 * (i & 1))) & 0xffffu;
    if constexpr (WG) {
      float du[kCW];
#pragma unroll
      for (int j = 0; j < kCW; j++) du[j] = (m >> j) & 1u ? g[j] : 0.0f;
      put_mn16(w->du, row, cg, du); put_mn16(w->g, row, cg, g);
      const float sb = warp_colsum16(du, lane), sc = warp_colsum16(g, lane);      // db_i, dbc_i
      if ((lane & 1) == 0) {
        const int col = kCW * cg + colsum_col(lane);
        atomicAdd(w->dpk + DW::o_b + 32 * i + col, sb); atomicAdd(w->dpk + DW::o_bc + 32 * i + col, sc);
      }
    }
    if constexpr (WG) {
#pragma unroll
      for (int k = 0; k < kKQ; k++) {
        if (xyz) tc::put4(g_hi, g_hi + TM * 32, row, kKQ * cg + k, 32, make_float4(g[4 * k], g[4 * k + 1], g[4 * k + 2], g[4 * k + 3]));
        tc::put4(du_hi, du_hi + TM * 32, row, kKQ * cg + k, 32,
                 make_float4((m >> (4 * k)) & 1u ? g[4 * k] : 0.0f, (m >> (4 * k + 1)) & 1u ? g[4 * k + 1] : 0.0f,
                             (m >> (4 * k + 2)) & 1u ? g[4 * k + 2] : 0.0f, (m >> (4 * k + 3)) & 1u ? g[4 * k + 3] : 0.0f));
      }
      NSB_PH(22);
      publish(t, 0);
    } else {
      float hi[kCW], lo[kCW];
      if (xyz) { split16(g, hi, lo); tmem_st16(tmem + kBwdGHi + my, hi); put16(g_hi + TM * 32, row, cg, lo); }
      float du[kCW];
#pragma unroll
      for (int j = 0; j < kCW; j++) du[j] = (m >> j) & 1u ? g[j] : 0.0f;
      split16(du, hi, lo);
      tmem_st16(tmem + kBwdDuHi + my, hi);
      put16(du_hi + TM * 32, row, cg, lo);
      NSB_PH(22);
      publish_tmem<true>(t, 0);
    }
    if (threadIdx.x < 32) issue_bwd_layer<!WG>(I, t, tmem, lv, i);
    NSB_PH(23);
    if constexpr (WG) {                                          // weight gradients of layer i (the chain's MMAs run meanwhile)
      if (i >= 1) {                                              // hidden input H_{i-1}
        float xr[kCW];
#pragma unroll
        for (int k = 0; k < kKQ; k++) {
          const float4 v = acts_row != nullptr ? __ldcg(reinterpret_cast<const float4*>(acts_row + (i - 1) * 32 + 4 * k)) : make_float4(0.f, 0.f, 0.f, 0.f);
          xr[4 * k] = v.x; xr[4 * k + 1] = v.y; xr[4 * k + 2] = v.z; xr[4 * k + 3] = v.w;
        }
        put_mn16(w->b, row, cg, xr);
        const int o_wh = i == 1 ? DW::o_W1 : i == 2 ? DW::o_W2 : i == 3 ? DW::o_W3H : DW::o_W4;
        wg_group(*w, tmem, 0, w->dpk + o_wh, DW::PH, 32);
      }
      put_mn16(w->b, row, cg, creg);                             // dWc_i = G_i^T C
      wg_group(*w, tmem, 1, w->dpk + DW::o_WC + 32 * i * DW::PC, DW::PC, 32);
      if (i == 3 || i == 0) {                                    // embedding part of W_0 / W_3
        const float* B = hdr + 464;
        for (int blk = 0; blk < 3; blk++) {
          float e[kCW];
#pragma unroll
          for (int j = 0; j < kCW; j++) {
            const int f = 32 * blk + kCW * cg + j;
            float x = G.pf[0] * B[f]; x = fmaf(G.pf[1], B[kEmbPad + f], x); x = fmaf(G.pf[2], B[2 * kEmbPad + f], x);
            e[j] = f < kEmb ? __sinf(reduce_2pi(x)) : 0.0f;
          }
          put_mn16(w->b, row, cg, e);
          wg_group(*w, tmem, 0, w->dpk + (i == 0 ? DW::o_W0 : DW::o_W3E) + 32 * blk, DW::PF, 32);
        }
      }
    }
    mbar_wait_b(t.bars + B_DONE, n & 1u); n++;
    tc::tc_fence_after();
    if (threadIdx.x == 0) loader_top_up(I.L, t, I.issued);       // slots of this layer are free: fetch the next layer's units under the epilogue
    NSB_PH(24);
    if (i >= 1) tmem_ld16(tmem + my, g);
    tc::tc_fence_before();
  }
  NSB_PH(22);
  // dL/dc rows -> a[0] (plain fp32 [128][cd]); every MMA reading the buffers has completed
  float* dcs = t.a[0];
  {
    float v[kCW];
    const int nch = xyz ? (cd >> 5) : 1;
    for (int c = 0; c < nch; c++) {
      tmem_ld16((xyz ? dcc : dfc) + 32u * c + my, v);
#pragma unroll
      for (int k = 0; k < kKQ; k++)
        *reinterpret_cast<float4*>(dcs + row * cd + 32 * c + kCW * cg + 4 * k) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
    }
  }
  float dpe[3] = {0.0f, 0.0f, 0.0f};
  if (xyz) {
    const float* B = hdr + 464;
    if constexpr (WG) {                                          // B tile of the dB groups: the point's coordinates in columns 0..2
      float pv[kCW];
#pragma unroll
      for (int j = 0; j < kCW; j++) pv[j] = (cg == 0 && j < 3) ? G.pf[j] : 0.0f;
      put_mn16(w->b, row, cg, pv);
    }
    for (int c = 0; c < 3; c++) {
      float v[kCW];
      tmem_ld16(dfc + 32u * c + my, v);
      float dxv[kCW];
#pragma unroll
      for (int j = 0; j < kCW; j++) {
        const int f = 32 * c + kCW * cg + j;
        dxv[j] = 0.0f;
        if (f < kEmb) {
          const float b0 = B[f], b1 = B[kEmbPad + f], b2 = B[2 * kEmbPad + f];
          float x = G.pf[0] * b0; x = fmaf(G.pf[1], b1, x); x = fmaf(G.pf[2], b2, x);
          const float dx = __cosf(reduce_2pi(x)) * v[j];
          dxv[j] = dx;
          dpe[0] = fmaf(b0, dx, dpe[0]); dpe[1] = fmaf(b1, dx, dpe[1]); dpe[2] = fmaf(b2, dx, dpe[2]);
        }
      }
      if constexpr (WG) {                                        // dB[a][f] = sum_p p_a cos(.) dE_f  (embedder._B is a parameter of the decoder)
        put_mn16(w->du, row, cg, dxv);
        const int nf = kEmb - 32 * c < 32 ? kEmb - 32 * c : 32;
        wg_group(*w, tmem, 0, w->dpk + DW::o_B + 32 * c, kEmbPad, nf, true);
      }
    }
  }
  *reinterpret_cast<float4*>(t.a[1] + (cg * TM + row) * 4) = make_float4(dpe[0], dpe[1], dpe[2], 0.0f);
  tc::tc_fence_before();
  NSB_PH(27);
}

// Backward of gather_tile (same warp -> rows mapping).  dcs = [128][cd] fp32.  emit(row, gx) once per point.
// (unlike gather_tile, making the channels-last test a compile-time property of this loop measured SLOWER -- profiles/README.md, r02k)
template <typename F>
__device__ __forceinline__ void scatter_tile(const nsb_grid& g, float* __restrict__ dgrid, const int32_t* __restrict__ slots,
                                             const float* dcs, int cd, const float xn[3], int warp, int lane, F&& emit) {
  const bool fast = grid_fast(g);
  const int q = lane & 7, qd = warp & 3, it0 = (warp >> 2) * 4;
#pragma unroll 1
  for (int it = it0; it < it0 + 4; it++) {
    const int src_lane = it * 4 + (lane >> 3);
    const int row = qd * 32 + src_lane;
    float x[3];
    x[0] = __shfl_sync(0xffffffffu, xn[0], src_lane); x[1] = __shfl_sync(0xffffffffu, xn[1], src_lane); x[2] = __shfl_sync(0xffffffffu, xn[2], src_lane);
    const Tri t = make_tri(x, g.W, g.H, g.D);
    const float4 d4 = *reinterpret_cast<const float4*>(dcs + row * cd + 4 * q);
    const float dc[4] = {d4.x, d4.y, d4.z, d4.w};
    float gi[3] = {0.f, 0.f, 0.f};
    float4 vv[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      int cx, cy, cz;
      tri_corner_clamped(t, k, g.W, g.H, g.D, cx, cy, cz);
      vv[k] = grid_load4(g, cz * g.stride_d + cy * g.stride_h + cx * g.stride_w, 4 * q, fast);
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
      int cx, cy, cz;
      if (tri_corner(t, k, g.W, g.H, g.D, cx, cy, cz)) {         // corners outside the grid get neither gradient nor a dot product
        const float4 v = vv[k];
        const float dot = v.x * dc[0] + v.y * dc[1] + v.z * dc[2] + v.w * dc[3];
        if (dgrid != nullptr) voxel_grad_add(g, dgrid, slots, cz * g.stride_d + cy * g.stride_h + cx * g.stride_w, cx, cy, cz, q, fast, tri_weight(t, k), dc);
        const float wx = (k & 1) ? t.w1[0] : t.w0[0], wy = (k & 2) ? t.w1[1] : t.w0[1], wz = (k & 4) ? t.w1[2] : t.w0[2];
        gi[0] += ((k & 1) ? 1.f : -1.f) * wy * wz * dot;
        gi[1] += ((k & 2) ? 1.f : -1.f) * wx * wz * dot;
        gi[2] += ((k & 4) ? 1.f : -1.f) * wx * wy * dot;
      }
    }
#pragma unroll
    for (int a = 0; a < 3; a++) {
      float v = gi[a];
      v += __shfl_xor_sync(0xffffffffu, v, 1); v += __shfl_xor_sync(0xffffffffu, v, 2); v += __shfl_xor_sync(0xffffffffu, v, 4);
      gi[a] = v;
    }
    if (q == 0) {
      const int size[3] = {g.W, g.H, g.D};
      float gx[3];
#pragma unroll
      for (int a = 0; a < 3; a++) gx[a] = t.clipg[a] * ((float)(size[a] - 1) * 0.5f) * gi[a];
      emit(row, gx);
    }
  }
}

// ---- tile <-> ray bookkeeping ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int tiles_of_ray(int ray, int S) {
  const long long p0 = (long long)ray * S;
  return (int)((p0 + S - 1) / TM - p0 / TM) + 1;
}
// Bump the completion counters of the rays [ray_lo, ray_lo + nr) this item touched; returns (CTA-uniform) how many of them this CTA
// completed, their indices in s_done[].  Every thread must call it, after its global writes.  target = items per tile (split).
__device__ __forceinline__ int complete_rays(int* ray_cnt, int ray_lo, int nr, int S, int per_tile, int* s_done, int* s_ndone) {
  __threadfence();
  if (threadIdx.x == 0) *s_ndone = 0;
  __syncthreads();
  if ((int)threadIdx.x < nr) {
    const int ray = ray_lo + threadIdx.x;
    const int target = tiles_of_ray(ray, S) * per_tile;
    const int old = atomicAdd(ray_cnt + ray, 1);
    if (old == target - 1) { ray_cnt[ray] = 0; s_done[atomicAdd(s_ndone, 1)] = ray; }
  }
  __syncthreads();
  const int nd = *s_ndone;
  if (nd > 0) __threadfence();
  return nd;
}

// raw2outputs_nerf_color of one completed ray by one warp (common.py:204-245 incl. the out-of-bound override of Renderer.py:57).
// scratch: per-warp shared memory, composite_scratch_bytes(S) bytes, 16-byte aligned: raw [S] float4 | z [S] f64 | w [S] f32.
__host__ __device__ inline size_t composite_scratch_bytes(int S) { return ((size_t)28 * S + 15) & ~size_t(15); }
__device__ __forceinline__ void composite_ray(const KParams& P, int ray, int lane, unsigned char* scratch) {
  const int S = P.S;
  float* rw = reinterpret_cast<float*>(scratch);
  double* zz = reinterpret_cast<double*>(rw + 4 * S);
  float* wq = reinterpret_cast<float*>(zz + S);
  float o[3], d[3];
#pragma unroll
  for (int a = 0; a < 3; a++) { o[a] = P.in.rays_o[3 * ray + a]; d[a] = P.in.rays_d[3 * ray + a]; }
  const long long g0 = (long long)ray * S, NS = (long long)P.in.n_rays * S;
  for (int s = lane; s < S; s += 32) {
    // (all loads of the sample first: with a run-time trip count they were issued one L2 round trip after the other)
    float4 pq[3];
#pragma unroll
    for (int q = 0; q < 3; q++) pq[q] = q < P.split ? __ldcg(P.tile_parts + q * NS + g0 + s) : make_float4(0.f, 0.f, 0.f, 0.f);
    const double z = __ldcg(P.fo.z_vals + g0 + s);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int q = 0; q < 3; q++) { v.x += pq[q].x; v.y += pq[q].y; v.z += pq[q].z; v.w += pq[q].w; }       // decoder order: occ = fine + middle, rgb = colour decoder (zeros elsewhere)
    PointGeom G; make_point(P.in.bound, P.in.coarse_bound, o, d, z, G);
    if (!G.inb) v.w = 100.0f;
    zz[s] = z;
    *reinterpret_cast<float4*>(rw + 4 * s) = v;
    *reinterpret_cast<float4*>(P.fo.raw + 4 * (g0 + s)) = v;
  }
  __syncwarp();
  ray_weights(rw, S, lane, wq, nullptr);
  __syncwarp();
  float c0 = 0.f, c1 = 0.f, c2 = 0.f; double dsum = 0.0;
  for (int s = lane; s < S; s += 32) {
    const float w = wq[s];
    c0 = fmaf(w, rw[4 * s], c0); c1 = fmaf(w, rw[4 * s + 1], c1); c2 = fmaf(w, rw[4 * s + 2], c2);
    dsum += (double)w * zz[s];
  }
  c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2); dsum = warp_sum(dsum);
  double v = 0.0;
  for (int s = lane; s < S; s += 32) { const double tt = zz[s] - dsum; v += (double)wq[s] * tt * tt; }
  v = warp_sum(v);
  if (lane == 0) {
    P.fo.depth[ray] = dsum; P.fo.var[ray] = v;
    P.fo.rgb[3 * ray] = c0; P.fo.rgb[3 * ray + 1] = c1; P.fo.rgb[3 * ray + 2] = c2;
  }
  __syncwarp();
}

}  // namespace tl

// ================================================================================================================================
// forward kernel
// ================================================================================================================================
template <bool H16>
__device__ __forceinline__ void render_fwd_tile_body(const KParams& P) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  using namespace tl;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row = tid & (TM - 1), cg = tid >> 7;            // (control warp: row/cg unused)
  TileSmem t; carve(smem_raw, t, false);
  __shared__ int s_ndone, s_done[kMaxTileRays], s_last;
  __shared__ float s_max[16];
  __shared__ uint32_t s_seq;

  const bool points = P.points != nullptr;
  const int nsplit = P.split;
  const int tile = blockIdx.x / nsplit, my = blockIdx.x - tile * nsplit;
  const int q0 = nsplit > 1 ? my : 0, q1 = nsplit > 1 ? my + 1 : P.n_dec;
  const long long NP = points ? (long long)P.n_points : (long long)P.in.n_rays * P.S;
  const long long gp0 = (long long)tile * TM;
  const int npts = (int)(NP - gp0 < TM ? NP - gp0 : TM);
  const int S = P.S;
  int ray_lo = 0, nr = 0;
  if (!points) { ray_lo = (int)(gp0 / S); nr = (int)((gp0 + npts - 1) / S) - ray_lo + 1; }

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(t.tmem)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  NSB_PH_RESET();
  Issuer I; I.L.P = &P; I.L.q = q0; I.L.q1 = q1; I.L.k = 0; I.L.loaded = 0; I.L.mode = H16 ? 2 : 0; I.issued = 0; I.g = 0;
  if (tid == 0) {
    for (int i = 0; i < kNumBars; i++) mbar_init(t.bars + i, (i == B_AREADY || i == B_AREADY + 1) ? kEpiThreads / 32 : 1);
    mbar_fence_init();
    load_header(P, t, P.dec[q0], 0);
    for (int i = 0; i < kSlots; i++) loader_issue(I.L, t);      // (every decoder has >= 6 units)
  }

  // ---- prologue: this tile's rays -> sorted sample depths -> this row's point
  PointGeom G;
  const int lp = row < npts ? row : npts - 1;
  if (points) {
    const long long gp = gp0 + lp;
    const double pin[3] = {P.points[3 * gp], P.points[3 * gp + 1], P.points[3 * gp + 2]};
    make_point_from_p(P.in.bound, P.in.coarse_bound, pin, G);
    __syncthreads();
  } else {
    float gtmax = 0.0f, gtmax12 = 0.0f;
    if (P.has_gt) {
      if (P.in.depth_max != nullptr) { gtmax = P.in.depth_max[0]; gtmax12 = P.in.depth_max[1]; }
      else {                                                      // small batches: every CTA reduces the sensor depths itself (Renderer.py:109,144)
        const bool whole = P.in.gt_depth_batch != nullptr;        // the depths of the whole (sharded) batch are known here: no exchange
        const float* gsrc = whole ? P.in.gt_depth_batch : P.in.gt_depth;
        const int gn = whole ? P.in.n_batch : P.in.n_rays;
        float m = -INFINITY;
        for (int i = tid; i < gn; i += kThreads) m = fmaxf(m, __ldg(gsrc + i));
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) s_max[warp] = m;
        __syncthreads();
        m = -INFINITY;
        for (int w = 0; w < kThreads / 32; w++) m = fmaxf(m, s_max[w]);
        if (P.fs.px.world > 1 && !whole) m = peer_max_all_ctas(P.fs.px, m, &s_seq);      // sharded batch: MAX over the ranks' shards (Renderer.py:109,144)
        gtmax = m; gtmax12 = __fmul_rn(m, 1.2f);
      }
    }
    NSB_PH(40);
    // scratch in the (still unused) operand buffers: ray table [nr][8] f32 + far [nr] f64 | unsorted z [nr*S] | sorted z [nr*S]
    float* rays = t.a[0];
    double* far = reinterpret_cast<double*>(t.a[0] + 8 * kMaxTileRays);
    double* zu = far + kMaxTileRays;
    double* zs = zu + (size_t)nr * S;
    for (int r = tid; r < nr; r += kThreads) {
      float o[3], d[3];
#pragma unroll
      for (int a = 0; a < 3; a++) { o[a] = P.in.rays_o[3 * (ray_lo + r) + a]; d[a] = P.in.rays_d[3 * (ray_lo + r) + a]; }
      const float gt = P.has_gt ? P.in.gt_depth[ray_lo + r] : 0.0f;
      const RaySampler rs = make_sampler(P.in.bound, o, d, P.has_gt, gt, gtmax12);
#pragma unroll
      for (int a = 0; a < 3; a++) { rays[8 * r + a] = o[a]; rays[8 * r + 3 + a] = d[a]; }
      rays[8 * r + 6] = rs.near; rays[8 * r + 7] = gt; far[r] = rs.far;
    }
    __syncthreads();
    NSB_PH(41);
    for (int i = tid; i < nr * S; i += kThreads) {
      const int r = i / S, s = i - r * S;
      RaySampler rs; rs.near = rays[8 * r + 6]; rs.gt = rays[8 * r + 7]; rs.far = far[r]; rs.has_gt = P.has_gt;
      zu[i] = sample_z(rs, s, P.in.n_samples, P.in.t_uniform, P.in.t_surface, gtmax);
    }
    __syncthreads();
    NSB_PH(42);
    // torch.sort of the concatenation [uniform | surface] (Renderer.py:168-170).  Both lists come out of linspace-style formulas and are
    // normally non-decreasing: then the stable rank of an element is its index in its own list plus a binary-search count in the other one
    // (merge by ranks).  A ray whose lists are not sorted (far < near, NaN) takes the general stable rank sort -- same values either way.
    int* unsorted = reinterpret_cast<int*>(zs + (size_t)nr * S);
    for (int r = tid; r < nr; r += kThreads) unsorted[r] = 0;
    __syncthreads();
    const int nu = P.in.n_samples < S ? P.in.n_samples : S;
    for (int i = tid; i < nr * S; i += kThreads) {
      const int r = i / S, s = i - r * S;
      if (s != 0 && s != nu) { const double a = zu[i - 1], b = zu[i]; if (!(a <= b)) unsorted[r] = 1; }
      else if (zu[i] != zu[i]) unsorted[r] = 1;
    }
    __syncthreads();
    for (int i = tid; i < nr * S; i += kThreads) {
      const int r = i / S, s = i - r * S;
      const double zi = zu[i];
      const double* zr = zu + r * S;
      int rank;
      if (!unsorted[r]) {
        // uniform element: + #{surface < z}; surface element: + #{uniform <= z} (cat order = uniform first, stable)
        const bool uni = s < nu;
        const double* other = uni ? zr + nu : zr;
        int lo = 0, hi = uni ? S - nu : nu;
        while (lo < hi) { const int mid = (lo + hi) >> 1; const double zm = other[mid]; if (uni ? (zm < zi) : (zm <= zi)) lo = mid + 1; else hi = mid; }
        rank = (uni ? s : s - nu) + lo;
      } else {
        rank = 0;
        for (int j = 0; j < S; j++) { const double zj = zr[j]; rank += (z_less(zj, zi) || (!z_less(zi, zj) && j < s)) ? 1 : 0; }
      }
      zs[r * S + rank] = zi;
    }
    __syncthreads();
    NSB_PH(43);
    {
      const long long gp = gp0 + lp;
      const int r = (int)(gp / S) - ray_lo, s = (int)(gp - (long long)(ray_lo + r) * S);
      const double z = zs[r * S + s];
      const float o[3] = {rays[8 * r], rays[8 * r + 1], rays[8 * r + 2]}, dd[3] = {rays[8 * r + 3], rays[8 * r + 4], rays[8 * r + 5]};
      make_point(P.in.bound, P.in.coarse_bound, o, dd, z, G);
      if (cg == 0 && row < npts && my == 0) P.fo.z_vals[gp] = z;
    }
    __syncthreads();                                              // the scratch is dead: the operand buffers may be written
  }
  tc::tc_fence_before();
  __syncthreads();                                                // TMEM address + barrier initialisation visible
  tc::tc_fence_after();
  const uint32_t tmem = *t.tmem;
  NSB_PH(44);

  float occ = 0.0f, c0 = 0.0f, c1 = 0.0f, c2 = 0.0f;
  {
    uint32_t n = 0;
    for (int qd = q0; qd < q1; qd++) {
      const int lv = P.dec[qd];
      float out[4];
      uint32_t* gm = (P.fo.masks != nullptr && row < npts) ? P.fo.masks + ((gp0 + row) * 15 + qd * 5) : nullptr;
      const int dq = qd - q0;
      if (tid == 0 && qd + 1 < q1) load_header(P, t, P.dec[qd + 1], (dq + 1) & 1);      // (decoder qd-1 ended with CTA barriers: its buffer is free)
      float* acts = (P.fo.acts != nullptr && lv == P.acts_lv && row < npts) ? P.fo.acts + ((gp0 + row) * 5) * 32 + kCW * cg : nullptr;
      epi_forward<H16>(P, t, I, lv, G, tmem, n, dq & 1, (dq >> 1) & 1u, out, gm, acts);
      if (lv == 3) { c0 = out[0]; c1 = out[1]; c2 = out[2]; } else occ += out[0];
      if (qd == 0 && cg == 0 && row < npts && P.fo.corner_idx != nullptr) {
        const nsb_grid& g = P.in.grid[lv];
        const Tri tr = make_tri(lv == 0 ? G.xnc : G.xn, g.W, g.H, g.D);
        const long long gp = gp0 + row;
        P.fo.corner_idx[3 * gp] = tr.i0[0]; P.fo.corner_idx[3 * gp + 1] = tr.i0[1]; P.fo.corner_idx[3 * gp + 2] = tr.i0[2];
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
  // the decoder chain of this item is done: a backward launched as a programmatic dependent may take the slots that free up from here on and
  // set up under the ray compositing / loss-seed tail (triggering at kernel start made the early backward CTAs compete with the chain: slower)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  NSB_PH(14);

  if (points) {                                                   // Renderer.eval_points: raw with the out-of-bound override
    if (cg == 0 && row < npts) *reinterpret_cast<float4*>(P.points_raw + 4 * (gp0 + row)) = make_float4(c0, c1, c2, G.inb ? occ : 100.0f);
    return;
  }
  if (cg == 0 && row < npts) P.tile_parts[(long long)my * NP + gp0 + row] = make_float4(c0, c1, c2, occ);
  const int nd = complete_rays(P.ray_cnt, ray_lo, nr, S, nsplit, s_done, &s_ndone);
  NSB_PH(15);
  for (int k = warp; k < nd; k += kThreads / 32) composite_ray(P, s_done[k], lane, smem_raw + (size_t)warp * composite_scratch_bytes(S));
  NSB_PH(16);
  // loss seeds: the last CTA of the grid to get here sees every ray composited
  if (P.fs.kind != 0 && grid_last_arrival(P.fs.counter, gridDim.x, &s_last)) {
    if (P.fs.kind == 1) {
      tracking_seeds_body(P.fo.depth, P.fo.var, P.fo.rgb, P.in.gt_depth, static_cast<const double*>(P.fs.gt_rgb), P.in.n_rays, P.fs.w_color,
                          P.fs.handle_dynamic, P.fs.use_color, nullptr, 0, P.fs.g_depth, P.fs.g_rgb, P.fs.loss, P.fs.res, P.fs.px, smem_raw);
      if (P.fs.px.world > 1 && P.in.depth_max == nullptr && P.in.gt_depth_batch == nullptr && tid == 0) peer_advance(P.fs.px, 0);      // every CTA is past the depth-max exchange
    } else {
      mapping_seeds_body(P.fo.depth, P.fo.rgb, P.fs.gt_depth_loss, static_cast<const float*>(P.fs.gt_rgb), P.in.n_rays, P.fs.w_color, P.fs.use_color,
                         P.fs.g_depth, P.fs.g_rgb, P.fs.loss, smem_raw);
    }
  }
}
__global__ void __launch_bounds__(tl::kThreads, 2) render_fwd_tile_kernel(const __grid_constant__ KParams P) { render_fwd_tile_body<false>(P); }
// forward with FP16 hi|lo operands (option fwd_f16; see mma_unit_h)
__global__ void __launch_bounds__(tl::kThreads, 2) render_fwd_tile_h16_kernel(const __grid_constant__ KParams P) { render_fwd_tile_body<true>(P); }

// ================================================================================================================================
// backward kernel (input gradients: rays + grid voxels)
// ================================================================================================================================
namespace tl {
struct BwdExtra {            // behind the common shared-memory part
  double dp[TM * 3];
  double z[TM];
  float gocc[TM];
  float wgt[TM];
  float gc[kMaxTileRays * 3];
};
}  // namespace tl

// WG = true: the item's decoder (the colour decoder) also gets its WEIGHT gradients (tensor-core contraction over the tile's points, see the
// "tensor-core weight gradients" helpers): 96 KB more shared memory in front of the common part -> one CTA per SM.
template <bool WG>
__device__ __forceinline__ void render_bwd_tile_body(const KParams& P) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  using namespace tl;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row = tid & (TM - 1), cg = tid >> 7;
  // (WG: the MN-major tiles need the 1024-byte alignment of their swizzle pattern: aligned by hand, 1 KB of slack in the launch size)
  unsigned char* sbase = WG ? smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u) : smem_raw;
  TileSmem t; carve(sbase + (WG ? kWgBytes : 0), t, true);
  BwdExtra& X = *reinterpret_cast<BwdExtra*>(t.extra);
  __shared__ int s_ndone, s_done[kMaxTileRays];
  __shared__ __align__(8) uint64_t s_wgbar;
  WgSmem wg;
  wg.du = reinterpret_cast<float*>(sbase); wg.g = wg.du + 2 * kMnTile; wg.b = wg.du + 4 * kMnTile; wg.bar = &s_wgbar; wg.phase = 0u;
  wg.dpk = WG ? P.d_packed[P.dec[0]] : nullptr;

  const int nsplit = P.split;
  const int tile = blockIdx.x / nsplit, my = blockIdx.x - tile * nsplit;
  const int q0 = nsplit > 1 ? my : 0, q1 = nsplit > 1 ? my + 1 : P.n_dec;
  const int S = P.S;
  const long long NP = (long long)P.in.n_rays * S;
  const long long gp0 = (long long)tile * TM;
  const int npts = (int)(NP - gp0 < TM ? NP - gp0 : TM);
  const int ray_lo = (int)(gp0 / S), nr = (int)((gp0 + npts - 1) / S) - ray_lo + 1;

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(t.tmem)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  NSB_PH_RESET();
  Issuer I; I.L.P = &P; I.L.q = q0; I.L.q1 = q1; I.L.k = 0; I.L.loaded = 0; I.L.mode = 1; I.issued = 0; I.g = 0;
  if (tid == 0) {
    for (int i = 0; i < kNumBars; i++) mbar_init(t.bars + i, (i == B_AREADY || i == B_AREADY + 1) ? kEpiThreads / 32 : 1);
    if (WG) mbar_init(&s_wgbar, 1);
    mbar_fence_init();
    load_header(P, t, P.dec[q0], 0);
    for (int i = 0; i < kSlots; i++) loader_issue(I.L, t);
  }

  for (int i = tid; i < TM * 3; i += kThreads) X.dp[i] = 0.0;
  // Launched as a programmatic dependent of the forward (nsb_render.cu): everything above ran under the forward's tail; nothing the forward
  // produces (raw, z_vals, ReLU bits, loss seeds, completion counters) is touched before the forward grid has completed.  (No-op otherwise.)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // ---- prologue: per ray of this tile, compositing weights and dL/d(occupancy logit) (SURVEY.md 8.1); scratch in the operand buffers
  for (int r = warp; r < nr; r += kThreads / 32) {
    const int ray = ray_lo + r;
    float* rw = t.a[0] + (size_t)warp * ((6 * S + 3) & ~3);       // per warp (16-byte aligned): raw [4S] | w [S] | go [S]
    float* wq = rw + 4 * S; float* go = wq + S;
    const long long g0 = (long long)ray * S;
    float o[3], d[3];
#pragma unroll
    for (int a = 0; a < 3; a++) { o[a] = P.in.rays_o[3 * ray + a]; d[a] = P.in.rays_d[3 * ray + a]; }
    for (int s = lane; s < S; s += 32) *reinterpret_cast<float4*>(rw + 4 * s) = *reinterpret_cast<const float4*>(P.bw.raw + 4 * (g0 + s));
    __syncwarp();
    const double gD = P.bw.g_depth != nullptr ? P.bw.g_depth[ray] : 0.0;
    const double gV = P.bw.g_var != nullptr ? P.bw.g_var[ray] : 0.0;
    float g3[3] = {0.f, 0.f, 0.f};
    if (P.bw.g_rgb != nullptr) { g3[0] = P.bw.g_rgb[3 * ray]; g3[1] = P.bw.g_rgb[3 * ray + 1]; g3[2] = P.bw.g_rgb[3 * ray + 2]; }
    if (lane == 0) { X.gc[3 * r] = g3[0]; X.gc[3 * r + 1] = g3[1]; X.gc[3 * r + 2] = g3[2]; }
    ray_weights(rw, S, lane, wq, go);                            // go[] temporarily holds T_s
    __syncwarp();
    const double* z = P.bw.z_vals + g0;
    double Dm = 0.0;
    for (int s = lane; s < S; s += 32) Dm += (double)wq[s] * z[s];
    Dm = warp_sum(Dm);
    double swt = 0.0;
    for (int s = lane; s < S; s += 32) swt += (double)wq[s] * (z[s] - Dm);
    swt = warp_sum(swt);
    const double gDe = gD + gV * (-2.0 * swt);
    float carry = 0.0f;
    const int nblk = (S + 31) / 32;
    for (int b = nblk - 1; b >= 0; b--) {
      const int s = b * 32 + lane;
      const bool v = s < S;
      float gw = 0.0f, al = 0.0f, T = 0.0f, w = 0.0f;
      if (v) {
        al = sigmoid_f(10.0f * rw[4 * s + 3]); T = go[s]; w = wq[s];
        const double tt = z[s] - Dm;
        gw = (float)(gDe * z[s] + gV * tt * tt) + g3[0] * rw[4 * s] + g3[1] * rw[4 * s + 1] + g3[2] * rw[4 * s + 2];
      }
      const float incl = warp_incl_suffix_sum(gw * w, lane);
      float excl = __shfl_down_sync(0xffffffffu, incl, 1);
      if (lane == 31) excl = 0.0f;
      const float R = carry + excl;
      if (v) {
        const long long gp = g0 + s;
        if (gp >= gp0 && gp < gp0 + npts) {                      // only the samples of this tile are needed
          PointGeom Gs; make_point(P.in.bound, P.in.coarse_bound, o, d, z[s], Gs);
          const float qd = (1.0f - al) + 1e-10f;
          const float ga = T * gw - R / qd;
          X.gocc[gp - gp0] = Gs.inb ? 10.0f * al * (1.0f - al) * ga : 0.0f;
          X.wgt[gp - gp0] = w;
        }
      }
      carry += __shfl_sync(0xffffffffu, incl, 0);
    }
  }
  NSB_PH(20);
  PointGeom G;
  const int lp = row < npts ? row : npts - 1;
  const long long gpr = gp0 + lp;
  const int rayr = (int)(gpr / S);
  {
    float o[3], d[3];
#pragma unroll
    for (int a = 0; a < 3; a++) { o[a] = P.in.rays_o[3 * rayr + a]; d[a] = P.in.rays_d[3 * rayr + a]; }
    const double z = P.bw.z_vals[gpr];
    make_point(P.in.bound, P.in.coarse_bound, o, d, z, G);
    if (cg == 0) X.z[row] = z;
  }
  tc::tc_fence_before();
  __syncthreads();                                                // prologue scratch dead, gocc / wgt / gc visible, TMEM address + barriers visible
  tc::tc_fence_after();
  const uint32_t tmem = *t.tmem;
  NSB_PH(21);

  {
    uint32_t n = 0;
    for (int qd = q0; qd < q1; qd++) {
      const int lv = P.dec[qd];
      const uint32_t* gm = P.bw.masks + ((gp0 + lp) * 15 + P.dec_pos[qd] * 5);
      float g_out[4] = {0.f, 0.f, 0.f, 0.f};
      if (row < npts) {
        if (lv == 3) { const float w = X.wgt[row]; const float* gc = X.gc + 3 * (rayr - ray_lo); g_out[0] = w * gc[0]; g_out[1] = w * gc[1]; g_out[2] = w * gc[2]; }
        else g_out[0] = X.gocc[row];
      }
      const int dq = qd - q0;
      if (tid == 0 && qd + 1 < q1) load_header(P, t, P.dec[qd + 1], (dq + 1) & 1);      // (the previous decoder ended with CTA barriers: its buffer is free)
      const float* acts_row = (WG && row < npts) ? P.bw.acts + ((gp0 + row) * 5) * 32 + kCW * cg : nullptr;
      epi_backward<WG>(P, t, I, lv, G, tmem, n, dq & 1, (dq >> 1) & 1u, g_out, gm, WG ? &wg : nullptr, acts_row);
      epi_sync();                                                 // dL/dc rows + embedding partials visible
      const double* bb = lv == 0 ? P.in.coarse_bound : P.in.bound;
      const double sc[3] = {2.0 / (bb[1] - bb[0]), 2.0 / (bb[3] - bb[2]), 2.0 / (bb[5] - bb[4])};      // d(normalised)/dp, common.py:280-282
      const float* xn = lv == 0 ? G.xnc : G.xn;
      scatter_tile(P.in.grid[lv], P.bw.d_grid[lv], P.bw.slot_map[lv], t.a[0], op_cd(lv), xn, warp, lane, [&](int prow, const float gx[3]) {
        if (prow < npts) {
          const float4 p0 = *reinterpret_cast<const float4*>(t.a[1] + prow * 4);
          const float4 p1 = *reinterpret_cast<const float4*>(t.a[1] + (TM + prow) * 4);
          const float dpe[3] = {p0.x + p1.x, p0.y + p1.y, p0.z + p1.z};
#pragma unroll
          for (int a = 0; a < 3; a++) X.dp[3 * prow + a] += (double)dpe[a] + (double)gx[a] * sc[a];
        }
      });
      epi_sync();                                                 // reads of a[0] / a[1] done before the next decoder overwrites them
      NSB_PH(29);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");

  // per-ray sums of this item: d rays_o = sum_s dp, d rays_d = sum_s z_s dp (pts = o + d z, Renderer.py:172-174) -> global scratch
  const int RT = P.tile_rays;                                     // rays a tile can touch: stride of the per-item parts
  double* parts = P.ray_parts + ((long long)tile * nsplit + my) * RT * 6;
  for (int i = tid; i < nr * 3; i += kThreads) {
    const int r = i / 3, a = i - 3 * r;
    const long long g0 = (long long)(ray_lo + r) * S;
    const int s0 = (int)(g0 > gp0 ? g0 - gp0 : 0), s1 = (int)(g0 + S - gp0 < npts ? g0 + S - gp0 : npts);
    double so = 0.0, sd = 0.0;
    for (int p = s0; p < s1; p++) { const double v = X.dp[3 * p + a]; so += v; sd += v * X.z[p]; }
    parts[r * 6 + a] = so; parts[r * 6 + 3 + a] = sd;
  }
  NSB_PH(30);
  const int nd = complete_rays(P.ray_cnt, ray_lo, nr, S, nsplit, s_done, &s_ndone);
  NSB_PH(31);
  for (int i = tid; i < nd * 3; i += kThreads) {                  // the completing CTA adds the parts in (tile, decoder) order
    const int ray = s_done[i / 3], a = i % 3;
    const long long p0 = (long long)ray * S;
    const int t0 = (int)(p0 / TM), t1 = (int)((p0 + S - 1) / TM);
    double so = 0.0, sd = 0.0;
    for (int tt = t0; tt <= t1; tt++) {
      const int rl = (int)(((long long)tt * TM) / S);
      for (int q = 0; q < nsplit; q++) {
        const double* pp = P.ray_parts + (((long long)tt * nsplit + q) * RT + (ray - rl)) * 6;
        so += __ldcg(pp + a); sd += __ldcg(pp + 3 + a);
      }
    }
    if (P.accumulate_rays) {
      if (P.bw.d_rays_o != nullptr) so += (double)P.bw.d_rays_o[3 * ray + a];
      if (P.bw.d_rays_d != nullptr) sd += (double)P.bw.d_rays_d[3 * ray + a];
    }
    if (P.bw.d_rays_o != nullptr) P.bw.d_rays_o[3 * ray + a] = (float)so;
    if (P.bw.d_rays_d != nullptr) P.bw.d_rays_d[3 * ray + a] = (float)sd;
  }
  NSB_PH(32);
  if (fused_pose_grad(P, gridDim.x, reinterpret_cast<double*>(smem_raw)) && P.tail.px.world > 1) {
    // sharded tracking batch: SUM over ranks of [loss | d c2w] by this (last) CTA -- identical bits on every rank
    __shared__ double tot[13];
    __shared__ uint32_t s_seq2;
    __syncthreads();
    if (tid == 0) tot[0] = P.tail.loss != nullptr ? P.tail.loss[0] : 0.0;
    if (tid < 12) tot[1 + tid] = P.bw.d_c2w[tid];
    __syncthreads();
    peer_sum13(P.tail.px, tot, 13, P.tail.out13, &s_seq2);
  }
}
__global__ void __launch_bounds__(tl::kThreads, 2) render_bwd_tile_kernel(const __grid_constant__ KParams P) { render_bwd_tile_body<false>(P); }
__global__ void __launch_bounds__(tl::kThreads, 1) render_bwd_wg_tile_kernel(const __grid_constant__ KParams P) { render_bwd_tile_body<true>(P); }

}  // namespace nsb
