// nsb_common.cuh -- shared constants, packed-decoder layout and PTX helpers for the sm_100a kernels.
//
// Packed decoder image = what one CTA stages into shared memory with a single TMA bulk copy
// (cp.async.bulk) before it evaluates that decoder.  Every matrix keeps the reference's [out][in]
// orientation (nn.Linear.weight, src/conv_onet/models/decoder.py:117-164) with the row pitch padded to
// pitch == 4 (mod 8) floats, which makes BOTH access patterns of the kernels bank-conflict free:
//   forward   acc[pt][n] += A[k][pt] * W[n][k]   (lanes stride rows n = og + 8j, float4 along k)
//   backward  dx[pt][i]  += DU[o][pt] * W[o][i]  (lanes read consecutive float4 along i in row o)
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include "../../include/nice_slam_b200.h"

namespace nsb {

constexpr int kHid = 32;
constexpr int kEmb = 93;
constexpr int kEmbPad = 96;
constexpr int kChunk = 16;          // points per warp work item
constexpr int kRowF = 16;           // floats per activation row (one value per point of the chunk)
constexpr int kMaxPtsPerBlock = 384;
constexpr int kMaxRaysPerBlock = 24;

// ---------------------------------------------------------------------------------------------
// Per-level decoder shape + packed layout (offsets in floats, every block 16-byte aligned)
// ---------------------------------------------------------------------------------------------
template <int LV>
struct Dec {
  static constexpr bool XYZ = LV != 0;                 // MLP (xyz + Fourier embedding) vs MLP_no_xyz
  static constexpr int CD = LV == 2 ? 64 : 32;         // fc_c input width (fine: [fine | middle] concat)
  static constexpr int NO = LV == 3 ? 4 : 1;           // outputs
  static constexpr int FIRST = XYZ ? kEmb : 32;        // width of the first-layer / skip input
  static constexpr int FIRSTP = XYZ ? kEmbPad : 32;    // padded to a multiple of 4
  static constexpr int PF = FIRSTP + 4;                // row pitch of W0 / W3E
  static constexpr int PH = kHid + 4;                  // row pitch of the 32-wide matrices
  static constexpr int PC = CD + 4;                    // row pitch of the fc_c matrices
  static constexpr int o_B = 0;                        // [3][96]
  static constexpr int o_W0 = XYZ ? 3 * kEmbPad : 0;   // [32][PF]
  static constexpr int o_W1 = o_W0 + 32 * PF;          // [32][PH]
  static constexpr int o_W2 = o_W1 + 32 * PH;
  static constexpr int o_W3E = o_W2 + 32 * PH;         // [32][PF]  skip part (embedding / coarse feature)
  static constexpr int o_W3H = o_W3E + 32 * PF;        // [32][PH]  hidden part
  static constexpr int o_W4 = o_W3H + 32 * PH;
  static constexpr int o_WC = o_W4 + 32 * PH;          // [5*32][PC]  (XYZ only)
  static constexpr int o_WO = o_WC + (XYZ ? 160 * PC : 0);   // [4][PH]   rows >= NO are zero
  static constexpr int o_b = o_WO + 4 * PH;            // [5][32]
  static constexpr int o_bc = o_b + 160;               // [5][32]    (XYZ only)
  static constexpr int o_bo = o_bc + (XYZ ? 160 : 0);  // [4]
  static constexpr int TOTAL = o_bo + 4;
  static_assert(TOTAL % 4 == 0, "packed image must be a multiple of 16 bytes");
  // activation rows per warp
  static constexpr int ROWS_FWD = 32 + 64 + 64;                 // E-scratch | C | HA | HB
  static constexpr int ROWS_BWD = 32 + 64 + 160 + 32 + 32;      // E-scratch | C | S1..S5 | DU | DU3
};

__host__ __device__ constexpr int packed_floats(int lv) {
  return lv == 0 ? Dec<0>::TOTAL : lv == 1 ? Dec<1>::TOTAL : lv == 2 ? Dec<2>::TOTAL : Dec<3>::TOTAL;
}
constexpr int kMaxPacked = Dec<2>::TOTAL;
constexpr int kRowsFwd = Dec<2>::ROWS_FWD;     // 160
constexpr int kRowsBwd = Dec<2>::ROWS_BWD;     // 320

// ---- tensor-core operand images (appended to the packed fp32 image of every decoder by nsb_pack_decoders) -----------------------
// Every MMA B operand is stored ready to use: the 3xTF32 split (hi | lo) of a K-major no-swizzle canonical tile ([row/8][k/4][row%8][k%4]),
// in the order the kernels consume them, so one TMA bulk copy per unit replaces all in-kernel staging.  Behind the fp32 image:
//   header (kHdrFloats): b[5][32] | bc[5][32] | bo[4] | pad[12] | Wo[4][32] | B[3][96] | pad
//   | v2 forward units | v2 backward units | v3 forward units (below)
constexpr int kHdrFloats = 768;
__host__ __device__ constexpr int op_cd(int lv) { return lv == 2 ? 64 : 32; }
__host__ __device__ constexpr int op_firstp(int lv) { return lv == 0 ? 32 : kEmbPad; }
__host__ __device__ constexpr int op_nblk(int lv) { return lv == 0 ? 1 : 3; }
__host__ __device__ constexpr int op_hdr_offset(int lv) { return packed_floats(lv); }
// ---- v2 operand images (tile kernels, nsb_tile.cuh): the matrices cut into UNITS that stream through a 4-slot ring ----------------
//   forward : FC_u, u < cd/8   : [160 x 8]  rows 32 i + o = Wc_i[o][8 u + k]                                  (2560 floats hi|lo)
//             L0_{b,h}, h < 2  : [64 x 16]  rows o = W0[o][32 b + 16 h + k], rows 32 + o = W3E[o][...]          (2048 floats)
//             H_i, i = 1..4    : [32 x 32]  rows o = W_i[o][hidden k]                                          (2048 floats)
//   backward: for i = 4..0: DC_{i,c2}, c2 < cd/32 : rows c = Wc_i[k][32 c2 + c] | D1_i (i >= 1): rows j = W_i[k][hidden j]
//             | DF_{i,fb} (i = 3, 0), fb < firstp/32 : rows f = W_i[k][first-input 32 fb + f]                  (all [32 x 32], 2048 floats)
__host__ __device__ constexpr int op2_fc_units(int lv) { return lv == 0 ? 0 : op_cd(lv) / 8; }
__host__ __device__ constexpr int op2_fwd_units(int lv) { return op2_fc_units(lv) + 2 * op_nblk(lv) + 4; }
__host__ __device__ constexpr int op2_fwd_floats(int lv) { return op2_fc_units(lv) * 2560 + (2 * op_nblk(lv) + 4) * 2048; }
__host__ __device__ constexpr int op2_bwd_layer_units(int lv, int i) {
  return (lv != 0 ? op_cd(lv) / 32 : 0) + (i >= 1 ? 1 : 0) + ((i == 3 || i == 0) ? op_firstp(lv) / 32 : 0);
}
__host__ __device__ constexpr int op2_bwd_units(int lv) {
  int n = 0;
  for (int i = 0; i < 5; i++) n += op2_bwd_layer_units(lv, i);
  return n;
}
__host__ __device__ constexpr int op2_bwd_floats(int lv) { return op2_bwd_units(lv) * 2048; }
__host__ __device__ constexpr int op2_fwd_offset(int lv) { return op_hdr_offset(lv) + kHdrFloats; }
__host__ __device__ constexpr int op2_bwd_offset(int lv) { return op2_fwd_offset(lv) + op2_fwd_floats(lv); }
// ---- v3 forward image (tile kernels, option fwd_f16): the forward units as FP16 hi | lo pairs (x = hi + lo, hi = fp16(x), lo = fp16(x - hi): the same
// ~22-bit effective mantissa as the 3xTF32 split at half the bytes; tcgen05 kind::f16 contracts K = 16 per instruction).  16-bit canonical K-major
// tile: [row/8][k/8][row%8][k%8] halves (core matrix = 8 rows x 16 bytes).  Sizes in FLOAT units (2 halves each):
//   FC_u, u < cd/16 : [160 x 16] (2560)   L0_b, b < nblk : [64 x 32] (2048)   H_i, i = 1..4 : [32 x 32] (1024)
__host__ __device__ constexpr int op3_fc_units(int lv) { return lv == 0 ? 0 : op_cd(lv) / 16; }
__host__ __device__ constexpr int op3_fwd_units(int lv) { return op3_fc_units(lv) + op_nblk(lv) + 4; }
__host__ __device__ constexpr int op3_fwd_floats(int lv) { return op3_fc_units(lv) * 2560 + op_nblk(lv) * 2048 + 4 * 1024; }
__host__ __device__ constexpr int op3_fwd_offset(int lv) { return op2_bwd_offset(lv) + op2_bwd_floats(lv); }
__host__ __device__ constexpr int packed_total_floats(int lv) { return op3_fwd_offset(lv) + op3_fwd_floats(lv); }

// canonical flat layout (include/nice_slam_b200.h): kind 0=B 1=W 2=b 3=Wc 4=bc 5=Wo 6=bo 7=total
__host__ __device__ inline int dec_in(int lv, int i) {
  if (lv == 0) return i == 3 ? 64 : 32;
  return i == 0 ? kEmb : (i == 3 ? kEmb + kHid : kHid);
}
__host__ __device__ inline long long flat_offset(int lv, int kind, int layer) {
  const bool xyz = lv != 0;
  const int cd = lv == 2 ? 64 : 32, no = lv == 3 ? 4 : 1;
  long long off = 0;
  if (xyz) { if (kind == 0) return off; off += 3 * kEmb; }
  for (int i = 0; i < 5; i++) {
    if (kind == 1 && layer == i) return off; off += (long long)kHid * dec_in(lv, i);
    if (kind == 2 && layer == i) return off; off += kHid;
  }
  if (xyz) for (int i = 0; i < 5; i++) {
    if (kind == 3 && layer == i) return off; off += (long long)kHid * cd;
    if (kind == 4 && layer == i) return off; off += kHid;
  }
  if (kind == 5) return off; off += (long long)no * kHid;
  if (kind == 6) return off; off += no;
  return off;
}

// ---------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA bulk copy (global -> shared), vector reductions
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// TMA bulk copy global -> shared::cta, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// 16-byte vector reduction into global memory (sm_90+): one L2 atomic transaction for 4 floats
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ float4 ldg_f4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// activation-row swizzle: element (row r, point pt) lives at r*16 + ((pt>>2) ^ (r>>1))&3)*4 + (pt&3)
__device__ __forceinline__ int swz(int r, int q) { return ((q ^ (r >> 1)) & 3) << 2; }
__device__ __forceinline__ int act_idx(int r, int pt) { return r * kRowF + swz(r, pt >> 2) + (pt & 3); }

// Loss seeds fused into the forward launch (small batches): the last CTA of the forward kernel to finish computes them (nsb_seeds.cuh).
// Internal to the library: nsb_tracking_iteration / nsb_mapping_iteration use it through render_forward_fused().
// exchange buffers of a ray-sharded iteration as the kernels see them (nsb_peers of the C ABI; helpers in nsb_seeds.cuh)
struct PeerX {
  int rank, world;                   // world <= 1: no exchange
  unsigned char* peer[NSB_MAX_PEERS];
  unsigned long long* counter;       // this rank's sequence counters, one per channel
  int max_n;                         // residual-pool capacity per rank
};
// What the LAST CTA of a sharded backward launch adds to the fused pose gradient: SUM over ranks of [loss | d c2w] -> out13
struct PeerTail { PeerX px; const double* loss; double* out13; };
struct FusedSeeds {
  int kind;                      // 0 = none, 1 = tracking (Tracker.py:108-123), 2 = mapping (Mapper.py:487-493)
  const void* gt_rgb;            // float64 [N,3] (tracking) / float32 [N,3] (mapping)
  const float* gt_depth_loss;    // mapping: the depth the loss supervises with
  double w_color;
  int handle_dynamic, use_color;
  double* g_depth; float* g_rgb; double* loss;
  double* res;                   // tracking: residual scratch [N]
  int* counter;                  // grid-wide arrival counter, zero between launches
  PeerX px;                      // world > 1: sharded tracking batch -- depth maxima and the median pool are exchanged inside the forward launch
};
int render_forward_fused(const nsb_render_inputs* in, const nsb_forward_outputs* out, const FusedSeeds* fs, void* stream);
int render_backward_tail(const nsb_render_inputs* in, const nsb_backward_args* bw, const PeerTail* tail, void* stream);
int make_peerx(const struct nsb_peers* p, PeerX* px);

// error plumbing shared by the API translation units
void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

}  // namespace nsb
