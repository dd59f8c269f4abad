// nsb_aux.cu -- small kernels on either side of the render kernels + library plumbing:
//   decoder packing / gradient unpacking, batch depth maxima, ray pre-filter, loss seeds.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cuda_fp16.h>
#include "nsb_common.cuh"
#include "nsb_seeds.cuh"
#include "nsb_geom.cuh"

namespace nsb {

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return NSB_OK;
  set_error("%s: %s", what, cudaGetErrorString(e));
  (void)cudaGetLastError();      // non-sticky errors must not leak into the next call's launch check
  return NSB_ERR_CUDA;
}

// ------------------------------------------------------------------------------------------------ pack / unpack
// Maps every element of the reference parameter tensors to its slot in the packed image (nsb_common.cuh).
// DIR = 0: packed[slot] = param[i] ; DIR = 1: flat_grad[flat_i] += packed_grad[slot]
struct PackArgs { nsb_decoder_params p[4]; float* packed[4]; float* flat[4]; int present[4]; };
// The pack kernels run blockIdx.x = decoder level, blockIdx.y = slice.  The work of a level is a SEQUENCE of small independent pieces (23
// parameter tensors; ~75 operand tiles / units of <= 5120 elements): piece number e belongs to slice e % gridDim.y, whose 256 threads stride
// over it.  (One CTA per level took 46 + 34 us of every colour-decoder optimiser step; striding every piece over all slices still walked the
// pieces one after the other -- ~1 us of load -> store latency each, 15 + 26 us; now a slice handles 2-3 pieces.)
__device__ __forceinline__ bool pk_mine(int& e) { return (e++ % (int)gridDim.y) == (int)blockIdx.y; }
constexpr int kPackSlices = 32;

template <int LV, int DIR>
__device__ void pack_level(const PackArgs& A) {
  using D = Dec<LV>;
  float* pk = A.packed[LV];
  const nsb_decoder_params& p = A.p[LV];
  float* fl = A.flat[LV];
  int e = 0;                                                      // (DIR == 0: the launcher has zeroed the image, pads included)
  auto xfer = [&](const float* src, long long flat_off, int n, auto slot) {
    if (!pk_mine(e)) return;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int s = slot(i);
      if (DIR == 0) pk[s] = src[i]; else fl[flat_off + i] += pk[s];
    }
  };
  if (D::XYZ) xfer(p.B, flat_offset(LV, 0, 0), 3 * kEmb, [](int i) { return D::o_B + (i / kEmb) * kEmbPad + i % kEmb; });
  for (int l = 0; l < 5; l++) {
    const int nin = dec_in(LV, l);
    if (l == 0) xfer(p.W[0], flat_offset(LV, 1, 0), 32 * nin, [=](int i) { return D::o_W0 + (i / nin) * D::PF + i % nin; });
    else if (l == 3) xfer(p.W[3], flat_offset(LV, 1, 3), 32 * nin, [=](int i) {
      const int o = i / nin, k = i % nin;
      return k < D::FIRST ? D::o_W3E + o * D::PF + k : D::o_W3H + o * D::PH + (k - D::FIRST); });
    else {
      const int ow = l == 1 ? D::o_W1 : l == 2 ? D::o_W2 : D::o_W4;
      xfer(p.W[l], flat_offset(LV, 1, l), 32 * 32, [=](int i) { return ow + (i / 32) * D::PH + i % 32; });
    }
    xfer(p.b[l], flat_offset(LV, 2, l), 32, [=](int i) { return D::o_b + l * 32 + i; });
    if (D::XYZ) {
      xfer(p.Wc[l], flat_offset(LV, 3, l), 32 * D::CD, [=](int i) { return D::o_WC + (l * 32 + i / D::CD) * D::PC + i % D::CD; });
      xfer(p.bc[l], flat_offset(LV, 4, l), 32, [=](int i) { return D::o_bc + l * 32 + i; });
    }
  }
  xfer(p.Wo, flat_offset(LV, 5, 0), D::NO * 32, [](int i) { return D::o_WO + (i / 32) * D::PH + i % 32; });
  xfer(p.bo, flat_offset(LV, 6, 0), D::NO, [](int i) { return D::o_bo + i; });
}

template <int DIR>
__global__ void pack_kernel(const __grid_constant__ PackArgs A) {
  const int lv = blockIdx.x;
  if (!A.present[lv]) return;
  switch (lv) {
    case 0: pack_level<0, DIR>(A); break;
    case 1: pack_level<1, DIR>(A); break;
    case 2: pack_level<2, DIR>(A); break;
    default: pack_level<3, DIR>(A); break;
  }
}

// ---- tensor-core operand images (layout: nsb_common.cuh) --------------------------------------------------------------------
// header: biases, output weights and the embedding matrix of one decoder, read by the tile kernels
template <int LV>
__device__ void pack_header_level(float* __restrict__ img /* packed image of this level: raw part already written */, int& e) {
  using D = Dec<LV>;
  const float* W = img;
  float* dst = img + op_hdr_offset(LV);
  if (pk_mine(e)) for (int i = threadIdx.x; i < kHdrFloats; i += blockDim.x) {
    float v = 0.0f;
    if (i < 160) v = W[D::o_b + i];
    else if (i < 320) v = D::XYZ ? W[D::o_bc + (i - 160)] : 0.0f;
    else if (i < 324) v = W[D::o_bo + (i - 320)];
    else if (i >= 336 && i < 464) v = W[D::o_WO + ((i - 336) >> 5) * D::PH + ((i - 336) & 31)];
    else if (i >= 464 && i < 464 + 3 * kEmbPad) v = D::XYZ ? W[D::o_B + (i - 464)] : 0.0f;
    dst[i] = v;
  }
}
// ---- v2 operand images: units for the tile kernels (layout: nsb_common.cuh op2_*) -------------------------------------------------
// hi | lo of a [R x KW] canonical tile ([row/8][k/4][row%8][k%4]) whose element (row, k) is get(row, k)
template <typename F>
__device__ __forceinline__ void emit_unit(float*& dst, int& e, int R, int KW, F&& get) {
  float* hi = dst; float* lo = dst + R * KW;
  dst += 2 * R * KW;
  if (!pk_mine(e)) return;
  for (int idx = threadIdx.x; idx < R * KW; idx += blockDim.x) {
    const int r = idx / KW, k = idx - r * KW;
    const float v = get(r, k);
    const float h = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
    const int o = ((r >> 3) * (KW >> 2) + (k >> 2)) * 32 + (r & 7) * 4 + (k & 3);
    hi[o] = h; lo[o] = v - h;
  }
}
template <int LV>
__device__ void pack_units_level(float* __restrict__ img, int& e) {
  using D = Dec<LV>;
  const float* W = img;
  constexpr int PH = D::PH;
  const int o_wh[5] = {0, D::o_W1, D::o_W2, D::o_W3H, D::o_W4};
  float* dst = img + op2_fwd_offset(LV);
  if (D::XYZ)
    for (int u = 0; u < D::CD / 8; u++)
      emit_unit(dst, e, 160, 8, [&](int r, int k) { return W[D::o_WC + r * D::PC + 8 * u + k]; });
  for (int b = 0; b < op_nblk(LV); b++)
    for (int h = 0; h < 2; h++)
      emit_unit(dst, e, 64, 16, [&](int r, int k) { return W[(r < 32 ? D::o_W0 : D::o_W3E) + (r & 31) * D::PF + 32 * b + 16 * h + k]; });
  for (int i = 1; i < 5; i++) emit_unit(dst, e, 32, 32, [&](int r, int k) { return W[o_wh[i] + r * PH + k]; });
  dst = img + op2_bwd_offset(LV);
  for (int i = 4; i >= 0; i--) {
    if (D::XYZ)
      for (int c2 = 0; c2 < D::CD / 32; c2++)
        emit_unit(dst, e, 32, 32, [&](int c, int k) { return W[D::o_WC + (i * 32 + k) * D::PC + 32 * c2 + c]; });
    if (i >= 1) emit_unit(dst, e, 32, 32, [&](int j, int k) { return W[o_wh[i] + k * PH + j]; });
    if (i == 3 || i == 0)
      for (int fb = 0; fb < D::FIRSTP / 32; fb++)
        emit_unit(dst, e, 32, 32, [&](int f, int k) { return W[(i == 0 ? D::o_W0 : D::o_W3E) + k * D::PF + 32 * fb + f]; });
  }
}
// ---- v3 forward image: FP16 hi | lo units (layout: nsb_common.cuh op3_*) ----------------------------------------------------------------
template <typename F>
__device__ __forceinline__ void emit_unit_h16(__half*& dst, int& e, int R, int KW, F&& get) {
  __half* hi = dst; __half* lo = dst + R * KW;
  dst += 2 * R * KW;
  if (!pk_mine(e)) return;
  for (int idx = threadIdx.x; idx < R * KW; idx += blockDim.x) {
    const int r = idx / KW, k = idx - r * KW;
    const float v = get(r, k);
    const __half h = __float2half_rn(v);
    const int o = ((r >> 3) * (KW >> 3) + (k >> 3)) * 64 + (r & 7) * 8 + (k & 7);
    hi[o] = h; lo[o] = __float2half_rn(v - __half2float(h));
  }
}
template <int LV>
__device__ void pack_units_h16_level(float* __restrict__ img, int& e) {
  using D = Dec<LV>;
  const float* W = img;
  constexpr int PH = D::PH;
  const int o_wh[5] = {0, D::o_W1, D::o_W2, D::o_W3H, D::o_W4};
  __half* dst = reinterpret_cast<__half*>(img + op3_fwd_offset(LV));
  if (D::XYZ)
    for (int u = 0; u < D::CD / 16; u++)
      emit_unit_h16(dst, e, 160, 16, [&](int r, int k) { return W[D::o_WC + r * D::PC + 16 * u + k]; });
  for (int b = 0; b < op_nblk(LV); b++)
    emit_unit_h16(dst, e, 64, 32, [&](int r, int k) { return W[(r < 32 ? D::o_W0 : D::o_W3E) + (r & 31) * D::PF + 32 * b + k]; });
  for (int i = 1; i < 5; i++) emit_unit_h16(dst, e, 32, 32, [&](int r, int k) { return W[o_wh[i] + r * PH + k]; });
}
__global__ void pack_operands_kernel(const __grid_constant__ PackArgs A) {
  const int lv = blockIdx.x;
  if (!A.present[lv]) return;
  int e = 0;                                                      // piece counter (pk_mine)
  switch (lv) {
    case 0: pack_header_level<0>(A.packed[0], e); pack_units_level<0>(A.packed[0], e); pack_units_h16_level<0>(A.packed[0], e); break;
    case 1: pack_header_level<1>(A.packed[1], e); pack_units_level<1>(A.packed[1], e); pack_units_h16_level<1>(A.packed[1], e); break;
    case 2: pack_header_level<2>(A.packed[2], e); pack_units_level<2>(A.packed[2], e); pack_units_h16_level<2>(A.packed[2], e); break;
    default: pack_header_level<3>(A.packed[3], e); pack_units_level<3>(A.packed[3], e); pack_units_h16_level<3>(A.packed[3], e); break;
  }
}

int launch_unpack_grads(float* const d_packed[4], float* const d_flat[4], cudaStream_t st) {
  PackArgs A; memset(&A, 0, sizeof(A));
  for (int l = 0; l < 4; l++) { A.packed[l] = d_packed[l]; A.flat[l] = d_flat[l]; A.present[l] = d_packed[l] != nullptr && d_flat[l] != nullptr; }
  pack_kernel<1><<<dim3(4, kPackSlices), 256, 0, st>>>(A);
  return check_cuda(cudaGetLastError(), "unpack_grads launch");
}

// ------------------------------------------------------------------------------------------------ batch max
__global__ void batch_max_kernel(const float* __restrict__ gt, int n, float* __restrict__ out2, const PeerX px) {
  __shared__ float red[32];
  float m = -INFINITY;
  for (int i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, gt[i]);
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : -INFINITY;
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) {
      if (n <= 0) m = 0.0f;
      out2[0] = m;                       // torch.max(gt_depth)            (Renderer.py:144)
      out2[1] = __fmul_rn(m, 1.2f);      // torch.max(gt_depth*1.2): x -> fl(1.2f*x) is monotone, so max commutes (Renderer.py:109)
    }
  }
  if (px.world > 1) {                    // MAX over the ray shards of all ranks (channel 0: one LL word {max | sequence number} per rank)
    __shared__ uint32_t s_seq;
    __syncthreads();
    const uint32_t seq = peer_begin(px, 0, &s_seq);
    const int par = seq & 1u;
    if ((int)threadIdx.x < px.world) ll_put_f32(px.peer[threadIdx.x] + kXMaxOff + ((size_t)par * NSB_MAX_PEERS + px.rank) * 16, out2[0], seq);
    if (threadIdx.x < 32) {
      float mm = -INFINITY;
      if ((int)threadIdx.x < px.world) mm = ll_get_f32(px.peer[px.rank] + kXMaxOff + ((size_t)par * NSB_MAX_PEERS + threadIdx.x) * 16, seq, px, 0);
      for (int o = 16; o > 0; o >>= 1) mm = fmaxf(mm, __shfl_xor_sync(0xffffffffu, mm, o));
      if (threadIdx.x == 0) { out2[0] = mm; out2[1] = __fmul_rn(mm, 1.2f); }
    }
    peer_end(px, 0, seq);
  }
}

// ------------------------------------------------------------------------------------------------ ray pre-filter
struct Bound6 { double b[6]; };
__global__ void prefilter_kernel(const float* __restrict__ ro, const float* __restrict__ rd, const float* __restrict__ gt,
                                 int n, const Bound6 B, uint8_t* __restrict__ keep) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float o[3] = {ro[3 * i], ro[3 * i + 1], ro[3 * i + 2]}, d[3] = {rd[3 * i], rd[3 * i + 1], rd[3 * i + 2]};
  const double t = ray_far_bb(B.b, o, d);
  keep[i] = (t >= (double)gt[i]) ? 1 : 0;          // Tracker.py:101 / Mapper.py:478
}

// ------------------------------------------------------------------------------------------------ loss seeds
// Stand-alone single-CTA kernels (large batches, sharded batches, direct C-ABI use).  nsb_seeds.cuh holds the same computations as
// device functions over caller-provided scratch for the tail of the forward kernels (small batches: no separate launch).
// Tracker.optimize_cam_in_batch loss (src/Tracker.py:108-123); single CTA, residuals staged in `res`.
__global__ void tracking_seeds_kernel(const double* __restrict__ depth, const double* __restrict__ var, const float* __restrict__ rgb,
                                      const float* __restrict__ gt, const double* __restrict__ gt_rgb, int n, double w_color,
                                      int handle_dynamic, int use_color, const double* __restrict__ pool, int n_pool,
                                      double* __restrict__ g_depth, float* __restrict__ g_rgb,
                                      double* __restrict__ loss, double* __restrict__ res, const PeerX px) {
  __shared__ __align__(16) unsigned char scratch[kSeedsScratchBytes];
  tracking_seeds_body(depth, var, rgb, gt, gt_rgb, n, w_color, handle_dynamic, use_color, pool, n_pool, g_depth, g_rgb, loss, res, px, scratch);
}

// Mapper.optimize_map loss (src/Mapper.py:487-493); single CTA (deterministic sum)
__global__ void mapping_seeds_kernel(const double* __restrict__ depth, const float* __restrict__ rgb, const float* __restrict__ gt,
                                     const float* __restrict__ gt_rgb, int n, double w_color, int use_color,
                                     double* __restrict__ g_depth, float* __restrict__ g_rgb, double* __restrict__ loss) {
  __shared__ __align__(16) unsigned char scratch[kSeedsScratchBytes];
  mapping_seeds_body(depth, rgb, gt, gt_rgb, n, w_color, use_color, g_depth, g_rgb, loss, scratch);
}


// d c2w from ray gradients (single CTA, deterministic)
__global__ void pose_grad_kernel(const float* __restrict__ dirs, const float* __restrict__ dro, const float* __restrict__ drd, int n,
                                 double* __restrict__ out, const double* __restrict__ loss_local, const PeerX px) {
  __shared__ double red[32];
  double acc[12];
#pragma unroll
  for (int k = 0; k < 12; k++) acc[k] = 0.0;
  for (int r = threadIdx.x; r < n; r += blockDim.x) {
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const double g = (double)drd[3 * r + i];
#pragma unroll
      for (int j = 0; j < 3; j++) acc[4 * i + j] += g * (double)dirs[3 * r + j];
      acc[4 * i + 3] += (double)dro[3 * r + i];
    }
  }
  __shared__ double tot[13];
  for (int k = 0; k < 12; k++) { const double t = block_sum(acc[k], red); if (threadIdx.x == 0) tot[k + 1] = t; }
  if (px.world <= 1) {
    if (threadIdx.x == 0) for (int k = 0; k < 12; k++) out[k] = tot[k + 1];
    return;
  }
  // SUM over ranks of [loss | d c2w] through peer memory (channel 2: slot = 13 doubles + flag in 128 bytes); out = 13 doubles.
  __shared__ uint32_t s_seq;
  if (threadIdx.x == 0) tot[0] = loss_local != nullptr ? loss_local[0] : 0.0;
  __syncthreads();
  peer_sum13(px, tot, 13, out, &s_seq);
}

// ---- masked voxel parameterisation (Mapper.py:317-333, :393-401, :511-519) --------------------------------------------
constexpr int kScanBlock = 1024;
__global__ void slots_count_kernel(const uint8_t* __restrict__ mask, long long n, int* __restrict__ block_count) {
  __shared__ int red[32];
  const long long i = (long long)blockIdx.x * kScanBlock + threadIdx.x;
  int v = (i < n && mask[i]) ? 1 : 0;
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    int t = red[threadIdx.x];
    for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) block_count[blockIdx.x] = t;
  }
}
// single CTA: exclusive scan of the block counts in place, total -> count[0]
__global__ void slots_scan_kernel(int* __restrict__ block_count, int n_blocks, int* __restrict__ count) {
  __shared__ int warp_tot[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n_blocks; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = i < n_blocks ? block_count[i] : 0;
    int inc = v;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if ((threadIdx.x & 31) >= o) inc += t; }
    if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
      int t = warp_tot[threadIdx.x];
      for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, t, o); if (threadIdx.x >= o) t += u; }
      warp_tot[threadIdx.x] = t;                               // inclusive over warps
    }
    __syncthreads();
    const int before = carry + ((threadIdx.x >> 5) ? warp_tot[(threadIdx.x >> 5) - 1] : 0) + inc - v;
    if (i < n_blocks) block_count[i] = before;
    __syncthreads();
    if (threadIdx.x == 0) carry += warp_tot[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) count[0] = carry;
}
__global__ void slots_write_kernel(const uint8_t* __restrict__ mask, long long n, const int* __restrict__ block_base, int32_t* __restrict__ slots) {
  __shared__ int warp_tot[32];
  const long long i = (long long)blockIdx.x * kScanBlock + threadIdx.x;
  const int v = (i < n && mask[i]) ? 1 : 0;
  const unsigned b = __ballot_sync(0xffffffffu, v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) warp_tot[warp] = __popc(b);
  __syncthreads();
  if (threadIdx.x < 32) {
    int t = warp_tot[threadIdx.x];
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, t, o); if (threadIdx.x >= o) t += u; }
    warp_tot[threadIdx.x] = t;
  }
  __syncthreads();
  if (i < n) slots[i] = v ? block_base[blockIdx.x] + (warp ? warp_tot[warp - 1] : 0) + __popc(b & ((1u << lane) - 1u)) : -1;
}
// one warp per voxel quad-row: lane -> channel; DIR 0: compact = grid[voxel], 1: grid[voxel] = compact
template <int DIR>
__global__ void masked_copy_kernel(nsb_grid g, const int32_t* __restrict__ slots, float* __restrict__ compact) {
  const long long n = (long long)g.D * g.H * g.W;
  const int lane = threadIdx.x & 31;
  for (long long v = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); v < n; v += (long long)gridDim.x * (blockDim.x >> 5)) {
    const int s = __ldg(slots + v);
    if (s < 0) continue;
    const int w = (int)(v % g.W), h = (int)((v / g.W) % g.H), d = (int)(v / ((long long)g.W * g.H));
    float* cell = const_cast<float*>(g.data) + d * g.stride_d + h * g.stride_h + w * g.stride_w + lane * g.stride_c;
    if (DIR == 0) compact[(long long)s * 32 + lane] = *cell; else *cell = compact[(long long)s * 32 + lane];
  }
}
__global__ void compact_transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, long long n, int to_ref) {
  __shared__ float tile[32][33];
  const long long v0 = (long long)blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;                         // 32 x 8 threads
  for (int r = ty; r < 32; r += 8) {
    const long long v = v0 + (to_ref ? r : tx);
    const int c = to_ref ? tx : r;
    if (v < n) tile[r][tx] = to_ref ? src[v * 32 + c] : src[(long long)c * n + v];
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const long long v = v0 + (to_ref ? tx : r);
    const int c = to_ref ? r : tx;
    if (v < n) { if (to_ref) dst[(long long)c * n + v] = tile[tx][r]; else dst[v * 32 + c] = tile[tx][r]; }
  }
}

// ---- frustum feature selection (Mapper.get_mask_from_c2w, Mapper.py:93-164) -------------------------------------------------------
struct FrustumArgs {
  float w2c[12];                    // rows 0..2 of inverse(c2w), float32 like the reference's numpy pipeline
  float cam_o[3];                   // c2w[:3,3]
  const float* xs; const float* ys; const float* zs;      // voxel-centre coordinates per axis (torch.linspace over the bound, Mapper.py:108-110)
  int D, H, W;
  const float* depth; int img_h, img_w;
  double fx, fy, cx, cy;
};
__device__ __forceinline__ float img_px(const float* __restrict__ img, int h, int w, int y, int x) {
  return (x >= 0 && x < w && y >= 0 && y < h) ? __ldg(img + (long long)y * w + x) : 0.0f;      // BORDER_CONSTANT 0
}
// cv2.remap(..., INTER_LINEAR) of a float32 image at float32 coordinates: 1/32-pixel fixed point + float32 bilinear table (remap.cpp)
__device__ __forceinline__ float remap_bilinear(const float* __restrict__ img, int h, int w, float x, float y) {
  const long long sx = llrint((double)x * 32.0), sy = llrint((double)y * 32.0);
  long long ixl = sx >> 5, iyl = sy >> 5;
  ixl = ixl < -32768 ? -32768 : (ixl > 32767 ? 32767 : ixl); iyl = iyl < -32768 ? -32768 : (iyl > 32767 ? 32767 : iyl);
  const int ix = (int)ixl, iy = (int)iyl;
  const float fx = __fdiv_rn((float)(sx & 31), 32.0f), fy = __fdiv_rn((float)(sy & 31), 32.0f);
  const float w00 = __fmul_rn(__fsub_rn(1.0f, fy), __fsub_rn(1.0f, fx)), w01 = __fmul_rn(__fsub_rn(1.0f, fy), fx);
  const float w10 = __fmul_rn(fy, __fsub_rn(1.0f, fx)), w11 = __fmul_rn(fy, fx);
  float r = __fmul_rn(img_px(img, h, w, iy, ix), w00);
  r = __fadd_rn(r, __fmul_rn(img_px(img, h, w, iy, ix + 1), w01));
  r = __fadd_rn(r, __fmul_rn(img_px(img, h, w, iy + 1, ix), w10));
  return __fadd_rn(r, __fmul_rn(img_px(img, h, w, iy + 1, ix + 1), w11));
}
struct FrustumPoint { float u, v; double z; float px, py, pz; };
__device__ __forceinline__ FrustumPoint frustum_project(const FrustumArgs& A, long long vox) {
  const int w = (int)(vox % A.W), h = (int)((vox / A.W) % A.H), d = (int)(vox / ((long long)A.W * A.H));
  FrustumPoint P; P.px = A.xs[w]; P.py = A.ys[h]; P.pz = A.zs[d];
  float c[3];
#pragma unroll
  for (int i = 0; i < 3; i++)      // float32 matrix-vector product, left to right (Mapper.py:121-122)
    c[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A.w2c[4 * i], P.px), __fmul_rn(A.w2c[4 * i + 1], P.py)), __fmul_rn(A.w2c[4 * i + 2], P.pz)), A.w2c[4 * i + 3]);
  c[0] = -c[0];                                                                     // :125
  const double uu = __dadd_rn(__dmul_rn(A.fx, (double)c[0]), __dmul_rn(A.cx, (double)c[2]));      // K @ cam in float64 (:126)
  const double vv = __dadd_rn(__dmul_rn(A.fy, (double)c[1]), __dmul_rn(A.cy, (double)c[2]));
  P.z = __dadd_rn((double)c[2], 1e-5);                                              // :127
  P.u = (float)__ddiv_rn(uu, P.z); P.v = (float)__ddiv_rn(vv, P.z);                 // :128-129
  return P;
}
// pass 1: looked-up depth of every voxel + its maximum (non-negative floats: the bit pattern is monotone)
__global__ void frustum_depth_kernel(const FrustumArgs A, float* __restrict__ depths, int* __restrict__ max_bits) {
  const long long n = (long long)A.D * A.H * A.W;
  float m = 0.0f;
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (long long)gridDim.x * blockDim.x) {
    const FrustumPoint P = frustum_project(A, v);
    const float dep = remap_bilinear(A.depth, A.img_h, A.img_w, P.u, P.v);
    depths[v] = dep;
    m = fmaxf(m, dep);
  }
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.0f) atomicMax(max_bits, __float_as_int(m));
}
// pass 2: image-bounds test, depth test (zeros replaced by the maximum, :144-147), ball around the camera centre (:153-161)
__global__ void frustum_mask_kernel(const FrustumArgs A, const float* __restrict__ depths, const int* __restrict__ max_bits, uint8_t* __restrict__ mask) {
  const long long n = (long long)A.D * A.H * A.W;
  const float dmax = __int_as_float(*max_bits);
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (long long)gridDim.x * blockDim.x) {
    const FrustumPoint P = frustum_project(A, v);
    float dep = depths[v];
    if (dep == 0.0f) dep = dmax;
    bool m = (P.u < (float)A.img_w) && (P.u > 0.0f) && (P.v < (float)A.img_h) && (P.v > 0.0f);
    const double nz = -P.z;
    m = m && (0.0 <= nz) && (nz <= (double)__fadd_rn(dep, 0.5f));                  // `depths + 0.5` stays float32 (numpy weak scalar), the comparison is float64
    const float dx = __fsub_rn(P.px, A.cam_o[0]), dy = __fsub_rn(P.py, A.cam_o[1]), dz = __fsub_rn(P.pz, A.cam_o[2]);
    const float dist = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    mask[v] = (m || dist < 0.25f) ? 1 : 0;
  }
}

// ---- fused Adam on the packed gradient block (torch.optim.Adam defaults; Mapper.py:365-379, :412-419, :504) ------------------------
struct AdamScalars { float w1, beta2, w2, inv_bc2_sqrt_div, eps, neg_step; };     // float32 casts of torch's python scalars
__device__ __forceinline__ float adam_update(float p, float g, float& m, float& v, const AdamScalars& a) {
  m = __fadd_rn(m, __fmul_rn(a.w1, __fsub_rn(g, m)));                                  // exp_avg.lerp_(grad, 1 - beta1)
  v = __fadd_rn(__fmul_rn(v, a.beta2), __fmul_rn(__fmul_rn(a.w2, g), g));              // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1-beta2)
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), a.inv_bc2_sqrt_div), a.eps);   // (exp_avg_sq.sqrt() / bias_correction2_sqrt).add_(eps)
  return __fadd_rn(p, __fmul_rn(a.neg_step, __fdiv_rn(m, denom)));                     // param.addcdiv_(exp_avg, denom, value=-step_size)
}
// one warp per voxel, lane = channel: the parameters ARE the selected voxels of the shared grid (updated in place)
__global__ void adam_masked_kernel(nsb_grid g, const int32_t* __restrict__ slots, const float* __restrict__ grad, float* __restrict__ em,
                                   float* __restrict__ ev, const AdamScalars a) {
  const long long n = (long long)g.D * g.H * g.W;
  const int lane = threadIdx.x & 31;
  for (long long vx = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); vx < n; vx += (long long)gridDim.x * (blockDim.x >> 5)) {
    const int s = __ldg(slots + vx);
    if (s < 0) continue;
    const int w = (int)(vx % g.W), h = (int)((vx / g.W) % g.H), d = (int)(vx / ((long long)g.W * g.H));
    float* cell = const_cast<float*>(g.data) + d * g.stride_d + h * g.stride_h + w * g.stride_w + lane * g.stride_c;
    const long long i = (long long)s * 32 + lane;
    float m = em[i], v = ev[i];
    *cell = adam_update(*cell, grad[i], m, v, a);
    em[i] = m; ev[i] = v;
  }
}
struct AdamTable { float* param[24]; int off[24]; int n[24]; int count; };
__global__ void adam_flat_kernel(const AdamTable T, const float* __restrict__ grad, float* __restrict__ em, float* __restrict__ ev, const AdamScalars a) {
  for (int t = 0; t < T.count; t++)
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < T.n[t]; i += gridDim.x * blockDim.x) {
      const int f = T.off[t] + i;
      float m = em[f], v = ev[f];
      T.param[t][i] = adam_update(T.param[t][i], grad[f], m, v, a);
      em[f] = m; ev[f] = v;
    }
}

// the mapper's whole optimiser step in ONE launch: CTAs [blk0[g], blk0[g+1]) update voxel group g, the last 32 CTAs the decoder
struct MapperAdamArgs {
  nsb_grid g[4]; const int32_t* slots[4]; const float* grad[4]; float* em[4]; float* ev[4]; AdamScalars a[4]; int blk0[5]; int n_groups;
  AdamTable T; const float* dgrad; float* dem; float* dev; AdamScalars da; int dec_blocks;
};
__global__ void adam_mapper_kernel(const __grid_constant__ MapperAdamArgs A) {
  const int b = blockIdx.x;
  if (b >= A.blk0[A.n_groups]) {                                   // decoder (adam_flat_kernel)
    const int bd = b - A.blk0[A.n_groups];
    for (int t = 0; t < A.T.count; t++)
      for (int i = bd * blockDim.x + threadIdx.x; i < A.T.n[t]; i += A.dec_blocks * blockDim.x) {
        const int f = A.T.off[t] + i;
        float m = A.dem[f], v = A.dev[f];
        A.T.param[t][i] = adam_update(A.T.param[t][i], A.dgrad[f], m, v, A.da);
        A.dem[f] = m; A.dev[f] = v;
      }
    return;
  }
  int q = 0;
  while (q + 1 < A.n_groups && b >= A.blk0[q + 1]) q++;
  const nsb_grid& g = A.g[q];
  const int nb = A.blk0[q + 1] - A.blk0[q], bq = b - A.blk0[q];
  const long long n = (long long)g.D * g.H * g.W;
  const int lane = threadIdx.x & 31;
  for (long long vx = (long long)bq * (blockDim.x >> 5) + (threadIdx.x >> 5); vx < n; vx += (long long)nb * (blockDim.x >> 5)) {      // (adam_masked_kernel)
    const int s = __ldg(A.slots[q] + vx);
    if (s < 0) continue;
    const int w = (int)(vx % g.W), h = (int)((vx / g.W) % g.H), d = (int)(vx / ((long long)g.W * g.H));
    float* cell = const_cast<float*>(g.data) + d * g.stride_d + h * g.stride_h + w * g.stride_w + lane * g.stride_c;
    const long long i = (long long)s * 32 + lane;
    float m = A.em[q][i], v = A.ev[q][i];
    *cell = adam_update(*cell, A.grad[q][i], m, v, A.a[q]);
    A.em[q][i] = m; A.ev[q][i] = v;
  }
}

// d c2w of every keyframe block (one CTA per frame)
__global__ void pose_grad_frames_kernel(const float* __restrict__ dirs, const float* __restrict__ dro, const float* __restrict__ drd,
                                        const int32_t* __restrict__ offs, float* __restrict__ out) {
  __shared__ double red[32];
  const int lo = offs[blockIdx.x], hi = offs[blockIdx.x + 1];
  double acc[12];
#pragma unroll
  for (int k = 0; k < 12; k++) acc[k] = 0.0;
  for (int r = lo + threadIdx.x; r < hi; r += blockDim.x) {
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const double g = (double)drd[3 * r + i];
#pragma unroll
      for (int j = 0; j < 3; j++) acc[4 * i + j] += g * (double)dirs[3 * r + j];
      acc[4 * i + 3] += (double)dro[3 * r + i];
    }
  }
  for (int k = 0; k < 12; k++) { const double t = block_sum(acc[k], red); if (threadIdx.x == 0) out[12 * blockIdx.x + k] = (float)t; }
}

}  // namespace nsb

using namespace nsb;

static PeerX no_peers() { PeerX px; memset(&px, 0, sizeof(px)); return px; }
static int make_peers(const nsb_peers* p, PeerX* px) {
  if (!p || p->world < 2 || p->world > NSB_MAX_PEERS || p->rank < 0 || p->rank >= p->world || !p->counters || p->max_rays < 1) {
    set_error("peer exchange: bad nsb_peers"); return NSB_ERR_ARG; }
  memset(px, 0, sizeof(*px));
  px->rank = p->rank; px->world = p->world; px->counter = p->counters; px->max_n = p->max_rays;
  for (int r = 0; r < p->world; r++) {
    if (!p->buffer[r]) { set_error("peer exchange: buffer[%d] is NULL", r); return NSB_ERR_ARG; }
    px->peer[r] = static_cast<unsigned char*>(p->buffer[r]);
  }
  return NSB_OK;
}
int nsb::make_peerx(const nsb_peers* p, PeerX* px) { return make_peers(p, px); }
extern "C" size_t nsb_peer_buffer_bytes(int max_rays) { return max_rays < 1 ? 0 : peer_buffer_bytes(max_rays); }

// ------------------------------------------------------------------------------------------------ small host <-> device blocks, copied by the SMs
// The per-iteration inputs of a tracking iteration are ~10 KB and its results ~5 KB (steps.IterationContext blocks).  As copy-engine nodes of a CUDA
// graph each of them costs a DMA launch + engine <-> SM synchronisation; one CTA whose threads each move one 16-byte word over the mapped view of the
// pinned host block has every word in flight at once: one PCIe round trip.  Either side may be device memory or mapped pinned host memory.
__global__ void __launch_bounds__(1024) block_copy_kernel(uint4* __restrict__ dst, const uint4* __restrict__ src, size_t n16, size_t tail_off, int tail) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) __stwt(dst + i, __ldcv(src + i));
  if (blockIdx.x == 0 && (int)threadIdx.x < tail)
    reinterpret_cast<unsigned char*>(dst)[tail_off + threadIdx.x] = reinterpret_cast<const volatile unsigned char*>(src)[tail_off + threadIdx.x];
  __threadfence_system();
}
extern "C" void* nsb_host_device_pointer(void* pinned_host) {
  void* d = nullptr;
  if (!pinned_host) { set_error("host_device_pointer: NULL"); return nullptr; }
  if (check_cuda(cudaHostGetDevicePointer(&d, pinned_host, 0), "cudaHostGetDevicePointer (is the block page-locked?)")) return nullptr;
  return d;
}
extern "C" int nsb_copy_block(void* dst, const void* src, size_t bytes, void* stream) {
  if (bytes == 0) return NSB_OK;
  if (!dst || !src || (((uintptr_t)dst | (uintptr_t)src) & 15)) { set_error("copy_block: pointers must be non-NULL and 16-byte aligned"); return NSB_ERR_ARG; }
  const size_t n16 = bytes >> 4;
  const int tail = (int)(bytes & 15);
  const int grid = (int)((n16 + 1023) / 1024 < 1 ? 1 : ((n16 + 1023) / 1024 > 64 ? 64 : (n16 + 1023) / 1024));
  block_copy_kernel<<<grid, 1024, 0, (cudaStream_t)stream>>>(static_cast<uint4*>(dst), static_cast<const uint4*>(src), n16, n16 << 4, tail);
  return check_cuda(cudaGetLastError(), "copy_block launch");
}

extern "C" int nsb_pose_grad(const float* dirs, const float* d_rays_o, const float* d_rays_d, int n, double* d_c2w, void* stream) {
  if (n < 0 || !d_c2w || (n > 0 && (!dirs || !d_rays_o || !d_rays_d))) { set_error("pose_grad: bad arguments"); return NSB_ERR_ARG; }
  pose_grad_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(dirs, d_rays_o, d_rays_d, n, d_c2w, nullptr, no_peers());
  return check_cuda(cudaGetLastError(), "pose_grad launch");
}
extern "C" int nsb_pose_grad_peers(const float* dirs, const float* d_rays_o, const float* d_rays_d, int n, const double* loss_local,
                                   double* loss_and_d_c2w, const nsb_peers* peers, void* stream) {
  if (n < 0 || !loss_and_d_c2w || (n > 0 && (!dirs || !d_rays_o || !d_rays_d))) { set_error("pose_grad_peers: bad arguments"); return NSB_ERR_ARG; }
  PeerX px; int rc = make_peers(peers, &px); if (rc) return rc;
  pose_grad_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(dirs, d_rays_o, d_rays_d, n, loss_and_d_c2w, loss_local, px);
  return check_cuda(cudaGetLastError(), "pose_grad_peers launch");
}

extern "C" size_t nsb_voxel_slots_workspace(long long n_voxels) {
  return n_voxels <= 0 ? 16 : (size_t)((n_voxels + kScanBlock - 1) / kScanBlock) * sizeof(int) + 16;
}
extern "C" int nsb_voxel_slots(const uint8_t* voxel_mask, long long n_voxels, int32_t* slot_map, int32_t* count,
                               void* workspace, size_t workspace_bytes, void* stream) {
  if (n_voxels < 0 || !count || (n_voxels > 0 && (!voxel_mask || !slot_map || !workspace))) { set_error("voxel_slots: bad arguments"); return NSB_ERR_ARG; }
  if (workspace_bytes < nsb_voxel_slots_workspace(n_voxels)) { set_error("voxel_slots: workspace too small"); return NSB_ERR_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  if (n_voxels == 0) return check_cuda(cudaMemsetAsync(count, 0, sizeof(int32_t), st), "voxel_slots memset");
  const int nb = (int)((n_voxels + kScanBlock - 1) / kScanBlock);
  int* bc = static_cast<int*>(workspace);
  slots_count_kernel<<<nb, kScanBlock, 0, st>>>(voxel_mask, n_voxels, bc);
  slots_scan_kernel<<<1, 1024, 0, st>>>(bc, nb, count);
  slots_write_kernel<<<nb, kScanBlock, 0, st>>>(voxel_mask, n_voxels, bc, slot_map);
  return check_cuda(cudaGetLastError(), "voxel_slots launch");
}
static int masked_copy(const nsb_grid* g, const int32_t* slots, float* compact, int dir, void* stream) {
  if (!g || !g->data || !slots || !compact || g->D <= 0 || g->H <= 0 || g->W <= 0) { set_error("masked gather/scatter: bad arguments"); return NSB_ERR_ARG; }
  const long long n = (long long)g->D * g->H * g->W;
  const int blocks = (int)((n + 7) / 8 < 148 * 16 ? (n + 7) / 8 : 148 * 16);
  if (dir == 0) masked_copy_kernel<0><<<blocks, 256, 0, (cudaStream_t)stream>>>(*g, slots, compact);
  else masked_copy_kernel<1><<<blocks, 256, 0, (cudaStream_t)stream>>>(*g, slots, compact);
  return check_cuda(cudaGetLastError(), "masked copy launch");
}
extern "C" int nsb_masked_gather(const nsb_grid* grid, const int32_t* slot_map, float* compact, void* stream) { return masked_copy(grid, slot_map, compact, 0, stream); }
extern "C" int nsb_masked_scatter(const nsb_grid* grid, const int32_t* slot_map, const float* compact, void* stream) {
  return masked_copy(grid, slot_map, const_cast<float*>(compact), 1, stream);
}
extern "C" int nsb_compact_transpose(const float* src, float* dst, long long n_selected, int to_reference, void* stream) {
  if (n_selected < 0 || (n_selected > 0 && (!src || !dst))) { set_error("compact_transpose: bad arguments"); return NSB_ERR_ARG; }
  if (n_selected == 0) return NSB_OK;
  compact_transpose_kernel<<<(unsigned)((n_selected + 31) / 32), 256, 0, (cudaStream_t)stream>>>(src, dst, n_selected, to_reference);
  return check_cuda(cudaGetLastError(), "compact_transpose launch");
}
static int adam_scalars(double lr, double beta1, double beta2, double eps, int step, AdamScalars* a) {
  if (step < 1 || !(beta1 >= 0.0 && beta1 < 1.0) || !(beta2 >= 0.0 && beta2 < 1.0) || !(eps >= 0.0)) { set_error("adam: bad hyper-parameters"); return NSB_ERR_ARG; }
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);      // python-float arithmetic of torch's _single_tensor_adam
  a->w1 = (float)(1.0 - beta1); a->beta2 = (float)beta2; a->w2 = (float)(1.0 - beta2);
  a->inv_bc2_sqrt_div = (float)sqrt(bc2); a->eps = (float)eps; a->neg_step = (float)(-(lr / bc1));
  return NSB_OK;
}
extern "C" int nsb_adam_masked_voxels(const nsb_grid* grid, const int32_t* slot_map, const float* grad, float* exp_avg, float* exp_avg_sq,
                                      double lr, double beta1, double beta2, double eps, int step, void* stream) {
  if (!grid || !grid->data || !slot_map || !grad || !exp_avg || !exp_avg_sq || grid->D < 1 || grid->H < 1 || grid->W < 1) {
    set_error("adam_masked_voxels: bad arguments"); return NSB_ERR_ARG; }
  AdamScalars a; int rc = adam_scalars(lr, beta1, beta2, eps, step, &a); if (rc) return rc;
  const long long n = (long long)grid->D * grid->H * grid->W;
  const int blocks = (int)((n + 7) / 8 < 148 * 16 ? (n + 7) / 8 : 148 * 16);
  adam_masked_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(*grid, slot_map, grad, exp_avg, exp_avg_sq, a);
  return check_cuda(cudaGetLastError(), "adam_masked_voxels launch");
}
static int adam_table(int level, const nsb_decoder_params* p, AdamTable* Tp) {
  AdamTable& T = *Tp; memset(&T, 0, sizeof(T));
  auto add = [&](const float* ptr, int kind, int layer, int n) { T.param[T.count] = const_cast<float*>(ptr); T.off[T.count] = (int)flat_offset(level, kind, layer); T.n[T.count] = n; T.count++; };
  const bool xyz = level != 0;
  const int cd = level == 2 ? 64 : 32, no = level == 3 ? 4 : 1;
  bool ok = p->Wo && p->bo;
  for (int i = 0; i < 5; i++) ok = ok && p->W[i] && p->b[i] && (!xyz || (p->Wc[i] && p->bc[i]));
  if (xyz) ok = ok && p->B;
  if (!ok) { set_error("adam_decoder: NULL parameter pointers"); return NSB_ERR_ARG; }
  if (xyz) add(p->B, 0, 0, 3 * kEmb);
  for (int i = 0; i < 5; i++) { add(p->W[i], 1, i, kHid * dec_in(level, i)); add(p->b[i], 2, i, kHid); }
  if (xyz) for (int i = 0; i < 5; i++) { add(p->Wc[i], 3, i, kHid * cd); add(p->bc[i], 4, i, kHid); }
  add(p->Wo, 5, 0, no * kHid); add(p->bo, 6, 0, no);
  return NSB_OK;
}
extern "C" int nsb_adam_decoder(int level, const nsb_decoder_params* p, const float* grad_flat, float* exp_avg, float* exp_avg_sq,
                                double lr, double beta1, double beta2, double eps, int step, void* stream) {
  if (level < 0 || level > 3 || !p || !grad_flat || !exp_avg || !exp_avg_sq) { set_error("adam_decoder: bad arguments"); return NSB_ERR_ARG; }
  AdamScalars a; int rc = adam_scalars(lr, beta1, beta2, eps, step, &a); if (rc) return rc;
  AdamTable T; if ((rc = adam_table(level, p, &T))) return rc;
  adam_flat_kernel<<<32, 256, 0, (cudaStream_t)stream>>>(T, grad_flat, exp_avg, exp_avg_sq, a);
  return check_cuda(cudaGetLastError(), "adam_decoder launch");
}
extern "C" int nsb_adam_mapper_step(const nsb_adam_voxel_group* groups, int n_groups, int dec_level, const nsb_decoder_params* dec_params,
                                    const float* dec_grad_flat, float* dec_exp_avg, float* dec_exp_avg_sq, double dec_lr, int dec_step,
                                    double beta1, double beta2, double eps, void* stream) {
  if (n_groups < 0 || n_groups > 4 || (n_groups > 0 && !groups)) { set_error("adam_mapper_step: 0..4 voxel groups"); return NSB_ERR_ARG; }
  MapperAdamArgs A; memset(&A, 0, sizeof(A));
  A.n_groups = n_groups;
  int rc;
  for (int q = 0; q < n_groups; q++) {
    const nsb_adam_voxel_group& G = groups[q];
    if (!G.grid.data || !G.slot_map || !G.grad || !G.exp_avg || !G.exp_avg_sq || G.grid.D < 1 || G.grid.H < 1 || G.grid.W < 1) {
      set_error("adam_mapper_step: bad voxel group %d", q); return NSB_ERR_ARG; }
    if ((rc = adam_scalars(G.lr, beta1, beta2, eps, G.step, &A.a[q]))) return rc;
    A.g[q] = G.grid; A.slots[q] = G.slot_map; A.grad[q] = G.grad; A.em[q] = G.exp_avg; A.ev[q] = G.exp_avg_sq;
    const long long n = (long long)G.grid.D * G.grid.H * G.grid.W;
    A.blk0[q + 1] = A.blk0[q] + (int)((n + 7) / 8 < 148 * 8 ? (n + 7) / 8 : 148 * 8);
  }
  if (dec_level >= 0) {
    if (dec_level > 3 || !dec_params || !dec_grad_flat || !dec_exp_avg || !dec_exp_avg_sq) { set_error("adam_mapper_step: bad decoder arguments"); return NSB_ERR_ARG; }
    if ((rc = adam_scalars(dec_lr, beta1, beta2, eps, dec_step, &A.da))) return rc;
    if ((rc = adam_table(dec_level, dec_params, &A.T))) return rc;
    A.dgrad = dec_grad_flat; A.dem = dec_exp_avg; A.dev = dec_exp_avg_sq; A.dec_blocks = 32;
  }
  const int blocks = A.blk0[n_groups] + A.dec_blocks;
  if (blocks == 0) return NSB_OK;
  adam_mapper_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(A);
  return check_cuda(cudaGetLastError(), "adam_mapper_step launch");
}

// ---- bundle-adjustment window: poses <-> rays (Mapper.py:346-363, :437-467, :521-540; common.py:74-89, :137-176) --------------------------
// quad2rotation (src/common.py:137-160), float32, same expression order; c2w row-major [3][4]
__device__ __forceinline__ void cam_to_c2w(const float* __restrict__ cam, float* __restrict__ m) {
  const float qr = cam[0], qi = cam[1], qj = cam[2], qk = cam[3];
  const float nn = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(qr, qr), __fmul_rn(qi, qi)), __fmul_rn(qj, qj)), __fmul_rn(qk, qk));
  const float s = __fdiv_rn(2.0f, nn);
  m[0] = __fsub_rn(1.0f, __fmul_rn(s, __fadd_rn(__fmul_rn(qj, qj), __fmul_rn(qk, qk))));
  m[1] = __fmul_rn(s, __fsub_rn(__fmul_rn(qi, qj), __fmul_rn(qk, qr)));
  m[2] = __fmul_rn(s, __fadd_rn(__fmul_rn(qi, qk), __fmul_rn(qj, qr)));
  m[4] = __fmul_rn(s, __fadd_rn(__fmul_rn(qi, qj), __fmul_rn(qk, qr)));
  m[5] = __fsub_rn(1.0f, __fmul_rn(s, __fadd_rn(__fmul_rn(qi, qi), __fmul_rn(qk, qk))));
  m[6] = __fmul_rn(s, __fsub_rn(__fmul_rn(qj, qk), __fmul_rn(qi, qr)));
  m[8] = __fmul_rn(s, __fsub_rn(__fmul_rn(qi, qk), __fmul_rn(qj, qr)));
  m[9] = __fmul_rn(s, __fadd_rn(__fmul_rn(qj, qk), __fmul_rn(qi, qr)));
  m[10] = __fsub_rn(1.0f, __fmul_rn(s, __fadd_rn(__fmul_rn(qi, qi), __fmul_rn(qj, qj))));
  m[3] = cam[4]; m[7] = cam[5]; m[11] = cam[6];
}
// poses of the window rows: row f uses camera tensor cam_row[f] (>= 0) or, for the fixed oldest frame (-1), fixed_c2w[f]
__global__ void window_poses_kernel(const float* __restrict__ cams, const int32_t* __restrict__ cam_row, const float* __restrict__ fixed_c2w,
                                    int n_frames, float* __restrict__ c2w_out) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_frames) return;
  float m[12];
  if (cam_row[f] >= 0) cam_to_c2w(cams + 7 * cam_row[f], m);
  else for (int k = 0; k < 12; k++) m[k] = fixed_c2w[12 * f + k];
  for (int k = 0; k < 12; k++) c2w_out[12 * f + k] = m[k];
}
// get_rays_from_uv (src/common.py:74-89): dirs = [(i-cx)/fx, -(j-cy)/fy, -1]; rays_d = sum_j dirs_j * R[:, j]; rays_o = t
__global__ void window_rays_kernel(const float* __restrict__ c2w, const float* __restrict__ pix_i, const float* __restrict__ pix_j,
                                   const int32_t* __restrict__ frame_of_ray, int n, float fx, float fy, float cx, float cy,
                                   float* __restrict__ rays_o, float* __restrict__ rays_d, float* __restrict__ dirs) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const float* m = c2w + 12 * frame_of_ray[r];
  const float d0 = __fdiv_rn(__fsub_rn(pix_i[r], cx), fx), d1 = -__fdiv_rn(__fsub_rn(pix_j[r], cy), fy), d2 = -1.0f;
#pragma unroll
  for (int a = 0; a < 3; a++) {
    rays_d[3 * r + a] = __fadd_rn(__fadd_rn(__fmul_rn(d0, m[4 * a]), __fmul_rn(d1, m[4 * a + 1])), __fmul_rn(d2, m[4 * a + 2]));
    rays_o[3 * r + a] = m[4 * a + 3];
  }
  if (dirs != nullptr) { dirs[3 * r] = d0; dirs[3 * r + 1] = d1; dirs[3 * r + 2] = d2; }
}
// d camera tensor = (d c2w / d camera tensor)^T d c2w  (backward of get_camera_from_tensor), then torch.optim.Adam's update in place.
// One thread per camera tensor (a window has <= a few dozen).  g: d c2w [3][4] of the tensor's window row.
__global__ void adam_poses_kernel(float* __restrict__ cams, const int32_t* __restrict__ cam_row, int n_frames, const float* __restrict__ d_c2w,
                                  float* __restrict__ em, float* __restrict__ ev, float* __restrict__ d_cams, const AdamScalars a) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_frames || cam_row[f] < 0) return;
  const int c = cam_row[f];
  const float* g = d_c2w + 12 * f;
  float* q = cams + 7 * c;
  const float r = q[0], i = q[1], j = q[2], k = q[3];
  const float nn = r * r + i * i + j * j + k * k, s = 2.0f / nn;
  const float G00 = g[0], G01 = g[1], G02 = g[2], G10 = g[4], G11 = g[5], G12 = g[6], G20 = g[8], G21 = g[9], G22 = g[10];
  // R = I - s A' (diagonal) / s A (off-diagonal);  dL/ds, then ds/dq = -s^2 q
  const float dLds = -(G00 * (j * j + k * k) + G11 * (i * i + k * k) + G22 * (i * i + j * j))
                     + G01 * (i * j - k * r) + G02 * (i * k + j * r) + G10 * (i * j + k * r) + G12 * (j * k - i * r) + G20 * (i * k - j * r) + G21 * (j * k + i * r);
  float dq[7];
  dq[0] = s * (-k * G01 + j * G02 + k * G10 - i * G12 - j * G20 + i * G21) - dLds * s * s * r;
  dq[1] = s * (-2.0f * i * (G11 + G22) + j * G01 + k * G02 + j * G10 - r * G12 + k * G20 + r * G21) - dLds * s * s * i;
  dq[2] = s * (-2.0f * j * (G00 + G22) + i * G01 + r * G02 + i * G10 + k * G12 - r * G20 + k * G21) - dLds * s * s * j;
  dq[3] = s * (-2.0f * k * (G00 + G11) - r * G01 + i * G02 + r * G10 + j * G12 + i * G20 + j * G21) - dLds * s * s * k;
  dq[4] = g[3]; dq[5] = g[7]; dq[6] = g[11];
#pragma unroll
  for (int t = 0; t < 7; t++) {
    const float gr = dq[t];
    if (d_cams != nullptr) d_cams[7 * c + t] = gr;
    float m = em[7 * c + t], v = ev[7 * c + t];
    q[t] = adam_update(q[t], gr, m, v, a);
    em[7 * c + t] = m; ev[7 * c + t] = v;
  }
}
extern "C" int nsb_window_rays(const float* cams, const int32_t* cam_row, const float* fixed_c2w, int n_frames,
                               const float* pix_i, const float* pix_j, const int32_t* frame_of_ray, int n_rays,
                               double fx, double fy, double cx, double cy, float* c2w_out, float* rays_o, float* rays_d, float* dirs, void* stream) {
  if (n_frames < 1 || !cam_row || !c2w_out || (!cams && !fixed_c2w) || n_rays < 0 || (n_rays > 0 && (!pix_i || !pix_j || !frame_of_ray || !rays_o || !rays_d))) {
    set_error("window_rays: bad arguments"); return NSB_ERR_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  window_poses_kernel<<<(n_frames + 63) / 64, 64, 0, st>>>(cams, cam_row, fixed_c2w, n_frames, c2w_out);
  if (n_rays > 0) window_rays_kernel<<<(n_rays + 255) / 256, 256, 0, st>>>(c2w_out, pix_i, pix_j, frame_of_ray, n_rays, (float)fx, (float)fy, (float)cx, (float)cy, rays_o, rays_d, dirs);
  return check_cuda(cudaGetLastError(), "window_rays launch");
}
extern "C" int nsb_adam_poses(float* cams, const int32_t* cam_row, int n_frames, const float* d_c2w, float* exp_avg, float* exp_avg_sq, float* d_cams,
                              double lr, double beta1, double beta2, double eps, int step, void* stream) {
  if (!cams || !cam_row || n_frames < 1 || !d_c2w || !exp_avg || !exp_avg_sq) { set_error("adam_poses: bad arguments"); return NSB_ERR_ARG; }
  AdamScalars a; int rc = adam_scalars(lr, beta1, beta2, eps, step, &a); if (rc) return rc;
  adam_poses_kernel<<<(n_frames + 63) / 64, 64, 0, (cudaStream_t)stream>>>(cams, cam_row, n_frames, d_c2w, exp_avg, exp_avg_sq, d_cams, a);
  return check_cuda(cudaGetLastError(), "adam_poses launch");
}

extern "C" size_t nsb_frustum_mask_workspace(long long n_voxels) { return n_voxels <= 0 ? 16 : (size_t)n_voxels * sizeof(float) + 16; }
extern "C" int nsb_frustum_mask(const float* c2w, const float* xs, const float* ys, const float* zs, int D, int H, int W,
                                const float* depth, int img_h, int img_w, double fx, double fy, double cx, double cy,
                                uint8_t* voxel_mask, void* workspace, size_t workspace_bytes, void* stream) {
  const long long n = (long long)D * H * W;
  if (!c2w || !xs || !ys || !zs || D < 1 || H < 1 || W < 1 || !depth || img_h < 1 || img_w < 1 || !voxel_mask || !workspace) {
    set_error("frustum_mask: bad arguments"); return NSB_ERR_ARG; }
  if (workspace_bytes < nsb_frustum_mask_workspace(n)) { set_error("frustum_mask: workspace too small"); return NSB_ERR_ARG; }
  // inverse of the rigid-or-not 4x4 pose in double (Gauss-Jordan with partial pivoting), rounded to float32 like the reference's w2c
  double a[4][8];
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) { a[i][j] = (double)c2w[4 * i + j]; a[i][4 + j] = i == j ? 1.0 : 0.0; }
  for (int col = 0; col < 4; col++) {
    int piv = col;
    for (int r = col + 1; r < 4; r++) if (fabs(a[r][col]) > fabs(a[piv][col])) piv = r;
    if (a[piv][col] == 0.0) { set_error("frustum_mask: singular c2w"); return NSB_ERR_ARG; }
    if (piv != col) for (int j = 0; j < 8; j++) { const double t = a[col][j]; a[col][j] = a[piv][j]; a[piv][j] = t; }
    const double inv = 1.0 / a[col][col];
    for (int j = 0; j < 8; j++) a[col][j] *= inv;
    for (int r = 0; r < 4; r++) if (r != col) { const double f = a[r][col]; if (f != 0.0) for (int j = 0; j < 8; j++) a[r][j] -= f * a[col][j]; }
  }
  FrustumArgs A;
  for (int i = 0; i < 3; i++) for (int j = 0; j < 4; j++) A.w2c[4 * i + j] = (float)a[i][4 + j];
  for (int i = 0; i < 3; i++) A.cam_o[i] = c2w[4 * i + 3];
  A.xs = xs; A.ys = ys; A.zs = zs; A.D = D; A.H = H; A.W = W; A.depth = depth; A.img_h = img_h; A.img_w = img_w;
  A.fx = fx; A.fy = fy; A.cx = cx; A.cy = cy;
  cudaStream_t st = (cudaStream_t)stream;
  float* depths = static_cast<float*>(workspace);
  int* max_bits = reinterpret_cast<int*>(static_cast<char*>(workspace) + (size_t)n * sizeof(float));
  if (check_cuda(cudaMemsetAsync(max_bits, 0, sizeof(int), st), "frustum memset")) return NSB_ERR_CUDA;
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  frustum_depth_kernel<<<blocks, 256, 0, st>>>(A, depths, max_bits);
  frustum_mask_kernel<<<blocks, 256, 0, st>>>(A, depths, max_bits, voxel_mask);
  return check_cuda(cudaGetLastError(), "frustum_mask launch");
}

extern "C" int nsb_pose_grad_frames(const float* dirs, const float* d_rays_o, const float* d_rays_d, const int32_t* frame_offsets,
                                    int n_frames, float* out, void* stream) {
  if (n_frames < 0 || (n_frames > 0 && (!dirs || !d_rays_o || !d_rays_d || !frame_offsets || !out))) { set_error("pose_grad_frames: bad arguments"); return NSB_ERR_ARG; }
  if (n_frames == 0) return NSB_OK;
  pose_grad_frames_kernel<<<n_frames, 256, 0, (cudaStream_t)stream>>>(dirs, d_rays_o, d_rays_d, frame_offsets, out);
  return check_cuda(cudaGetLastError(), "pose_grad_frames launch");
}

extern "C" int nsb_version(void) { return NSB_VERSION; }
extern "C" const char* nsb_last_error(void) { return g_err; }
extern "C" size_t nsb_flat_decoder_floats(int level) { return level < 0 || level > 3 ? 0 : (size_t)flat_offset(level, 7, 0); }
extern "C" long long nsb_flat_offset(int level, int kind, int layer) { return level < 0 || level > 3 ? -1 : flat_offset(level, kind, layer); }
extern "C" size_t nsb_packed_decoder_floats(int level) { return level < 0 || level > 3 ? 0 : (size_t)packed_total_floats(level); }

extern "C" int nsb_pack_decoders(const nsb_decoder_params* const params[4], float* const packed[4], void* stream) {
  if (!params || !packed) { set_error("params / packed NULL"); return NSB_ERR_ARG; }
  PackArgs A; memset(&A, 0, sizeof(A));
  for (int l = 0; l < 4; l++) {
    if (!params[l]) continue;
    if (!packed[l]) { set_error("packed[%d] NULL", l); return NSB_ERR_ARG; }
    const nsb_decoder_params& p = *params[l];
    bool ok = p.Wo && p.bo;
    for (int i = 0; i < 5; i++) ok = ok && p.W[i] && p.b[i] && (l == 0 || (p.Wc[i] && p.bc[i]));
    if (l != 0) ok = ok && p.B;
    if (!ok) { set_error("decoder %d has NULL parameter pointers", l); return NSB_ERR_ARG; }
    A.p[l] = p; A.packed[l] = packed[l]; A.present[l] = 1;
  }
  for (int l = 0; l < 4; l++)
    if (A.present[l] && check_cuda(cudaMemsetAsync(A.packed[l], 0, (size_t)packed_floats(l) * 4, (cudaStream_t)stream), "pack memset")) return NSB_ERR_CUDA;
  pack_kernel<0><<<dim3(4, kPackSlices), 256, 0, (cudaStream_t)stream>>>(A);
  pack_operands_kernel<<<dim3(4, kPackSlices), 256, 0, (cudaStream_t)stream>>>(A);   // tensor-core operand images behind the fp32 image
  return check_cuda(cudaGetLastError(), "pack_decoders launch");
}

extern "C" int nsb_batch_max_depth(const float* gt_depth, int n, float* out2, void* stream) {
  if (!out2 || (n > 0 && !gt_depth) || n < 0) { set_error("batch_max_depth: bad arguments"); return NSB_ERR_ARG; }
  batch_max_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(gt_depth, n, out2, no_peers());
  return check_cuda(cudaGetLastError(), "batch_max launch");
}
extern "C" int nsb_batch_max_depth_peers(const float* gt_depth, int n, float* out2, const nsb_peers* peers, void* stream) {
  if (!out2 || (n > 0 && !gt_depth) || n < 0) { set_error("batch_max_depth_peers: bad arguments"); return NSB_ERR_ARG; }
  PeerX px; int rc = make_peers(peers, &px); if (rc) return rc;
  batch_max_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(gt_depth, n, out2, px);
  return check_cuda(cudaGetLastError(), "batch_max_peers launch");
}

extern "C" int nsb_bbox_prefilter(const float* rays_o, const float* rays_d, const float* gt_depth, int n,
                                  const double bound[6], uint8_t* keep, void* stream) {
  if (n < 0 || (n > 0 && (!rays_o || !rays_d || !gt_depth || !keep || !bound))) { set_error("bbox_prefilter: bad arguments"); return NSB_ERR_ARG; }
  if (n == 0) return NSB_OK;
  Bound6 B; for (int i = 0; i < 6; i++) B.b[i] = bound[i];
  prefilter_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rays_o, rays_d, gt_depth, n, B, keep);
  return check_cuda(cudaGetLastError(), "prefilter launch");
}

// ------------------------------------------------------------------------------------------------ keyframe store (SURVEY.md 8f-4)
// Mapper.keyframe_selection_overlap (src/Mapper.py:186-218): the n_samples points of every sampled ray of the current frame, between
// 0.8 * gt_depth and gt_depth + 0.5, are projected into every keyframe; counts[k] = points inside keyframe k's (edge-cropped) image and in
// front of its camera.  One CTA per keyframe.  float32 points and w2c product, float64 intrinsics product, float32 pixel compare -- the
// dtype flow of the reference's torch / numpy code.
__global__ void keyframe_overlap_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ gt_depth,
                                        int n_rays, const float* __restrict__ t_vals, int n_samples, const float* __restrict__ w2c,
                                        int H, int W, double fx, double fy, double cx, double cy, int edge, int32_t* __restrict__ counts) {
  __shared__ int red[32];
  const float* m = w2c + (size_t)blockIdx.x * 16;
  float M[12];
#pragma unroll
  for (int i = 0; i < 12; i++) M[i] = m[i];
  int cnt = 0;
  const int np = n_rays * n_samples;
  for (int p = threadIdx.x; p < np; p += blockDim.x) {
    const int r = p / n_samples, s = p - r * n_samples;
    const float gd = gt_depth[r], t = t_vals[s];
    const float z = __fadd_rn(__fmul_rn(__fmul_rn(gd, 0.8f), __fsub_rn(1.0f, t)), __fmul_rn(__fadd_rn(gd, 0.5f), t));      // Mapper.py:189-192
    float x[3];
#pragma unroll
    for (int a = 0; a < 3; a++) x[a] = __fadd_rn(rays_o[3 * r + a], __fmul_rn(rays_d[3 * r + a], z));                          // :193-194
    float c[3];
#pragma unroll
    for (int a = 0; a < 3; a++)                                                                                                // w2c @ [x, 1], :203
      c[a] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(M[4 * a], x[0]), __fmul_rn(M[4 * a + 1], x[1])), __fmul_rn(M[4 * a + 2], x[2])), M[4 * a + 3]);
    const double X = -(double)c[0], Y = (double)c[1], Z = (double)c[2];                                                        // :207
    const double uz = Z + 1e-5;                                                                                                // K @ cam, :208-209
    const float u = (float)((fx * X + cx * Z) / uz), v = (float)((fy * Y + cy * Z) / uz);                                      // :210-211
    const bool in = u < (float)(W - edge) && u > (float)edge && v < (float)(H - edge) && v > (float)edge && uz < 0.0;          // :213-215
    cnt += in ? 1 : 0;
  }
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x < 32) {
    int t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) counts[blockIdx.x] = t;
  }
}
extern "C" int nsb_keyframe_overlap(const float* rays_o, const float* rays_d, const float* gt_depth, int n_rays, const float* t_vals, int n_samples,
                                    const float* w2c, int n_keyframes, int H, int W, double fx, double fy, double cx, double cy, int edge,
                                    int32_t* counts, void* stream) {
  if (n_rays < 0 || n_samples < 1 || n_keyframes < 0 || (n_keyframes > 0 && (!w2c || !counts)) || (n_rays > 0 && (!rays_o || !rays_d || !gt_depth || !t_vals))) {
    set_error("keyframe_overlap: bad arguments"); return NSB_ERR_ARG; }
  if (n_keyframes == 0) return NSB_OK;
  keyframe_overlap_kernel<<<n_keyframes, 256, 0, (cudaStream_t)stream>>>(rays_o, rays_d, gt_depth, n_rays, t_vals, n_samples, w2c, H, W, fx, fy, cx, cy, edge, counts);
  return check_cuda(cudaGetLastError(), "keyframe_overlap launch");
}

// Per-frame pixel samples of a mapping window from the device-resident keyframe store (what Mapper.py:437-462 obtains with a host->device copy of
// the full keyframe images followed by get_samples' indexing): out_depth[f][k] = depth[slot[f]][j][i], out_color likewise (3 channels).
__global__ void keyframe_gather_kernel(const float* __restrict__ depth, const float* __restrict__ color, const int32_t* __restrict__ slot,
                                       const int32_t* __restrict__ pix_i, const int32_t* __restrict__ pix_j, int n_frames, int n_pix, int H, int W,
                                       float* __restrict__ out_depth, float* __restrict__ out_color) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_frames * n_pix) return;
  const int f = idx / n_pix;
  const size_t px = ((size_t)slot[f] * H + pix_j[idx]) * W + pix_i[idx];
  out_depth[idx] = depth[px];
  out_color[3 * idx] = color[3 * px]; out_color[3 * idx + 1] = color[3 * px + 1]; out_color[3 * idx + 2] = color[3 * px + 2];
}
extern "C" int nsb_keyframe_gather(const float* depth, const float* color, const int32_t* slot, const int32_t* pix_i, const int32_t* pix_j,
                                   int n_frames, int n_pix, int H, int W, float* out_depth, float* out_color, void* stream) {
  if (n_frames < 0 || n_pix < 0 || H < 1 || W < 1 || (n_frames * n_pix > 0 && (!depth || !color || !slot || !pix_i || !pix_j || !out_depth || !out_color))) {
    set_error("keyframe_gather: bad arguments"); return NSB_ERR_ARG; }
  const int n = n_frames * n_pix;
  if (n == 0) return NSB_OK;
  keyframe_gather_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(depth, color, slot, pix_i, pix_j, n_frames, n_pix, H, W, out_depth, out_color);
  return check_cuda(cudaGetLastError(), "keyframe_gather launch");
}

extern "C" size_t nsb_tracking_seeds_workspace(int n) { return (size_t)(n > 0 ? n : 1) * sizeof(double); }

__global__ void residuals_kernel(const double* __restrict__ depth, const double* __restrict__ var, const float* __restrict__ gt,
                                 int n, double* __restrict__ res) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) res[i] = fabs((double)gt[i] - depth[i]) / sqrt(var[i] + 1e-10);
}
extern "C" int nsb_tracking_residuals(const double* depth, const double* var, const float* gt_depth, int n, double* res, void* stream) {
  if (n < 0 || (n > 0 && (!depth || !var || !gt_depth || !res))) { set_error("tracking_residuals: bad arguments"); return NSB_ERR_ARG; }
  if (n == 0) return NSB_OK;
  residuals_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(depth, var, gt_depth, n, res);
  return check_cuda(cudaGetLastError(), "residuals launch");
}

extern "C" int nsb_tracking_seeds(const double* depth, const double* var, const float* rgb, const float* gt_depth,
                                  const double* gt_rgb, int n, double w_color, int handle_dynamic, int use_color,
                                  const double* median_pool, int n_pool,
                                  double* g_depth, float* g_rgb, double* loss, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  if (n < 0 || !loss || (n > 0 && (!depth || !var || !rgb || !gt_depth || !g_depth || !g_rgb || (use_color && !gt_rgb)))) {
    set_error("tracking_seeds: bad arguments"); return NSB_ERR_ARG; }
  if (!workspace || workspace_bytes < nsb_tracking_seeds_workspace(n)) { set_error("tracking_seeds: workspace too small"); return NSB_ERR_ARG; }
  if (median_pool != nullptr && n_pool < 1) { set_error("tracking_seeds: empty median pool"); return NSB_ERR_ARG; }
  tracking_seeds_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(depth, var, rgb, gt_depth, gt_rgb, n, w_color, handle_dynamic, use_color,
                                                               median_pool, n_pool, g_depth, g_rgb, loss, (double*)workspace, no_peers());
  return check_cuda(cudaGetLastError(), "tracking_seeds launch");
}
extern "C" int nsb_tracking_seeds_peers(const double* depth, const double* var, const float* rgb, const float* gt_depth,
                                        const double* gt_rgb, int n, double w_color, int handle_dynamic, int use_color,
                                        const nsb_peers* peers, double* g_depth, float* g_rgb, double* loss,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  if (n < 1 || !loss || !depth || !var || !rgb || !gt_depth || !g_depth || !g_rgb || (use_color && !gt_rgb)) {
    set_error("tracking_seeds_peers: bad arguments"); return NSB_ERR_ARG; }
  if (!workspace || workspace_bytes < nsb_tracking_seeds_workspace(n)) { set_error("tracking_seeds_peers: workspace too small"); return NSB_ERR_ARG; }
  PeerX px; int rc = make_peers(peers, &px); if (rc) return rc;
  if (n > px.max_n) { set_error("tracking_seeds_peers: n exceeds the exchange buffer capacity"); return NSB_ERR_ARG; }
  tracking_seeds_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(depth, var, rgb, gt_depth, gt_rgb, n, w_color, handle_dynamic, use_color,
                                                               nullptr, 0, g_depth, g_rgb, loss, (double*)workspace, px);
  return check_cuda(cudaGetLastError(), "tracking_seeds_peers launch");
}

extern "C" int nsb_mapping_seeds(const double* depth, const float* rgb, const float* gt_depth, const float* gt_rgb, int n,
                                 double w_color, int use_color, double* g_depth, float* g_rgb, double* loss, void* stream) {
  if (n < 0 || !loss || (n > 0 && (!depth || !rgb || !gt_depth || !g_depth || !g_rgb || (use_color && !gt_rgb)))) {
    set_error("mapping_seeds: bad arguments"); return NSB_ERR_ARG; }
  mapping_seeds_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(depth, rgb, gt_depth, gt_rgb, n, w_color, use_color, g_depth, g_rgb, loss);
  return check_cuda(cudaGetLastError(), "mapping_seeds launch");
}
