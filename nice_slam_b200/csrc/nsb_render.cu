// nsb_render.cu -- the render-and-backprop kernels and their C-ABI entry points.
//
//   render_fwd_kernel : sample -> trilinear gather -> decoders -> alpha-composite      (Renderer.render_batch_ray,
//                       src/utils/Renderer.py:63-198; eval_points :23-61; raw2outputs_nerf_color, src/common.py:204-245)
//   render_bwd_kernel : recompute + hand-rolled backward into rays, grid voxels and decoder weights
//                       (what loss.backward() does at src/Tracker.py:125 / src/Mapper.py:503; SURVEY.md 8.1)
//
// Work decomposition: a CTA owns `rays_per_block` consecutive rays (all S samples of each, so compositing and
// the per-ray scan stay inside the CTA); its points are cut into chunks of 16 that the warps process
// independently (nsb_mlp.cuh).  Decoders are evaluated one after the other; each decoder's packed weight image
// is staged into shared memory with one TMA bulk copy that overlaps with the first chunk's feature gather.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include "nsb_common.cuh"
#include "nsb_geom.cuh"
#include "nsb_mlp.cuh"
#include "nsb_seeds.cuh"

namespace nsb {

// ------------------------------------------------------------------------------------------------
// trilinear gather / scatter of one chunk (8 lanes per point, 16-byte channel quads, 4 points per pass)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool grid_fast(const nsb_grid& g) { return g.stride_c == 1; }

__device__ __forceinline__ float4 grid_load4(const nsb_grid& g, long long off, int c0, bool fast) {
  if (fast) return ldg_f4(g.data + off + c0);
  return make_float4(__ldg(g.data + off + (long long)c0 * g.stride_c), __ldg(g.data + off + (long long)(c0 + 1) * g.stride_c),
                     __ldg(g.data + off + (long long)(c0 + 2) * g.stride_c), __ldg(g.data + off + (long long)(c0 + 3) * g.stride_c));
}

// rows [row0,row0+32) <- features of the 16 points; xn = normalised coords of point (lane & 15).
// All eight corner loads of a pass are issued before any of them is consumed (branch-free clamped addressing).
__device__ __forceinline__ void gather_chunk(const nsb_grid& g, float* __restrict__ act, int row0, const float xn[3], int lane) {
  const bool fast = grid_fast(g);
  const int q = lane & 7;
#pragma unroll 2
  for (int it = 0; it < 4; it++) {
    const int pt = it * 4 + (lane >> 3);
    float x[3];
    x[0] = __shfl_sync(0xffffffffu, xn[0], pt); x[1] = __shfl_sync(0xffffffffu, xn[1], pt); x[2] = __shfl_sync(0xffffffffu, xn[2], pt);
    const Tri t = make_tri(x, g.W, g.H, g.D);
    float4 v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      int cx, cy, cz;
      tri_corner_clamped(t, k, g.W, g.H, g.D, cx, cy, cz);
      v[k] = grid_load4(g, cz * g.stride_d + cy * g.stride_h + cx * g.stride_w, 4 * q, fast);
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const float w = tri_weight(t, k);
      acc.x = fmaf(v[k].x, w, acc.x); acc.y = fmaf(v[k].y, w, acc.y); acc.z = fmaf(v[k].z, w, acc.z); acc.w = fmaf(v[k].w, w, acc.w);
    }
    act[act_idx(row0 + 4 * q + 0, pt)] = acc.x; act[act_idx(row0 + 4 * q + 1, pt)] = acc.y;
    act[act_idx(row0 + 4 * q + 2, pt)] = acc.z; act[act_idx(row0 + 4 * q + 3, pt)] = acc.w;
  }
}

// w * dc -> gradient of voxel (cx,cy,cz), channels [4q,4q+4): dense buffer with the grid's strides, or -- masked voxel
// parameterisation (Mapper.py:317-333) -- the compact [n_selected][32] buffer through the voxel -> slot table
__device__ __forceinline__ void voxel_grad_add(const nsb_grid& g, float* __restrict__ dgrid, const int32_t* __restrict__ slots, long long off,
                                               int cx, int cy, int cz, int q, bool fast, float w, const float dc[4]) {
  if (slots != nullptr) {
    const int s = __ldg(slots + ((long long)cz * g.H + cy) * g.W + cx);
    if (s >= 0) red_add_v4(dgrid + (long long)s * 32 + 4 * q, w * dc[0], w * dc[1], w * dc[2], w * dc[3]);
  } else if (fast) {
    red_add_v4(dgrid + off + 4 * q, w * dc[0], w * dc[1], w * dc[2], w * dc[3]);
  } else {
#pragma unroll
    for (int c = 0; c < 4; c++) atomicAdd(dgrid + off + (long long)(4 * q + c) * g.stride_c, w * dc[c]);
  }
}

// Backward of gather_chunk: rows [row0,row0+32) hold dL/dc.  Scatter-adds w_k * dc into dgrid (if non-null)
// and returns through gx (valid in lanes with (lane&7)==0, for point it*4 + lane>>3 of pass `it`) the gradient
// w.r.t. the normalised coordinate (grid_sampler_3d_backward incl. the clip multiplier, GridSampler.h:66-82).
template <typename F>
__device__ __forceinline__ void scatter_chunk(const nsb_grid& g, float* __restrict__ dgrid, const int32_t* __restrict__ slots,
                                              const float* __restrict__ act, int row0, const float xn[3], int lane, F&& emit) {
  const bool fast = grid_fast(g);
  const int q = lane & 7;
#pragma unroll 1
  for (int it = 0; it < 4; it++) {
    const int pt = it * 4 + (lane >> 3);
    float x[3];
    x[0] = __shfl_sync(0xffffffffu, xn[0], pt); x[1] = __shfl_sync(0xffffffffu, xn[1], pt); x[2] = __shfl_sync(0xffffffffu, xn[2], pt);
    const Tri t = make_tri(x, g.W, g.H, g.D);
    float dc[4];
#pragma unroll
    for (int c = 0; c < 4; c++) dc[c] = act[act_idx(row0 + 4 * q + c, pt)];
    float gi[3] = {0.f, 0.f, 0.f};
    long long offs[8]; float4 vv[8]; bool ins[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {                                // all corner loads first (branch-free clamped addressing)
      int cx, cy, cz;
      ins[k] = tri_corner(t, k, g.W, g.H, g.D, cx, cy, cz);
      tri_corner_clamped(t, k, g.W, g.H, g.D, cx, cy, cz);
      offs[k] = cz * g.stride_d + cy * g.stride_h + cx * g.stride_w;
      vv[k] = grid_load4(g, offs[k], 4 * q, fast);
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
      if (ins[k]) {                                              // corners outside the grid get neither gradient nor a dot product
        const float4 v = vv[k];
        const float dot = v.x * dc[0] + v.y * dc[1] + v.z * dc[2] + v.w * dc[3];
        if (dgrid != nullptr) {
          int cx, cy, cz;
          tri_corner(t, k, g.W, g.H, g.D, cx, cy, cz);
          voxel_grad_add(g, dgrid, slots, offs[k], cx, cy, cz, q, fast, tri_weight(t, k), dc);
        }
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
      emit(pt, gx);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// kernel parameters
// ------------------------------------------------------------------------------------------------
struct KParams {
  nsb_render_inputs in;
  nsb_forward_outputs fo;       // forward
  nsb_backward_args bw;         // backward
  float* d_packed[4];           // backward: packed-layout weight-gradient images (WGRAD decoders)
  const double* points;         // points-only mode: f64 [P,3]
  float* points_raw;            // points-only mode: f32 [P,4]
  int n_points;
  int rays_per_block;
  int S;                        // samples per ray actually used
  int has_gt;
  int n_dec;                    // decoders of this stage, in the reference's evaluation order
  int dec[3];
  int dec_pos[3];               // position of dec[i] in the stage's full decoder list (slot of its saved ReLU masks)
  int accumulate_rays;          // backward: add to d_rays_o / d_rays_d instead of overwriting (second launch of a split backward)
  // tile kernels (nsb_tile.cuh): item = (128-point tile, decoder); `split` items per tile
  int split;                    // 1 = one CTA evaluates all decoders of its tile; n_dec = CTA j of a tile evaluates decoder dec[j] only
  double* ray_parts;            // backward: [tiles * split][tile_rays][6] per-item ray-gradient sums
  int* ray_cnt;                 // [N] completion counters of the rays, zero between launches (the completing CTA resets them)
  float4* tile_parts;           // forward: [split][N*S] per-item decoder outputs (split == 1: aliases fo.raw)
  int tile_rays;                // backward: rays one tile can touch (stride of ray_parts per item)
  FusedSeeds fs;                // forward: loss seeds computed by the last CTA to finish (kind 0 = not fused)
  PeerTail tail;                // backward: sum of [loss | d c2w] over ranks by the last CTA (px.world <= 1: none)
  int acts_lv;                  // forward: decoder level whose layer outputs go to fo.acts (-1: none)
  int wbytes;                   // bytes reserved for the weight image in shared memory
  int max_pts, max_rays;        // per-CTA capacities the shared-memory carve-up was sized for
};

struct Smem {                   // carve-up of dynamic shared memory (all offsets 16-byte aligned)
  float* wt; uint64_t* bar; float* rays; double* far; double* zs; float* raw; double* dp; float* gocc; float* wgt;
  unsigned char* inb; float* act;
};
__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~size_t(15); }
__host__ __device__ inline size_t smem_layout(int wbytes, int max_pts, int max_rays, int warps, int rows, bool bwd, Smem* s, unsigned char* base) {
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o = align16(o + bytes); return r; };
  size_t o_wt = take(wbytes), o_bar = take(16), o_rays = take(sizeof(float) * 8 * max_rays), o_far = take(sizeof(double) * max_rays);
  size_t o_zs = take(sizeof(double) * max_pts), o_raw = take(sizeof(float) * 4 * max_pts);
  size_t o_dp = bwd ? take(sizeof(double) * 3 * max_pts) : 0, o_gocc = bwd ? take(sizeof(float) * max_pts) : 0, o_wgt = take(sizeof(float) * max_pts);
  size_t o_inb = take(max_pts);
  size_t o_act = take((size_t)warps * rows * kRowF * sizeof(float));
  if (s) {
    s->wt = (float*)(base + o_wt); s->bar = (uint64_t*)(base + o_bar); s->rays = (float*)(base + o_rays); s->far = (double*)(base + o_far);
    s->zs = (double*)(base + o_zs); s->raw = (float*)(base + o_raw); s->dp = (double*)(base + o_dp); s->gocc = (float*)(base + o_gocc);
    s->wgt = (float*)(base + o_wgt); s->inb = base + o_inb; s->act = (float*)(base + o_act);
  }
  return o;
}

// rays[r*8 + {0,1,2}] = o, {3,4,5} = d, 6 = near(f32), 7 = gt ; far[r] (f64)
__device__ __forceinline__ void block_setup_rays(const KParams& P, const Smem& sm, int r0, int nr, float gtmax12) {
  for (int r = threadIdx.x; r < nr; r += blockDim.x) {
    float o[3], d[3];
#pragma unroll
    for (int a = 0; a < 3; a++) { o[a] = P.in.rays_o[3 * (r0 + r) + a]; d[a] = P.in.rays_d[3 * (r0 + r) + a]; }
    const float gt = P.has_gt ? P.in.gt_depth[r0 + r] : 0.0f;
    const RaySampler rs = make_sampler(P.in.bound, o, d, P.has_gt, gt, gtmax12);
#pragma unroll
    for (int a = 0; a < 3; a++) { sm.rays[8 * r + a] = o[a]; sm.rays[8 * r + 3 + a] = d[a]; }
    sm.rays[8 * r + 6] = rs.near; sm.rays[8 * r + 7] = gt; sm.far[r] = rs.far;
  }
}

__device__ __forceinline__ void issue_weights(const KParams& P, const Smem& sm, int lv) {
  // one elected thread: order prior generic-proxy reads of the buffer before the async-proxy overwrite, then TMA
  fence_proxy_async();
  const uint32_t bytes = (uint32_t)packed_floats(lv) * 4u;
  mbar_expect_tx(sm.bar, bytes);
  const char* src = reinterpret_cast<const char*>(P.in.packed[lv]);
  char* dst = reinterpret_cast<char*>(sm.wt);
  for (uint32_t off = 0; off < bytes; off += 32768u) {
    const uint32_t n = bytes - off < 32768u ? bytes - off : 32768u;
    tma_bulk_g2s(dst + off, src + off, n, sm.bar);
  }
}

// geometry of this lane's point (lane & 15) of chunk `chunk`
__device__ __forceinline__ void chunk_point(const KParams& P, const Smem& sm, int chunk, int Pb, int lane, int& lp, PointGeom& G) {
  lp = chunk * kChunk + (lane & 15);
  const int lpc = lp < Pb ? lp : Pb - 1;
  if (P.points != nullptr) {
    const long long gp = (long long)blockIdx.x * P.rays_per_block + lpc;      // points mode: rays_per_block == points per block
    const double pin[3] = {P.points[3 * gp], P.points[3 * gp + 1], P.points[3 * gp + 2]};
    make_point_from_p(P.in.bound, P.in.coarse_bound, pin, G);
  } else {
    const int ray = lpc / P.S;
    const float* rr = sm.rays + 8 * ray;
    const float o[3] = {rr[0], rr[1], rr[2]}, d[3] = {rr[3], rr[4], rr[5]};
    make_point(P.in.bound, P.in.coarse_bound, o, d, sm.zs[lpc], G);
  }
}

__device__ __forceinline__ void chunk_forward(const KParams& P, const Smem& sm, float* act, int chunk, int Pb,
                                              const LaneId& L, uint32_t parity, bool first_dec, const int lv, const DecRT& d) {
  int lp; PointGeom G;
  chunk_point(P, sm, chunk, Pb, L.lane, lp, G);
  const float* xn = lv == 0 ? G.xnc : G.xn;
  gather_chunk(P.in.grid[lv], act, R_C, xn, L.lane);
  if (lv == 2) gather_chunk(P.in.grid[1], act, R_C + 32, G.xn, L.lane);   // no_grad middle concat (decoder.py:182-187)
  mbar_wait(sm.bar, parity);
  __syncwarp();
  Masks masks; float out[4];
  mlp_forward<false>(d, sm.wt, act, L, G.pf, masks, out);
  if (L.lane < 16 && lp < Pb) {
    if (lv == 3) { sm.raw[4 * lp] = out[0]; sm.raw[4 * lp + 1] = out[1]; sm.raw[4 * lp + 2] = out[2]; }
    else sm.raw[4 * lp + 3] += out[0];
    if (first_dec) {
      sm.inb[lp] = (unsigned char)G.inb;
      if (P.fo.corner_idx != nullptr) {
        const nsb_grid& g = P.in.grid[lv];
        const Tri t = make_tri(xn, g.W, g.H, g.D);
        const long long gp = ((long long)blockIdx.x * P.rays_per_block) * P.S + lp;
        P.fo.corner_idx[3 * gp] = t.i0[0]; P.fo.corner_idx[3 * gp + 1] = t.i0[1]; P.fo.corner_idx[3 * gp + 2] = t.i0[2];
      }
    }
  }
  __syncwarp();
}

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

// warp-wide helpers for the per-ray compositing scans (one warp per ray, lanes over samples)
__device__ __forceinline__ float warp_incl_prod(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v *= t; }
  return v;
}
__device__ __forceinline__ float warp_incl_suffix_sum(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_down_sync(0xffffffffu, v, o); if (lane + o < 32) v += t; }
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// alpha_s = sigmoid(10 occ_s), T_s = prod_{j<s} (1 - alpha_j + 1e-10), w_s = alpha_s T_s  (common.py:233-240).
// Writes w to wq[] and (optionally) T to tq[].  All lanes of one warp call it for one ray.
__device__ __forceinline__ void ray_weights(const float* __restrict__ rw, int S, int lane, float* __restrict__ wq, float* __restrict__ tq) {
  float carry = 1.0f;
  for (int base = 0; base < S; base += 32) {
    const int s = base + lane;
    const bool v = s < S;
    const float al = v ? sigmoid_f(10.0f * rw[4 * s + 3]) : 0.0f;
    const float q = v ? (1.0f - al) + 1e-10f : 1.0f;
    const float incl = warp_incl_prod(q, lane);
    float excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.0f;
    const float T = carry * excl;
    if (v) { wq[s] = al * T; if (tq) tq[s] = T; }
    carry *= __shfl_sync(0xffffffffu, incl, 31);
  }
}

// ------------------------------------------------------------------------------------------------
// forward kernel
// ------------------------------------------------------------------------------------------------
struct BlockRange { int r0, nr, Pb; };
__device__ __forceinline__ BlockRange block_range(const KParams& P, int bid) {
  BlockRange b; b.r0 = 0; b.nr = 0;
  if (P.points != nullptr) {
    const long long p0 = (long long)bid * P.rays_per_block;
    b.Pb = (int)((P.n_points - p0) < P.rays_per_block ? (P.n_points - p0) : P.rays_per_block);
  } else {
    b.r0 = bid * P.rays_per_block;
    b.nr = P.in.n_rays - b.r0 < P.rays_per_block ? P.in.n_rays - b.r0 : P.rays_per_block;
    b.Pb = b.nr * P.S;
  }
  return b;
}
// stratified + near-surface sampling and the stable merge (Renderer.py:82-170); leaves sorted z in sm.zs and zeroes sm.raw
__device__ __forceinline__ void fwd_sample_sort(const KParams& P, const Smem& sm, const BlockRange& b) {
  if (P.points == nullptr) {
    float gtmax = 0.0f, gtmax12 = 0.0f;
    if (P.has_gt) {
      if (P.in.depth_max != nullptr) { gtmax = P.in.depth_max[0]; gtmax12 = P.in.depth_max[1]; }
      else {
        // small batches: every CTA reduces the batch's sensor depths itself (n_rays <= kInlineMaxRays floats from L2) instead of waiting
        // for a separate single-CTA kernel: torch.max(gt_depth) and torch.max(gt_depth*1.2) = fl(1.2f * max)  (Renderer.py:109,144)
        __shared__ float s_max[32];
        const bool whole = P.in.gt_depth_batch != nullptr;        // the depths of the whole (sharded) batch are known here: no exchange
        const float* gsrc = whole ? P.in.gt_depth_batch : P.in.gt_depth;
        const int gn = whole ? P.in.n_batch : P.in.n_rays;
        float m = -INFINITY;
        for (int i = threadIdx.x; i < gn; i += blockDim.x) m = fmaxf(m, __ldg(gsrc + i));
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
        __syncthreads();
        m = -INFINITY;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) m = fmaxf(m, s_max[w]);
        if (P.fs.px.world > 1 && !whole) { __shared__ uint32_t s_seq; m = peer_max_all_ctas(P.fs.px, m, &s_seq); }      // sharded batch: MAX over the ranks' shards
        gtmax = m; gtmax12 = __fmul_rn(m, 1.2f);
      }
    }
    block_setup_rays(P, sm, b.r0, b.nr, gtmax12);
    __syncthreads();
    double* zu = reinterpret_cast<double*>(sm.raw);              // unsorted samples (raw is not live yet)
    for (int lp = threadIdx.x; lp < b.Pb; lp += blockDim.x) {
      const int ray = lp / P.S, i = lp - ray * P.S;
      RaySampler rs; rs.near = sm.rays[8 * ray + 6]; rs.gt = sm.rays[8 * ray + 7]; rs.far = sm.far[ray]; rs.has_gt = P.has_gt;
      zu[lp] = sample_z(rs, i, P.in.n_samples, P.in.t_uniform, P.in.t_surface, gtmax);
    }
    __syncthreads();
    // torch.sort of [uniform | surface] (Renderer.py:168-170): both lists are normally non-decreasing -> merge by ranks (own index + binary-search
    // count in the other list); a ray whose lists are not sorted (far < near, NaN) takes the general stable rank sort (same values either way)
    __shared__ int s_unsorted[kMaxRaysPerBlock];
    for (int r = threadIdx.x; r < b.nr; r += blockDim.x) s_unsorted[r] = 0;
    __syncthreads();
    const int nu = P.in.n_samples < P.S ? P.in.n_samples : P.S;
    for (int lp = threadIdx.x; lp < b.Pb; lp += blockDim.x) {
      const int ray = lp / P.S, i = lp - ray * P.S;
      if (i != 0 && i != nu) { if (!(zu[lp - 1] <= zu[lp])) s_unsorted[ray] = 1; }
      else if (zu[lp] != zu[lp]) s_unsorted[ray] = 1;
    }
    __syncthreads();
    for (int lp = threadIdx.x; lp < b.Pb; lp += blockDim.x) {
      const int ray = lp / P.S, i = lp - ray * P.S;
      const double zi = zu[lp];
      const double* zr = zu + ray * P.S;
      int rank;
      if (!s_unsorted[ray]) {
        const bool uni = i < nu;
        const double* other = uni ? zr + nu : zr;
        int lo = 0, hi = uni ? P.S - nu : nu;
        while (lo < hi) { const int mid = (lo + hi) >> 1; const double zm = other[mid]; if (uni ? (zm < zi) : (zm <= zi)) lo = mid + 1; else hi = mid; }
        rank = (uni ? i : i - nu) + lo;
      } else {
        rank = 0;
        for (int j = 0; j < P.S; j++) { const double zj = zr[j]; rank += (z_less(zj, zi) || (!z_less(zi, zj) && j < i)) ? 1 : 0; }
      }
      sm.zs[ray * P.S + rank] = zi;
    }
  }
  __syncthreads();
  for (int lp = threadIdx.x; lp < b.Pb; lp += blockDim.x) { sm.raw[4 * lp] = 0.f; sm.raw[4 * lp + 1] = 0.f; sm.raw[4 * lp + 2] = 0.f; sm.raw[4 * lp + 3] = 0.f; }
}
// out-of-bound override, compositing and the stores of the forward pass (call after a __syncthreads())
__device__ __forceinline__ void fwd_composite_store(const KParams& P, const Smem& sm, const BlockRange& b, int warp, int warps, int lane) {
  const int r0 = b.r0, nr = b.nr, Pb = b.Pb;
  if (P.points != nullptr) {                                     // Renderer.eval_points: raw with the OOB override
    for (int lp = threadIdx.x; lp < Pb; lp += blockDim.x) {
      const long long gp = (long long)blockIdx.x * P.rays_per_block + lp;
      float4 v = *reinterpret_cast<float4*>(sm.raw + 4 * lp);
      if (!sm.inb[lp]) v.w = 100.0f;
      *reinterpret_cast<float4*>(P.points_raw + 4 * gp) = v;
    }
    return;
  }
  // out-of-bound override (Renderer.py:57), then raw2outputs_nerf_color, occupancy branch (common.py:233-244)
  for (int lp = threadIdx.x; lp < Pb; lp += blockDim.x) if (!sm.inb[lp]) sm.raw[4 * lp + 3] = 100.0f;
  __syncthreads();
  for (int r = warp; r < nr; r += warps) {                       // one warp per ray, lanes over samples
    const float* rw = sm.raw + 4 * r * P.S;
    const double* z = sm.zs + r * P.S;
    float* wq = sm.wgt + r * P.S;
    ray_weights(rw, P.S, lane, wq, nullptr);
    __syncwarp();
    float c0 = 0.f, c1 = 0.f, c2 = 0.f; double dsum = 0.0;
    for (int s = lane; s < P.S; s += 32) {
      const float w = wq[s];
      c0 = fmaf(w, rw[4 * s], c0); c1 = fmaf(w, rw[4 * s + 1], c1); c2 = fmaf(w, rw[4 * s + 2], c2);
      dsum += (double)w * z[s];
    }
    c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2); dsum = warp_sum(dsum);
    double v = 0.0;
    for (int s = lane; s < P.S; s += 32) { const double t = z[s] - dsum; v += (double)wq[s] * t * t; }
    v = warp_sum(v);
    if (lane == 0) {
      P.fo.depth[r0 + r] = dsum; P.fo.var[r0 + r] = v;
      P.fo.rgb[3 * (r0 + r)] = c0; P.fo.rgb[3 * (r0 + r) + 1] = c1; P.fo.rgb[3 * (r0 + r) + 2] = c2;
    }
  }
  const long long g0 = (long long)r0 * P.S;
  if (P.fo.z_vals != nullptr) for (int lp = threadIdx.x; lp < Pb; lp += blockDim.x) P.fo.z_vals[g0 + lp] = sm.zs[lp];
  if (P.fo.raw != nullptr)
    for (int lp = threadIdx.x; lp < Pb; lp += blockDim.x)
      *reinterpret_cast<float4*>(P.fo.raw + 4 * (g0 + lp)) = *reinterpret_cast<float4*>(sm.raw + 4 * lp);
}

// Loss seeds fused into the forward launch: the last of `n_participants` CTAs (those that stored ray outputs) reads every ray's
// depth / variance / colour back and runs the single-CTA seed computation.  scratch = dead dynamic shared memory of this CTA.
__device__ __forceinline__ void fused_seeds_tail(const KParams& P, int n_participants, unsigned char* scratch) {
  if (P.fs.kind == 0) return;
  __shared__ int s_seeds_last;
  if (!grid_last_arrival(P.fs.counter, n_participants, &s_seeds_last)) return;
  if (P.fs.kind == 1) {
    // (sharded batch: the residual pool of the median is exchanged inside; then every CTA of this grid is past the depth-max exchange)
    tracking_seeds_body(P.fo.depth, P.fo.var, P.fo.rgb, P.in.gt_depth, static_cast<const double*>(P.fs.gt_rgb), P.in.n_rays, P.fs.w_color,
                        P.fs.handle_dynamic, P.fs.use_color, nullptr, 0, P.fs.g_depth, P.fs.g_rgb, P.fs.loss, P.fs.res, P.fs.px, scratch);
    if (P.fs.px.world > 1 && P.in.depth_max == nullptr && P.in.gt_depth_batch == nullptr && threadIdx.x == 0) peer_advance(P.fs.px, 0);
  } else {
    mapping_seeds_body(P.fo.depth, P.fo.rgb, P.fs.gt_depth_loss, static_cast<const float*>(P.fs.gt_rgb), P.in.n_rays, P.fs.w_color, P.fs.use_color,
                       P.fs.g_depth, P.fs.g_rgb, P.fs.loss, scratch);
  }
}

// ------------------------------------------------------------------------------------------------
// forward kernel, FP32-FMA (SIMT) decoders
__global__ void __launch_bounds__(256, 1) render_fwd_kernel(const __grid_constant__ KParams P) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5;
  const LaneId L = make_lane(threadIdx.x & 31);
  Smem sm;
  smem_layout(P.wbytes, P.max_pts, P.max_rays, warps, kRowsFwd, false, &sm, smem_raw);
  float* act = sm.act + (size_t)warp * kRowsFwd * kRowF;
  const BlockRange b = block_range(P, blockIdx.x);
  const int Pb = b.Pb;
  if (threadIdx.x == 0) { mbar_init(sm.bar, 1); mbar_fence_init(); }
  fwd_sample_sort(P, sm, b);

  const int nchunks = (Pb + kChunk - 1) / kChunk;
  uint32_t parity = 0;
  for (int qd = 0; qd < P.n_dec; qd++) {
    const int lv = P.dec[qd];
    __syncthreads();                                             // previous weight image no longer in use
    if (threadIdx.x == 0) issue_weights(P, sm, lv);
    const DecRT d = make_dec(lv);
#pragma unroll 1
    for (int chunk = warp; chunk < nchunks; chunk += warps) chunk_forward(P, sm, act, chunk, Pb, L, parity, qd == 0, lv, d);
    parity ^= 1u;
  }
  __syncthreads();
  fwd_composite_store(P, sm, b, warp, warps, L.lane);
  fused_seeds_tail(P, gridDim.x, smem_raw);
}

// ------------------------------------------------------------------------------------------------
// backward kernel
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void chunk_backward(const KParams& P, const Smem& sm, float* act, int chunk, int Pb,
                                               const LaneId& L, uint32_t parity, const float* gC /*[R][3] smem*/,
                                               const int lv, const DecRT& d) {
  int lp; PointGeom G;
  chunk_point(P, sm, chunk, Pb, L.lane, lp, G);
  const float* xn = lv == 0 ? G.xnc : G.xn;
  gather_chunk(P.in.grid[lv], act, R_C, xn, L.lane);
  if (lv == 2) gather_chunk(P.in.grid[1], act, R_C + 32, G.xn, L.lane);
  mbar_wait(sm.bar, parity);
  __syncwarp();
  Masks masks; float out[4];
  mlp_forward<true>(d, sm.wt, act, L, G.pf, masks, out);

  float g_out[4] = {0.f, 0.f, 0.f, 0.f};
  if (lp < Pb) {
    if (lv == 3) { const int ray = lp / P.S; const float w = sm.wgt[lp];
      g_out[0] = w * gC[3 * ray]; g_out[1] = w * gC[3 * ray + 1]; g_out[2] = w * gC[3 * ray + 2]; }
    else g_out[0] = sm.gocc[lp];
  }
  float pfq[4][3], dpe[4][3];
#pragma unroll
  for (int p = 0; p < 4; p++)
#pragma unroll
    for (int a = 0; a < 3; a++) pfq[p][a] = __shfl_sync(0xffffffffu, G.pf[a], 4 * L.pg + p);
  mlp_backward(d, sm.wt, act, L, G.pf, masks, g_out, pfq, dpe, P.d_packed[lv]);

  if (d.xyz && L.og == 0) {                                       // embedding chain -> dL/dp
#pragma unroll
    for (int p = 0; p < 4; p++) { const int l2 = chunk * kChunk + 4 * L.pg + p;
      if (l2 < Pb) { sm.dp[3 * l2] += (double)dpe[p][0]; sm.dp[3 * l2 + 1] += (double)dpe[p][1]; sm.dp[3 * l2 + 2] += (double)dpe[p][2]; } }
  }
  __syncwarp();
  const double* bb = lv == 0 ? P.in.coarse_bound : P.in.bound;
  // rows of padding points (lp >= Pb) carry zero gradients because their g_out is zero
  scatter_chunk(P.in.grid[lv], P.bw.d_grid[lv], P.bw.slot_map[lv], act, R_C, xn, L.lane, [&](int pt, const float gx[3]) {
    const int l2 = chunk * kChunk + pt;
    if (l2 < Pb) {
#pragma unroll
      for (int a = 0; a < 3; a++) sm.dp[3 * l2 + a] += ((double)gx[a] * 2.0) / (bb[2 * a + 1] - bb[2 * a]);   // d normalise / dp, common.py:280-282
    }
  });
  __syncwarp();
}

// load the forward state, in-bound flags, and the per-ray scans
__device__ __forceinline__ void bwd_prologue(const KParams& P, const Smem& sm, int r0, int nr, int Pb, int warp, int warps, int lane, float* gC) {
  const long long g0 = (long long)r0 * P.S;
  block_setup_rays(P, sm, r0, nr, 0.0f);                         // only o, d are used below (z comes from forward)
  for (int lp = threadIdx.x; lp < Pb; lp += blockDim.x) {
    sm.zs[lp] = P.bw.z_vals[g0 + lp];
    *reinterpret_cast<float4*>(sm.raw + 4 * lp) = *reinterpret_cast<const float4*>(P.bw.raw + 4 * (g0 + lp));
    sm.dp[3 * lp] = 0.0; sm.dp[3 * lp + 1] = 0.0; sm.dp[3 * lp + 2] = 0.0;
  }
  __syncthreads();
  for (int lp = threadIdx.x; lp < Pb; lp += blockDim.x) {        // in-bound flags (Renderer.py:43-46)
    const int ray = lp / P.S; const float* rr = sm.rays + 8 * ray;
    const float o[3] = {rr[0], rr[1], rr[2]}, d[3] = {rr[3], rr[4], rr[5]};
    PointGeom G; make_point(P.in.bound, P.in.coarse_bound, o, d, sm.zs[lp], G);
    sm.inb[lp] = (unsigned char)G.inb;
  }
  __syncthreads();
  // per-ray: compositing weights and dL/d(occupancy logit)   (SURVEY.md 8.1; cumprod backward in division form)
  for (int r = warp; r < nr; r += warps) {                       // one warp per ray, lanes over samples
    const float* rw = sm.raw + 4 * r * P.S;
    const double* z = sm.zs + r * P.S;
    float* wq = sm.wgt + r * P.S; float* go = sm.gocc + r * P.S;
    const double gD = P.bw.g_depth != nullptr ? P.bw.g_depth[r0 + r] : 0.0;
    const double gV = P.bw.g_var != nullptr ? P.bw.g_var[r0 + r] : 0.0;
    float g3[3] = {0.f, 0.f, 0.f};
    if (P.bw.g_rgb != nullptr) { g3[0] = P.bw.g_rgb[3 * (r0 + r)]; g3[1] = P.bw.g_rgb[3 * (r0 + r) + 1]; g3[2] = P.bw.g_rgb[3 * (r0 + r) + 2]; }
    if (lane == 0) { gC[3 * r] = g3[0]; gC[3 * r + 1] = g3[1]; gC[3 * r + 2] = g3[2]; }
    ray_weights(rw, P.S, lane, wq, go);                        // go[] temporarily holds T_s
    __syncwarp();
    double Dm = 0.0;
    for (int s = lane; s < P.S; s += 32) Dm += (double)wq[s] * z[s];
    Dm = warp_sum(Dm);
    double swt = 0.0;
    for (int s = lane; s < P.S; s += 32) swt += (double)wq[s] * (z[s] - Dm);
    swt = warp_sum(swt);
    const double gDe = gD + gV * (-2.0 * swt);                   // var reaches depth through tmp = z - depth
    // dL/dalpha_s = T_s g_w_s - (sum_{k>s} g_w_k w_k) / q_s   (cumprod backward in division form, SURVEY 8.1)
    float carry = 0.0f;
    const int nblk = (P.S + 31) / 32;
    for (int b = nblk - 1; b >= 0; b--) {
      const int s = b * 32 + lane;
      const bool v = s < P.S;
      float gw = 0.0f, al = 0.0f, T = 0.0f, w = 0.0f;
      if (v) {
        al = sigmoid_f(10.0f * rw[4 * s + 3]); T = go[s]; w = wq[s];
        const double t = z[s] - Dm;
        gw = (float)(gDe * z[s] + gV * t * t) + g3[0] * rw[4 * s] + g3[1] * rw[4 * s + 1] + g3[2] * rw[4 * s + 2];
      }
      const float incl = warp_incl_suffix_sum(gw * w, lane);
      float excl = __shfl_down_sync(0xffffffffu, incl, 1);       // exclusive suffix sum inside the block (no cancellation)
      if (lane == 31) excl = 0.0f;
      const float R = carry + excl;
      if (v) {
        const float qd = (1.0f - al) + 1e-10f;
        const float ga = T * gw - R / qd;
        go[s] = sm.inb[r * P.S + s] ? 10.0f * al * (1.0f - al) * ga : 0.0f;
      }
      carry += __shfl_sync(0xffffffffu, incl, 0);
    }
  }

}
// d rays_o = sum_s dp ; d rays_d = sum_s z_s dp   (pts = o + d*z, Renderer.py:172-174)
__device__ __forceinline__ void bwd_ray_reduce(const KParams& P, const Smem& sm, int r0, int nr) {
  if (P.bw.d_rays_o != nullptr || P.bw.d_rays_d != nullptr) {
    for (int t = threadIdx.x; t < nr * 3; t += blockDim.x) {
      const int r = t / 3, a = t - 3 * r;
      double so = 0.0, sd = 0.0;
      for (int s = 0; s < P.S; s++) { const double v = sm.dp[3 * (r * P.S + s) + a]; so += v; sd += v * sm.zs[r * P.S + s]; }
      if (P.accumulate_rays) {                                   // this ray's earlier contribution was written by the first launch
        if (P.bw.d_rays_o != nullptr) so += (double)P.bw.d_rays_o[3 * (r0 + r) + a];
        if (P.bw.d_rays_d != nullptr) sd += (double)P.bw.d_rays_d[3 * (r0 + r) + a];
      }
      if (P.bw.d_rays_o != nullptr) P.bw.d_rays_o[3 * (r0 + r) + a] = (float)so;
      if (P.bw.d_rays_d != nullptr) P.bw.d_rays_d[3 * (r0 + r) + a] = (float)sd;
    }
  }
}

// Fused pose gradient (optional): every CTA that has written ray gradients arrives on a grid-wide counter; the last one reduces
// d c2w = [sum_r d_rays_d[r] (x) dirs[r] | sum_r d_rays_o[r]] over the whole batch (fixed thread mapping -> deterministic) and resets
// the counter.  Saves the separate single-CTA pose_grad launch of a tracking iteration.
__device__ __forceinline__ bool fused_pose_grad(const KParams& P, int n_writers, double* __restrict__ s_pose /* [16][12] scratch in dynamic shared memory */) {
  if (P.bw.pose_dirs == nullptr) return false;
  __shared__ int s_pose_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int old = atomicAdd(P.bw.pose_counter, 1);
    s_pose_last = old == n_writers - 1;
    if (s_pose_last) *P.bw.pose_counter = 0;
  }
  __syncthreads();
  if (!s_pose_last) return false;
  __threadfence();
  double acc[12];
#pragma unroll
  for (int k = 0; k < 12; k++) acc[k] = 0.0;
  for (int r = threadIdx.x; r < P.in.n_rays; r += blockDim.x) {
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const double g = (double)__ldcg(P.bw.d_rays_d + 3 * r + i);
#pragma unroll
      for (int j = 0; j < 3; j++) acc[4 * i + j] += g * (double)__ldg(P.bw.pose_dirs + 3 * r + j);
      acc[4 * i + 3] += (double)__ldcg(P.bw.d_rays_o + 3 * r + i);
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 12; k++) {
    double v = acc[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0 && warp < 16) s_pose[warp * 12 + k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    double v = 0.0;
    const int nw = (int)(blockDim.x >> 5) < 16 ? (int)(blockDim.x >> 5) : 16;
    for (int w = 0; w < nw; w++) v += s_pose[w * 12 + threadIdx.x];
    P.bw.d_c2w[threadIdx.x] = v;
  }
  if (P.bw.result_dst != nullptr) {
    // read-back without a copy node: this CTA is the last writer of everything the caller wants back (ray gradients by the completing CTAs --
    // fenced above --, the loss by the forward launch, d c2w just now), so it stores the result block to its destination (the mapped view of a
    // pinned host block) itself.
    __syncthreads();
    const uint4* src = static_cast<const uint4*>(P.bw.result_src);
    uint4* dst = static_cast<uint4*>(P.bw.result_dst);
    const size_t n16 = P.bw.result_bytes >> 4;
    for (size_t i = threadIdx.x; i < n16; i += blockDim.x) __stwt(dst + i, __ldcg(src + i));
    const int tail = (int)(P.bw.result_bytes & 15);
    if ((int)threadIdx.x < tail)
      reinterpret_cast<unsigned char*>(dst)[(n16 << 4) + threadIdx.x] = __ldcg(reinterpret_cast<const unsigned char*>(src) + (n16 << 4) + threadIdx.x);
    __threadfence_system();
  }
  return true;                                                   // this CTA was the last one: d_c2w is complete (written by threads 0..11)
}

__global__ void __launch_bounds__(256, 1) render_bwd_kernel(const __grid_constant__ KParams P) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5;
  const LaneId L = make_lane(threadIdx.x & 31);
  Smem sm;
  smem_layout(P.wbytes, P.max_pts, P.max_rays, warps, kRowsBwd, true, &sm, smem_raw);
  float* act = sm.act + (size_t)warp * kRowsBwd * kRowF;
  __shared__ float gC[kMaxRaysPerBlock * 3];

  const int r0 = blockIdx.x * P.rays_per_block;
  const int nr = P.in.n_rays - r0 < P.rays_per_block ? P.in.n_rays - r0 : P.rays_per_block;
  const int Pb = nr * P.S;
  if (threadIdx.x == 0) { mbar_init(sm.bar, 1); mbar_fence_init(); }
  bwd_prologue(P, sm, r0, nr, Pb, warp, warps, L.lane, gC);

  const int nchunks = (Pb + kChunk - 1) / kChunk;
  uint32_t parity = 0;
  for (int qd = 0; qd < P.n_dec; qd++) {
    const int lv = P.dec[qd];
    const DecRT d = make_dec(lv);
    __syncthreads();
    if (threadIdx.x == 0) issue_weights(P, sm, lv);
#pragma unroll 1
    for (int chunk = warp; chunk < nchunks; chunk += warps) chunk_backward(P, sm, act, chunk, Pb, L, parity, gC, lv, d);
    parity ^= 1u;
  }
  __syncthreads();
  bwd_ray_reduce(P, sm, r0, nr);
}

}  // namespace nsb
#include "nsb_tc.cuh"
#include "nsb_tile.cuh"
namespace nsb {

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int stage_decoders(int stage, int dec[3]) {   // NICE.forward evaluation order, decoder.py:317-342
  switch (stage) {
    case NSB_STAGE_COARSE: dec[0] = NSB_COARSE; return 1;
    case NSB_STAGE_MIDDLE: dec[0] = NSB_MIDDLE; return 1;
    case NSB_STAGE_FINE: dec[0] = NSB_FINE; dec[1] = NSB_MIDDLE; return 2;
    default: dec[0] = NSB_FINE; dec[1] = NSB_COLOR; dec[2] = NSB_MIDDLE; return 3;
  }
}

static int validate_inputs(const nsb_render_inputs* in, bool need_rays) {
  if (!in) { set_error("inputs == NULL"); return NSB_ERR_ARG; }
  if (in->stage < 0 || in->stage > 3) { set_error("bad stage %d", in->stage); return NSB_ERR_ARG; }
  if (need_rays) {
    if (in->n_rays < 0) { set_error("n_rays < 0"); return NSB_ERR_ARG; }
    if (in->n_rays > 0 && (!in->rays_o || !in->rays_d)) { set_error("rays_o / rays_d are NULL"); return NSB_ERR_ARG; }
    if (in->n_samples < 1 || !in->t_uniform) { set_error("n_samples < 1 or t_uniform NULL"); return NSB_ERR_ARG; }
    if (in->gt_depth_batch && (!in->gt_depth || in->n_batch < 1 || in->n_batch > NSB_MAX_BATCH_DEPTHS)) {
      set_error("gt_depth_batch needs gt_depth and 1 <= n_batch <= %d (got %d)", NSB_MAX_BATCH_DEPTHS, in->n_batch); return NSB_ERR_ARG; }
    if (in->gt_depth && !in->depth_max && !in->gt_depth_batch && in->n_rays > NSB_INLINE_MAX_RAYS) {
      set_error("gt_depth given without depth_max: batches of more than %d rays need nsb_batch_max_depth", NSB_INLINE_MAX_RAYS); return NSB_ERR_ARG; }
  }
  int dec[3]; const int nd = stage_decoders(in->stage, dec);
  for (int i = 0; i < nd; i++) {
    const nsb_grid& g = in->grid[dec[i]];
    if (!g.data || g.D < 1 || g.H < 1 || g.W < 1) { set_error("grid %d missing", dec[i]); return NSB_ERR_ARG; }
    if (g.stride_c == 1 && (g.stride_w % 4 || g.stride_h % 4 || g.stride_d % 4 || ((uintptr_t)g.data & 15))) {
      set_error("channels-last grid %d must be 16-byte aligned with strides multiple of 4", dec[i]); return NSB_ERR_ARG; }
    if (!in->packed[dec[i]]) { set_error("packed decoder %d missing (call nsb_pack_decoders)", dec[i]); return NSB_ERR_ARG; }
    if ((uintptr_t)in->packed[dec[i]] & 15) { set_error("packed decoder %d not 16-byte aligned", dec[i]); return NSB_ERR_ARG; }
  }
  return NSB_OK;
}

static void fill_common(KParams& K, const nsb_render_inputs* in) {
  K.in = *in;
  K.has_gt = (in->gt_depth != nullptr && in->stage != NSB_STAGE_COARSE) ? 1 : 0;    // Renderer.py:88-92
  K.S = in->n_samples + (K.has_gt ? in->n_surface : 0);
  K.n_dec = stage_decoders(in->stage, K.dec);
  for (int i = 0; i < 3; i++) K.dec_pos[i] = i;
  K.accumulate_rays = 0;
  K.split = 1; K.ray_parts = nullptr; K.ray_cnt = nullptr; K.tile_parts = nullptr; K.tile_rays = 0;
  memset(&K.fs, 0, sizeof(K.fs)); memset(&K.tail, 0, sizeof(K.tail));
  int wb = 0;
  for (int i = 0; i < K.n_dec; i++) { const int b = packed_floats(K.dec[i]) * 4; wb = b > wb ? b : wb; }
  K.wbytes = wb;
  K.points = nullptr; K.points_raw = nullptr; K.n_points = 0;
  K.acts_lv = in->stage == NSB_STAGE_COLOR ? 3 : -1;      // the colour decoder is the only one whose weights the mapper optimises (Mapper.py:339-341)
  for (int l = 0; l < 4; l++) K.d_packed[l] = nullptr;
}

// per-device caches (one process may drive several GPUs: the reference configures tracker and mapper devices separately)
constexpr int kMaxDevices = 64;
static int g_sm_count[kMaxDevices] = {0};
static int current_device() { int dev = 0; cudaGetDevice(&dev); return dev >= 0 && dev < kMaxDevices ? dev : 0; }
static int sm_count() {
  const int dev = current_device();
  if (g_sm_count[dev] == 0) { cudaDeviceGetAttribute(&g_sm_count[dev], cudaDevAttrMultiProcessorCount, dev); if (g_sm_count[dev] <= 0) g_sm_count[dev] = 148; }
  return g_sm_count[dev];
}

// choose rays per CTA and warps per CTA: fill all SMs once before growing CTAs (latency-bound small batches),
// cap CTA size by the shared-memory budget (227 KB per CTA, 1 KB kept for static shared memory)
constexpr size_t kSmemCap = 226u * 1024u;
static void choose_config(int n_items, int S, int rows, bool bwd, int wbytes, int max_warps, KParams* K, int* warps, size_t* smem) {
  const int sms = sm_count();
  int r_cap = kMaxPtsPerBlock / S; if (r_cap < 1) r_cap = 1; if (r_cap > kMaxRaysPerBlock) r_cap = kMaxRaysPerBlock;
  int r = (n_items + sms - 1) / sms; if (r < 1) r = 1; if (r > r_cap) r = r_cap;
  const int max_pts = ((r * S + kChunk - 1) / kChunk) * kChunk;
  const int chunks = max_pts / kChunk;
  int w = chunks < max_warps ? chunks : max_warps;
  while (w > 1 && smem_layout(wbytes, max_pts, r, w, rows, bwd, nullptr, nullptr) > kSmemCap) w--;
  const int rounds = (chunks + w - 1) / w;
  w = (chunks + rounds - 1) / rounds;                    // same number of rounds with balanced warps
  K->rays_per_block = r; K->max_pts = max_pts; K->max_rays = r;
  *warps = w;
  *smem = smem_layout(wbytes, max_pts, r, w, rows, bwd, nullptr, nullptr);
}

static int g_split_model = 1;      // tile kernels: per-decoder items only while they beat all-decoder items by wave efficiency (0: split whenever N*S <= kSplitMaxPts)
static int g_fwd_f16 = 0;          // tile-kernel forward with FP16 hi|lo operands (kind::f16, K = 16 per MMA) instead of 3xTF32; see nsb_tile.cuh mma_unit_h
static int g_wgrad_tc = 1;         // decoder weight gradients on the tensor cores when the forward kept the layer outputs (0: FP32-FMA pass)
static int g_mlp_backend = 0;      // 0 = auto (tile kernels where S >= 8, otherwise FP32-FMA), 1 = FP32-FMA
// ---- tile kernels: workspace = [16 B | ray completion counters (N ints) | per-item scratch] -----------------------------------------
// per-item scratch: forward = decoder outputs [split][N*S] float4 (only when items are split per decoder; otherwise they live in fo.raw),
// backward = ray-gradient parts [tiles * split][kMaxTileRays][6] f64.  Items are split per decoder for batches of up to kSplitMaxPts points
// (finer granularity for small and medium batches); larger batches evaluate all decoders of a tile in one CTA.
constexpr long long kSplitMaxPts = 262144;
struct TileWs { int split; int* ray_cnt; void* scratch; };
static long long tile_count(long long n_points) { return (n_points + tc::TM - 1) / tc::TM; }
static int tile_rays(int S) { const int r = (tc::TM - 1) / S + 2; return r < tl::kMaxTileRays ? r : tl::kMaxTileRays; }
// Layout: [scratch ... | ray counters (N ints) at the very END of the buffer].  The counters must stay zero between launches (the completing
// CTA resets them) while the scratch is left dirty; anchoring the counters at the end keeps the two apart when one buffer, sized for a
// capacity, serves batches of varying size (the mapper's bbox pre-filter changes N every iteration): counters of any N <= capacity live
// in the last 4 * capacity bytes, which no scratch of a batch <= capacity reaches (the sizing below is monotone in N).
static size_t tile_scratch_bytes(int N, int S, int split, bool bwd) {
  const long long NS = (long long)N * S;
  return bwd ? (size_t)tile_count(NS) * split * tile_rays(S) * 6 * sizeof(double) : (split > 1 ? (size_t)split * NS * sizeof(float4) : 0);
}
static size_t tile_ws_need(int N, int S, int split, bool bwd) { return 16 + align16((size_t)N * sizeof(int)) + align16(tile_scratch_bytes(N, S, split, bwd)); }
static bool tile_ws_plan(void* ws, size_t bytes, int N, int S, int n_dec, bool bwd, TileWs* out) {
  if (!ws || (reinterpret_cast<uintptr_t>(ws) & 15)) return false;
  bytes &= ~size_t(15);
  int split = ((long long)N * S <= kSplitMaxPts && n_dec > 1) ? n_dec : 1;
  if (split > 1 && g_split_model) {
    // Splitting a tile's decoders over CTAs buys parallelism for batches that do not fill the GPU, at the price of one prologue / ray-completion
    // pass per decoder: measured on the configs[4] sweep, a per-decoder item sustains ~0.81x (three decoders) of the throughput of the same work
    // inside all-decoder items.  Once the tiles alone fill the resident slots (two CTAs per SM), compare the two forms by their wave efficiency.
    const long long tiles = tile_count((long long)N * S), slots = 2ll * sm_count();
    auto wave_eff = [&](long long items) { const long long waves = (items + slots - 1) / slots; return (double)items / (double)(waves * slots); };
    const double eff_one = wave_eff(tiles), eff_split = wave_eff(tiles * n_dec) * (1.0 - 0.095 * (n_dec - 1));
    if (tiles >= slots && eff_one >= eff_split) split = 1;
  }
  if (bytes < tile_ws_need(N, S, split, bwd)) split = 1;
  if (bytes < tile_ws_need(N, S, split, bwd)) return false;
  out->split = split;
  out->ray_cnt = reinterpret_cast<int*>(static_cast<char*>(ws) + bytes - align16((size_t)N * sizeof(int)));
  out->scratch = static_cast<char*>(ws);
  return true;
}
extern "C" size_t nsb_split_workspace_bytes(int n_rays, int S) {
  if (n_rays < 1 || S < 1) return 0;
  auto need_exact = [&](int n, int s) {
    const int split = (long long)n * s <= kSplitMaxPts ? 3 : 1;
    const size_t a = tile_scratch_bytes(n, s, split, false), b = tile_scratch_bytes(n, s, split, true);
    return align16(a > b ? a : b);
  };
  auto need = [&](int s) {                                  // monotone in n_rays: also covers the largest batch that still splits per decoder
    const long long n_small = kSplitMaxPts / s;
    const size_t a = need_exact(n_rays, s), b = need_exact((int)(n_small < n_rays ? (n_small > 0 ? n_small : 1) : n_rays), s);
    return a > b ? a : b;
  };
  size_t m = need(S);
  if (S >= NSB_MAX_SAMPLES) for (int s = tl::kMinSamples; s < NSB_MAX_SAMPLES; s++) { const size_t v = need(s); if (v > m) m = v; }   // "any S" sizing (nsb_iteration_workspace_bytes)
  return m + 16 + align16((size_t)n_rays * sizeof(int));
}
static size_t tile_smem_bytes(bool bwd) { return tl::common_bytes(bwd) + (bwd ? sizeof(tl::BwdExtra) : 0); }
static size_t tile_wg_smem_bytes() { return tl::kWgBytes + ((tile_smem_bytes(true) + 1023) & ~size_t(1023)) + 1024; }
// Tensor-core tile kernels or FP32-FMA kernels.  A tile may touch at most kMaxTileRays rays, which bounds S from below; smaller S runs on the
// FP32-FMA kernels.  Forward and backward of an iteration see the same S and so pick the same family (the saved ReLU bits are laid out per family).
static bool use_tile_kernels(int S) { return g_mlp_backend == 0 && S >= tl::kMinSamples && S <= NSB_MAX_SAMPLES; }
static bool g_attr_set[kMaxDevices] = {false};
static int set_attrs() {
  const int dev = current_device();
  if (g_attr_set[dev]) return NSB_OK;
  if (check_cuda(cudaFuncSetAttribute(render_fwd_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem_bytes(false)), "fwd tile smem attr")) return NSB_ERR_CUDA;
  if (check_cuda(cudaFuncSetAttribute(render_fwd_tile_h16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem_bytes(false)), "fwd tile (f16) smem attr")) return NSB_ERR_CUDA;
  if (check_cuda(cudaFuncSetAttribute(render_fwd_tile_h16_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared), "fwd tile (f16) carveout")) return NSB_ERR_CUDA;
  if (check_cuda(cudaFuncSetAttribute(render_bwd_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem_bytes(true)), "bwd tile smem attr")) return NSB_ERR_CUDA;
  if (check_cuda(cudaFuncSetAttribute(render_bwd_wg_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_wg_smem_bytes()), "bwd wg tile smem attr")) return NSB_ERR_CUDA;
  // two CTAs per SM need the full shared-memory carve-out (2 x ~111 KB of the 228 KB)
  if (check_cuda(cudaFuncSetAttribute(render_fwd_tile_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared), "fwd tile carveout")) return NSB_ERR_CUDA;
  if (check_cuda(cudaFuncSetAttribute(render_bwd_tile_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared), "bwd tile carveout")) return NSB_ERR_CUDA;
  if (check_cuda(cudaFuncSetAttribute(render_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap), "fwd smem attr")) return NSB_ERR_CUDA;
  if (check_cuda(cudaFuncSetAttribute(render_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap), "bwd smem attr")) return NSB_ERR_CUDA;
  g_attr_set[dev] = true;
  return NSB_OK;
}

}  // namespace nsb

using namespace nsb;

extern "C" int nsb_set_option(const char* key, int value) {
  if (key && !strcmp(key, "wgrad_tc")) { g_wgrad_tc = value != 0; return NSB_OK; }
  if (key && !strcmp(key, "fwd_f16")) { g_fwd_f16 = value != 0; return NSB_OK; }
  if (key && !strcmp(key, "split_model")) { g_split_model = value != 0; return NSB_OK; }
  if (key && !strcmp(key, "mlp_backend")) { if (value < 0 || value > 1) { set_error("mlp_backend must be 0 (auto = tile kernels) or 1 (FP32-FMA)"); return NSB_ERR_ARG; } g_mlp_backend = value; return NSB_OK; }
  set_error("unknown option %s", key ? key : "(null)"); return NSB_ERR_ARG;
}

extern "C" int nsb_render_forward(const nsb_render_inputs* in, const nsb_forward_outputs* out, void* stream) {
  return nsb::render_forward_fused(in, out, nullptr, stream);
}
int nsb::render_forward_fused(const nsb_render_inputs* in, const nsb_forward_outputs* out, const nsb::FusedSeeds* fs, void* stream) {
  int rc = validate_inputs(in, true); if (rc) return rc;
  if (!out || !out->depth || !out->var || !out->rgb) { set_error("forward outputs missing"); return NSB_ERR_ARG; }
  if (in->n_rays == 0) return NSB_OK;
  KParams K; fill_common(K, in); K.fo = *out; memset(&K.bw, 0, sizeof(K.bw));
  if (fs != nullptr) K.fs = *fs;
  const bool tile = use_tile_kernels(K.S);
  if (!tile) K.fo.masks = nullptr;                                // only the tensor-core forward produces masks
  if (K.S > NSB_MAX_SAMPLES) { set_error("n_samples+n_surface = %d exceeds %d", K.S, NSB_MAX_SAMPLES); return NSB_ERR_UNSUPPORTED; }
  if (K.has_gt && in->n_surface > 0 && !in->t_surface) { set_error("t_surface NULL"); return NSB_ERR_ARG; }
  if ((rc = set_attrs())) return rc;
  if (K.fs.px.world > 1 && !(tile && in->gt_depth != nullptr)) {
    set_error("in-kernel exchanges of a sharded forward need the tile kernels (mlp_backend 0, n_samples+n_surface >= %d) and gt_depth", tl::kMinSamples); return NSB_ERR_UNSUPPORTED; }
  if (tile) {                                             // tile kernels: item = (128-point tile, decoder), two CTAs per SM
    if (!out->z_vals || !out->raw) { set_error("the tensor-core forward needs z_vals and raw outputs"); return NSB_ERR_ARG; }
    TileWs w;
    if (!tile_ws_plan(out->split_workspace, out->split_workspace_bytes, in->n_rays, K.S, K.n_dec, false, &w)) {
      set_error("split_workspace missing or smaller than nsb_split_workspace_bytes(%d, %d)", in->n_rays, K.S); return NSB_ERR_ARG; }
    K.split = w.split; K.ray_cnt = w.ray_cnt;
    K.tile_parts = w.split > 1 ? static_cast<float4*>(w.scratch) : reinterpret_cast<float4*>(out->raw);
    const long long grid_t = tile_count((long long)in->n_rays * K.S) * K.split;
    if (g_fwd_f16) render_fwd_tile_h16_kernel<<<(unsigned)grid_t, tl::kThreads, tile_smem_bytes(false), (cudaStream_t)stream>>>(K);
    else render_fwd_tile_kernel<<<(unsigned)grid_t, tl::kThreads, tile_smem_bytes(false), (cudaStream_t)stream>>>(K);
    return check_cuda(cudaGetLastError(), "render_fwd_tile_kernel launch");
  }
  int warps; size_t smem;
  choose_config(in->n_rays, K.S, kRowsFwd, false, K.wbytes, 8, &K, &warps, &smem);
  if (smem > kSmemCap) { set_error("shared-memory budget exceeded (%zu bytes)", smem); return NSB_ERR_UNSUPPORTED; }
  const int grid = (in->n_rays + K.rays_per_block - 1) / K.rays_per_block;
  render_fwd_kernel<<<grid, warps * 32, smem, (cudaStream_t)stream>>>(K);
  return check_cuda(cudaGetLastError(), "render_fwd_kernel launch");
}

extern "C" int nsb_eval_points(const nsb_render_inputs* in, const double* points, int n_points, float* raw, void* stream) {
  int rc = validate_inputs(in, false); if (rc) return rc;
  if (n_points < 0 || (n_points > 0 && (!points || !raw))) { set_error("points / raw missing"); return NSB_ERR_ARG; }
  if (n_points == 0) return NSB_OK;
  KParams K; fill_common(K, in); memset(&K.fo, 0, sizeof(K.fo)); memset(&K.bw, 0, sizeof(K.bw));
  K.points = points; K.points_raw = raw; K.n_points = n_points; K.S = 1; K.has_gt = 0;
  if ((rc = set_attrs())) return rc;
  // points mode: "rays_per_block" = points per CTA
  const int sms = sm_count();
  int ppb = (n_points + sms - 1) / sms; ppb = ((ppb + kChunk - 1) / kChunk) * kChunk;
  if (ppb > kMaxPtsPerBlock) ppb = kMaxPtsPerBlock;
  if (ppb < kChunk) ppb = kChunk;
  int warps = ppb / kChunk < 8 ? ppb / kChunk : 8;
  while (warps > 1 && smem_layout(K.wbytes, ppb, 1, warps, kRowsFwd, false, nullptr, nullptr) > kSmemCap) warps--;
  const size_t smem = smem_layout(K.wbytes, ppb, 1, warps, kRowsFwd, false, nullptr, nullptr);
  K.rays_per_block = ppb; K.max_pts = ppb; K.max_rays = 1;
  const int grid = (n_points + ppb - 1) / ppb;
  if (g_mlp_backend == 0) {
    K.split = 1;
    if (g_fwd_f16) render_fwd_tile_h16_kernel<<<(unsigned)tile_count(n_points), tl::kThreads, tile_smem_bytes(false), (cudaStream_t)stream>>>(K);
    else render_fwd_tile_kernel<<<(unsigned)tile_count(n_points), tl::kThreads, tile_smem_bytes(false), (cudaStream_t)stream>>>(K);
    return check_cuda(cudaGetLastError(), "render_fwd_tile_kernel(points) launch");
  }
  render_fwd_kernel<<<grid, warps * 32, smem, (cudaStream_t)stream>>>(K);
  return check_cuda(cudaGetLastError(), "render_fwd_kernel(points) launch");
}

namespace nsb { int launch_unpack_grads(float* const d_packed[4], float* const d_flat[4], cudaStream_t st); }

extern "C" size_t nsb_backward_workspace_bytes(void) {
  size_t t = 0; for (int l = 0; l < 4; l++) t += align16((size_t)packed_floats(l) * 4); return t;
}

extern "C" int nsb_render_backward(const nsb_render_inputs* in, const nsb_backward_args* bw, void* stream) {
  return nsb::render_backward_tail(in, bw, nullptr, stream);
}
int nsb::render_backward_tail(const nsb_render_inputs* in, const nsb_backward_args* bw, const nsb::PeerTail* tail, void* stream) {
  int rc = validate_inputs(in, true); if (rc) return rc;
  if (!bw || !bw->z_vals || !bw->raw) { set_error("backward needs z_vals and raw from the forward pass"); return NSB_ERR_ARG; }
  if (in->n_rays == 0) return NSB_OK;
  KParams K; fill_common(K, in); K.bw = *bw; memset(&K.fo, 0, sizeof(K.fo));
  if (K.S > NSB_MAX_SAMPLES) { set_error("n_samples+n_surface = %d exceeds %d", K.S, NSB_MAX_SAMPLES); return NSB_ERR_UNSUPPORTED; }
  cudaStream_t st = (cudaStream_t)stream;
  bool any_w = false;
  const bool want_pose = bw->pose_dirs != nullptr;
  if (want_pose && (!bw->d_c2w || !bw->pose_counter || !bw->d_rays_o || !bw->d_rays_d)) {
    set_error("pose_dirs given without d_c2w / pose_counter / d_rays_o / d_rays_d"); return NSB_ERR_ARG; }
  if (bw->result_dst != nullptr) {
    if (!want_pose) { set_error("result_dst needs pose_dirs (the block is stored by the CTA that produces d c2w)"); return NSB_ERR_ARG; }
    if (tail != nullptr && tail->px.world > 1) { set_error("result_dst is not supported by the sharded backward tail"); return NSB_ERR_ARG; }
    if (!bw->result_src || ((reinterpret_cast<uintptr_t>(bw->result_dst) | reinterpret_cast<uintptr_t>(bw->result_src)) & 15)) {
      set_error("result_dst / result_src must be non-NULL and 16-byte aligned"); return NSB_ERR_ARG; }
  }
  K.bw.pose_dirs = nullptr;                                        // fused only into the LAST launch that writes ray gradients (below)
  for (int l = 0; l < 4; l++) {
    if (bw->slot_map[l] != nullptr && bw->d_grid[l] != nullptr && (reinterpret_cast<uintptr_t>(bw->d_grid[l]) & 15) != 0) {
      set_error("compact d_grid[%d] must be 16-byte aligned", l); return NSB_ERR_ARG;
    }
  }
  for (int i = 0; i < K.n_dec; i++) {
    const int l = K.dec[i];
    if (bw->d_flat[l] != nullptr) {
      if (!bw->workspace) { set_error("d_flat requested but workspace is NULL (nsb_backward_workspace_bytes)"); return NSB_ERR_ARG; }
      size_t off = 0; for (int m = 0; m < l; m++) off += align16((size_t)packed_floats(m) * 4);
      K.d_packed[l] = reinterpret_cast<float*>(reinterpret_cast<char*>(bw->workspace) + off);
      if (check_cuda(cudaMemsetAsync(K.d_packed[l], 0, (size_t)packed_floats(l) * 4, st), "memset d_packed")) return NSB_ERR_CUDA;
      any_w = true;
    }
  }
  // grids/weights that are not part of this stage get no gradient
  for (int l = 0; l < 4; l++) { bool used = false; for (int i = 0; i < K.n_dec; i++) used |= K.dec[i] == l; if (!used) { K.bw.d_grid[l] = nullptr; } }
  if ((rc = set_attrs())) return rc;
  int warps; size_t smem;
  choose_config(in->n_rays, K.S, kRowsBwd, true, K.wbytes, 8, &K, &warps, &smem);
  if (smem > kSmemCap) { set_error("shared-memory budget exceeded (%zu bytes)", smem); return NSB_ERR_UNSUPPORTED; }
  const bool sharded = tail != nullptr && tail->px.world > 1;
  if (bw->masks != nullptr && use_tile_kernels(K.S)) {            // (no saved ReLU masks -> FP32 kernel, which recomputes the forward)
    // Tensor-core kernel for the decoders that only need input gradients (rays, voxels).  Decoders whose WEIGHT gradients are
    // requested (the colour decoder in the mapper's colour stage, Mapper.py:339-341) go through the FP32-FMA kernel in a second
    // launch that adds its share of the ray gradients.
    KParams T = K;
    T.n_dec = 0;
    int n_w = 0, wdec[3], wpos[3];
    for (int i = 0; i < K.n_dec; i++) {
      if (bw->d_flat[K.dec[i]] != nullptr) { wdec[n_w] = K.dec[i]; wpos[n_w] = i; n_w++; }
      else { T.dec[T.n_dec] = K.dec[i]; T.dec_pos[T.n_dec] = i; T.n_dec++; }
    }
    // Weight gradients on the tensor cores: the colour decoder, when the forward kept its layer outputs (acts) -- a second tile launch with one item
    // per tile (one CTA per SM) after the input-gradient launch of the other decoders; it adds its share of the ray gradients.
    const bool wg_tc = n_w == 1 && wdec[0] == 3 && bw->acts != nullptr && g_wgrad_tc && !sharded;
    if (T.n_dec > 0) {
      if (n_w == 0 && want_pose) T.bw.pose_dirs = bw->pose_dirs;   // the tensor-core launch is the last writer of the ray gradients
      TileWs w;
      if (!tile_ws_plan(bw->split_workspace, bw->split_workspace_bytes, in->n_rays, T.S, T.n_dec, true, &w)) {
        set_error("split_workspace missing or smaller than nsb_split_workspace_bytes(%d, %d)", in->n_rays, T.S); return NSB_ERR_ARG; }
      T.split = w.split; T.ray_cnt = w.ray_cnt; T.ray_parts = static_cast<double*>(w.scratch); T.tile_rays = tile_rays(T.S);
      if (sharded) {
        if (n_w != 0 || T.bw.pose_dirs == nullptr) { set_error("sharded backward tail needs pose_dirs and no decoder weight gradients"); return NSB_ERR_ARG; }
        T.tail = *tail;
      }
      const long long grid_t = tile_count((long long)in->n_rays * T.S) * T.split;
      render_bwd_tile_kernel<<<(unsigned)grid_t, tl::kThreads, tile_smem_bytes(true), st>>>(T);
      if ((rc = check_cuda(cudaGetLastError(), "render_bwd_tile_kernel launch"))) return rc;
      if (n_w == 0) return NSB_OK;
      K.accumulate_rays = 1;
    }
    if (wg_tc) {
      KParams W = K;
      W.n_dec = 1; W.dec[0] = wdec[0]; W.dec_pos[0] = wpos[0];
      W.accumulate_rays = T.n_dec > 0 ? 1 : 0;
      W.bw.pose_dirs = want_pose ? bw->pose_dirs : nullptr;          // last writer of the ray gradients: d c2w by its last CTA
      TileWs w;
      if (!tile_ws_plan(bw->split_workspace, bw->split_workspace_bytes, in->n_rays, W.S, 1, true, &w)) {
        set_error("split_workspace missing or smaller than nsb_split_workspace_bytes(%d, %d)", in->n_rays, W.S); return NSB_ERR_ARG; }
      W.split = 1; W.ray_cnt = w.ray_cnt; W.ray_parts = static_cast<double*>(w.scratch); W.tile_rays = tile_rays(W.S);
      render_bwd_wg_tile_kernel<<<(unsigned)tile_count((long long)in->n_rays * W.S), tl::kThreads, tile_wg_smem_bytes(), st>>>(W);
      if ((rc = check_cuda(cudaGetLastError(), "render_bwd_wg_tile_kernel launch"))) return rc;
      return launch_unpack_grads(W.d_packed, bw->d_flat, st);
    }
    if (T.n_dec > 0) {
      K.n_dec = n_w;
      for (int i = 0; i < n_w; i++) { K.dec[i] = wdec[i]; K.dec_pos[i] = wpos[i]; }
      int wb = 0;
      for (int i = 0; i < K.n_dec; i++) { const int b = packed_floats(K.dec[i]) * 4; wb = b > wb ? b : wb; }
      K.wbytes = wb;
      choose_config(in->n_rays, K.S, kRowsBwd, true, K.wbytes, 8, &K, &warps, &smem);
      if (smem > kSmemCap) { set_error("shared-memory budget exceeded (%zu bytes)", smem); return NSB_ERR_UNSUPPORTED; }
    }
  }
  const int grid = (in->n_rays + K.rays_per_block - 1) / K.rays_per_block;
  render_bwd_kernel<<<grid, warps * 32, smem, st>>>(K);
  if ((rc = check_cuda(cudaGetLastError(), "render_bwd_kernel launch"))) return rc;
  if (any_w && (rc = launch_unpack_grads(K.d_packed, bw->d_flat, st))) return rc;
  if (want_pose) {                                                 // FP32 path: separate launches
    if ((rc = nsb_pose_grad(bw->pose_dirs, bw->d_rays_o, bw->d_rays_d, in->n_rays, bw->d_c2w, stream))) return rc;
    if (bw->result_dst != nullptr) return nsb_copy_block(bw->result_dst, bw->result_src, bw->result_bytes, stream);
  }
  return NSB_OK;
}

// resident CTAs per SM of the tile kernels (diagnostic; 2 = the design point)
extern "C" int nsb_debug_occupancy(int* fwd, int* bwd) {
  int rc = set_attrs(); if (rc) return rc;
  if (check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(fwd, render_fwd_tile_kernel, tl::kThreads, tile_smem_bytes(false)), "occupancy fwd")) return NSB_ERR_CUDA;
  if (check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(bwd, render_bwd_tile_kernel, tl::kThreads, tile_smem_bytes(true)), "occupancy bwd")) return NSB_ERR_CUDA;
  return NSB_OK;
}

#ifdef NSB_PHASE_TIMING
extern "C" int nsb_debug_phases(long long* out64, int reset) {
  cudaError_t e = cudaMemcpyFromSymbol(out64, nsb::tc::g_phase, sizeof(long long) * 64);
  if (e == cudaSuccess && reset) { long long z[64] = {0}; e = cudaMemcpyToSymbol(nsb::tc::g_phase, z, sizeof(z)); }
  return e == cudaSuccess ? 0 : 1;
}
#endif
