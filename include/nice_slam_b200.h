/*
 * nice_slam_b200.h -- C ABI of the B200-native render-and-backprop path for NICE-SLAM.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference (cvg/nice-slam) has no FFI layer:
 * its operator boundary is the Python object `slam.renderer` (src/NICE_SLAM.py:91) whose methods
 * Renderer.render_batch_ray / eval_points / render_img (src/utils/Renderer.py:63,23,200) are called by
 * Tracker.optimize_cam_in_batch (src/Tracker.py:106) and Mapper.optimize_map (src/Mapper.py:482).
 * The functions below are what a ctypes binding of that object calls (see INTEGRATION.md); every
 * pointer is a raw device pointer owned by the caller (torch storage), every size is a plain integer,
 * no torch types cross this boundary.  All entry points return 0 on success and a negative nsb_status
 * on failure; nsb_last_error() gives the message (the Python side raises RuntimeError, the reference's
 * own convention being plain Python exceptions).
 *
 * Threading: calls are asynchronous on the given cudaStream_t (pass the caller's current stream); the
 * library keeps no per-call state and allocates nothing persistent, so the three reference processes
 * (tracker, mapper, coarse mapper; src/NICE_SLAM.py:288-307) can each dlopen it independently.
 */
#ifndef NICE_SLAM_B200_H_
#define NICE_SLAM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NSB_VERSION 100           /* 1.0.0 */
#define NSB_C_DIM 32              /* feature channels per grid     (configs/nice_slam.yaml:113) */
#define NSB_HIDDEN 32             /* decoder width                 (src/conv_onet/models/decoder.py:293) */
#define NSB_EMBED 93              /* Gaussian-Fourier mapping size (src/conv_onet/models/decoder.py:133) */
#define NSB_MAX_BATCH_DEPTHS 8192 /* nsb_render_inputs.n_batch: every CTA reduces the list itself (L2-resident) */
#define NSB_INLINE_MAX_RAYS 1024  /* up to this batch size nsb_render_inputs.depth_max may be NULL: the kernels reduce gt_depth themselves */
#define NSB_MAX_SAMPLES 256       /* N_samples + N_surface per ray supported by the kernels */

typedef enum { NSB_OK = 0, NSB_ERR_ARG = -1, NSB_ERR_CUDA = -2, NSB_ERR_UNSUPPORTED = -3 } nsb_status;

/* stage of NICE.forward (src/conv_onet/models/decoder.py:312-342) */
typedef enum { NSB_STAGE_COARSE = 0, NSB_STAGE_MIDDLE = 1, NSB_STAGE_FINE = 2, NSB_STAGE_COLOR = 3 } nsb_stage;
/* decoder / grid slot indices used by every array-of-4 below */
typedef enum { NSB_COARSE = 0, NSB_MIDDLE = 1, NSB_FINE = 2, NSB_COLOR = 3 } nsb_level;

/* One hierarchical feature grid, logical shape [1, 32, D, H, W] (src/NICE_SLAM.py:192-250; D=z, H=y, W=x).
 * Strides are in elements.  Fast path: channels-last (stride_c == 1, stride_w == 32), 128 B per voxel.
 * The reference's contiguous NCDHW layout is accepted too (slow gathers). */
typedef struct {
  const float* data;
  int32_t D, H, W;
  int64_t stride_c, stride_d, stride_h, stride_w;
} nsb_grid;

/* Device pointers to one decoder's parameter tensors exactly as the reference's nn.Module holds them
 * (contiguous fp32).  MLP (middle/fine/color): src/conv_onet/models/decoder.py:117-164;
 * MLP_no_xyz (coarse): :224-253 (B, Wc, bc are NULL).
 *   B      embedder._B              [3][93]
 *   W[i]   pts_linears.i.weight     [32][in_i]   in = 93,32,32,125,32   (coarse: 32,32,32,64,32)
 *   b[i]   pts_linears.i.bias       [32]
 *   Wc[i]  fc_c.i.weight            [32][c_dim]  c_dim = 32 (middle,color) / 64 (fine)
 *   bc[i]  fc_c.i.bias              [32]
 *   Wo/bo  output_linear            [n_out][32], [n_out]   n_out = 1 (occupancy) / 4 (color)     */
typedef struct {
  const float* B;
  const float* W[5];
  const float* b[5];
  const float* Wc[5];
  const float* bc[5];
  const float* Wo;
  const float* bo;
} nsb_decoder_params;

/* Canonical flat order of one decoder's parameters / parameter gradients:
 *   [B] [W0 b0 W1 b1 W2 b2 W3 b3 W4 b4] [Wc0 bc0 ... Wc4 bc4] [Wo bo]      (row-major as above) */
size_t nsb_flat_decoder_floats(int level);
/* Offset (in floats) of a named block inside the flat order.  kind: 0=B 1=W 2=b 3=Wc 4=bc 5=Wo 6=bo */
long long nsb_flat_offset(int level, int kind, int layer);
/* Size (in floats) of the kernel-side packed weight image of one decoder (padded, TMA-stageable). */
size_t nsb_packed_decoder_floats(int level);

int nsb_version(void);
const char* nsb_last_error(void);
/* Process-wide options.  "mlp_backend": 0 = auto (default: tcgen05 tile kernels, 3xTF32, two CTAs per SM; FP32-FMA decoders where
 * n_samples + n_surface < 8), 1 = FP32-FMA decoders; other values return NSB_ERR_ARG.  "split_model": 1 (default) = a tile's decoders are
 * spread over CTAs only while that beats one CTA per tile by wave efficiency, 0 = always for batches of <= 262144 points.  "wgrad_tc",
 * "fwd_f16": DESIGN.md. */
int nsb_set_option(const char* key, int value);

/* Diagnostic: resident CTAs per SM of the tile-centric tensor-core kernels (2 = the design point: two tiles in flight per SM). */
int nsb_debug_occupancy(int* fwd_ctas_per_sm, int* bwd_ctas_per_sm);

/* Pack decoders' parameters into the kernels' shared-memory image (one launch for all four).
 * params[l] == NULL skips level l.  packed[l] must hold nsb_packed_decoder_floats(l) floats.
 * Must be re-run whenever the parameters changed (the mapper's Adam mutates them in place,
 * src/Mapper.py:339-341,504; the tracker deep-copies them, src/Tracker.py:138). */
int nsb_pack_decoders(const nsb_decoder_params* const params[4], float* const packed[4], void* stream);

/* Batch-global depth maxima used by the sampler: out[0] = max(gt_depth), out[1] = max(gt_depth*1.2f)
 * (src/utils/Renderer.py:109,144).  n may be 0 (out := 0). */
int nsb_batch_max_depth(const float* gt_depth, int n, float* out2, void* stream);

/* Ray pre-filter (src/Tracker.py:95-104, src/Mapper.py:471-481): keep[i] = (t_exit(ray i) >= gt_depth[i]). */
int nsb_bbox_prefilter(const float* rays_o, const float* rays_d, const float* gt_depth, int n,
                       const double bound[6], uint8_t* keep, void* stream);

typedef struct {
  int32_t stage;                 /* nsb_stage */
  int32_t n_rays;
  int32_t n_samples;             /* cfg rendering.N_samples (32) */
  int32_t n_surface;             /* cfg rendering.N_surface (16); forced 0 when gt_depth==NULL or stage coarse */
  double bound[6];               /* scene bound x_lo,x_hi,y_lo,y_hi,z_lo,z_hi as float64 (slam.bound) */
  double coarse_bound[6];        /* bound * coarse_bound_enlarge (src/NICE_SLAM.py:157) */
  const float* rays_o;           /* [N,3] */
  const float* rays_d;           /* [N,3] (not normalised) */
  const float* gt_depth;         /* [N] or NULL */
  const float* depth_max;        /* device float[2] from nsb_batch_max_depth; NULL if gt_depth is NULL, and optionally NULL for batches
                                    of <= NSB_INLINE_MAX_RAYS rays (then every CTA reduces gt_depth itself: one launch less) */
  const float* t_uniform;        /* device f32[n_samples]  = torch.linspace(0,1,n_samples) */
  const double* t_surface;       /* device f64[n_surface]  = torch.linspace(0,1,n_surface).double() */
  nsb_grid grid[4];              /* indexed by nsb_level; only the stage's grids are read */
  const float* packed[4];        /* packed decoders (nsb_pack_decoders) */
  const float* gt_depth_batch;   /* optional device f32[n_batch]: the sensor depths of the WHOLE batch this call renders a shard of (a ray-sharded
                                    tracker splits a pixel list every rank knows).  When given (depth_max NULL), the batch depth maxima
                                    (Renderer.py:109,144) are reduced over this list inside the kernel: no separate launch, no exchange. */
  int32_t n_batch;               /* 1 .. NSB_MAX_BATCH_DEPTHS */
} nsb_render_inputs;

typedef struct {
  double* depth;                 /* [N]   rendered depth      (float64 like the reference) */
  double* var;                   /* [N]   depth variance */
  float* rgb;                    /* [N,3] */
  double* z_vals;                /* [N,S] sorted sample depths; required if backward will run, else optional */
  float* raw;                    /* [N,S,4] (r,g,b,occ logit with the out-of-bound override); same rule */
  int32_t* corner_idx;           /* optional [N,S,3]: (ix0,iy0,iz0) of the stage's finest occupancy grid */
  uint32_t* masks;               /* optional [N,S,15]: ReLU sign bits of the 5 layers of up to 3 decoders (stage order); when the
                                    backward pass receives them it does not recompute the forward (tensor-core backend only) */
  void* split_workspace;         /* device scratch of nsb_split_workspace_bytes(N, S) bytes, ZEROED ONCE by the caller (the library
                                    leaves it clean): ray completion counters and per-item partial results of the tile kernels, which
                                    need it; the FP32-FMA kernels (S < 8, mlp_backend 1) do not read it */
  size_t split_workspace_bytes;
  float* acts;                   /* optional [N,S,5,32] float32: outputs of the five hidden layers of the decoder whose WEIGHT gradients the
                                    backward will be asked for (the colour decoder in stage color, src/Mapper.py:339-341).  When the forward
                                    keeps them, the backward computes those weight gradients on the tensor cores (dW = dU^T X contracted over
                                    the points of a tile) instead of the FP32-FMA pass that recomputes the forward.  NULL = not kept. */
} nsb_forward_outputs;

/* Bytes of split_workspace for n_rays rays of n_samples_total samples (NSB_MAX_SAMPLES: any S up to it); 0 for an empty batch. */
size_t nsb_split_workspace_bytes(int n_rays, int n_samples_total);

/* Forward: sample -> gather -> decode -> composite  (Renderer.render_batch_ray, src/utils/Renderer.py:63-198) */
int nsb_render_forward(const nsb_render_inputs* in, const nsb_forward_outputs* out, void* stream);

typedef struct {
  const double* z_vals;          /* [N,S] from forward */
  const float* raw;              /* [N,S,4] from forward */
  const double* g_depth;         /* [N]   dL/d depth */
  const double* g_var;           /* [N]   dL/d var   or NULL (0) */
  const float* g_rgb;            /* [N,3] dL/d rgb   or NULL (0) */
  float* d_rays_o;               /* [N,3] or NULL */
  float* d_rays_d;               /* [N,3] or NULL */
  float* d_grid[4];              /* dense gradient, same shape+strides as grid[l]; ACCUMULATED (caller zeroes); NULL = skip */
  float* d_flat[4];              /* decoder parameter gradients, canonical flat order; ACCUMULATED; NULL = skip */
  void* workspace;               /* device scratch of nsb_backward_workspace_bytes() bytes, 16-byte aligned;
                                    required iff any d_flat[l] != NULL (the library zeroes and consumes it) */
  const uint32_t* masks;         /* [N,S,15] from forward, or NULL (recompute) */
  const int32_t* slot_map[4];    /* masked (frustum-selected) voxel parameterisation, src/Mapper.py:317-333: when slot_map[l] != NULL
                                    it is the [D*H*W] voxel -> slot table of nsb_voxel_slots() and d_grid[l] is the COMPACT gradient
                                    [n_selected][32] (slot-major, 32 channels contiguous) of the selected voxels only; voxels with
                                    slot -1 are not parameters and receive nothing.  NULL = d_grid[l] is dense. */
  void* split_workspace;         /* as in nsb_forward_outputs (the same buffer may be passed to both) */
  size_t split_workspace_bytes;
  const float* pose_dirs;        /* optional [N,3] camera-frame ray directions: when given, d_c2w[12] (float64, row-major [3][4], as
                                    nsb_pose_grad) is produced by the backward itself -- by the last CTA to finish, through the
                                    zero-initialised, self-resetting device counter pose_counter -- instead of a separate launch */
  double* d_c2w;
  int* pose_counter;
  const float* acts;             /* nsb_forward_outputs.acts of the same forward, or NULL */
  void* result_dst;              /* optional (needs pose_dirs): once d_c2w is written, the same last CTA copies result_bytes bytes from result_src */
  const void* result_src;        /* to result_dst -- e.g. the block [d_rays_o | d_rays_d | loss | d c2w] to the device view of pinned host memory   */
  size_t result_bytes;           /* (nsb_host_device_pointer): the iteration's read-back without a copy node.  Both pointers 16-byte aligned.        */
} nsb_backward_args;

size_t nsb_backward_workspace_bytes(void);

/* Backward of the same path (what loss.backward() does at src/Tracker.py:125 / src/Mapper.py:503). */
int nsb_render_backward(const nsb_render_inputs* in, const nsb_backward_args* bw, void* stream);

/* Loss seeds.  Tracking (src/Tracker.py:108-123): residual r = |gt-depth|/sqrt(var+1e-10), mask =
 * (r < 10*median(r)) & (gt>0) when handle_dynamic else gt>0; loss = sum_mask r + w_color*sum_mask|gt_rgb-rgb|.
 * Mapping (src/Mapper.py:487-493): loss = sum_{gt>0}|gt-depth| (+ w_color*sum|gt_rgb-rgb| in stage color).
 * gt_rgb is float64 [N,3] for tracking (dataset colour is f64) and float32 for mapping (Mapper.py:462).
 * Writes g_depth[N] (f64), g_rgb[N,3] (f32) and loss[1] (f64). */
int nsb_tracking_seeds(const double* depth, const double* var, const float* rgb, const float* gt_depth,
                       const double* gt_rgb, int n, double w_color, int handle_dynamic, int use_color,
                       const double* median_pool, int n_pool,
                       double* g_depth, float* g_rgb, double* loss, void* workspace, size_t workspace_bytes,
                       void* stream);
/* r_i = |gt_i - depth_i| / sqrt(var_i + 1e-10) (src/Tracker.py:112).  When a tracking batch is sharded over several
 * GPUs the median of Tracker.py:113 must be taken over ALL shards: all-gather these residuals and pass them to
 * nsb_tracking_seeds as median_pool / n_pool (NULL / 0 = use this call's own rays). */
int nsb_tracking_residuals(const double* depth, const double* var, const float* gt_depth, int n, double* res, void* stream);
int nsb_mapping_seeds(const double* depth, const float* rgb, const float* gt_depth, const float* gt_rgb, int n,
                      double w_color, int use_color, double* g_depth, float* g_rgb, double* loss, void* stream);
size_t nsb_tracking_seeds_workspace(int n);

/* ---- masked voxel parameterisation (src/Mapper.py:317-333 val_grad = val[mask]; :393-401 / :511-519 val[mask] = val_grad) ----
 * voxel_mask: uint8 [D*H*W] (the reference's bool mask is the same for all 32 channels: Mapper.py:319-320 repeats it).
 * nsb_voxel_slots: slot_map[v] = rank of voxel v among the selected ones (d,h,w order), -1 if not selected; count[0] = n_selected.
 * The reference orders val[mask] channel-major ([32][n_selected]); the compact buffers here are slot-major ([n_selected][32],
 * one 128-byte line per voxel = what one red.global.add.v4 quad of the scatter touches): nsb_compact_transpose converts. */
size_t nsb_voxel_slots_workspace(long long n_voxels);
int nsb_voxel_slots(const uint8_t* voxel_mask, long long n_voxels, int32_t* slot_map, int32_t* count,
                    void* workspace, size_t workspace_bytes, void* stream);
int nsb_masked_gather(const nsb_grid* grid, const int32_t* slot_map, float* compact, void* stream);        /* compact = val[mask] */
int nsb_masked_scatter(const nsb_grid* grid, const int32_t* slot_map, const float* compact, void* stream); /* val[mask] = compact */
/* to_reference != 0: [n][32] -> [32][n] (the reference's val[mask] order); 0: the inverse. */
int nsb_compact_transpose(const float* src, float* dst, long long n_selected, int to_reference, void* stream);

/* Fused Adam steps (torch.optim.Adam with its defaults -- no weight decay, no amsgrad -- as the mapper uses it, src/Mapper.py:365-379,
 * per-group learning rates set per stage :412-419, step :504), float32 arithmetic in torch's operation order.  `step` = 1-based count of
 * updates of these parameters; exp_avg / exp_avg_sq: caller-owned state, zeroed at creation.
 * nsb_adam_masked_voxels: the parameters are the frustum-selected voxels of `grid`, updated IN PLACE on the shared grid storage from
 * the compact gradient [n_selected][32] -- replaces val_grad = val[mask] ... step ... val[mask] = val_grad (:324, :399, :517).
 * nsb_adam_decoder: the parameter tensors of one decoder, from its flat gradient (canonical order, nsb_flat_offset). */
int nsb_adam_masked_voxels(const nsb_grid* grid, const int32_t* slot_map, const float* grad, float* exp_avg, float* exp_avg_sq,
                           double lr, double beta1, double beta2, double eps, int step, void* stream);
/* The mapper's whole optimiser.step() (Mapper.py:504) in one launch: up to four voxel groups (as nsb_adam_masked_voxels, each with its own
 * learning rate and step count) and optionally one decoder (as nsb_adam_decoder; dec_level < 0: none). */
typedef struct nsb_adam_voxel_group {
  nsb_grid grid; const int32_t* slot_map; const float* grad; float* exp_avg; float* exp_avg_sq; double lr; int step;
} nsb_adam_voxel_group;
int nsb_adam_mapper_step(const nsb_adam_voxel_group* groups, int n_groups, int dec_level, const nsb_decoder_params* dec_params,
                         const float* dec_grad_flat, float* dec_exp_avg, float* dec_exp_avg_sq, double dec_lr, int dec_step,
                         double beta1, double beta2, double eps, void* stream);
int nsb_adam_decoder(int level, const nsb_decoder_params* params, const float* grad_flat, float* exp_avg, float* exp_avg_sq,
                     double lr, double beta1, double beta2, double eps, int step, void* stream);

/* Frustum feature selection (Mapper.get_mask_from_c2w, src/Mapper.py:93-164) of one grid, on the device: every voxel centre is
 * projected into the current frame (float32 camera transform, float64 intrinsics, like the reference's numpy code), the sensor
 * depth is looked up with OpenCV's INTER_LINEAR remap arithmetic (1/32-pixel fixed point, BORDER_CONSTANT 0), zero look-ups are
 * replaced by the maximum look-up, and the voxel is selected when it projects inside the image with 0 <= depth_cam <= sensor + 0.5,
 * or lies within 0.5 of the camera centre.  c2w: HOST float[16] row-major.  xs/ys/zs: DEVICE voxel-centre coordinates per axis
 * (W, H, D values: torch.linspace over the scene bound, Mapper.py:108-110).  depth: DEVICE float32 [img_h, img_w].
 * voxel_mask: DEVICE uint8 [D*H*W] (d,h,w order) -- the input of nsb_voxel_slots.  ('grid_coarse' is always fully selected, :114-116:
 * the caller fills ones.)  workspace: nsb_frustum_mask_workspace(D*H*W) bytes. */
size_t nsb_frustum_mask_workspace(long long n_voxels);
int nsb_frustum_mask(const float* c2w, const float* xs, const float* ys, const float* zs, int D, int H, int W,
                     const float* depth, int img_h, int img_w, double fx, double fy, double cx, double cy,
                     uint8_t* voxel_mask, void* workspace, size_t workspace_bytes, void* stream);

/* d c2w per keyframe of a bundle-adjustment window (src/Mapper.py:437-467 concatenates per-frame ray blocks):
 * frame f owns rays [frame_offsets[f], frame_offsets[f+1]); out[f][12] (float32, row-major [3][4]) as nsb_pose_grad. */
int nsb_pose_grad_frames(const float* dirs, const float* d_rays_o, const float* d_rays_d, const int32_t* frame_offsets,
                         int n_frames, float* out, void* stream);

/* ---- keyframe store (SURVEY.md 8f-4; src/Mapper.py:166-228 overlap selection, :437-462 per-frame samples) -----------------------------------
 * nsb_keyframe_overlap: for each of n_keyframes world-to-camera matrices w2c[k] (row-major [4][4] float32 = numpy.linalg.inv(est_c2w), as the
 * reference computes it on the host), counts[k] = number of the n_rays * n_samples points  o + d * (0.8 gt (1 - t) + (gt + 0.5) t)  that project
 * to  edge < u < W - edge, edge < v < H - edge  in front of the camera (Mapper.py:186-216; percent_inside = counts[k] / (n_rays * n_samples)).
 * t_vals = torch.linspace(0, 1, n_samples) (float32, device).
 * nsb_keyframe_gather: out_depth[f][k] = depth[slot[f]][pix_j[f][k]][pix_i[f][k]] (and the 3 colour channels) from keyframe images kept
 * resident on the device ([n_slots][H][W] float32, [n_slots][H][W][3] float32) instead of Mapper.py:439-440's per-iteration host->device copy. */
int nsb_keyframe_overlap(const float* rays_o, const float* rays_d, const float* gt_depth, int n_rays, const float* t_vals, int n_samples,
                         const float* w2c, int n_keyframes, int H, int W, double fx, double fy, double cx, double cy, int edge,
                         int32_t* counts, void* stream);
int nsb_keyframe_gather(const float* depth, const float* color, const int32_t* slot, const int32_t* pix_i, const int32_t* pix_j,
                        int n_frames, int n_pix, int H, int W, float* out_depth, float* out_color, void* stream);

/* ---- bundle-adjustment window (src/Mapper.py:346-363 camera tensors, :437-467 per-frame get_samples, :521-540 write-back) -----------------
 * A window has n_frames rows (the selected keyframes + the current frame).  Row f is either optimised -- its pose is camera tensor
 * cams[cam_row[f]] = [qw,qx,qy,qz,tx,ty,tz] (get_tensor_from_camera, src/common.py:179-200) -- or fixed (cam_row[f] = -1: the oldest frame,
 * Mapper.py:350; its pose is fixed_c2w[f], row-major [3][4]).
 * nsb_window_rays: c2w_out[f] = get_camera_from_tensor(cams[cam_row[f]]) (quad2rotation, src/common.py:137-176) or fixed_c2w[f]; then for
 * every ray r of frame frame_of_ray[r] at pixel (pix_i, pix_j): get_rays_from_uv (src/common.py:74-89) -> rays_o, rays_d and (optional)
 * the camera-frame direction `dirs` that nsb_pose_grad_frames needs.  All float32, the reference's operation order.
 * nsb_adam_poses: d_c2w[f] ([3][4] float32 per window row, from nsb_pose_grad_frames) is chained through quad2rotation to the gradient of
 * the camera tensors (written to d_cams [n_cams][7] if non-NULL) and torch.optim.Adam's update is applied to `cams` in place. */
int nsb_window_rays(const float* cams, const int32_t* cam_row, const float* fixed_c2w, int n_frames,
                    const float* pix_i, const float* pix_j, const int32_t* frame_of_ray, int n_rays,
                    double fx, double fy, double cx, double cy, float* c2w_out, float* rays_o, float* rays_d, float* dirs, void* stream);
int nsb_adam_poses(float* cams, const int32_t* cam_row, int n_frames, const float* d_c2w, float* exp_avg, float* exp_avg_sq, float* d_cams,
                   double lr, double beta1, double beta2, double eps, int step, void* stream);

/* ---- exchanges of a ray-sharded tracking iteration through NVLink peer memory (SURVEY.md 8e) ---------------------------------
 * A batch sharded over `world` GPUs (equal shards) needs three batch-global quantities: max(gt_depth) (Renderer.py:109,144), the
 * median of the residuals (Tracker.py:113) and the sums of loss and pose gradient.  The *_peers variants of the three single-CTA
 * kernels exchange them inside the kernel: every rank owns an exchange buffer of nsb_peer_buffer_bytes(max_rays) bytes, zeroed once,
 * mapped on all ranks (CUDA IPC / torch symmetric memory); buffer[r] is rank r's buffer as addressable from THIS device.
 * counters: device uint64[4] of this rank, zeroed once TOGETHER with the buffers (sequence numbers; advanced by the kernels -> CUDA-graph
 * replay safe; every 8-byte word of an exchange carries its sequence number next to 4 bytes of payload, so data and arrival flag are one
 * atomic word and no system-scope fence sits on the path).  Buffers: 16-byte aligned.
 * All ranks must enqueue the same sequence of *_peers calls; the kernels of one call spin until every rank has arrived. */
#define NSB_MAX_PEERS 8
typedef struct nsb_peers {
  int rank, world;
  void* buffer[NSB_MAX_PEERS];
  unsigned long long* counters;
  int max_rays;                  /* per-rank capacity of the residual pool the buffers were sized for */
} nsb_peers;
size_t nsb_peer_buffer_bytes(int max_rays);
int nsb_batch_max_depth_peers(const float* gt_depth, int n, float* out2, const nsb_peers* peers, void* stream);
/* as nsb_tracking_seeds with the median taken over ALL ranks' residuals (all-gathered through the exchange buffers); loss[0] = this
 * rank's partial loss. */
int nsb_tracking_seeds_peers(const double* depth, const double* var, const float* rgb, const float* gt_depth,
                             const double* gt_rgb, int n, double w_color, int handle_dynamic, int use_color,
                             const nsb_peers* peers, double* g_depth, float* g_rgb, double* loss,
                             void* workspace, size_t workspace_bytes, void* stream);
/* loss_and_d_c2w[13] = sum over ranks of [loss_local[0] | d c2w (12)], identical bits on every rank. */
int nsb_pose_grad_peers(const float* dirs, const float* d_rays_o, const float* d_rays_d, int n, const double* loss_local,
                        double* loss_and_d_c2w, const nsb_peers* peers, void* stream);

/* Points-only decode (Renderer.eval_points, src/utils/Renderer.py:23-61): p f64 [P,3] -> raw f32 [P,4]. */
int nsb_eval_points(const nsb_render_inputs* in, const double* points, int n_points, float* raw, void* stream);

/* Pose-gradient reduction: rays_d = sum_j dirs_j * R[:,j], rays_o = t (get_rays_from_uv, src/common.py:74-89) =>
 * d c2w[i][j] = sum_r d_rays_d[r][i] * dirs[r][j] (j<3), d c2w[i][3] = sum_r d_rays_o[r][i].  dirs: [N,3] camera-frame
 * directions.  d_c2w: float64 [3][4], OVERWRITTEN.  The quaternion chain (quad2rotation, src/common.py:137-160) stays in
 * PyTorch on these 12 numbers. */
int nsb_pose_grad(const float* dirs, const float* d_rays_o, const float* d_rays_d, int n, double* d_c2w, void* stream);

/* ---- per-iteration host blocks ----
 * The reference moves every batch tensor with its own `.to(device)` and reads the loss with `.item()` (src/Tracker.py:94-105,124-131,
 * src/Mapper.py:439-462,505-507).  Here the inputs of an iteration are ONE pinned host block and its results ONE block (see
 * nice_slam_b200/steps.py); nsb_copy_block moves such a block with the SMs (one 16-byte word per thread, all in flight: one PCIe round
 * trip) instead of a copy-engine transfer -- inside a CUDA graph that is a kernel node between kernel nodes.  Either pointer may be device
 * memory or the device view of page-locked host memory (nsb_host_device_pointer: NULL + nsb_last_error() if the block is not page-locked);
 * both must be 16-byte aligned.  Ordinary stream semantics: the copy is complete when the stream reaches the next operation. */
void* nsb_host_device_pointer(void* pinned_host);
int nsb_copy_block(void* dst, const void* src, size_t bytes, void* stream);

/* ---- one optimisation iteration = batch max -> forward -> loss seeds -> backward, enqueued by ONE call ----
 * (what Tracker.optimize_cam_in_batch, src/Tracker.py:106-125, and one joint_iter of Mapper.optimize_map,
 * src/Mapper.py:482-503, do around the optimiser step).  All buffers are caller-owned device memory. */
typedef struct {
  double* depth;  double* var;  float* rgb;      /* [N], [N], [N,3]   rendered outputs            */
  double* z_vals; float* raw;                    /* [N,S], [N,S,4]    forward state kept for backward */
  uint32_t* masks;                               /* [N,S,15] or NULL  ReLU sign bits (see nsb_forward_outputs) */
  double* g_depth; float* g_rgb;                 /* [N], [N,3]        loss seeds                  */
  double* loss;                                  /* [1]               scalar loss (float64)       */
  float* depth_max;                              /* [2]               batch depth maxima          */
  void* workspace; size_t workspace_bytes;       /* >= nsb_iteration_workspace_bytes(N)           */
  void* event_bwd_begin; void* event_bwd_end;    /* optional cudaEvent_t recorded around the backward launch (profiling hook) */
  float* acts;                                   /* [N,S,5,32] or NULL (see nsb_forward_outputs.acts): needed for tensor-core weight gradients */
} nsb_iteration_buffers;

/* The workspace must be ZEROED ONCE after allocation (it contains the split_workspace counters, see nsb_forward_outputs). */
size_t nsb_iteration_workspace_bytes(int n_rays);

/* `in->depth_max` is ignored (batches of more than NSB_INLINE_MAX_RAYS rays: computed into buf->depth_max; smaller ones: reduced
 * inside the render kernel).  `grads` supplies only the OUTPUT pointers of
 * nsb_backward_args (d_rays_o, d_rays_d, d_grid, d_flat); its z_vals, raw, seed and workspace fields are ignored. */
int nsb_tracking_iteration(const nsb_render_inputs* in, const nsb_iteration_buffers* buf, const double* gt_rgb,
                           double w_color, int handle_dynamic, int use_color, const nsb_backward_args* grads, void* stream);
/* gt_depth_loss: the depth the loss compares against (the coarse mapper renders with in->gt_depth == NULL but still
 * supervises with the sensor depth, src/Mapper.py:484-489); NULL = in->gt_depth. */
int nsb_mapping_iteration(const nsb_render_inputs* in, const nsb_iteration_buffers* buf, const float* gt_depth_loss,
                          const float* gt_rgb, double w_color, const nsb_backward_args* grads, void* stream);

/* The whole ray-sharded tracking iteration of one rank in TWO kernel launches (<= 512 rays per rank, equal shard sizes): the forward launch
 * exchanges the depth maxima (every CTA waits for all ranks' values before it samples) and, in its last CTA, the residual pool of the
 * median, then computes this shard's loss seeds; the last CTA of the backward launch sums [loss | d c2w] over the ranks in rank order
 * (loss_and_d_c2w[13], identical bits on every rank).  Arguments as nsb_tracking_iteration; grads->pose_dirs / d_c2w / pose_counter are
 * required.  Waits on a missing rank are bounded (the launch fails instead of hanging).  If in->depth_max is given (the maxima of the FULL batch,
 * nsb_batch_max_depth over all ranks' sensor depths, which every rank of a sharded tracker knows) the depth-max exchange is skipped. */
int nsb_tracking_iteration_peers(const nsb_render_inputs* in, const nsb_iteration_buffers* buf, const double* gt_rgb,
                                 double w_color, int handle_dynamic, int use_color, const nsb_backward_args* grads,
                                 const nsb_peers* peers, double* loss_and_d_c2w, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NICE_SLAM_B200_H_ */
