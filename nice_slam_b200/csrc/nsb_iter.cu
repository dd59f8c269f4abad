// nsb_iter.cu -- one optimisation iteration enqueued by a single C call:
//   batch depth maxima -> render forward -> loss seeds -> render backward
// (Tracker.optimize_cam_in_batch, src/Tracker.py:106-125; one joint_iter of Mapper.optimize_map, src/Mapper.py:482-503).
#include <cstring>
#include "nsb_common.cuh"

using namespace nsb;

static size_t a16(size_t x) { return (x + 15) & ~size_t(15); }

// workspace = [fused-seeds counter (16 B) | tracking-seeds scratch | packed weight-gradient images | tile-kernel workspace = the rest].
// Only the first 16 bytes and the END of the buffer (ray completion counters, nsb_render.cu) hold state that must stay zero between calls,
// so one buffer sized for a capacity serves batches of varying size.
static size_t split_bytes(int n_rays) { return nsb_split_workspace_bytes(n_rays, NSB_MAX_SAMPLES); }
extern "C" size_t nsb_iteration_workspace_bytes(int n_rays) {
  return 16 + a16(nsb_tracking_seeds_workspace(n_rays)) + a16(nsb_backward_workspace_bytes()) + a16(split_bytes(n_rays));
}
static int* seeds_counter(const nsb_iteration_buffers* b, int) { return reinterpret_cast<int*>(b->workspace); }
static void* seeds_scratch(const nsb_iteration_buffers* b) { return reinterpret_cast<char*>(b->workspace) + 16; }
static size_t split_offset(int n_rays) { return 16 + a16(nsb_tracking_seeds_workspace(n_rays)) + a16(nsb_backward_workspace_bytes()); }
static void* split_ptr(const nsb_iteration_buffers* b, int n_rays) { return reinterpret_cast<char*>(b->workspace) + split_offset(n_rays); }
static size_t split_room(const nsb_iteration_buffers* b, int n_rays) { return b->workspace_bytes - split_offset(n_rays); }

static int check_buffers(const nsb_render_inputs* in, const nsb_iteration_buffers* b, const nsb_backward_args* g) {
  if (!in || !b || !g) { set_error("iteration: NULL argument"); return NSB_ERR_ARG; }
  if (!b->depth || !b->var || !b->rgb || !b->z_vals || !b->raw || !b->g_depth || !b->g_rgb || !b->loss || !b->depth_max || !b->workspace) {
    set_error("iteration: incomplete nsb_iteration_buffers"); return NSB_ERR_ARG; }
  if (b->workspace_bytes < nsb_iteration_workspace_bytes(in->n_rays)) { set_error("iteration: workspace too small"); return NSB_ERR_ARG; }
  return NSB_OK;
}

static int forward_part(const nsb_render_inputs* in, const nsb_iteration_buffers* b, nsb_render_inputs* in2, const FusedSeeds* fs, void* stream,
                        bool keep_depth_max = false) {
  *in2 = *in;
  int rc;
  if (keep_depth_max && in->depth_max != nullptr) {                // the caller supplies the batch depth maxima (sharded batch: maxima of the FULL batch)
    nsb_forward_outputs fo = {b->depth, b->var, b->rgb, b->z_vals, b->raw, nullptr, b->masks, split_ptr(b, in->n_rays), split_room(b, in->n_rays), b->acts};
    return render_forward_fused(in2, &fo, fs, stream);
  }
  in2->depth_max = nullptr;
  if (in->gt_depth && in->gt_depth_batch == nullptr && in->n_rays > NSB_INLINE_MAX_RAYS) {          // small batches: the render kernel reduces gt_depth itself
    if ((rc = nsb_batch_max_depth(in->gt_depth, in->n_rays, b->depth_max, stream))) return rc;
    in2->depth_max = b->depth_max;
  }
  nsb_forward_outputs fo = {b->depth, b->var, b->rgb, b->z_vals, b->raw, nullptr, b->masks, split_ptr(b, in->n_rays), split_room(b, in->n_rays), b->acts};
  return render_forward_fused(in2, &fo, fs, stream);
}

static int backward_part(const nsb_render_inputs* in2, const nsb_iteration_buffers* b, const nsb_backward_args* g, void* stream, const PeerTail* tail = nullptr) {
  nsb_backward_args bw = *g;
  bw.z_vals = b->z_vals; bw.raw = b->raw; bw.g_depth = b->g_depth; bw.g_var = nullptr; bw.g_rgb = b->g_rgb; bw.masks = b->masks; bw.acts = b->acts;
  bw.workspace = reinterpret_cast<char*>(b->workspace) + 16 + a16(nsb_tracking_seeds_workspace(in2->n_rays));
  bw.split_workspace = split_ptr(b, in2->n_rays); bw.split_workspace_bytes = split_room(b, in2->n_rays);
  if (b->event_bwd_begin) cudaEventRecord((cudaEvent_t)b->event_bwd_begin, (cudaStream_t)stream);
  const int rc = render_backward_tail(in2, &bw, tail, stream);
  if (b->event_bwd_end) cudaEventRecord((cudaEvent_t)b->event_bwd_end, (cudaStream_t)stream);
  return rc;
}

extern "C" int nsb_tracking_iteration(const nsb_render_inputs* in, const nsb_iteration_buffers* buf, const double* gt_rgb,
                                      double w_color, int handle_dynamic, int use_color, const nsb_backward_args* grads, void* stream) {
  int rc = check_buffers(in, buf, grads); if (rc) return rc;
  if (!in->gt_depth) { set_error("tracking iteration needs gt_depth"); return NSB_ERR_ARG; }
  nsb_render_inputs in2;
  // small batches: the last CTA of the forward launch computes the loss seeds itself (no separate single-CTA launch)
  const bool fuse = in->n_rays > 0 && in->n_rays <= 512;          // (the median by direct rank counting, nsb_seeds.cuh)
  FusedSeeds fs; memset(&fs, 0, sizeof(fs));
  if (fuse) {
    fs.kind = 1; fs.gt_rgb = gt_rgb; fs.w_color = w_color; fs.handle_dynamic = handle_dynamic; fs.use_color = use_color;
    fs.g_depth = buf->g_depth; fs.g_rgb = buf->g_rgb; fs.loss = buf->loss; fs.res = static_cast<double*>(seeds_scratch(buf));
    fs.counter = seeds_counter(buf, in->n_rays);
    if (use_color && !gt_rgb) { set_error("tracking iteration: use_color without gt_rgb"); return NSB_ERR_ARG; }
  }
  if ((rc = forward_part(in, buf, &in2, fuse ? &fs : nullptr, stream))) return rc;
  if (!fuse && (rc = nsb_tracking_seeds(buf->depth, buf->var, buf->rgb, in->gt_depth, gt_rgb, in->n_rays, w_color, handle_dynamic, use_color,
                                        nullptr, 0, buf->g_depth, buf->g_rgb, buf->loss, seeds_scratch(buf), nsb_tracking_seeds_workspace(in->n_rays), stream))) return rc;
  return backward_part(&in2, buf, grads, stream);
}

// Ray-sharded tracking iteration in TWO launches per rank: the forward exchanges the depth maxima (every CTA) and the residual pool of the
// median (last CTA, which then computes the loss seeds); the backward's last CTA sums [loss | d c2w] over the ranks.
extern "C" int nsb_tracking_iteration_peers(const nsb_render_inputs* in, const nsb_iteration_buffers* buf, const double* gt_rgb,
                                            double w_color, int handle_dynamic, int use_color, const nsb_backward_args* grads,
                                            const nsb_peers* peers, double* loss_and_d_c2w, void* stream) {
  int rc = check_buffers(in, buf, grads); if (rc) return rc;
  if (!in->gt_depth || !loss_and_d_c2w) { set_error("sharded tracking iteration needs gt_depth and an output for [loss | d c2w]"); return NSB_ERR_ARG; }
  if (in->n_rays < 1 || in->n_rays > 512) { set_error("sharded tracking iteration: 1..512 rays per rank (got %d)", in->n_rays); return NSB_ERR_UNSUPPORTED; }
  if (!grads->pose_dirs || !grads->d_c2w || !grads->pose_counter) { set_error("sharded tracking iteration needs pose_dirs / d_c2w / pose_counter"); return NSB_ERR_ARG; }
  if (use_color && !gt_rgb) { set_error("tracking iteration: use_color without gt_rgb"); return NSB_ERR_ARG; }
  PeerX px;
  if ((rc = make_peerx(peers, &px))) return rc;
  if (in->n_rays > px.max_n) { set_error("sharded tracking iteration: %d rays exceed the exchange buffers' capacity %d", in->n_rays, px.max_n); return NSB_ERR_ARG; }
  FusedSeeds fs; memset(&fs, 0, sizeof(fs));
  fs.kind = 1; fs.gt_rgb = gt_rgb; fs.w_color = w_color; fs.handle_dynamic = handle_dynamic; fs.use_color = use_color;
  fs.g_depth = buf->g_depth; fs.g_rgb = buf->g_rgb; fs.loss = buf->loss; fs.res = static_cast<double*>(seeds_scratch(buf));
  fs.counter = seeds_counter(buf, in->n_rays);
  fs.px = px;
  nsb_render_inputs in2;
  if ((rc = forward_part(in, buf, &in2, &fs, stream, true))) return rc;      // in->depth_max given: no depth-max exchange inside the forward
  PeerTail tail; tail.px = px; tail.loss = buf->loss; tail.out13 = loss_and_d_c2w;
  return backward_part(&in2, buf, grads, stream, &tail);
}

extern "C" int nsb_mapping_iteration(const nsb_render_inputs* in, const nsb_iteration_buffers* buf, const float* gt_depth_loss,
                                     const float* gt_rgb, double w_color, const nsb_backward_args* grads, void* stream) {
  int rc = check_buffers(in, buf, grads); if (rc) return rc;
  const float* gtl = gt_depth_loss ? gt_depth_loss : in->gt_depth;
  if (!gtl) { set_error("mapping iteration needs a depth to supervise with"); return NSB_ERR_ARG; }
  nsb_render_inputs in2;
  const int use_color = in->stage == NSB_STAGE_COLOR;                      // Mapper.py:490
  const bool fuse = in->n_rays > 0 && in->n_rays <= NSB_INLINE_MAX_RAYS;
  FusedSeeds fs; memset(&fs, 0, sizeof(fs));
  if (fuse) {
    if (use_color && !gt_rgb) { set_error("mapping iteration: colour stage without gt_rgb"); return NSB_ERR_ARG; }
    fs.kind = 2; fs.gt_rgb = gt_rgb; fs.gt_depth_loss = gtl; fs.w_color = w_color; fs.use_color = use_color;
    fs.g_depth = buf->g_depth; fs.g_rgb = buf->g_rgb; fs.loss = buf->loss; fs.counter = seeds_counter(buf, in->n_rays);
  }
  if ((rc = forward_part(in, buf, &in2, fuse ? &fs : nullptr, stream))) return rc;
  if (!fuse && (rc = nsb_mapping_seeds(buf->depth, buf->rgb, gtl, gt_rgb, in->n_rays, w_color, use_color, buf->g_depth, buf->g_rgb, buf->loss, stream))) return rc;
  return backward_part(&in2, buf, grads, stream);
}
