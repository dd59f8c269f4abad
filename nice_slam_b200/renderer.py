"""FusedRenderer -- drop-in for the reference's `Renderer` (src/utils/Renderer.py) on the B200 path.

Same constructor and method set (SURVEY.md section 8b):
    FusedRenderer(cfg, args, slam, points_batch_size=500000, ray_batch_size=100000)
    .render_batch_ray(c, decoders, rays_d, rays_o, device, stage, gt_depth=None) -> (depth f64, uncertainty f64, color f32)
    .eval_points(p, decoders, c=None, stage='color', device='cuda:0') -> raw [N,4]
    .render_img(c, decoders, c2w, device, stage, gt_depth=None)
    .regulation(...)   # iMAP-only in the reference; raises here
Swap point: `self.renderer = Renderer(cfg, args, self)` at src/NICE_SLAM.py:91.

render_batch_ray is differentiable w.r.t. rays_o, rays_d, the grids in `c` and the decoders' parameters
(Tracker.optimize_cam_in_batch, src/Tracker.py:106-125; Mapper.optimize_map, src/Mapper.py:482-503): the
forward and the hand-written backward are the CUDA kernels behind include/nice_slam_b200.h.  There is no
PyTorch / CPU fallback: tensors that are not on a CUDA device raise.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import LEVELS, STAGES, STAGE_DECODERS
from .decoders import named_params

_VP = C.c_void_p


def _ptr(t):
    return _VP(t.data_ptr()) if t is not None else _VP(None)


def _stream():
    return _VP(torch.cuda.current_stream().cuda_stream)


def _require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError("nice_slam_b200: %s is on %s; the fused path runs on CUDA only (no CPU fallback)" % (what, t.device))


def grid_struct(t):
    """nsb_grid view of a [1,32,D,H,W] fp32 CUDA tensor (any strides; channels_last_3d is the fast path)."""
    if t.dim() != 5 or t.shape[0] != 1 or t.shape[1] != 32 or t.dtype != torch.float32:
        raise RuntimeError("feature grid must be float32 [1,32,D,H,W], got %s %s" % (tuple(t.shape), t.dtype))
    _require_cuda(t, "feature grid")
    s = t.stride()
    return _lib.Grid(t.data_ptr(), t.shape[2], t.shape[3], t.shape[4], s[1], s[2], s[3], s[4])


def to_channels_last(grids):
    """In-place (dict) conversion of the shared grids to channels_last_3d: logical shape, values, val[mask],
    torch.save and F.grid_sample behaviour are unchanged; physical layout becomes 128 B per voxel."""
    for k, v in list(grids.items()):
        if v.is_cuda and v.dim() == 5 and v.stride(1) != 1:
            grids[k] = v.contiguous(memory_format=torch.channels_last_3d)
    return grids


class _PackCache:
    """Packed (shared-memory image) copies of the decoders, rebuilt when a parameter's storage or version
    changes (the mapper's Adam mutates them in place; the tracker deep-copies them: SURVEY 8b traps)."""

    def __init__(self):
        self.key = {}
        self.buf = {}

    def get(self, decoders, levels, device):
        L = _lib.lib()
        need = []
        params = {}
        for lvl in levels:
            p = named_params(decoders, lvl)
            params[lvl] = p
            key = tuple((k, v.data_ptr(), v._version) for k, v in sorted(p.items()))
            if self.key.get(lvl) != key or lvl not in self.buf or self.buf[lvl].device != device:
                need.append((lvl, key))
        if need:
            arr_p = (C.POINTER(_lib.DecoderParams) * 4)()
            arr_o = (_VP * 4)()
            keep = []
            for lvl, key in need:
                li = LEVELS.index(lvl)
                p = params[lvl]
                dp = _lib.DecoderParams()
                for t in p.values():
                    _require_cuda(t, "decoder parameter")
                    if t.dtype != torch.float32 or not t.is_contiguous():
                        raise RuntimeError("decoder parameters must be contiguous float32")
                if li != 0:
                    dp.B = p["embedder._B"].data_ptr()
                for i in range(5):
                    dp.W[i] = p["pts_linears.%d.weight" % i].data_ptr()
                    dp.b[i] = p["pts_linears.%d.bias" % i].data_ptr()
                    if li != 0:
                        dp.Wc[i] = p["fc_c.%d.weight" % i].data_ptr()
                        dp.bc[i] = p["fc_c.%d.bias" % i].data_ptr()
                dp.Wo = p["output_linear.weight"].data_ptr()
                dp.bo = p["output_linear.bias"].data_ptr()
                buf = torch.empty(L.nsb_packed_decoder_floats(li), dtype=torch.float32, device=device)
                keep.append(dp)
                arr_p[li] = C.pointer(dp)
                arr_o[li] = buf.data_ptr()
                self.buf[lvl] = buf
                self.key[lvl] = key
            _lib.check(L.nsb_pack_decoders(arr_p, arr_o, _stream()), "nsb_pack_decoders")
        return {lvl: self.buf[lvl] for lvl in levels}, params


class _Call:
    """Non-tensor arguments of one render call."""
    __slots__ = ("stage", "levels", "bound", "cbound", "n_samples", "n_surface", "gt_depth", "packed", "param_names",
                 "aux", "masked", "grid_data")


INLINE_MAX_RAYS = 1024          # NSB_INLINE_MAX_RAYS of include/nice_slam_b200.h


def _inputs(call, rays_o, rays_d, depth_max, t_u, t_s, grids):
    inp = _lib.RenderInputs()
    inp.stage = STAGES[call.stage]
    inp.n_rays = rays_o.shape[0]
    inp.n_samples, inp.n_surface = call.n_samples, call.n_surface
    for i in range(6):
        inp.bound[i] = call.bound[i]
        inp.coarse_bound[i] = call.cbound[i]
    inp.rays_o, inp.rays_d = rays_o.data_ptr(), rays_d.data_ptr()
    if call.gt_depth is not None:
        inp.gt_depth = call.gt_depth.data_ptr()
        inp.depth_max = depth_max.data_ptr() if depth_max is not None else None      # None: reduced inside the kernel (small batches)
    inp.t_uniform = t_u.data_ptr()
    inp.t_surface = t_s.data_ptr() if t_s is not None else None
    for lvl, g in zip(call.levels, grids):
        li = LEVELS.index(lvl)
        inp.grid[li] = grid_struct(g)
        inp.packed[li] = call.packed[lvl].data_ptr()
    return inp


_LINSPACE = {}


def _linspaces(n_samples, n_surface, device):
    key = (n_samples, n_surface, str(device))
    if key not in _LINSPACE:
        t_u = torch.linspace(0., 1., steps=n_samples, device=device)                       # Renderer.py:152
        t_s = torch.linspace(0., 1., steps=n_surface).double().to(device) if n_surface > 0 else None   # Renderer.py:131-132
        _LINSPACE[key] = (t_u, t_s)
    return _LINSPACE[key]


class _RenderFn(torch.autograd.Function):
    """forward/backward = nsb_render_forward / nsb_render_backward."""

    @staticmethod
    def forward(ctx, call, rays_o, rays_d, *tensors):
        L = _lib.lib()
        n_lvl = len(call.levels)
        grids, params = tensors[:n_lvl], tensors[n_lvl:]
        dev = rays_o.device
        ro = rays_o.detach().contiguous().float()
        rd = rays_d.detach().contiguous().float()
        n = ro.shape[0]
        has_gt = call.gt_depth is not None and call.stage != "coarse"
        S = call.n_samples + (call.n_surface if has_gt else 0)
        depth_max = None
        if call.gt_depth is not None and n > INLINE_MAX_RAYS:             # smaller batches: the render kernel reduces gt_depth itself
            depth_max = torch.empty(2, dtype=torch.float32, device=dev)
            _lib.check(L.nsb_batch_max_depth(_ptr(call.gt_depth), n, _ptr(depth_max), _stream()), "nsb_batch_max_depth")
        t_u, t_s = _linspaces(call.n_samples, call.n_surface, dev)
        # a grid argument is either the grid itself or, for a frustum-masked grid (see FusedRenderer._masked_leaf), the mapper's 1-D leaf
        # `val_grad`; the data the kernels read is always the full grid
        data = [call.grid_data[j] if call.masked[j] is not None else grids[j].detach() for j in range(n_lvl)]
        inp = _inputs(call, ro, rd, depth_max, t_u, t_s, data)
        depth = torch.empty(n, dtype=torch.float64, device=dev)
        var = torch.empty(n, dtype=torch.float64, device=dev)
        rgb = torch.empty(n, 3, dtype=torch.float32, device=dev)
        z_vals = torch.empty(n, S, dtype=torch.float64, device=dev)
        raw = torch.empty(n, S, 4, dtype=torch.float32, device=dev)
        masks = torch.empty(n, S, 15, dtype=torch.int32, device=dev)      # ReLU sign bits: lets backward skip the forward recompute
        nsplit = L.nsb_split_workspace_bytes(n, S)                        # tile kernels: ray completion counters + per-item scratch
        split = torch.zeros(nsplit, dtype=torch.uint8, device=dev) if nsplit else None
        # colour-decoder parameters that need a gradient (the mapper's colour stage, Mapper.py:339-341): keep the decoder's layer outputs so that
        # the backward computes the weight gradients on the tensor cores
        acts = None
        if call.stage == "color":
            k0 = 3 + n_lvl + sum(len(call.param_names[l]) for l in call.levels[: call.levels.index("color")])
            if any(ctx.needs_input_grad[k0 + i] for i in range(len(call.param_names["color"]))):
                acts = torch.empty(n, S, 5, 32, dtype=torch.float32, device=dev)
        out = _lib.ForwardOutputs(depth.data_ptr(), var.data_ptr(), rgb.data_ptr(), z_vals.data_ptr(), raw.data_ptr(), None, masks.data_ptr(),
                                  split.data_ptr() if nsplit else None, nsplit, acts.data_ptr() if acts is not None else None)
        corner = None
        if call.aux is not None:
            corner = torch.empty(n, S, 3, dtype=torch.int32, device=dev)
            out.corner_idx = corner.data_ptr()
        if n > 0:                                                         # (an empty batch has no storage to point at)
            _lib.check(L.nsb_render_forward(C.byref(inp), C.byref(out), _stream()), "nsb_render_forward")
        if call.aux is not None:
            call.aux.update(z_vals=z_vals, raw=raw, corner_idx=corner)
        ctx.call = call
        ctx.n_lvl = n_lvl
        ctx.keep = (ro, rd, depth_max, t_u, t_s, z_vals, raw, masks, split)
        ctx.acts = acts
        ctx.grids = data
        ctx.param_shapes = [tuple(p.shape) for p in params]
        return depth, var, rgb

    @staticmethod
    def backward(ctx, g_depth, g_var, g_rgb):
        L = _lib.lib()
        call = ctx.call
        ro, rd, depth_max, t_u, t_s, z_vals, raw, masks, split = ctx.keep
        dev = ro.device
        n = ro.shape[0]
        n_lvl = ctx.n_lvl
        needs = ctx.needs_input_grad          # (call, rays_o, rays_d, *grids, *params)
        inp = _inputs(call, ro, rd, depth_max, t_u, t_s, ctx.grids)
        bw = _lib.BackwardArgs()
        bw.z_vals, bw.raw, bw.masks = z_vals.data_ptr(), raw.data_ptr(), masks.data_ptr()
        if split is not None:
            bw.split_workspace, bw.split_workspace_bytes = split.data_ptr(), split.numel()
        if ctx.acts is not None:
            bw.acts = ctx.acts.data_ptr()
        gd = g_depth.detach().contiguous().double() if g_depth is not None else torch.zeros(n, dtype=torch.float64, device=dev)
        gv = g_var.detach().contiguous().double() if g_var is not None else None
        gc = g_rgb.detach().contiguous().float() if g_rgb is not None else None
        bw.g_depth, bw.g_var, bw.g_rgb = gd.data_ptr(), (gv.data_ptr() if gv is not None else None), (gc.data_ptr() if gc is not None else None)
        d_o = d_d = None
        if needs[1] or needs[2]:
            d_o = torch.empty(n, 3, dtype=torch.float32, device=dev)
            d_d = torch.empty(n, 3, dtype=torch.float32, device=dev)
            bw.d_rays_o, bw.d_rays_d = d_o.data_ptr(), d_d.data_ptr()
        d_grids = [None] * n_lvl
        compact = {}
        for j, lvl in enumerate(call.levels):
            if needs[3 + j] and call.masked[j] is not None:
                # frustum-masked parameterisation (Mapper.py:321-333): COMPACT gradient of the selected voxels only -- no dense zero-fill, no
                # index_put backward; converted to the reference's `val[mask]` order below
                mv = call.masked[j]
                dg = torch.zeros(max(mv.count, 1), 32, dtype=torch.float32, device=dev)
                compact[j] = dg
                li = LEVELS.index(lvl)
                bw.d_grid[li], bw.slot_map[li] = dg.data_ptr(), mv.slot_map.data_ptr()
            elif needs[3 + j]:
                g = ctx.grids[j]
                dg = torch.zeros_like(g)
                if dg.stride() != g.stride():
                    dg = torch.empty_strided(g.size(), g.stride(), dtype=g.dtype, device=dev).zero_()
                d_grids[j] = dg
                bw.d_grid[LEVELS.index(lvl)] = dg.data_ptr()
        # decoder parameter gradients: one flat buffer per decoder, returned as views in the reference's names
        d_params = [None] * (len(needs) - 3 - n_lvl)
        flats = {}
        k = 0
        for lvl in call.levels:
            names = call.param_names[lvl]
            if any(needs[3 + n_lvl + k + i] for i in range(len(names))):
                li = LEVELS.index(lvl)
                flat = torch.zeros(L.nsb_flat_decoder_floats(li), dtype=torch.float32, device=dev)
                flats[lvl] = flat
                bw.d_flat[li] = flat.data_ptr()
                lay = {nm: (off, cnt) for nm, off, cnt in _lib.flat_layout(li)}
                for i, nm in enumerate(names):
                    if needs[3 + n_lvl + k + i]:
                        off, cnt = lay[nm]
                        d_params[k + i] = flat[off:off + cnt].view(ctx.param_shapes[k + i])
            k += len(names)
        ws = None
        if flats:
            ws = torch.empty(L.nsb_backward_workspace_bytes(), dtype=torch.uint8, device=dev)
            bw.workspace = ws.data_ptr()
        if n > 0:
            _lib.check(L.nsb_render_backward(C.byref(inp), C.byref(bw), _stream()), "nsb_render_backward")
        elif d_o is not None:
            d_o.zero_(); d_d.zero_()
        for j, dg in compact.items():
            mv = call.masked[j]
            d_grids[j] = mv.to_reference(dg[: mv.count]) if mv.count > 0 else torch.zeros(0, dtype=torch.float32, device=dev)
        return (None, d_o if needs[1] else None, d_d if needs[2] else None, *d_grids, *d_params)


class FusedRenderer(object):
    def __init__(self, cfg, args, slam, points_batch_size=500000, ray_batch_size=100000, convert_grids=True):
        self.ray_batch_size = ray_batch_size
        self.points_batch_size = points_batch_size
        r = cfg["rendering"]
        self.lindisp, self.perturb = r["lindisp"], r["perturb"]
        self.N_samples, self.N_surface, self.N_importance = r["N_samples"], r["N_surface"], r["N_importance"]
        self.scale = cfg["scale"]
        self.occupancy = cfg["occupancy"]
        self.nice = slam.nice
        self.bound = slam.bound
        self.H, self.W, self.fx, self.fy, self.cx, self.cy = slam.H, slam.W, slam.fx, slam.fy, slam.cx, slam.cy
        self.coarse_bound_enlarge = cfg["model"]["coarse_bound_enlarge"]
        if not self.nice or not self.occupancy:
            raise RuntimeError("FusedRenderer implements the NICE (occupancy) path only; iMAP* stays on the reference Renderer")
        if self.lindisp or self.perturb > 0 or self.N_importance > 0:
            raise RuntimeError("FusedRenderer supports lindisp=False, perturb=0, N_importance=0 (configs/nice_slam.yaml:105-110)")
        if convert_grids and getattr(slam, "shared_c", None) is not None:
            to_channels_last(slam.shared_c)        # layout conversion point, before Mapper/Tracker capture the dict
        self._cache = _PackCache()
        self._mask_cache = {}
        self.detect_masked_grids = True

    def __getstate__(self):                        # pickled into spawned processes: no device state travels
        d = dict(self.__dict__)
        d["_cache"] = None
        d["_mask_cache"] = {}
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        self._cache = _PackCache()

    # ------------------------------------------------------------------ helpers
    def invalidate_decoders(self, levels=None):
        """Force a re-pack of the decoders' packed / operand images on the next call (needed only after parameter updates that bypass
        torch's version counters, e.g. optim.FusedMapperAdam.step_decoder)."""
        for lvl in (levels or list(self._cache.key.keys())):
            self._cache.key.pop(lvl, None)

    def _bounds(self):
        b = self.bound.detach().cpu().double().reshape(6)
        return b.tolist(), (b * self.coarse_bound_enlarge).tolist()

    def _call(self, c, decoders, stage, gt_depth, device, aux=None):
        if stage not in STAGES:
            raise RuntimeError("unknown stage %r" % (stage,))
        call = _Call()
        call.stage = stage
        call.levels = STAGE_DECODERS[stage]
        call.bound, call.cbound = self._bounds()
        call.n_samples, call.n_surface = self.N_samples, self.N_surface
        call.gt_depth = None
        if gt_depth is not None and stage != "coarse":
            _require_cuda(gt_depth, "gt_depth")
            call.gt_depth = gt_depth.detach().reshape(-1).contiguous().float()
        call.packed, params = self._cache.get(decoders, call.levels, torch.device(device) if not isinstance(device, torch.device) else device)
        call.param_names = {lvl: [nm for nm, _, _ in _lib.flat_layout(LEVELS.index(lvl))] for lvl in call.levels}
        call.aux = aux
        call.masked, call.grid_data = [None] * len(call.levels), [None] * len(call.levels)
        grids = [c["grid_" + lvl] for lvl in call.levels]
        plist = [params[lvl][nm] for lvl in call.levels for nm in call.param_names[lvl]]
        return call, grids, plist

    # ------------------------------------------------------------------ reference API
    def render_batch_ray(self, c, decoders, rays_d, rays_o, device, stage, gt_depth=None, aux=None):
        """Render depth, uncertainty and colour of a batch of rays (Renderer.render_batch_ray, Renderer.py:63-198).
        `aux` (optional dict) receives z_vals / raw / corner_idx for the parity tests."""
        _require_cuda(rays_o, "rays_o")
        _require_cuda(rays_d, "rays_d")
        call, grids, plist = self._call(c, decoders, stage, gt_depth, rays_o.device, aux)
        if self.detect_masked_grids and torch.is_grad_enabled():
            for j, g in enumerate(grids):
                sel = self._masked_leaf(g)
                if sel is not None:                        # the mapper's `val[mask] = val_grad`: route the gradient to val_grad directly
                    grids[j], call.masked[j], call.grid_data[j] = sel[0], sel[1], g.detach()
        return _RenderFn.apply(call, rays_o, rays_d, *grids, *plist)

    def _masked_leaf(self, g):
        """Detects the reference mapper's frustum-masked parameterisation at the boundary (src/Mapper.py:393-401): `val[mask] = val_grad; c[key] = val`
        makes c[key] the output of an in-place index_put whose only differentiable input is the leaf `val_grad`.  Autograd would then need the DENSE
        gradient of the grid (a 23-59 MB zero-fill + scatter per grid and iteration) just to gather `grad[mask]` back out of it.  When the pattern is
        recognised -- IndexPutBackward0 with one boolean mask of the grid's shape that selects whole voxels (all 32 channels), a non-differentiable
        target and a leaf of matching size -- returns (val_grad, MaskedVoxels): render_batch_ray then differentiates with respect to val_grad itself
        and the backward kernel scatters into a compact [n_selected, 32] buffer.  Anything else returns None (dense path, same results)."""
        fn = g.grad_fn
        if fn is None or type(fn).__name__ != "IndexPutBackward0" or not g.is_cuda or g.dim() != 5:
            return None
        try:
            idx, acc, nxt = fn._saved_indices, fn._saved_accumulate, fn.next_functions
        except (AttributeError, RuntimeError):
            return None
        if acc or len(idx) != 1 or idx[0] is None or idx[0].dtype != torch.bool or tuple(idx[0].shape) != tuple(g.shape):
            return None
        if len(nxt) != 2 or nxt[0][0] is not None or nxt[1][0] is None or not hasattr(nxt[1][0], "variable"):
            return None
        leaf, mask = nxt[1][0].variable, idx[0]
        key = (mask.data_ptr(), mask._version, tuple(mask.shape), str(mask.device))
        mv = self._mask_cache.get(key)
        if mv is None:
            vm = mask[0, 0]
            if not bool((mask == vm).all()):             # the reference repeats one voxel mask over the channels (Mapper.py:319-320)
                self._mask_cache[key] = False
                return None
            from .masked import MaskedVoxels
            mv = MaskedVoxels(g.detach(), vm)
            if len(self._mask_cache) >= 16:
                self._mask_cache.pop(next(iter(self._mask_cache)))
            self._mask_cache[key] = mv
        if mv is False or leaf.dim() != 1 or leaf.numel() != 32 * mv.count or leaf.dtype != torch.float32 or leaf.device != g.device:
            return None
        return leaf, mv

    def eval_points(self, p, decoders, c=None, stage="color", device="cuda:0"):
        """Occupancy/colour of free points (Renderer.eval_points, Renderer.py:23-61).  No autograd: inside
        render_batch_ray the decode is fused; this entry serves meshing / visualisation style bulk queries."""
        _require_cuda(p, "p")
        L = _lib.lib()
        call, grids, _ = self._call(c, decoders, stage, None, p.device)
        pts = p.detach().reshape(-1, 3).contiguous().double()
        n = pts.shape[0]
        dummy = torch.zeros(1, 3, dtype=torch.float32, device=p.device)
        t_u, t_s = _linspaces(self.N_samples, self.N_surface, p.device)
        inp = _inputs(call, dummy, dummy, None, t_u, t_s, [g.detach() for g in grids])
        raw = torch.empty(n, 4, dtype=torch.float32, device=p.device)
        for i in range(0, n, self.points_batch_size):
            m = min(self.points_batch_size, n - i)
            _lib.check(L.nsb_eval_points(C.byref(inp), _VP(pts.data_ptr() + i * 24), m, _VP(raw.data_ptr() + i * 16), _stream()),
                       "nsb_eval_points")
        return raw

    def render_img(self, c, decoders, c2w, device, stage, gt_depth=None):
        """Full-image render in ray batches under no_grad (Renderer.render_img, Renderer.py:200-255)."""
        with torch.no_grad():
            H, W = self.H, self.W
            dev = torch.device(device)
            if not torch.is_tensor(c2w):
                c2w = torch.as_tensor(c2w)
            c2w = c2w.to(dev).float()
            # get_rays (src/common.py:248-266): pixel grid -> camera dirs -> world rays
            i, j = torch.meshgrid(torch.linspace(0, W - 1, W, device=dev), torch.linspace(0, H - 1, H, device=dev), indexing="ij")
            i, j = i.t(), j.t()
            dirs = torch.stack([(i - self.cx) / self.fx, -(j - self.cy) / self.fy, -torch.ones_like(i)], -1)
            rays_d = torch.sum(dirs.reshape(H, W, 1, 3) * c2w[:3, :3], -1).reshape(-1, 3)
            rays_o = c2w[:3, -1].expand(rays_d.shape)
            gt = gt_depth.reshape(-1) if gt_depth is not None else None
            ds, us, cs = [], [], []
            for s in range(0, rays_d.shape[0], self.ray_batch_size):
                e = s + self.ray_batch_size
                d, u, col = self.render_batch_ray(c, decoders, rays_d[s:e], rays_o[s:e].contiguous(), device, stage,
                                                  gt_depth=None if gt is None else gt[s:e])
                ds.append(d.double()); us.append(u.double()); cs.append(col)
            return torch.cat(ds).reshape(H, W), torch.cat(us).reshape(H, W), torch.cat(cs).reshape(H, W, 3)

    def regulation(self, *a, **k):
        raise RuntimeError("regulation() is iMAP*-only (src/utils/Renderer.py:258-296) and is not part of the NICE path")
