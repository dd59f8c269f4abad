"""ctypes binding of the C-ABI library (include/nice_slam_b200.h).

The product path has NO fallback: if libnsb.so is missing, or a call fails, a RuntimeError is raised.
The handle is loaded lazily per process (the reference pickles its Renderer into three spawned
processes, src/NICE_SLAM.py:288-307), nothing CUDA-related lives in picklable state.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NSB_LIB") or os.path.join(_HERE, "libnsb.so")      # NSB_LIB: instrumented build for tools/phase_timing.py

LEVELS = ("coarse", "middle", "fine", "color")
STAGES = {"coarse": 0, "middle": 1, "fine": 2, "color": 3}
STAGE_DECODERS = {"coarse": ("coarse",), "middle": ("middle",), "fine": ("fine", "middle"),
                  "color": ("fine", "color", "middle")}          # NICE.forward order, decoder.py:317-342


class Grid(C.Structure):
    _fields_ = [("data", C.c_void_p), ("D", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("stride_c", C.c_int64), ("stride_d", C.c_int64), ("stride_h", C.c_int64), ("stride_w", C.c_int64)]


class AdamVoxelGroup(C.Structure):
    _fields_ = [("grid", Grid), ("slot_map", C.c_void_p), ("grad", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
                ("lr", C.c_double), ("step", C.c_int)]


class DecoderParams(C.Structure):
    _fields_ = [("B", C.c_void_p), ("W", C.c_void_p * 5), ("b", C.c_void_p * 5),
                ("Wc", C.c_void_p * 5), ("bc", C.c_void_p * 5), ("Wo", C.c_void_p), ("bo", C.c_void_p)]


class RenderInputs(C.Structure):
    _fields_ = [("stage", C.c_int32), ("n_rays", C.c_int32), ("n_samples", C.c_int32), ("n_surface", C.c_int32),
                ("bound", C.c_double * 6), ("coarse_bound", C.c_double * 6),
                ("rays_o", C.c_void_p), ("rays_d", C.c_void_p), ("gt_depth", C.c_void_p), ("depth_max", C.c_void_p),
                ("t_uniform", C.c_void_p), ("t_surface", C.c_void_p),
                ("grid", Grid * 4), ("packed", C.c_void_p * 4), ("gt_depth_batch", C.c_void_p), ("n_batch", C.c_int32)]


class ForwardOutputs(C.Structure):
    _fields_ = [("depth", C.c_void_p), ("var", C.c_void_p), ("rgb", C.c_void_p),
                ("z_vals", C.c_void_p), ("raw", C.c_void_p), ("corner_idx", C.c_void_p), ("masks", C.c_void_p),
                ("split_workspace", C.c_void_p), ("split_workspace_bytes", C.c_size_t), ("acts", C.c_void_p)]


class BackwardArgs(C.Structure):
    _fields_ = [("z_vals", C.c_void_p), ("raw", C.c_void_p), ("g_depth", C.c_void_p), ("g_var", C.c_void_p),
                ("g_rgb", C.c_void_p), ("d_rays_o", C.c_void_p), ("d_rays_d", C.c_void_p),
                ("d_grid", C.c_void_p * 4), ("d_flat", C.c_void_p * 4), ("workspace", C.c_void_p), ("masks", C.c_void_p),
                ("slot_map", C.c_void_p * 4), ("split_workspace", C.c_void_p), ("split_workspace_bytes", C.c_size_t),
                ("pose_dirs", C.c_void_p), ("d_c2w", C.c_void_p), ("pose_counter", C.c_void_p), ("acts", C.c_void_p),
                ("result_dst", C.c_void_p), ("result_src", C.c_void_p), ("result_bytes", C.c_size_t)]


class IterationBuffers(C.Structure):
    _fields_ = [("depth", C.c_void_p), ("var", C.c_void_p), ("rgb", C.c_void_p), ("z_vals", C.c_void_p), ("raw", C.c_void_p),
                ("masks", C.c_void_p), ("g_depth", C.c_void_p), ("g_rgb", C.c_void_p), ("loss", C.c_void_p), ("depth_max", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
                ("event_bwd_begin", C.c_void_p), ("event_bwd_end", C.c_void_p), ("acts", C.c_void_p)]


class Peers(C.Structure):
    _fields_ = [("rank", C.c_int), ("world", C.c_int), ("buffer", C.c_void_p * 8), ("counters", C.c_void_p), ("max_rays", C.c_int)]


# every symbol include/nice_slam_b200.h declares: (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "nsb_version": (C.c_int, []),
    "nsb_last_error": (C.c_char_p, []),
    "nsb_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "nsb_debug_occupancy": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "nsb_flat_decoder_floats": (C.c_size_t, [C.c_int]),
    "nsb_flat_offset": (C.c_longlong, [C.c_int, C.c_int, C.c_int]),
    "nsb_packed_decoder_floats": (C.c_size_t, [C.c_int]),
    "nsb_pack_decoders": (C.c_int, [C.POINTER(C.POINTER(DecoderParams)), C.POINTER(_P), _P]),
    "nsb_batch_max_depth": (C.c_int, [_P, C.c_int, _P, _P]),
    "nsb_bbox_prefilter": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(C.c_double), _P, _P]),
    "nsb_render_forward": (C.c_int, [C.POINTER(RenderInputs), C.POINTER(ForwardOutputs), _P]),
    "nsb_backward_workspace_bytes": (C.c_size_t, []),
    "nsb_render_backward": (C.c_int, [C.POINTER(RenderInputs), C.POINTER(BackwardArgs), _P]),
    "nsb_tracking_seeds": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_double, C.c_int, C.c_int, _P, C.c_int, _P, _P, _P, _P, C.c_size_t, _P]),
    "nsb_tracking_residuals": (C.c_int, [_P, _P, _P, C.c_int, _P, _P]),
    "nsb_pose_grad": (C.c_int, [_P, _P, _P, C.c_int, _P, _P]),
    "nsb_iteration_workspace_bytes": (C.c_size_t, [C.c_int]),
    "nsb_tracking_iteration": (C.c_int, [C.POINTER(RenderInputs), C.POINTER(IterationBuffers), _P, C.c_double, C.c_int, C.c_int, C.POINTER(BackwardArgs), _P]),
    "nsb_tracking_iteration_peers": (C.c_int, [C.POINTER(RenderInputs), C.POINTER(IterationBuffers), _P, C.c_double, C.c_int, C.c_int, C.POINTER(BackwardArgs),
                                               C.POINTER(Peers), _P, _P]),
    "nsb_mapping_iteration": (C.c_int, [C.POINTER(RenderInputs), C.POINTER(IterationBuffers), _P, _P, C.c_double, C.POINTER(BackwardArgs), _P]),
    "nsb_mapping_seeds": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_double, C.c_int, _P, _P, _P, _P]),
    "nsb_tracking_seeds_workspace": (C.c_size_t, [C.c_int]),
    "nsb_host_device_pointer": (C.c_void_p, [_P]),
    "nsb_copy_block": (C.c_int, [_P, _P, C.c_size_t, _P]),
    "nsb_eval_points": (C.c_int, [C.POINTER(RenderInputs), _P, C.c_int, _P, _P]),
    "nsb_voxel_slots_workspace": (C.c_size_t, [C.c_longlong]),
    "nsb_voxel_slots": (C.c_int, [_P, C.c_longlong, _P, _P, _P, C.c_size_t, _P]),
    "nsb_masked_gather": (C.c_int, [C.POINTER(Grid), _P, _P, _P]),
    "nsb_masked_scatter": (C.c_int, [C.POINTER(Grid), _P, _P, _P]),
    "nsb_compact_transpose": (C.c_int, [_P, _P, C.c_longlong, C.c_int, _P]),
    "nsb_pose_grad_frames": (C.c_int, [_P, _P, _P, _P, C.c_int, _P, _P]),
    "nsb_split_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "nsb_adam_masked_voxels": (C.c_int, [C.POINTER(Grid), _P, _P, _P, _P, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int, _P]),
    "nsb_adam_mapper_step": (C.c_int, [C.POINTER(AdamVoxelGroup), C.c_int, C.c_int, C.POINTER(DecoderParams), _P, _P, _P, C.c_double, C.c_int,
                                       C.c_double, C.c_double, C.c_double, _P]),
    "nsb_adam_decoder": (C.c_int, [C.c_int, C.POINTER(DecoderParams), _P, _P, _P, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int, _P]),
    "nsb_frustum_mask_workspace": (C.c_size_t, [C.c_longlong]),
    "nsb_frustum_mask": (C.c_int, [C.POINTER(C.c_float), _P, _P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int, C.c_int,
                                   C.c_double, C.c_double, C.c_double, C.c_double, _P, _P, C.c_size_t, _P]),
    "nsb_keyframe_overlap": (C.c_int, [_P, _P, _P, C.c_int, _P, C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double,
                                       C.c_int, _P, _P]),
    "nsb_keyframe_gather": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "nsb_window_rays": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, _P, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, _P, _P, _P, _P, _P]),
    "nsb_adam_poses": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int, _P]),
    "nsb_peer_buffer_bytes": (C.c_size_t, [C.c_int]),
    "nsb_batch_max_depth_peers": (C.c_int, [_P, C.c_int, _P, C.POINTER(Peers), _P]),
    "nsb_tracking_seeds_peers": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_double, C.c_int, C.c_int, C.POINTER(Peers), _P, _P, _P, _P, C.c_size_t, _P]),
    "nsb_pose_grad_peers": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, C.POINTER(Peers), _P]),
}

_LIB = None


def lib():
    """Load libnsb.so (once per process) and type its entry points.  Raises if it is not built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "nice_slam_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or make -C nice_slam_b200/csrc).  There is no CPU / PyTorch fallback." % LIB_PATH)
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(h, name)          # AttributeError if the library does not export a declared symbol
            f.restype, f.argtypes = res, args
        backend = os.environ.get("NSB_MLP_BACKEND")          # 1 = FP32-FMA decoders (default 0: tile kernels where S >= 8)
        if backend is not None and h.nsb_set_option(b"mlp_backend", int(backend)) != 0:
            raise RuntimeError("bad NSB_MLP_BACKEND=%r" % backend)
        wg = os.environ.get("NSB_WGRAD_TC")                  # 0 = decoder weight gradients by the FP32-FMA pass (default: tensor cores)
        if wg is not None:
            h.nsb_set_option(b"wgrad_tc", int(wg))
        f16 = os.environ.get("NSB_FWD_F16")                  # 1 = forward decoders with FP16 hi|lo operands (kind::f16) instead of 3xTF32
        if f16 is not None:
            h.nsb_set_option(b"fwd_f16", int(f16))
        sm = os.environ.get("NSB_SPLIT_MODEL")               # 0 = per-decoder items for every batch of <= 262144 points (default: by wave efficiency)
        if sm is not None:
            h.nsb_set_option(b"split_model", int(sm))
        _LIB = h
    return _LIB


def check(rc, what):
    if rc != 0:
        msg = lib().nsb_last_error().decode("utf-8", "replace")
        raise RuntimeError("nice_slam_b200.%s failed (status %d): %s" % (what, rc, msg))


def flat_layout(level):
    """[(reference parameter name, offset, numel)] of the canonical flat order of decoder `level`."""
    L = lib()
    kinds = [("embedder._B", 0, None), ("pts_linears.%d.weight", 1, 5), ("pts_linears.%d.bias", 2, 5),
             ("fc_c.%d.weight", 3, 5), ("fc_c.%d.bias", 4, 5), ("output_linear.weight", 5, None),
             ("output_linear.bias", 6, None)]
    offs = []
    for name, kind, n in kinds:
        if level == 0 and kind in (0, 3, 4):
            continue
        for i in (range(n) if n else [0]):
            offs.append((name % i if n else name, L.nsb_flat_offset(level, kind, i)))
    offs.sort(key=lambda t: t[1])
    total = L.nsb_flat_decoder_floats(level)
    return [(nm, off, (offs[j + 1][1] if j + 1 < len(offs) else total) - off) for j, (nm, off) in enumerate(offs)]
