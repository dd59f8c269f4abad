"""CPU: the C-ABI library builds, loads and exports every symbol include/nice_slam_b200.h declares; the host-side
layout helpers agree with the oracle's.  No compute calls (no GPU here)."""
import ctypes as C
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "nice_slam_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nsb_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_expected_entry_points():
    syms = declared_symbols()
    for s in ("nsb_render_forward", "nsb_render_backward", "nsb_pack_decoders", "nsb_eval_points", "nsb_batch_max_depth",
              "nsb_bbox_prefilter", "nsb_tracking_seeds", "nsb_mapping_seeds", "nsb_last_error", "nsb_version"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    from nice_slam_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "build with __graft_entry__.build()"
    h = C.CDLL(_lib.LIB_PATH)
    for s in declared_symbols():
        assert hasattr(h, s), "libnsb.so does not export %s" % s
    assert set(declared_symbols()) == set(_lib.SYMBOLS.keys())      # the ctypes binding covers the whole header
    L = _lib.lib()
    assert L.nsb_version() == 100
    assert L.nsb_last_error() is not None


def test_flat_layout_matches_oracle_and_reference_shapes():
    from nice_slam_b200 import _lib
    from oracle import c_oracle as co
    import scene_util as su
    dec = su.load_decoders("init")
    for li, lvl in enumerate(_lib.LEVELS):
        mine, theirs = _lib.flat_layout(li), co.flat_layout(li)
        assert mine == theirs
        assert sum(n for _, _, n in mine) == _lib.lib().nsb_flat_decoder_floats(li)
        for name, off, n in mine:
            assert dec[lvl][name].numel() == n, (lvl, name)
    L = _lib.lib()
    assert [L.nsb_flat_decoder_floats(i) for i in range(4)] == [6337, 15800, 20920, 15899]     # SURVEY 8a parameter counts
    assert all(L.nsb_packed_decoder_floats(i) % 4 == 0 for i in range(4))


def test_struct_sizes_match_the_header():
    """sizeof() of the ctypes mirrors == sizeof() of the C structs (compiled on the fly with gcc)."""
    import subprocess, tempfile
    from nice_slam_b200 import _lib
    prog = r'''
#include <stdio.h>
#include "nice_slam_b200.h"
int main(){ printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(nsb_grid), sizeof(nsb_decoder_params), sizeof(nsb_render_inputs),
                   sizeof(nsb_forward_outputs), sizeof(nsb_backward_args), sizeof(nsb_iteration_buffers), sizeof(nsb_peers), sizeof(nsb_adam_voxel_group)); return 0; }
'''
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "s.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    mine = [C.sizeof(x) for x in (_lib.Grid, _lib.DecoderParams, _lib.RenderInputs, _lib.ForwardOutputs, _lib.BackwardArgs, _lib.IterationBuffers,
                                   _lib.Peers, _lib.AdamVoxelGroup)]
    assert sizes == mine


def test_product_path_fails_loudly_without_cuda():
    from types import SimpleNamespace
    import scene_util as su
    from gpu_util import make_cfg
    from nice_slam_b200.decoders import NICEDecoders
    from nice_slam_b200.renderer import FusedRenderer
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    sc = su.load_scenes()["room0"]
    grids = su.make_grids(sc, "init", keys=("grid_middle",))
    slam = SimpleNamespace(nice=True, bound=su.scene_bound(sc), shared_c=grids, H=1, W=1, fx=1, fy=1, cx=0, cy=0)
    r = FusedRenderer(make_cfg(sc), SimpleNamespace(nice=True), slam)
    dec = NICEDecoders.from_state(su.load_decoders("init"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        r.render_batch_ray(grids, dec, torch.zeros(4, 3), torch.zeros(4, 3), "cpu", "middle", gt_depth=torch.ones(4))


def test_renderer_pickles_without_device_state_and_keeps_reference_surface():
    import pickle
    from types import SimpleNamespace
    import scene_util as su
    from gpu_util import make_cfg
    from nice_slam_b200.renderer import FusedRenderer
    sc = su.load_scenes()["room0"]
    slam = SimpleNamespace(nice=True, bound=su.scene_bound(sc), shared_c={}, H=680, W=1200, fx=600., fy=600., cx=599.5, cy=339.5)
    r = FusedRenderer(make_cfg(sc), SimpleNamespace(nice=True), slam)
    r2 = pickle.loads(pickle.dumps(r))
    for attr in ("ray_batch_size", "points_batch_size", "lindisp", "perturb", "N_samples", "N_surface", "N_importance", "scale",
                 "occupancy", "nice", "bound", "H", "W", "fx", "fy", "cx", "cy"):            # Renderer.__init__, Renderer.py:6-21
        assert hasattr(r2, attr)
    for meth in ("eval_points", "render_batch_ray", "render_img", "regulation"):
        assert callable(getattr(r2, meth))


def test_decoder_container_has_reference_state_dict_keys():
    import scene_util as su
    from nice_slam_b200.decoders import NICEDecoders
    st = su.load_decoders("init")
    m = NICEDecoders.from_state(st)
    for lvl, sd in st.items():
        mine = dict(getattr(m, lvl + "_decoder").named_parameters())
        assert set(mine.keys()) == set(sd.keys())
        for k in sd:
            assert torch.equal(mine[k].detach(), sd[k])


def test_bench_reference_arm_prints_one_contract_line():
    """bench.py --impl reference (the CPU arm the driver launches beside the native one): exactly one JSON line on stdout, with the
    keys of the bench contract."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "rays/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_iteration_context_block_layouts_on_cpu():
    """Host-side layout logic of steps.IterationContext (no kernel runs): the single-copy input / result blocks and the packed gradient block."""
    from types import SimpleNamespace
    from nice_slam_b200 import _lib
    from nice_slam_b200.steps import IterationContext, packed_layout
    r = SimpleNamespace(N_samples=32, N_surface=16)
    for kind, col_dt in (("track", torch.float64), ("map", torch.float32)):
        n = 37
        x = IterationContext(r, n, "color", "cpu", kind=kind, grad_decoders=("color",) if kind == "map" else (), n_frames=3 if kind == "map" else 0)
        ro, rd, gd, gc = x.device_views()
        assert ro.shape == (n, 3) and rd.shape == (n, 3) and gd.shape == (n,) and gc.shape == (n, 3) and gc.dtype == col_dt
        x.d_in.zero_(); gc.fill_(1.0); assert float(ro.abs().sum() + rd.abs().sum() + gd.abs().sum()) == 0.0      # colour does not overlap the rays
        ro.fill_(2.0); rd.fill_(3.0); gd.fill_(4.0); assert float(gc.sum()) == 3 * n
        assert gc.data_ptr() % 8 == 0 and x.loss.data_ptr() % 8 == 0 and x.d_c2w.data_ptr() == x.loss.data_ptr() + 8
        assert x.d_rays_o.data_ptr() == x.d_res.data_ptr() and x.d_rays_d.data_ptr() == x.d_res.data_ptr() + 12 * n
        assert x.h2d_bytes == x.d_in.numel() and x.d2h_bytes == x.d_res.numel()
        if kind == "map":
            sect, total = packed_layout(3, ("color",), [("grid_fine", 10)])
            assert sect["frames"] == (4, 36) and sect["dec_color"][0] == 40 and sect["dec_color"][1] == _lib.lib().nsb_flat_decoder_floats(3)
            assert sect["grid_fine"][0] % 4 == 0 and total == sect["grid_fine"][0] + 320          # voxel sections are 16-byte aligned
            assert x.packed.numel() == 40 + ((15899 + 3) // 4) * 4 and x.d_frames.shape == (3, 12) and x.d_flat["color"].numel() == 15899


def test_set_option_accepts_only_the_supported_decoder_backends():
    """mlp_backend takes 0 (auto: tile kernels, FP32-FMA where S < 8) and 1 (FP32-FMA); other values and unknown keys are rejected."""
    from nice_slam_b200 import _lib
    L = _lib.lib()
    NSB_ERR_ARG = -1
    configured = int(os.environ.get("NSB_MLP_BACKEND", "0"))
    try:
        assert L.nsb_set_option(b"mlp_backend", 0) == 0
        assert L.nsb_set_option(b"mlp_backend", 1) == 0
        for value in (2, 3, -1):
            assert L.nsb_set_option(b"mlp_backend", value) == NSB_ERR_ARG
            assert b"mlp_backend" in L.nsb_last_error()
        for key in (b"small_rays", b"pdl"):
            assert L.nsb_set_option(key, 0) == NSB_ERR_ARG
            assert b"unknown option" in L.nsb_last_error()
    finally:
        assert L.nsb_set_option(b"mlp_backend", configured) == 0
