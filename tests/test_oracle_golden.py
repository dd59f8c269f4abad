"""CPU: both oracles (oracle/torch_port.py, oracle/nsb_oracle.c) against the fixtures produced by the real
reference (tests/make_golden.py).  This is what pins the oracle wherever /root/reference is absent."""
import glob
import os

import numpy as np
import pytest
import torch

import scene_util as su
from oracle import c_oracle as co
from oracle import torch_port as tp

RENDER_CASES = sorted(glob.glob(os.path.join(su.GOLDEN, "render_*.pt")))
LV = {"coarse": ["coarse"], "middle": ["middle"], "fine": ["fine", "middle"], "color": ["fine", "color", "middle"]}
TOL = 1e-4      # north_star tolerance (rel) -- the oracles actually agree to ~1e-6
# Saturated scene ('init': alpha == 1 at the first sample): the occupancy decoders' weight gradients are ~1e-7 and
# dominated by f32 rounding of (1 - alpha); the reference's own f32 run differs from its f64 evaluation by 8e-4 there
# (measured, DESIGN.md "tolerances"), so those tensors get a noise-floor tolerance instead of 1e-4.
TOL_SATURATED = 3e-3
# The fixtures hold the reference's float32 bits as PyTorch computed them with 8 CPU threads.  MKL's sgemm splits its sums by the
# thread count, so any other count changes the bits: the bit-exact comparisons run on exactly 8 threads, whatever the machine's
# core count.  (By default MKL runs at most one thread per physical core: this needs a machine with 8 cores or more.)
FIXTURE_THREADS = 8


@pytest.fixture(autouse=True, scope="module")
def fixture_thread_count():
    n = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    yield
    torch.set_num_threads(n)


def dec_tol(variant, lvl):
    return TOL_SATURATED if (variant == "init" and lvl in ("fine", "middle", "coarse")) else TOL


def rel(a, b):
    a = torch.as_tensor(np.asarray(a)).double()
    b = torch.as_tensor(np.asarray(b)).double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def load_case(path):
    case = torch.load(path, map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    grids = su.make_grids(sc, case["variant"])
    dec = su.load_decoders(case["variant"])
    return case, sc, grids, dec


@pytest.mark.parametrize("path", RENDER_CASES, ids=[os.path.basename(p)[:-3] for p in RENDER_CASES])
def test_torch_port_matches_reference_fixture(path):
    case, sc, grids, dec = load_case(path)
    bound = su.scene_bound(sc)
    stage = case["stage"]
    ro = case["rays_o"].clone().requires_grad_(True)
    rd = case["rays_d"].clone().requires_grad_(True)
    g = {k: v.clone().requires_grad_(k[5:] in LV[stage]) for k, v in grids.items()}
    dw = {n: {k: v.clone().requires_grad_(True) for k, v in W.items()} for n, W in dec.items()}
    d, u, c, aux = tp.render_batch_ray(g, dw, rd, ro, stage, case["gt_depth"], bound, return_aux=True)
    assert torch.equal(aux["z_vals"], case["z_vals"])                      # bit-exact sample positions
    assert torch.equal(d.detach(), case["depth"]) and torch.equal(u.detach(), case["var"]) and torch.equal(c.detach(), case["rgb"])
    ((d * case["g_depth"]).sum() + (u * case["g_var"]).sum() + (c * case["g_rgb"]).sum()).backward()
    assert torch.equal(ro.grad, case["d_rays_o"]) and torch.equal(rd.grad, case["d_rays_d"])
    for k, summ in case["d_grid"].items():
        mine = su.grid_summary(g[k].grad)
        assert mine["nnz"] == summ["nnz"] and torch.equal(mine["val"], summ["val"])
    for lvl, gd in case["d_dec"].items():
        for k, v in gd.items():
            assert torch.equal(dw[lvl][k].grad, v), (lvl, k)


@pytest.mark.parametrize("path", RENDER_CASES, ids=[os.path.basename(p)[:-3] for p in RENDER_CASES])
def test_c_oracle_matches_reference_fixture(path):
    case, sc, grids, dec = load_case(path)
    stage = case["stage"]
    scene = co.Scene(grids, dec, su.scene_bound(sc), coarse_enlarge=sc["coarse_bound_enlarge"],
                     n_samples=sc["rendering"]["N_samples"], n_surface=sc["rendering"]["N_surface"])
    f = scene.forward(stage, case["rays_o"], case["rays_d"], case["gt_depth"])
    assert np.array_equal(f["z_vals"], case["z_vals"].numpy())               # bit-exact
    assert np.array_equal(f["corner_idx"], case["corner_idx"].numpy().astype(np.int32))   # bit-exact voxel indices
    assert rel(f["depth"], case["depth"]) < TOL and rel(f["var"], case["var"]) < TOL
    if stage == "color":
        assert rel(f["rgb"], case["rgb"]) < TOL
    b = scene.backward(stage, case["rays_o"], case["rays_d"], case["gt_depth"], case["g_depth"], case["g_var"], case["g_rgb"],
                       grad_grids=["grid_" + x for x in LV[stage]], grad_decoders=LV[stage])
    assert rel(b["d_rays_o"], case["d_rays_o"]) < TOL and rel(b["d_rays_d"], case["d_rays_d"]) < TOL
    for k, summ in case["d_grid"].items():
        mine = b["d_" + k].reshape(-1)[summ["idx"]]
        assert rel(mine, summ["val"]) < TOL, k
        assert abs(float(b["d_" + k].double().norm()) - summ["norm"]) < TOL * summ["norm"]
    for lvl, gd in case["d_dec"].items():
        fl = co.unflatten_decoder(co.LEVELS.index(lvl), b["d_flat_" + lvl], dec[lvl])
        for k, v in gd.items():
            assert rel(fl[k], v) < dec_tol(case["variant"], lvl), (lvl, k)


def test_tracker_boundary_capture():
    """Real Tracker.optimize_cam_in_batch (src/Tracker.py:71-128) captured at the renderer boundary: the port, fed the
    captured rays, reproduces outputs exactly and -- through the restated glue -- the camera gradient."""
    case = torch.load(os.path.join(su.GOLDEN, "tracker_color.pt"), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    grids, dec, bound = su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"]), su.scene_bound(sc)
    d, u, c = tp.render_batch_ray(grids, dec, case["rays_d"], case["rays_o"], "color", case["gt_depth"], bound)
    assert torch.equal(d, case["depth"]) and torch.equal(u, case["var"]) and torch.equal(c, case["rgb"])
    import glue
    out = glue.tracking_iteration_cpu(sc, case, grids, dec)
    assert abs(out["loss"] - case["loss"]) < 1e-9 * abs(case["loss"])
    assert torch.allclose(out["d_camera"], case["d_camera"], rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("stage", ["coarse", "middle", "fine", "color"])
def test_mapper_boundary_capture(stage):
    """Real Mapper.optimize_map (src/Mapper.py:230-540) iterations captured at the renderer boundary."""
    case = torch.load(os.path.join(su.GOLDEN, "mapper_%s.pt" % stage), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    grids, dec, bound = su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"]), su.scene_bound(sc)
    import glue
    out = glue.mapping_iteration_cpu(sc, case, grids, dec)
    assert torch.equal(out["depth"], case["depth"]) and torch.equal(out["color"], case["rgb"])
    for k, summ in case["masked_grads"].items():
        dense = out["d_" + k]
        m = case["masks"][k]
        masked = dense[m.unsqueeze(0).unsqueeze(0).expand_as(dense)]
        mine = su.grid_summary(masked, n_sample=4096)
        assert mine["nnz"] == summ["nnz"] and torch.equal(mine["val"], summ["val"]), k
    for k, v in case["d_color_decoder"].items():
        assert torch.equal(out["d_dec"]["color"][k], v), k


def test_frustum_oracle_matches_real_mapper_masks_and_cv2_remap():
    """oracle/frustum.py against (a) the masks the REAL Mapper.get_mask_from_c2w produced (stored with the mapper captures) and
    (b) cv2.remap itself for the bilinear look-up."""
    import numpy as np
    from oracle import frustum as fr
    sc = su.load_scenes()["room0"]
    case = torch.load(os.path.join(su.GOLDEN, "mapper_color.pt"), map_location="cpu", weights_only=False)
    depth, _ = su.make_frame(sc, case["frame_seed"])
    c2w = su.make_pose(sc, 1)
    bound = su.scene_bound(sc)
    for key, want in case["masks"].items():
        got = fr.frustum_mask(c2w, key, tuple(want.shape), depth.numpy(), bound, sc["cam"])
        assert torch.equal(got, want), key
        assert key == "grid_coarse" or 0 < int(want.sum()) < want.numel()
    cv2 = pytest.importorskip("cv2")
    g = np.random.default_rng(0)
    x = (g.random(20000) * 1300 - 50).astype(np.float32)
    y = (g.random(20000) * 800 - 60).astype(np.float32)
    assert np.array_equal(cv2.remap(depth.numpy(), x, y, interpolation=cv2.INTER_LINEAR)[:, 0], fr.remap_bilinear(depth.numpy(), x, y))


def test_oracle_reproduces_five_real_mapper_iterations_with_adam():
    """tests/golden/mapper_loop.pt (real Mapper.optimize_map, real torch Adam, 3 x middle + fine + color) replayed with the oracle port:
    frustum masks from oracle/frustum.py, masked leaf parameters val[mask] as in Mapper.py:317-333, the port's render + mapping loss,
    torch Adam with the per-stage learning rates.  Pins the whole chain the native mapping loop (nice_slam_b200/mapping.py) replaces."""
    from oracle import frustum as fr
    case = torch.load(os.path.join(su.GOLDEN, "mapper_loop.pt"), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    grids, dec = su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"])
    depth, _ = su.make_frame(sc, case["frame_seed"])
    c2w = su.make_pose(sc, case["pose_seed"])
    bound = su.scene_bound(sc)
    keys = ("grid_middle", "grid_fine", "grid_color")
    m5 = {k: fr.frustum_mask(c2w, k, tuple(grids[k].shape[2:]), depth.numpy(), bound, sc["cam"]).unsqueeze(0).unsqueeze(0).expand_as(grids[k])
          for k in keys}
    val_grad = {k: grids[k][m5[k]].clone().requires_grad_(True) for k in keys}
    dw = {n: {k: v.clone().requires_grad_(n == "color") for k, v in W.items()} for n, W in dec.items()}
    opt = torch.optim.Adam([{"params": list(dw["color"].values()), "lr": 0}] + [{"params": [val_grad[k]], "lr": 0} for k in keys])
    lv = {"middle": ("grid_middle",), "fine": ("grid_fine", "grid_middle"), "color": keys}
    for it in case["iterations"]:
        opt.param_groups[0]["lr"] = it["lr"]["decoders"]
        for gi, k in enumerate(keys):
            opt.param_groups[1 + gi]["lr"] = it["lr"][k[5:]]
        g = {k: v.clone() for k, v in grids.items()}
        for k in keys:
            g[k][m5[k]] = val_grad[k]                                   # Mapper.py:393-401
        opt.zero_grad()
        d, _, col = tp.render_batch_ray(g, dw, it["rays_d"], it["rays_o"], it["stage"], it["gt_depth"], bound)
        tp.mapping_loss(d, col, it["gt_depth_loss"], it["gt_color"], it["stage"], case["w_color_loss"]).backward()
        for k in keys:
            if k not in lv[it["stage"]]:
                assert val_grad[k].grad is None or not bool(val_grad[k].grad.any())
        opt.step()
        for k in keys:
            grids[k][m5[k]] = val_grad[k].detach()                       # Mapper.py:511-519
    for k, fin in case["final"].items():
        got = val_grad[k].detach()[fin["idx"]]
        assert torch.allclose(got, fin["val"], rtol=1e-5, atol=1e-6), (k, float((got - fin["val"]).abs().max()))
    for k, v in case["color_decoder"].items():
        assert torch.allclose(dw["color"][k].detach(), v, rtol=1e-5, atol=1e-6), k


def _ba_fixed_row(case_window_c2w, cams):
    """The window row that has no camera tensor (the oldest frame, Mapper.py:350): the one whose pose no tensor reproduces."""
    poses = tp.camera_from_tensor(cams)
    for r in range(case_window_c2w.shape[0]):
        if not any(torch.allclose(poses[k], case_window_c2w[r], atol=1e-5) for k in range(poses.shape[0])):
            return r
    raise AssertionError("no fixed row")


@pytest.mark.parametrize("stage", ["middle", "fine", "color"])
def test_oracle_reproduces_ba_window_gradients(stage):
    """tests/golden/mapper_ba_grads.pt: REAL Mapper.optimize_map with BA=True on a window of 5 keyframes + the current frame
    (src/Mapper.py:346-363,437-467).  The oracle chain camera tensor -> c2w -> rays -> render -> loss reproduces camera_tensor.grad of
    every non-fixed frame, the masked voxel gradients and the colour-decoder gradients."""
    case = torch.load(os.path.join(su.GOLDEN, "mapper_ba_grads.pt"), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    grids, dec, bound = su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"]), su.scene_bound(sc)
    cam = sc["cam"]
    st = case["stages"][stage]
    cams = case["camera_tensors"].clone().requires_grad_(True)
    fixed = _ba_fixed_row(case["window_c2w"], case["camera_tensors"])
    ro, rd = tp.ba_window_rays(cams, case["window_c2w"][fixed], fixed, st["pix_i"], st["pix_j"], st["frame_of_ray"], cam["fx"], cam["fy"], cam["cx"], cam["cy"])
    assert torch.equal(ro.detach(), st["rays_o"]) and torch.equal(rd.detach(), st["rays_d"])          # ray generation is bit-exact
    keys = {"middle": ("grid_middle",), "fine": ("grid_middle", "grid_fine"), "color": ("grid_middle", "grid_fine", "grid_color")}[stage]
    g = {k: v.clone().requires_grad_(k in keys) for k, v in grids.items()}
    dw = {n: {k: v.clone().requires_grad_(n == "color") for k, v in W.items()} for n, W in dec.items()}
    d, _, col = tp.render_batch_ray(g, dw, rd, ro, stage, st["gt_depth"], bound)
    assert torch.equal(d.detach(), st["depth"]) and torch.equal(col.detach(), st["rgb"])
    tp.mapping_loss(d, col, st["gt_depth_loss"], st["gt_color"], stage).backward()
    assert rel(cams.grad, st["d_cameras"]) < 1e-5, rel(cams.grad, st["d_cameras"])
    assert float(st["d_cameras"].abs().min()) > 0                                                  # every non-fixed frame gets a gradient
    for k, summ in st["masked_grads"].items():
        m = case["masks"][k]
        mine = su.grid_summary(g[k].grad[m.unsqueeze(0).unsqueeze(0).expand_as(g[k])], n_sample=4096)
        assert mine["nnz"] == summ["nnz"] and torch.allclose(mine["val"], summ["val"], rtol=1e-5, atol=1e-9), k
    for k, v in st["d_color_decoder"].items():
        assert torch.allclose(dw["color"][k].grad, v, rtol=1e-4, atol=1e-7), k


def test_oracle_reproduces_ba_loop_with_adam():
    """tests/golden/mapper_ba_loop.pt: eight REAL joint iterations with bundle adjustment and the real torch Adam (4 x middle, fine, 3 x color;
    the pose group has lr = BA_cam_lr in stage color only, Mapper.py:417-424, but its Adam state advances in every iteration).  Replayed with
    the oracle: per-iteration rays regenerated from the CURRENT camera tensors and the recorded pixel draws, bbox pre-filter, masked leaf
    voxels, port render + loss, torch Adam with the six parameter groups.  Checks the poses the mapper wrote back (Mapper.py:521-540)."""
    from oracle import frustum as fr
    case = torch.load(os.path.join(su.GOLDEN, "mapper_ba_loop.pt"), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    cam = sc["cam"]
    grids, dec = su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"])
    depth, _ = su.make_frame(sc, case["frame_seed"])
    c2w_cur = su.make_pose(sc, case["pose_seed"])
    bound = su.scene_bound(sc)
    keys = ("grid_middle", "grid_fine", "grid_color")
    m5 = {k: fr.frustum_mask(c2w_cur, k, tuple(grids[k].shape[2:]), depth.numpy(), bound, sc["cam"]).unsqueeze(0).unsqueeze(0).expand_as(grids[k])
          for k in keys}
    val_grad = {k: grids[k][m5[k]].clone().requires_grad_(True) for k in keys}
    dw = {n: {k: v.clone().requires_grad_(n == "color") for k, v in W.items()} for n, W in dec.items()}
    win = case["window_keyframes"]
    fixed = win.index(min(k for k in win if k >= 0))                       # oldest keyframe of the window is fixed (Mapper.py:262,350)
    # start from the camera tensors the reference derived from the keyframes' est_c2w (get_tensor_from_camera, src/common.py:179-200): the L1
    # losses make the pose gradients discontinuous, so a 1e-8 difference in the starting quaternion shows up at the 1e-4 level in the gradients
    cams = [case["camera_tensors"][k].clone().requires_grad_(True) for k in range(5)]
    opt = torch.optim.Adam([{"params": list(dw["color"].values()), "lr": 0}, {"params": [], "lr": 0}] + [{"params": [val_grad[k]], "lr": 0} for k in keys]
                           + [{"params": cams, "lr": 0}])
    for it, (stage, lr, dr) in enumerate(zip(case["stages"], case["lrs"], case["draws"])):
        opt.param_groups[0]["lr"] = lr["decoders"]
        for gi, k in enumerate(keys):
            opt.param_groups[2 + gi]["lr"] = lr[k[5:]]
        if stage == "color":
            opt.param_groups[5]["lr"] = case["BA_cam_lr"]
        g = {k: v.clone() for k, v in grids.items()}
        for k in keys:
            g[k][m5[k]] = val_grad[k]
        opt.zero_grad()
        n = dr["i"].shape[1]
        fid = torch.arange(6).repeat_interleave(n)
        ro, rd = tp.ba_window_rays(torch.stack(cams), case["window_c2w"][fixed], fixed, dr["i"].reshape(-1), dr["j"].reshape(-1), fid,
                                   cam["fx"], cam["fy"], cam["cx"], cam["cy"])
        gd, gc = dr["depth"].reshape(-1), dr["color"].reshape(-1, 3)
        keep = tp.bbox_prefilter(ro, rd, gd, bound)
        d, _, col = tp.render_batch_ray(g, dw, rd[keep], ro[keep], stage, gd[keep], bound)
        tp.mapping_loss(d, col, gd[keep], gc[keep], stage, case["w_color_loss"]).backward()
        hist = case["camera_history"][it]
        assert rel(torch.stack([c.detach() for c in cams]), hist["cam"]) < 1e-6 and rel(torch.stack([c.grad for c in cams]), hist["grad"]) < 1e-4, it
        opt.step()
        for k in keys:
            grids[k][m5[k]] = val_grad[k].detach()
    got = tp.camera_from_tensor(torch.stack([c.detach() for c in cams]))
    want = torch.stack([case["final_c2w"][r] for r in range(6) if r != fixed])
    moved = (want - torch.stack([case["window_c2w"][r] for r in range(6) if r != fixed])).abs().amax((1, 2))
    assert float(moved.min()) > 5e-4                                       # the poses did move
    assert float((got - want).abs().max()) < 2e-5, float((got - want).abs().max())
    for k, fin in case["final"].items():
        gotv = val_grad[k].detach()[fin["idx"]]
        assert torch.allclose(gotv, fin["val"], rtol=1e-4, atol=2e-5), (k, float((gotv - fin["val"]).abs().max()))


def test_keyframe_overlap_oracle_matches_real_mapper():
    """oracle/keyframes.py against the REAL Mapper.keyframe_selection_overlap (tests/golden/keyframe_overlap.pt): the same percent_inside for
    every keyframe (exact counts) and, under the same numpy seed, the same selected keyframes."""
    import numpy as np
    from oracle import keyframes as kf
    case = torch.load(os.path.join(su.GOLDEN, "keyframe_overlap.pt"), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    cam = sc["cam"]
    pts = kf.overlap_points(case["rays_o"], case["rays_d"], case["gt_depth"])
    per = [kf.percent_inside(pts, c2w, cam["H"], cam["W"], cam["fx"], cam["fy"], cam["cx"], cam["cy"])[0] for c2w in case["keyframe_c2w"]]
    assert [float(p) for p in per] == case["percent_inside"]
    assert sum(p == 0 for p in per) >= 3 and sum(p > 0 for p in per) > case["k"]
    # the reference draws its pixels with the torch RNG first; only the numpy stream matters for the permutation
    rng = np.random.RandomState(case["numpy_seed"])
    assert [int(x) for x in kf.select(per, case["k"], rng)] == case["selected"]


@pytest.mark.parametrize("stage,n_samples,n_surface,n_rays", [("color", 5, 3, 37), ("fine", 32, 16, 1), ("middle", 16, 16, 61),
                                                              ("color", 80, 16, 9), ("coarse", 32, 16, 23), ("color", 32, 0, 19)])
def test_the_two_oracles_agree_on_ragged_shapes(stage, n_samples, n_surface, n_rays):
    """Shapes the reference fixtures do not hold (other sample counts, a single ray, no near-surface samples, some zero sensor depths):
    the C restatement against the torch port -- z_vals bit-exact, outputs and gradients at the path's tolerance.  (The torch port is the one
    pinned bit for bit to the reference; this keeps the C oracle, which smoke() and the GPU tests use at these shapes, honest.)"""
    sc = su.load_scenes()["room0"]
    grids, dec, bound = su.make_grids(sc, "soft"), su.load_decoders("soft"), su.scene_bound(sc)
    ro, rd, gd, _ = su.make_rays(sc, n_rays, seed=1000 + n_rays)
    gd = gd.clone()
    gd[::5] = 0.0                                                        # rays without a sensor depth (Renderer.py:133-149)
    with_depth = stage != "coarse" and n_surface > 0
    gt = gd if with_depth else None
    g = torch.Generator().manual_seed(n_samples)
    s_d = torch.randn(n_rays, dtype=torch.float64, generator=g)
    s_v = torch.randn(n_rays, dtype=torch.float64, generator=g)
    s_c = torch.randn(n_rays, 3, generator=g)
    r_o = ro.clone().requires_grad_(True); r_d = rd.clone().requires_grad_(True)
    gg = {k: v.clone().requires_grad_(k[5:] in LV[stage]) for k, v in grids.items()}
    d, u, c, aux = tp.render_batch_ray(gg, dec, r_d, r_o, stage, gt, bound, n_samples=n_samples, n_surface=n_surface, return_aux=True)
    ((d * s_d).sum() + (u * s_v).sum() + (c * s_c).sum()).backward()
    scene = co.Scene(grids, dec, bound, coarse_enlarge=sc["coarse_bound_enlarge"], n_samples=n_samples, n_surface=n_surface)
    f = scene.forward(stage, ro, rd, gt)
    assert np.array_equal(f["z_vals"], aux["z_vals"].numpy())
    assert rel(f["depth"], d.detach()) < TOL and rel(f["var"], u.detach()) < TOL
    if stage == "color":
        assert rel(f["rgb"], c.detach()) < TOL
    b = scene.backward(stage, ro, rd, gt, s_d, s_v, s_c, grad_grids=["grid_" + x for x in LV[stage]], grad_decoders=[])
    assert rel(b["d_rays_o"], r_o.grad) < TOL and rel(b["d_rays_d"], r_d.grad) < TOL
    for x in LV[stage]:
        assert rel(b["d_grid_" + x], gg["grid_" + x].grad) < TOL, x
