"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C-ABI library
(nice_slam_b200/libnsb.so) via FusedRenderer; the checker is the oracle (oracle/torch_port.py, oracle/nsb_oracle.c)
run live on the host CPU plus the committed reference fixtures (tests/golden).

Bars: bit-exact sample positions (z_vals) and voxel-corner indices; 1e-4 relative (max-norm) on rendered
depth / variance / RGB and on every gradient (TOL); the saturated-scene occupancy-decoder weight gradients use the
measured f32 noise floor (TOL_SATURATED, see tests/test_oracle_golden.py)."""
import glob
import os

import pytest
import torch

import glue
import scene_util as su
from gpu_util import LV, l2rel, make_renderer, rel
from oracle import torch_port as tp

pytestmark = pytest.mark.gpu
TOL = 1e-4
TOL_SATURATED = 3e-3
RENDER_CASES = sorted(glob.glob(os.path.join(su.GOLDEN, "render_*.pt")))
DEV = "cuda"


def load_case(path):
    case = torch.load(path, map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    return case, sc, su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"])


def run_render(renderer, c, dec, case, stage, grads=True):
    ro = case["rays_o"].to(DEV).requires_grad_(grads)
    rd = case["rays_d"].to(DEV).requires_grad_(grads)
    gt = case["gt_depth"].to(DEV) if case["gt_depth"] is not None else None
    for k in c:
        c[k] = c[k].detach().requires_grad_(grads and k[5:] in LV[stage])
    for p in dec.parameters():
        p.grad = None
        p.requires_grad_(grads)
    aux = {}
    d, u, col = renderer.render_batch_ray(c, dec, rd, ro, DEV, stage, gt_depth=gt, aux=aux)
    if grads:
        ((d * case["g_depth"].to(DEV)).sum() + (u * case["g_var"].to(DEV)).sum() + (col * case["g_rgb"].to(DEV)).sum()).backward()
    return d, u, col, aux, ro, rd


@pytest.mark.parametrize("layout", ["channels_last", "ncdhw"])
@pytest.mark.parametrize("path", RENDER_CASES, ids=[os.path.basename(p)[:-3] for p in RENDER_CASES])
def test_render_against_reference_fixture(path, layout):
    case, sc, grids, dec_state = load_case(path)
    stage, variant = case["stage"], case["variant"]
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV, channels_last=(layout == "channels_last"))
    d, u, col, aux, ro, rd = run_render(renderer, c, dec, case, stage)
    assert d.dtype == torch.float64 and u.dtype == torch.float64 and col.dtype == torch.float32
    # bit-exact sampling and voxel indices
    assert torch.equal(aux["z_vals"].cpu(), case["z_vals"])
    assert torch.equal(aux["corner_idx"].cpu().to(torch.int16), case["corner_idx"])
    assert rel(d, case["depth"]) < TOL and rel(u, case["var"]) < TOL
    if stage == "color":
        assert rel(col, case["rgb"]) < TOL
    assert rel(ro.grad, case["d_rays_o"]) < TOL and rel(rd.grad, case["d_rays_d"]) < TOL
    # dense grid gradients: fingerprints from the reference + the full tensor from the oracle run live
    bound = su.scene_bound(sc)
    o_grids = {k: v.clone().requires_grad_(k[5:] in LV[stage]) for k, v in grids.items()}
    o_ro, o_rd = case["rays_o"].clone().requires_grad_(True), case["rays_d"].clone().requires_grad_(True)
    od, ou, oc = tp.render_batch_ray(o_grids, dec_state, o_rd, o_ro, stage, case["gt_depth"], bound)
    ((od * case["g_depth"]).sum() + (ou * case["g_var"]).sum() + (oc * case["g_rgb"]).sum()).backward()
    for k, summ in case["d_grid"].items():
        g = c[k].grad
        assert g is not None, k
        assert rel(g.reshape(-1).cpu()[summ["idx"]], summ["val"]) < TOL, k
        assert abs(float(g.double().norm()) - summ["norm"]) < TOL * summ["norm"], k
        assert rel(g, o_grids[k].grad) < TOL and l2rel(g, o_grids[k].grad) < TOL, k
    for lvl, gd in case["d_dec"].items():
        tol = TOL_SATURATED if (variant == "init" and lvl in ("fine", "middle", "coarse")) else TOL
        mine = dict(getattr(dec, lvl + "_decoder").named_parameters())
        for k, v in gd.items():
            assert mine[k].grad is not None, (lvl, k)
            assert rel(mine[k].grad, v) < tol, (lvl, k, rel(mine[k].grad, v))


def test_tracker_iteration_against_real_tracker_capture():
    """camera_tensor.grad of one Tracker.optimize_cam_in_batch iteration (captured from the real Tracker on CPU)."""
    case = torch.load(os.path.join(su.GOLDEN, "tracker_color.pt"), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    renderer, c, dec = make_renderer(sc, su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"]), DEV)
    bound = su.scene_bound(sc)
    out = glue.tracking_iteration(sc, case, lambda rd, ro, stage, gd: renderer.render_batch_ray(c, dec, rd, ro, DEV, stage, gt_depth=gd),
                                  bound, device=DEV)
    assert torch.equal(out["rays_o"], case["rays_o"])
    assert rel(out["depth"], case["depth"]) < TOL
    assert abs(out["loss"] - case["loss"]) < TOL * abs(case["loss"])
    assert rel(out["d_camera"], case["d_camera"]) < TOL, (out["d_camera"], case["d_camera"])


@pytest.mark.parametrize("stage", ["coarse", "middle", "fine", "color"])
def test_mapper_iteration_against_real_mapper_capture(stage):
    """Masked voxel gradients + colour-decoder gradients of real Mapper.optimize_map iterations (captured on CPU)."""
    case = torch.load(os.path.join(su.GOLDEN, "mapper_%s.pt" % stage), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    renderer, c, dec = make_renderer(sc, su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"]), DEV)
    for k in c:
        c[k] = c[k].detach().requires_grad_(k[5:] in LV[stage])
    for n, p in dec.named_parameters():
        p.requires_grad_(stage == "color" and n.startswith("color_decoder"))
    gt = case["gt_depth"].to(DEV) if case["gt_depth"] is not None else None
    d, u, col = renderer.render_batch_ray(c, dec, case["rays_d"].to(DEV), case["rays_o"].to(DEV), DEV, stage, gt_depth=gt)
    assert rel(d, case["depth"]) < TOL and rel(u, case["var"]) < TOL
    loss = tp.mapping_loss(d, col, case["gt_depth_loss"].to(DEV), case["gt_color"].to(DEV), stage, sc["mapping"]["w_color_loss"])
    loss.backward()
    for k, summ in case["masked_grads"].items():
        dense = c[k].grad.cpu()
        m = case["masks"][k]
        masked = dense[m.unsqueeze(0).unsqueeze(0).expand_as(dense)]
        assert rel(masked.reshape(-1)[summ["idx"]], summ["val"]) < TOL, k
        assert abs(float(masked.double().norm()) - summ["norm"]) < TOL * summ["norm"], k
    mine = dict(dec.color_decoder.named_parameters())
    for k, v in case["d_color_decoder"].items():
        assert rel(mine[k].grad, v) < TOL, (k, rel(mine[k].grad, v))


@pytest.mark.parametrize("backend", [1])
def test_other_decoder_backends_match_the_default_one(backend):
    """mlp_backend 1 (FP32-FMA decoders, render_fwd_kernel / render_bwd_kernel) against the default tile kernels on one tracking and one
    colour-stage mapping iteration, in this process (the whole suite also runs under NSB_MLP_BACKEND=1 in tools/gpu_round.sh / gpu_final.sh;
    this keeps the other back-end inside the default `pytest -m gpu` run)."""
    from nice_slam_b200 import _lib
    from nice_slam_b200.steps import IterationContext
    L = _lib.lib()
    sc = su.load_scenes()["room0"]
    renderer, c, dec = make_renderer(sc, su.make_grids(sc, "soft"), su.load_decoders("soft"), DEV)
    n = 150
    ro, rd, gd, gc = su.make_rays(sc, n, seed=404)
    dirs = torch.randn(n, 3, generator=torch.Generator().manual_seed(3)).to(DEV)
    keys = ("grid_fine", "grid_color", "grid_middle")
    out = {}
    try:
        for b in (0, backend):
            assert L.nsb_set_option(b"mlp_backend", b) == 0
            t = IterationContext(renderer, n, "color", DEV, kind="track")
            t.run(c, dec, ro.to(DEV), rd.to(DEV), gd.to(DEV), gc.double().to(DEV), dirs=dirs)
            m = IterationContext(renderer, n, "color", DEV, kind="map", grad_grids=keys, grad_decoders=("color",))
            m.run(c, dec, ro.to(DEV), rd.to(DEV), gd.to(DEV), gc.float().to(DEV))
            torch.cuda.synchronize()
            out[b] = dict(z=t.z_vals.clone(), depth=t.depth.clone(), rgb=t.rgb.clone(), loss=float(t.loss), d_c2w=t.d_c2w.clone(),
                          rays=torch.cat([t.d_rays_o, t.d_rays_d], 1).clone(), mloss=float(m.loss), flat=m.d_flat["color"].clone(),
                          grid={k: m.d_grid[k].clone() for k in keys})
    finally:
        L.nsb_set_option(b"mlp_backend", 0)
    a, w = out[backend], out[0]
    assert torch.equal(a["z"], w["z"])
    assert rel(a["depth"], w["depth"]) < 2e-5 and rel(a["rgb"], w["rgb"]) < 2e-5
    assert abs(a["loss"] - w["loss"]) <= 2e-5 * abs(w["loss"]) and abs(a["mloss"] - w["mloss"]) <= 2e-5 * abs(w["mloss"])
    # (an L1 residual within ~1e-6 of zero flips the sign of that ray's gradient between two arithmetics: a knife edge of the loss, not an error)
    flipped = int(((a["rays"] - w["rays"]).abs().amax(dim=1) > 1e-4 * float(w["rays"].abs().max())).sum())
    assert flipped <= 1, flipped
    if flipped == 0:
        assert rel(a["d_c2w"], w["d_c2w"]) < 1e-4 and rel(a["flat"], w["flat"]) < 1e-4
        for k in keys:
            assert rel(a["grid"][k], w["grid"][k]) < 1e-4, k


def test_coarse_mapper_iteration_in_the_native_loop_against_real_mapper_capture():
    """The coarse mapper's joint iteration (Mapper.py:403-404,484: stage 'coarse', gt_depth=None for the renderer, sensor depth in the loss) through
    the native loop's pieces -- frustum-masked parameterisation of grid_coarse, fused mapping iteration with compact gradients, fused Adam -- against
    the real coarse Mapper.optimize_map capture (tests/golden/mapper_coarse.pt): rendered depth, the masked voxel gradient, and one Adam step."""
    from nice_slam_b200.mapping import FusedMappingLoop
    from nice_slam_b200.masked import MaskedVoxels
    case = torch.load(os.path.join(su.GOLDEN, "mapper_coarse.pt"), map_location="cpu", weights_only=False)
    assert case["coarse_mapper"] and case["gt_depth"] is None
    sc = su.load_scenes()[case["scene"]]
    renderer, c, dec = make_renderer(sc, su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"]), DEV)
    depth1, _ = su.make_frame(sc, 1)
    loop = FusedMappingLoop(renderer, c, dec, su.make_pose(sc, 1), depth1.to(DEV), keys=("grid_coarse",), w_color=sc["mapping"]["w_color_loss"])
    mask = case["masks"]["grid_coarse"].to(DEV)
    loop.masked["grid_coarse"] = MaskedVoxels(c["grid_coarse"], mask)          # the real mapper's selection (the on-GPU mask has its own test)
    before = c["grid_coarse"].detach().clone()
    ro, rd = case["rays_o"].to(DEV), case["rays_d"].to(DEV)
    loop.iteration("coarse", ro, rd, case["gt_depth_loss"].to(DEV), case["gt_color"].to(DEV), dict(decoders=0.0, coarse=0.001))
    torch.cuda.synchronize()
    ctx = loop._ctx["coarse"]
    n = ro.shape[0]
    assert ctx.z_vals.shape[1] == renderer.N_samples                 # no surface samples: the renderer got no depth
    assert rel(ctx.depth[:n], case["depth"]) < TOL and rel(ctx.var[:n], case["var"]) < TOL
    summ = case["masked_grads"]["grid_coarse"]
    got = ctx.d_grid["grid_coarse"][: int(mask.sum())].t().reshape(-1).cpu()     # the reference's val[mask] order is channel-major
    assert rel(got[summ["idx"]], summ["val"]) < TOL
    assert abs(float(got.double().norm()) - summ["norm"]) < TOL * summ["norm"]
    # first Adam step on the selected voxels only: -lr * sign-like update where the gradient is non-zero, everything else untouched
    delta = (c["grid_coarse"].detach() - before)
    sel = mask.unsqueeze(0).unsqueeze(0).expand_as(delta)
    assert int((delta[~sel] != 0).sum()) == 0                        # (the coarse selection is the whole grid, Mapper.py:113-116: nothing outside)
    g = ctx.d_grid["grid_coarse"][: int(mask.sum())].t().reshape(-1)
    want = -0.001 * g / (g.abs() + 1e-8)
    assert rel(delta[sel], want) < 1e-4


def test_eval_points_matches_oracle():
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    bound = su.scene_bound(sc)
    g = torch.Generator().manual_seed(5)
    lo, hi = bound[:, 0] - 0.3, bound[:, 1] + 0.3
    p = lo + (hi - lo) * torch.rand(3001, 3, generator=g, dtype=torch.float64)
    for stage in ("coarse", "middle", "fine", "color"):
        want = tp.eval_points(p, grids, dec_state, stage, bound)
        got = renderer.eval_points(p.to(DEV), dec, c, stage, DEV)
        assert rel(got, want) < TOL, stage
        assert torch.equal(got[:, 3].cpu() == 100, want[:, 3] == 100)


@pytest.mark.parametrize("n", [777, 200, 5000])      # radix-select median (> 512 residuals), direct rank counting, radix again
def test_seed_kernels_match_reference_losses(n):
    import ctypes as C
    from nice_slam_b200 import _lib
    L = _lib.lib()
    g = torch.Generator().manual_seed(9)
    depth = torch.rand(n, generator=g, dtype=torch.float64) * 3
    var = torch.rand(n, generator=g, dtype=torch.float64) * 0.1
    rgb = torch.rand(n, 3, generator=g)
    gt = torch.rand(n, generator=g) * 3
    gt[::13] = 0
    gt_rgb = torch.rand(n, 3, generator=g, dtype=torch.float64)
    # tracking
    d1 = depth.clone().requires_grad_(True); c1 = rgb.clone().requires_grad_(True)
    loss = tp.tracking_loss(d1, var, c1, gt, gt_rgb, 0.5)
    loss.backward()
    dev = lambda t: t.to(DEV)
    gD = torch.empty(n, dtype=torch.float64, device=DEV); gC = torch.empty(n, 3, device=DEV); lo = torch.empty(1, dtype=torch.float64, device=DEV)
    ws = torch.empty(L.nsb_tracking_seeds_workspace(n), dtype=torch.uint8, device=DEV)
    t = [dev(depth), dev(var), dev(rgb), dev(gt), dev(gt_rgb)]
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.nsb_tracking_seeds(*[C.c_void_p(x.data_ptr()) for x in t], n, 0.5, 1, 1, None, 0, C.c_void_p(gD.data_ptr()), C.c_void_p(gC.data_ptr()),
                                    C.c_void_p(lo.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(), st), "tracking_seeds")
    assert abs(float(lo) - float(loss)) < 1e-9 * abs(float(loss))
    assert rel(gD, d1.grad) < 1e-12 and rel(gC, c1.grad) < 1e-6
    # median over an external pool (the all-gathered residuals of a sharded batch): mask = r < 10 * median(pool)
    pool = torch.rand(1601, generator=g, dtype=torch.float64) * 2.0
    res = torch.abs(gt.double() - depth) / torch.sqrt(var + 1e-10)
    m = (res < 10 * pool.median()) & (gt > 0)
    want = res[m].sum() + 0.5 * torch.abs(gt_rgb - rgb.double())[m].sum()
    pool_d = dev(pool)
    _lib.check(L.nsb_tracking_seeds(*[C.c_void_p(x.data_ptr()) for x in t], n, 0.5, 1, 1, C.c_void_p(pool_d.data_ptr()), pool.numel(),
                                    C.c_void_p(gD.data_ptr()), C.c_void_p(gC.data_ptr()), C.c_void_p(lo.data_ptr()), C.c_void_p(ws.data_ptr()),
                                    ws.numel(), st), "tracking_seeds(pool)")
    assert float(want) > 0 and abs(float(lo) - float(want)) < 1e-9 * abs(float(want))
    # mapping
    d2 = depth.clone().requires_grad_(True); c2 = rgb.clone().requires_grad_(True)
    loss2 = tp.mapping_loss(d2, c2, gt, gt_rgb.float(), "color", 0.2)
    loss2.backward()
    t2 = [dev(depth), dev(rgb), dev(gt), dev(gt_rgb.float())]
    _lib.check(L.nsb_mapping_seeds(*[C.c_void_p(x.data_ptr()) for x in t2], n, 0.2, 1, C.c_void_p(gD.data_ptr()), C.c_void_p(gC.data_ptr()),
                                   C.c_void_p(lo.data_ptr()), st), "mapping_seeds")
    assert abs(float(lo) - float(loss2)) < 1e-6 * abs(float(loss2))
    assert rel(gD, d2.grad) < 1e-12 and rel(gC, c2.grad) < 1e-6


def test_prefilter_and_batch_max():
    import ctypes as C
    from nice_slam_b200 import _lib
    L = _lib.lib()
    sc = su.load_scenes()["room0"]
    bound = su.scene_bound(sc)
    ro, rd, gd, _ = su.make_rays(sc, 5000, seed=1)
    keep = tp.bbox_prefilter(ro, rd, gd, bound)
    k = torch.empty(5000, dtype=torch.uint8, device=DEV)
    b6 = (C.c_double * 6)(*bound.reshape(6).tolist())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ro_d, rd_d, gd_d = ro.to(DEV), rd.to(DEV), gd.to(DEV)
    _lib.check(L.nsb_bbox_prefilter(C.c_void_p(ro_d.data_ptr()), C.c_void_p(rd_d.data_ptr()), C.c_void_p(gd_d.data_ptr()), 5000, b6,
                                    C.c_void_p(k.data_ptr()), st), "prefilter")
    assert torch.equal(k.cpu().bool(), keep)
    out = torch.empty(2, device=DEV)
    _lib.check(L.nsb_batch_max_depth(C.c_void_p(gd_d.data_ptr()), 5000, C.c_void_p(out.data_ptr()), st), "batch_max")
    assert float(out[0]) == float(torch.max(gd)) and float(out[1]) == float(torch.max(gd * 1.2))


# ------------------------------------------------------------------------------------ edge cases & properties
# (4, 2, 37): S = 6 is below the tile kernels' minimum of 8 samples per ray and runs on the FP32-FMA kernels
@pytest.mark.parametrize("n_samples,n_surface,n_rays", [(5, 3, 37), (4, 2, 37), (32, 16, 1), (16, 16, 333), (80, 16, 50), (32, 0, 64)])
def test_ragged_shapes_against_oracle(n_samples, n_surface, n_rays):
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV, n_samples=n_samples, n_surface=n_surface)
    bound = su.scene_bound(sc)
    ro, rd, gd, gc = su.make_rays(sc, n_rays, seed=n_rays)
    gd[::5] = 0                                    # zero-depth branch of the surface sampler (Renderer.py:143-150)
    out = tp.iteration("map", grids, dec_state, ro, rd, gd, gc.float(), "color", bound, n_samples, n_surface,
                       grad_grids=("grid_fine", "grid_color", "grid_middle"), grad_decoders=("color",))
    for k in c:
        c[k] = c[k].detach().requires_grad_(k != "grid_coarse")
    for n, p in dec.named_parameters():
        p.requires_grad_(n.startswith("color_decoder"))
    r1, r2 = ro.to(DEV).requires_grad_(True), rd.to(DEV).requires_grad_(True)
    aux = {}
    d, u, col = renderer.render_batch_ray(c, dec, r2, r1, DEV, "color", gt_depth=gd.to(DEV), aux=aux)
    z = tp.sample_z_vals(ro, rd, gd, bound, n_samples, n_surface, "color")
    assert torch.equal(aux["z_vals"].cpu(), z)
    tp.mapping_loss(d, col, gd.to(DEV), gc.float().to(DEV), "color").backward()
    assert rel(d, out["depth"]) < TOL and rel(col, out["color"]) < TOL and rel(u, out["var"]) < TOL
    assert rel(r1.grad, out["d_rays_o"]) < TOL and rel(r2.grad, out["d_rays_d"]) < TOL
    for k in ("grid_fine", "grid_color", "grid_middle"):
        assert rel(c[k].grad, out["d_" + k]) < TOL, k
    mine = dict(dec.color_decoder.named_parameters())
    for k, v in out["d_dec"]["color"].items():
        assert rel(mine[k].grad, v) < TOL, k


def test_all_rays_outside_bound_and_zero_depth():
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    bound = su.scene_bound(sc)
    ro, rd, gd, _ = su.make_rays(sc, 64, seed=2)
    ro = ro + 100.0                  # every sample out of bound -> occ logit 100 -> alpha 1 at the first sample
    gd = torch.zeros_like(gd)        # no sensor depth anywhere
    want = tp.render_batch_ray(grids, dec_state, rd, ro, "color", gd, bound)
    got = renderer.render_batch_ray(c, dec, rd.to(DEV), ro.to(DEV), DEV, "color", gt_depth=gd.to(DEV))
    for a, b in zip(got, want):
        assert torch.allclose(a.cpu().double(), b.double(), rtol=1e-4, atol=1e-7)


def test_large_batch_properties():
    """BASELINE sweep size (65536 rays x 48): size-independent properties instead of an oracle run."""
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    n = 65536
    ro, rd, gd, gc = su.make_rays(sc, n, seed=77)
    ro, rd, gd = ro.to(DEV), rd.to(DEV), gd.to(DEV)
    aux = {}
    d, u, col = renderer.render_batch_ray(c, dec, rd, ro, DEV, "color", gt_depth=gd, aux=aux)
    z = aux["z_vals"]
    assert bool((z[:, 1:] >= z[:, :-1]).all())                       # sortedness
    assert bool(torch.isfinite(d).all() and torch.isfinite(col).all() and (u >= 0).all())
    # permutation equivariance + split invariance (same batch-global depth max in both halves by construction)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(1)).to(DEV)
    imax = int(torch.argmax(gd))
    d2, u2, col2 = renderer.render_batch_ray(c, dec, rd[perm], ro[perm], DEV, "color", gt_depth=gd[perm])
    assert torch.equal(d2, d[perm]) and torch.equal(col2, col[perm]) and torch.equal(u2, u[perm])
    half = torch.cat([torch.arange(0, n // 2, device=DEV), torch.tensor([imax], device=DEV)])
    d3, _, col3 = renderer.render_batch_ray(c, dec, rd[half], ro[half], DEV, "color", gt_depth=gd[half])
    assert torch.equal(d3[:-1], d[: n // 2]) and torch.equal(col3[:-1], col[: n // 2])
    # linearity of the backward pass in the output seeds
    sub = slice(0, 4096)
    r1 = ro[sub].clone().requires_grad_(True); r2 = rd[sub].clone().requires_grad_(True)
    dd, uu, cc = renderer.render_batch_ray(c, dec, r2, r1, DEV, "color", gt_depth=gd[sub])
    g = torch.Generator(device=DEV).manual_seed(3)
    s1 = torch.randn(4096, dtype=torch.float64, device=DEV, generator=g); s2 = torch.randn(4096, 3, device=DEV, generator=g)
    ga = torch.autograd.grad((dd * s1).sum(), (r1, r2), retain_graph=True)
    gb = torch.autograd.grad((cc * s2).sum(), (r1, r2), retain_graph=True)
    gab = torch.autograd.grad((dd * s1).sum() + (cc * s2).sum(), (r1, r2))
    for x, y, zz in zip(ga, gb, gab):
        assert rel(x + y, zz) < 1e-5


# ------------------------------------------------------------------------------------ fused iterations (what bench.py times)
def _flat_named(level, flat):
    from nice_slam_b200 import _lib
    return {nm: flat[off:off + cnt] for nm, off, cnt in _lib.flat_layout(level)}


@pytest.mark.parametrize("n_rays", [200, 37])
def test_fused_tracking_iteration_matches_oracle(n_rays):
    """nsb_tracking_iteration (one C call: batch max, forward, median-gated loss seeds, backward) + nsb_pose_grad, eager,
    replayed from a CUDA graph, and through the split-phase sharded iteration at world size 1."""
    from nice_slam_b200.dist import ShardedTrackingIteration
    from nice_slam_b200.steps import IterationContext
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    bound = su.scene_bound(sc)
    ro, rd, gd, gc = su.make_rays(sc, n_rays, seed=5 + n_rays)
    out = tp.iteration("track", grids, dec_state, ro, rd, gd, gc.double(), "color", bound)
    dirs = torch.randn(n_rays, 3, generator=torch.Generator().manual_seed(1))
    want_pose = torch.cat([(out["d_rays_d"].double()[:, :, None] * dirs.double()[:, None, :]).sum(0),
                           out["d_rays_o"].double().sum(0)[:, None]], 1)             # d c2w[:3,:3] | d c2w[:3,3]
    ctx = IterationContext(renderer, n_rays, "color", DEV, kind="track")
    dev_in = [t.to(DEV) for t in (ro, rd, gd, gc.double())]
    dirs_d = dirs.to(DEV)

    def check(loss, d_o, d_d, pose):
        assert abs(float(loss) - float(out["loss"])) < TOL * abs(float(out["loss"]))
        assert rel(d_o, out["d_rays_o"]) < TOL and rel(d_d, out["d_rays_d"]) < TOL
        assert rel(pose, want_pose) < TOL

    ctx.run(c, dec, *dev_in)
    check(ctx.loss, ctx.d_rays_o, ctx.d_rays_d, ctx.pose_grad(dirs_d))
    assert rel(ctx.depth, out["depth"]) < TOL and rel(ctx.rgb, out["color"]) < TOL and rel(ctx.var, out["var"]) < TOL
    # CUDA graph replay (device inputs, then pinned-host inputs)
    ctx.load_device_inputs(*dev_in)
    g = ctx.build_graph(c, dec, dirs=dirs_d)
    ctx.loss.zero_(); ctx.d_out.zero_(); ctx.d_c2w.zero_()
    g.replay(); torch.cuda.synchronize()
    check(ctx.loss, ctx.d_rays_o, ctx.d_rays_d, ctx.d_c2w)
    ctx.stage_host_inputs(ro, rd, gd, gc.double())
    loss, d_rays = ctx.run_host(c, dec)
    check(loss, d_rays[0], d_rays[1], ctx.pose_grad(dirs_d))
    # the end-to-end graph forms: copy-engine transfers, nsb_copy_block kernels and the backward's own store deliver the same result block to pinned host memory
    blocks = []
    for mode in (True, "sm", "sm_push"):
        ge = ctx.build_graph(c, dec, dirs=dirs_d, host_io=mode)
        ctx.d_in.zero_(); ctx.h_res.zero_()
        ge.replay(); torch.cuda.synchronize()
        check(ctx.h_loss[0], ctx.h_out.view(2, n_rays, 3)[0], ctx.h_out.view(2, n_rays, 3)[1], ctx.h_pose)
        blocks.append(ctx.h_res.clone())
    assert torch.equal(blocks[0], blocks[1]) and torch.equal(blocks[0], blocks[2])
    # split-phase sharded iteration without a process group == the fused one
    sh = ShardedTrackingIteration(ctx)
    packed = sh.run(c, dec, *dev_in[:2], dirs_d, *dev_in[2:]).clone()
    check(packed[0], ctx.d_rays_o, ctx.d_rays_d, packed[1:].view(3, 4))
    gs = sh.build_graph()
    assert gs is not None
    sh.packed.zero_()
    gs.replay(); torch.cuda.synchronize()
    check(sh.packed[0], ctx.d_rays_o, ctx.d_rays_d, sh.packed[1:].view(3, 4))


@pytest.mark.parametrize("stage", ["middle", "color"])
def test_fused_mapping_iteration_matches_oracle(stage):
    """nsb_mapping_iteration: dense voxel gradients of the stage's grids + (stage color) colour-decoder gradients."""
    from nice_slam_b200.steps import IterationContext
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    bound = su.scene_bound(sc)
    n_rays = 300
    ro, rd, gd, gc = su.make_rays(sc, n_rays, seed=99)
    gg = tuple("grid_" + l for l in LV[stage])
    gdec = ("color",) if stage == "color" else ()
    out = tp.iteration("map", grids, dec_state, ro, rd, gd, gc.float(), stage, bound, grad_grids=gg, grad_decoders=gdec)
    ctx = IterationContext(renderer, n_rays, stage, DEV, kind="map", grad_grids=gg, grad_decoders=gdec)
    for rep in range(2):                            # second run: the accumulation buffers are re-zeroed
        ctx.run(c, dec, ro.to(DEV), rd.to(DEV), gd.to(DEV), gc.float().to(DEV))
    assert abs(float(ctx.loss) - float(out["loss"])) < TOL * abs(float(out["loss"]))
    assert rel(ctx.d_rays_o, out["d_rays_o"]) < TOL and rel(ctx.d_rays_d, out["d_rays_d"]) < TOL
    for k in gg:
        assert rel(ctx.d_grid[k], out["d_" + k]) < TOL, k
    for lvl in gdec:
        from nice_slam_b200._lib import LEVELS
        mine = _flat_named(LEVELS.index(lvl), ctx.d_flat[lvl])
        for k, v in out["d_dec"][lvl].items():
            if k in mine:
                assert rel(mine[k], v.reshape(-1)) < TOL, (lvl, k)


# ------------------------------------------------------------------------------------ masked voxel parameterisation (Mapper.py:317-333)
def _random_masks(grids, keys, frac=0.5, seed=11):
    g = torch.Generator().manual_seed(seed)
    return {k: torch.rand(grids[k].shape[2:], generator=g) < frac for k in keys}


@pytest.mark.parametrize("layout", ["channels_last", "ncdhw"])
def test_masked_voxels_gather_scatter_match_reference_indexing(layout):
    """val_grad = val[mask] (Mapper.py:324) and val[mask] = val_grad (:399, :517) with the reference's repeated [1,32,D,H,W] mask."""
    from nice_slam_b200.masked import MaskedVoxels
    sc = su.load_scenes()["room0"]
    grids = su.make_grids(sc, "soft")
    renderer, c, dec = make_renderer(sc, grids, su.load_decoders("soft"), DEV, channels_last=(layout == "channels_last"))
    for key, vm in _random_masks(grids, ("grid_middle", "grid_color")).items():
        val = c[key]
        mask5 = vm.to(DEV).unsqueeze(0).unsqueeze(0).repeat(1, 32, 1, 1, 1)          # Mapper.py:319-320
        mv = MaskedVoxels(val, mask5)
        assert mv.count == int(vm.sum())
        slots = mv.slot_map.view(vm.shape).cpu()
        assert torch.equal(slots >= 0, vm) and torch.equal(slots[vm], torch.arange(mv.count, dtype=torch.int32))
        compact = mv.gather(val)
        assert torch.equal(mv.to_reference(compact), val[mask5])
        assert torch.equal(mv.from_reference(val[mask5]), compact)
        new = torch.randn(mv.count, 32, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
        want = val.clone()
        want[mask5] = mv.to_reference(new)
        mv.scatter(val, new)
        assert torch.equal(val, want)
    empty = MaskedVoxels(c["grid_middle"], torch.zeros(grids["grid_middle"].shape[2:], dtype=torch.bool))
    assert empty.count == 0 and bool((empty.slot_map == -1).all())


@pytest.mark.parametrize("backend_decoder_grads", [False, True])
def test_masked_mapping_iteration_packed_block(backend_decoder_grads):
    """Compact voxel gradients == the dense ones restricted to the mask; the packed block [loss | keyframe pose grads | decoder grads |
    voxel grads]; the sharded mapping iteration (world size 1) and its CUDA graph give the same block."""
    from nice_slam_b200._lib import LEVELS
    from nice_slam_b200.dist import ShardedMappingIteration
    from nice_slam_b200.masked import MaskedVoxels
    from nice_slam_b200.steps import IterationContext
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    n_rays, n_frames = 330, 3
    ro, rd, gd, gc = su.make_rays(sc, n_rays, seed=123)
    dev_in = [t.to(DEV) for t in (ro, rd, gd, gc.float())]
    dirs = torch.randn(n_rays, 3, generator=torch.Generator().manual_seed(7)).to(DEV)
    offs = torch.tensor([0, 100, 230, 330], dtype=torch.int32, device=DEV)
    keys = ("grid_fine", "grid_color", "grid_middle")
    gdec = ("color",) if backend_decoder_grads else ()           # decoder grads -> FP32-FMA backward kernel, none -> tensor-core kernel
    masks = _random_masks(grids, keys, 0.6)
    dense = IterationContext(renderer, n_rays, "color", DEV, kind="map", grad_grids=keys, grad_decoders=gdec)
    dense.run(c, dec, *dev_in)
    mv = {k: MaskedVoxels(c[k], masks[k]) for k in keys}
    ctx = IterationContext(renderer, n_rays, "color", DEV, kind="map", grad_grids=keys, grad_decoders=gdec, masked=mv, n_frames=n_frames)
    for rep in range(2):
        ctx.run(c, dec, *dev_in)
    packed = ctx.finish_packed(dirs, offs).clone()
    assert abs(float(packed[0]) - float(dense.loss)) < 1e-6 * abs(float(dense.loss))
    for k in keys:
        want = dense.d_grid[k][masks[k].to(DEV).unsqueeze(0).unsqueeze(0).expand_as(dense.d_grid[k])]
        assert float(want.abs().max()) > 0
        assert rel(mv[k].to_reference(ctx.d_grid[k]), want) < 1e-5, k
        o, cnt = ctx.sections[k]
        assert torch.equal(packed[o:o + cnt].view(-1, 32), ctx.d_grid[k])
    for lvl in gdec:
        assert rel(ctx.d_flat[lvl], dense.d_flat[lvl]) < 1e-5
    for f in range(n_frames):
        lo, hi = int(offs[f]), int(offs[f + 1])
        want = torch.cat([ctx.d_rays_d[lo:hi].double().t() @ dirs[lo:hi].double(), ctx.d_rays_o[lo:hi].double().sum(0, keepdim=True).t()], 1)
        assert rel(ctx.d_frames[f].view(3, 4), want) < 1e-5
    # split-phase sharded iteration, no process group: same block; then replayed from a CUDA graph
    ctx.load_device_inputs(*dev_in)
    sh = ShardedMappingIteration(ctx)
    sh.prepare(c, dec, dirs, offs)
    got = sh.enqueue().clone()
    assert rel(got, packed) < 1e-5
    g = sh.build_graph()
    assert g is not None
    ctx.packed.fill_(7.0)
    g.replay(); torch.cuda.synchronize()
    assert rel(ctx.packed, packed) < 1e-5


# ------------------------------------------------------------------------------------ more edge cases
@pytest.mark.parametrize("stage,n_rays", [("color", 200), ("middle", 333), ("color", 1500)])
def test_fp16_split_forward_matches_3xtf32_forward(stage, n_rays):
    """Option fwd_f16: the forward's decoder GEMMs with FP16 hi | lo operands (tcgen05 kind::f16, K = 16 per instruction; nsb_tile.cuh mma_unit_h)
    against the default 3xTF32 forward on the same inputs -- raw decoder outputs, rendered depth / colour, loss and the gradients that the
    (unchanged, 3xTF32) backward derives from them.  Both sit ~1e-6 from the FP32 reference; the path's tolerance is 1e-4 (north_star)."""
    from nice_slam_b200 import _lib
    from nice_slam_b200.steps import IterationContext
    L = _lib.lib()
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    ro, rd, gd, gc = su.make_rays(sc, n_rays, seed=77 + n_rays)
    dev_in = [t.to(DEV) for t in (ro, rd, gd, gc.float())]
    keys = ("grid_fine", "grid_color", "grid_middle") if stage == "color" else ("grid_middle",)
    out = {}
    try:
        for mode in (1, 0):
            assert L.nsb_set_option(b"fwd_f16", mode) == 0
            ctx = IterationContext(renderer, n_rays, stage, DEV, kind="map", grad_grids=keys)
            for _ in range(2):
                ctx.run(c, dec, *dev_in)
            torch.cuda.synchronize()
            out[mode] = dict(raw=ctx.raw.clone(), depth=ctx.depth.clone(), rgb=ctx.rgb.clone(), loss=float(ctx.loss), z=ctx.z_vals.clone(),
                             d_o=ctx.d_rays_o.clone(), grid={k: ctx.d_grid[k].clone() for k in keys})
    finally:
        L.nsb_set_option(b"fwd_f16", 0)
    a, b = out[1], out[0]
    assert torch.equal(a["z"], b["z"])                                # sampling does not depend on the decoder arithmetic
    assert torch.isfinite(a["raw"]).all()
    assert float((a["raw"] - b["raw"]).abs().max()) > 0               # the option took effect (another arithmetic, not the same kernel)
    assert rel(a["raw"], b["raw"]) < 1e-5
    assert rel(a["depth"], b["depth"]) < 1e-5 and rel(a["rgb"], b["rgb"]) < 1e-5
    assert abs(a["loss"] - b["loss"]) <= 1e-5 * abs(b["loss"])
    # gradients: the L1 losses make a ray whose residual sits within ~1e-6 of zero flip the sign of its whole gradient between two arithmetics
    # (a knife edge of the loss, not an error): allow a couple of such rays, everything else must agree
    scale = float(b["d_o"].abs().max())
    flipped = int(((a["d_o"] - b["d_o"]).abs().amax(dim=1) > 1e-4 * scale).sum())
    assert flipped <= max(2, n_rays // 500), flipped
    for k in keys:
        if flipped == 0:
            assert rel(a["grid"][k], b["grid"][k]) < 1e-4, k
        else:
            assert l2rel(a["grid"][k], b["grid"][k]) < 0.1 * flipped, k


@pytest.mark.parametrize("n_rays", [96, 437, 1200])
def test_tensor_core_weight_gradients_match_fp32_pass_and_oracle(n_rays):
    """Colour-decoder weight gradients of a mapping iteration (src/Mapper.py:339-341,503): the tensor-core contraction over the points of a tile
    (render_bwd_wg_tile_kernel, layer outputs kept by the forward) against the FP32-FMA pass that recomputes the forward (option wgrad_tc = 0)
    and against the oracle; ragged last tile (n_rays * 48 is not a multiple of 128) and more tiles than SMs included."""
    from nice_slam_b200 import _lib
    from nice_slam_b200.steps import IterationContext
    L = _lib.lib()
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    ro, rd, gd, gc = su.make_rays(sc, n_rays, seed=31 + n_rays)
    dev_in = [t.to(DEV) for t in (ro, rd, gd, gc.float())]
    keys = ("grid_fine", "grid_color", "grid_middle")
    out = {}
    try:
        for mode in (1, 0):
            assert L.nsb_set_option(b"wgrad_tc", mode) == 0
            ctx = IterationContext(renderer, n_rays, "color", DEV, kind="map", grad_grids=keys, grad_decoders=("color",))
            for _ in range(2):                                        # twice: accumulation buffers are re-zeroed per run
                ctx.run(c, dec, *dev_in)
            torch.cuda.synchronize()
            out[mode] = dict(flat=ctx.d_flat["color"].clone(), d_o=ctx.d_rays_o.clone(), d_d=ctx.d_rays_d.clone(), loss=float(ctx.loss),
                             grid={k: ctx.d_grid[k].clone() for k in keys})
    finally:
        L.nsb_set_option(b"wgrad_tc", 1)
    a, b = out[1], out[0]
    assert abs(a["loss"] - b["loss"]) <= 1e-9 * abs(b["loss"])
    assert float(b["flat"].abs().max()) > 0
    lay = {nm: (off, cnt) for nm, off, cnt in _lib.flat_layout(_lib.LEVELS.index("color"))}
    for nm, (off, cnt) in lay.items():                               # every parameter tensor on its own scale (weights, biases, embedding matrix)
        assert rel(a["flat"][off:off + cnt], b["flat"][off:off + cnt]) < 2e-5, nm
    assert rel(a["d_o"], b["d_o"]) < 5e-5 and rel(a["d_d"], b["d_d"]) < 5e-5      # (the colour decoder's share is summed in another order)
    for k in keys:
        assert rel(a["grid"][k], b["grid"][k]) < 1e-5, k
    if n_rays <= 437:                                                # oracle (CPU autograd) on the smaller batches
        bound = su.scene_bound(sc)
        want = tp.iteration("map", grids, dec_state, ro, rd, gd, gc.float(), "color", bound, grad_grids=keys, grad_decoders=("color",))
        flat = a["flat"].cpu()
        for nm, v in want["d_dec"]["color"].items():
            off, cnt = lay[nm]
            assert rel(flat[off:off + cnt].view(v.shape), v) < 1e-4, nm


def test_unmodified_mapper_indexing_gets_compact_gradients():
    """The reference mapper's own parameterisation at the renderer boundary (src/Mapper.py:317-333,393-401): `val_grad = Variable(val[mask])`,
    then every iteration `val[mask] = val_grad; c[key] = val`.  FusedRenderer recognises the index_put and differentiates with respect to val_grad
    directly (compact gradients, no dense zero-fill); the result equals the generic dense autograd path (detection switched off) and the oracle."""
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c0, dec = make_renderer(sc, grids, dec_state, DEV)
    n = 160
    ro, rd, gd, gc = [t.to(DEV) for t in su.make_rays(sc, n, seed=77)]
    keys = ("grid_middle", "grid_fine", "grid_color")
    masks = _random_masks(grids, keys, 0.5)
    for p in dec.parameters():
        p.requires_grad_(False)
    got = {}
    for detect in (True, False):
        renderer.detect_masked_grids = detect
        c, leaves = {}, {}
        for k, v in c0.items():
            val = v.detach().clone(memory_format=torch.preserve_format)
            if k in keys:
                mask = masks[k].to(DEV).unsqueeze(0).unsqueeze(0).repeat(1, val.shape[1], 1, 1, 1)      # Mapper.py:319-320
                val_grad = val[mask].clone().requires_grad_(True)                                      # :321-325
                val[mask] = val_grad                                                                   # :399
                leaves[k] = val_grad
            c[k] = val
        d, u, col = renderer.render_batch_ray(c, dec, rd, ro, DEV, "color", gt_depth=gd)
        loss = torch.abs(gd - d)[gd > 0].sum() + 0.2 * torch.abs(gc.float() - col).sum()               # :487-493
        loss.backward()
        got[detect] = dict(loss=float(loss), grads={k: leaves[k].grad.clone() for k in keys})
    renderer.detect_masked_grids = True
    assert len(renderer._mask_cache) == 3 and all(v is not False for v in renderer._mask_cache.values())        # the pattern WAS recognised
    assert abs(got[True]["loss"] - got[False]["loss"]) <= 1e-12 * abs(got[False]["loss"])
    for k in keys:
        a, b = got[True]["grads"][k], got[False]["grads"][k]
        assert a.shape == b.shape and float(b.abs().max()) > 0
        assert rel(a, b) < 1e-5, k
    # oracle: dense CPU autograd restricted to the mask
    want = tp.iteration("map", grids, dec_state, ro.cpu(), rd.cpu(), gd.cpu(), gc.float().cpu(), "color", su.scene_bound(sc), grad_grids=keys, grad_decoders=())
    for k in keys:
        m = masks[k].unsqueeze(0).unsqueeze(0).expand_as(grids[k])
        assert rel(got[True]["grads"][k], want["d_" + k][m]) < 1e-4, k


def test_render_img_matches_oracle_per_ray_batch():
    """Renderer.render_img (Renderer.py:200-255): full image in ray_batch_size chunks; the batch-global depth maxima are per chunk,
    exactly as in the reference."""
    from types import SimpleNamespace
    from gpu_util import make_cfg
    from nice_slam_b200.decoders import NICEDecoders
    from nice_slam_b200.renderer import FusedRenderer
    sc = dict(su.load_scenes()["room0"])
    H, W = 12, 20
    cam = dict(sc["cam"]); cam.update(H=H, W=W, fx=15.0, fy=15.0, cx=9.5, cy=5.5)
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    c = {k: v.to(DEV) for k, v in grids.items()}
    slam = SimpleNamespace(nice=True, bound=su.scene_bound(sc), shared_c=c, H=H, W=W, fx=cam["fx"], fy=cam["fy"], cx=cam["cx"], cy=cam["cy"])
    r = FusedRenderer(make_cfg(sc), SimpleNamespace(nice=True), slam, ray_batch_size=100)
    dec = NICEDecoders.from_state(dec_state, DEV)
    c2w = su.make_pose(sc, 4)
    g = torch.Generator().manual_seed(12)
    gt = torch.rand(H, W, generator=g) * 3 + 0.5
    gt[2, 3] = 0
    d, u, col = r.render_img(slam.shared_c, dec, c2w.to(DEV), DEV, "color", gt_depth=gt.to(DEV))
    assert d.shape == (H, W) and u.shape == (H, W) and col.shape == (H, W, 3)
    # oracle: same rays (get_rays, common.py:248-266), same chunking
    i, j = torch.meshgrid(torch.linspace(0, W - 1, W), torch.linspace(0, H - 1, H), indexing="ij")
    i, j = i.t(), j.t()
    dirs = torch.stack([(i - cam["cx"]) / cam["fx"], -(j - cam["cy"]) / cam["fy"], -torch.ones_like(i)], -1)
    rd = torch.sum(dirs.reshape(H, W, 1, 3) * c2w[:3, :3], -1).reshape(-1, 3)
    ro = c2w[:3, -1].expand(rd.shape)
    bound = su.scene_bound(sc)
    wd, wu, wc = [], [], []
    for s in range(0, H * W, 100):
        a, b_, cc = tp.render_batch_ray(grids, dec_state, rd[s:s + 100], ro[s:s + 100], "color", gt.reshape(-1)[s:s + 100], bound)
        wd.append(a); wu.append(b_); wc.append(cc)
    assert rel(d.reshape(-1), torch.cat(wd)) < TOL and rel(u.reshape(-1), torch.cat(wu)) < TOL and rel(col.reshape(-1, 3), torch.cat(wc)) < TOL


def test_empty_batch_and_sample_count_limits():
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    z3 = torch.zeros(0, 3, device=DEV)
    d, u, col = renderer.render_batch_ray(c, dec, z3.clone().requires_grad_(True), z3.clone().requires_grad_(True), DEV, "color",
                                          gt_depth=torch.zeros(0, device=DEV))
    assert d.shape == (0,) and u.shape == (0,) and col.shape == (0, 3)
    (d.sum() + col.sum()).backward()                                   # empty backward is a no-op, not an error
    # the largest supported sample count (256 per ray) against the oracle; one more raises
    bound = su.scene_bound(sc)
    ro, rd, gd, _ = su.make_rays(sc, 9, seed=8)
    r2, c2, dec2 = make_renderer(sc, grids, dec_state, DEV, n_samples=240, n_surface=16)
    want = tp.render_batch_ray(grids, dec_state, rd, ro, "color", gd, bound, 240, 16)
    got = r2.render_batch_ray(c2, dec2, rd.to(DEV), ro.to(DEV), DEV, "color", gt_depth=gd.to(DEV))
    for a, b in zip(got, want):
        assert rel(a, b) < TOL
    r3, c3, dec3 = make_renderer(sc, grids, dec_state, DEV, n_samples=241, n_surface=16)
    with pytest.raises(RuntimeError, match="exceeds"):
        r3.render_batch_ray(c3, dec3, rd.to(DEV), ro.to(DEV), DEV, "color", gt_depth=gd.to(DEV))


@pytest.mark.parametrize("scene", ["scene0000", "apartment"])
def test_other_scene_volumes_against_oracle(scene):
    """ScanNet scene0000 / Apartment bounds and grid shapes (SURVEY.md section 8 table): forward + backward of a small batch."""
    sc = su.load_scenes()[scene]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    bound = su.scene_bound(sc)
    ro, rd, gd, gc = su.make_rays(sc, 40, seed=17)
    out = tp.iteration("track", grids, dec_state, ro, rd, gd, gc.double(), "color", bound)
    r1, r2 = ro.to(DEV).requires_grad_(True), rd.to(DEV).requires_grad_(True)
    aux = {}
    d, u, col = renderer.render_batch_ray(c, dec, r2, r1, DEV, "color", gt_depth=gd.to(DEV), aux=aux)
    assert torch.equal(aux["z_vals"].cpu(), tp.sample_z_vals(ro, rd, gd, bound, 32, 16, "color"))
    tp.tracking_loss(d, u, col, gd.to(DEV), gc.double().to(DEV)).backward()
    assert rel(d, out["depth"]) < TOL and rel(col, out["color"]) < TOL and rel(u, out["var"]) < TOL
    assert rel(r1.grad, out["d_rays_o"]) < TOL and rel(r2.grad, out["d_rays_d"]) < TOL


def test_frustum_mask_matches_real_mapper_masks():
    """nsb_frustum_mask against the masks of the real Mapper.get_mask_from_c2w (tests/golden/mapper_*.pt); a voxel may differ only if it
    sits on a decision boundary (the oracle reports how far every voxel is from each threshold)."""
    import numpy as np
    from oracle import frustum as fr
    from nice_slam_b200.masked import MaskedVoxels, frustum_voxel_mask
    sc = su.load_scenes()["room0"]
    case = torch.load(os.path.join(su.GOLDEN, "mapper_color.pt"), map_location="cpu", weights_only=False)
    depth, _ = su.make_frame(sc, case["frame_seed"])
    c2w = su.make_pose(sc, 1)
    renderer, c, dec = make_renderer(sc, su.make_grids(sc, "soft"), su.load_decoders("soft"), DEV)
    bound = su.scene_bound(sc)
    for key, want in case["masks"].items():
        got = frustum_voxel_mask(renderer, c2w, key, c[key], depth.to(DEV)).cpu()
        diff = got != want
        if bool(diff.any()):
            mg = {}
            fr.frustum_mask(c2w, key, tuple(want.shape), depth.numpy(), bound, sc["cam"], margins=mg)
            W_, H_, D_ = want.shape[2], want.shape[1], want.shape[0]
            near = np.minimum.reduce([mg["uv"], mg["z"], mg["ball"]]).reshape(W_, H_, D_).transpose(2, 1, 0)
            assert float(near[diff.numpy()].max()) < 1e-4, (key, int(diff.sum()))
        assert int(diff.sum()) <= 2, (key, int(diff.sum()))
        assert MaskedVoxels(c[key], got.to(DEV)).count == int(got.sum())


def test_fused_adam_matches_torch_adam():
    """nsb_adam_masked_voxels / nsb_adam_decoder against torch.optim.Adam on the reference's parameterisation (val_grad = val[mask] as a
    leaf, the colour decoder's parameters), three steps with changing gradients and learning rates (Mapper.py:365-379, :412-419, :504)."""
    from nice_slam_b200._lib import LEVELS, flat_layout
    from nice_slam_b200.masked import MaskedVoxels
    from nice_slam_b200.optim import FusedMapperAdam
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    key = "grid_middle"
    vm = _random_masks(grids, (key,), 0.4)[key]
    mv = MaskedVoxels(c[key], vm)
    mask5 = vm.to(DEV).unsqueeze(0).unsqueeze(0).repeat(1, 32, 1, 1, 1)
    # reference side: leaf parameter vectors + torch Adam
    val_ref = c[key].clone()
    val_grad = val_ref[mask5].clone().requires_grad_(True)
    dec_ref = {k: v.detach().clone().requires_grad_(True) for k, v in dict(dec.color_decoder.named_parameters()).items()}
    opt = torch.optim.Adam([{"params": [val_grad], "lr": 0.0}, {"params": list(dec_ref.values()), "lr": 0.0}])
    fused = FusedMapperAdam()
    lay = flat_layout(LEVELS.index("color"))
    n_flat = sum(cnt for _, _, cnt in lay)
    g = torch.Generator(device=DEV).manual_seed(4)
    for step, (lr_v, lr_d) in enumerate([(0.1, 0.005), (0.005, 0.005), (0.005, 0.0)]):
        gv = torch.randn(mv.count, 32, device=DEV, generator=g) * (10.0 ** (-step))
        gflat = torch.randn(n_flat, device=DEV, generator=g) * 0.1
        opt.param_groups[0]["lr"], opt.param_groups[1]["lr"] = lr_v, lr_d
        val_grad.grad = mv.to_reference(gv)
        for name, off, cnt in lay:
            dec_ref[name].grad = gflat[off:off + cnt].view_as(dec_ref[name]).clone()
        opt.step()
        fused.step_voxels(key, c[key], mv, gv, lr_v)
        fused.step_decoder("color", dec, gflat, lr_d, renderer=renderer)
        want = val_ref.clone()
        want[mask5] = val_grad.detach()
        assert rel(c[key], want) < 1e-6, step
        assert torch.equal(c[key][~mask5], val_ref[~mask5])                    # unselected voxels untouched
        mine = dict(dec.color_decoder.named_parameters())
        for name in dec_ref:
            assert rel(mine[name], dec_ref[name]) < 1e-6, (step, name)
    # the renderer sees the updated colour decoder (its packed image was invalidated)
    ro, rd, gd, _ = su.make_rays(sc, 16, seed=1)
    got = renderer.render_batch_ray(c, dec, rd.to(DEV), ro.to(DEV), DEV, "color", gt_depth=gd.to(DEV))
    st = {lvl: dict(v) for lvl, v in dec_state.items()}
    st["color"] = {k: v.detach().cpu() for k, v in dec_ref.items()}
    want = tp.render_batch_ray({k: v.cpu().contiguous() for k, v in c.items()}, st, rd, ro, "color", gd, su.scene_bound(sc))
    assert rel(got[2], want[2]) < TOL and rel(got[0], want[0]) < TOL


def test_fused_mapping_loop_against_five_real_mapper_iterations():
    """Five joint iterations (3 x middle, fine, color) of the REAL Mapper.optimize_map with the real torch Adam (tests/golden/mapper_loop.pt,
    ray batches captured at the renderer boundary) against the native loop: on-GPU frustum mask + slot tables + fused iterations +
    fused Adam in place on the grids.  Adam's first steps are sign-like (lr 0.1 on the middle grid), so a handful of voxels whose
    gradient is at rounding level may land elsewhere: the bulk must agree tightly, the outliers must be few."""
    from nice_slam_b200.mapping import FusedMappingLoop
    case = torch.load(os.path.join(su.GOLDEN, "mapper_loop.pt"), map_location="cpu", weights_only=False)
    sc = su.load_scenes()[case["scene"]]
    renderer, c, dec = make_renderer(sc, su.make_grids(sc, case["variant"]), su.load_decoders(case["variant"]), DEV)
    depth, _ = su.make_frame(sc, case["frame_seed"])
    c2w = su.make_pose(sc, case["pose_seed"])
    start = {k: v.clone() for k, v in c.items()}
    loop = FusedMappingLoop(renderer, c, dec, c2w, depth.to(DEV), w_color=case["w_color_loss"])
    for it in case["iterations"]:
        loss = loop.iteration(it["stage"], it["rays_o"].to(DEV), it["rays_d"].to(DEV), it["gt_depth"].to(DEV), it["gt_color"].to(DEV), it["lr"])
        assert bool(torch.isfinite(loss).all())
    for key, fin in case["final"].items():
        mv = loop.masked[key]
        after = mv.to_reference(mv.gather(c[key])).cpu()
        before = mv.to_reference(mv.gather(start[key])).cpu()
        got, want = after[fin["idx"]], fin["val"]
        close = (got - want).abs() <= 1e-3 * (1 + want.abs())
        assert float(close.float().mean()) > 0.995, (key, float(close.float().mean()))
        dn = float((after - before).double().norm())
        assert abs(dn - fin["delta_norm"]) < 0.02 * fin["delta_norm"], (key, dn, fin["delta_norm"])
        m5 = (mv.slot_map.view(c[key].shape[2:]) >= 0).unsqueeze(0).unsqueeze(0).expand_as(c[key])
        assert torch.equal(c[key][~m5], start[key][~m5])                        # nothing outside the frustum selection moved
    mine = dict(dec.color_decoder.named_parameters())
    for k, v in case["color_decoder"].items():
        close = (mine[k].detach().cpu() - v).abs() <= 1e-3 * (1 + v.abs())
        assert float(close.float().mean()) > 0.99, (k, float(close.float().mean()))


@pytest.mark.parametrize("nbytes", [16, 104, 4904, 10400, 70000, 3 << 20])
def test_copy_block_moves_pinned_host_blocks_both_ways(nbytes):
    """nsb_copy_block (SM copy over the mapped view of page-locked host memory): host -> device -> host round trip, bytes preserved,
    neighbours untouched; a misaligned pointer is refused."""
    import ctypes as C
    from nice_slam_b200 import _lib
    L = _lib.lib()
    g = torch.Generator().manual_seed(nbytes)
    src = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, generator=g).pin_memory()
    back = torch.zeros(nbytes + 32, dtype=torch.uint8).pin_memory()
    dev = torch.zeros(nbytes + 32, dtype=torch.uint8, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    hs, hb = L.nsb_host_device_pointer(C.c_void_p(src.data_ptr())), L.nsb_host_device_pointer(C.c_void_p(back.data_ptr()))
    assert hs and hb
    _lib.check(L.nsb_copy_block(C.c_void_p(dev.data_ptr() + 16), C.c_void_p(hs), nbytes, st), "nsb_copy_block")
    _lib.check(L.nsb_copy_block(C.c_void_p(hb + 16), C.c_void_p(dev.data_ptr() + 16), nbytes, st), "nsb_copy_block")
    torch.cuda.synchronize()
    assert torch.equal(dev[16: 16 + nbytes].cpu(), src)
    assert torch.equal(back[16: 16 + nbytes], src)
    assert int(dev[:16].sum()) == 0 and int(dev[16 + nbytes:].sum()) == 0 and int(back[:16].sum()) == 0 and int(back[16 + nbytes:].sum()) == 0
    assert L.nsb_copy_block(C.c_void_p(dev.data_ptr() + 4), C.c_void_p(hs), 16, st) != 0          # misaligned destination
    pageable = torch.zeros(64, dtype=torch.uint8)
    if not L.nsb_host_device_pointer(C.c_void_p(pageable.data_ptr())):      # (a system with pageable-memory access may accept it)
        assert b"page-locked" in L.nsb_last_error()


@pytest.mark.parametrize("stage,n_rays", [("color", 4096), ("fine", 2500)])
def test_item_split_policy_does_not_change_the_bits(stage, n_rays):
    """Medium batches: one CTA per tile (all decoders) vs one CTA per (tile, decoder) -- the dispatch picks by wave efficiency (option
    split_model); both forms evaluate the same arithmetic: outputs bit-identical, ray gradients equal up to the order of their float64 partial sums."""
    from nice_slam_b200 import _lib
    L = _lib.lib()
    sc = su.load_scenes()["room0"]
    grids, dec_state = su.make_grids(sc, "soft"), su.load_decoders("soft")
    renderer, c, dec = make_renderer(sc, grids, dec_state, DEV)
    ro, rd, gd, gc = su.make_rays(sc, n_rays, seed=4242)
    ro, rd, gd = ro.to(DEV), rd.to(DEV), gd.to(DEV)
    g = torch.Generator(device=DEV).manual_seed(5)
    s1 = torch.randn(n_rays, dtype=torch.float64, device=DEV, generator=g); s2 = torch.randn(n_rays, 3, device=DEV, generator=g)
    res = []
    try:
        for model in (1, 0):
            assert L.nsb_set_option(b"split_model", model) == 0
            r1 = ro.clone().requires_grad_(True); r2 = rd.clone().requires_grad_(True)
            d, u, col = renderer.render_batch_ray(c, dec, r2, r1, DEV, stage, gt_depth=gd)
            ga = torch.autograd.grad((d * s1).sum() + (col * s2).sum() + u.sum(), (r1, r2))
            res.append((d.detach(), u.detach(), col.detach(), ga[0], ga[1]))
    finally:
        L.nsb_set_option(b"split_model", 1)
    for a, b in zip(res[0][:3], res[1][:3]):
        assert torch.equal(a, b)
    for a, b in zip(res[0][3:], res[1][3:]):        # per-ray sums: float64 partial sums added in a different order before the cast to float32
        assert rel(a, b) < 1e-6
