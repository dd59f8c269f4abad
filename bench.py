#!/usr/bin/env python
"""bench.py -- rendered rays/sec of one NICE-SLAM tracking iteration (fwd + loss + bwd) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json metric "rendered rays/sec (200px x 48samp batch) ... ms/tracking-iter"): Replica room0 geometry,
full coarse/middle/fine/color grids (48.5 MB, channels-last), pretrained middle/fine decoders + seeded colour decoder,
stage 'color', 200 rays x (32 uniform + 16 near-surface) samples per GPU, one Tracker.optimize_cam_in_batch-style
iteration = batch depth maxima -> render forward -> tracking loss (median-gated) -> render backward -> pose-gradient
reduction.  N > 1: the global batch of 200*N rays is ray-sharded (weak scaling) with the exchanges the reference's
batch-global ops require (depth maxima MAX, residual all-gather for the median, SUM of loss + pose gradient) over NCCL.
The Adam step on the 7 pose numbers stays in PyTorch and is outside the timed region of both arms.

`value` : rays/s with inputs resident in HBM; `e2e`: the same iteration through IterationContext.build_graph(host_io=...): pinned host
inputs -> device, iteration, loss + ray / pose gradients -> pinned host, all inside the timed region, followed by a stream synchronize (the
caller reads the result).  The two host blocks can travel as copy-engine nodes ("dma"), as nsb_copy_block kernels over the mapped pinned
memory ("sm"), or with the result stored by the backward's last CTA ("sm_push"); all three are timed, checked to deliver identical bytes, and
the fastest is reported (`e2e.ms_per_step_by_transport` keeps the three figures).  --impl reference times the reference algorithm's CPU path (oracle port, PyTorch CPU, all host
threads) on the same batch.  Every timed quantity uses CUDA events on the launching stream, max over ranks.

--dump-outputs DIR: after the timed steps, what the last timed step handed its caller is written as DIR/<name>.npy (float32 / float64, rank 0):
one GPU: loss, d_c2w, depth, var, rgb, d_rays_o, d_rays_d of the 200-ray iteration; N > 1: the summed loss and d_c2w; --impl reference: loss
and d_c2w.  The inputs are generated from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

RAYS_PER_GPU = 200
STAGE = "color"
BYTES_PER_RAY = 48 * 3 * 1024            # SURVEY 8d: S x G(stage) x 1024 B gathered per ray (tracking: no scatter) = 147456
MAC_PER_POINT = 51653                    # SURVEY 8a: forward MACs per sample point in stage color (fine + color + middle decoders)
# tracking iteration: forward + input-gradient backward (~ the same MACs), 2 flops per MAC; the tensor cores execute 3x that (3xTF32 split)
FLOPS_PER_RAY = 48 * MAC_PER_POINT * 2 * 2
METRIC = "rendered rays/sec"
WORKLOAD = "room0 tracking iteration (fwd+loss+bwd), 200 rays x 48 samples (32+16) per GPU, stage color, full grids"


# ------------------------------------------------------------------------------------------------ helpers
def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak():
    """TF32 dense tensor peak in TFLOP/s: half the measured bf16 cuBLAS burst figure (TF32 runs at half the bf16 rate on B200)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("bf16_tflops", 1590.0) / 2, "0.5 x measured bf16 burst (MEASURED_PEAKS.json bf16_tflops)"
    return 1590.0 / 2, "0.5 x fallback bf16 (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.2] or [r for _, r in self.rows]
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def build_scene(device):
    import scene_util as su
    from gpu_util import make_renderer
    sc = su.load_scenes()["room0"]
    renderer, c, dec = make_renderer(sc, su.make_grids(sc, "soft"), su.load_decoders("soft"), device)
    for p in dec.parameters():
        p.requires_grad_(False)
    return sc, renderer, c, dec


def make_batch(sc, n, seed):
    """n rays that pass the bbox pre-filter (host tensors): rays_o, rays_d, camera-frame dirs, gt_depth f32, gt_color f64."""
    import scene_util as su
    depth, color = su.make_frame(sc, seed)
    c2w = su.make_pose(sc, seed)
    cam = sc["cam"]
    g = torch.Generator().manual_seed(31000 + seed)
    idx = torch.randint(cam["H"] * cam["W"], (4 * n,), generator=g)
    i, j = (idx % cam["W"]).float(), (idx // cam["W"]).float()
    dirs = torch.stack([(i - cam["cx"]) / cam["fx"], -(j - cam["cy"]) / cam["fy"], -torch.ones_like(i)], -1)
    rd = torch.sum(dirs.reshape(-1, 1, 3) * c2w[:3, :3], -1)
    ro = c2w[:3, -1].expand(rd.shape).contiguous()
    gd, gc = depth.reshape(-1)[idx], color.reshape(-1, 3)[idx]
    keep = su.prefilter_host(ro, rd, gd, su.scene_bound(sc))
    sel = torch.nonzero(keep).reshape(-1)[:n]
    assert sel.numel() == n, "not enough rays survive the pre-filter"
    return ro[sel].contiguous(), rd[sel].contiguous(), dirs[sel].contiguous(), gd[sel].contiguous(), gc[sel].contiguous()


def workload_config(world):
    """`config` of BOTH arms: the reference arm times the reference's CPU implementation on this arm's configuration, so the two lines carry
    the same dict; what is specific to a run (launch form, exchange back-end, the reference arm's bounded sample) sits next to it (`run`)."""
    return {"workload": WORKLOAD, "rays_per_step": RAYS_PER_GPU * world,
            "l2": "flushed between steps on the GPU (256 MiB memset outside the event pair)",
            "batch": "every step replays the same synthetic ray batch (fixed seed); grids and decoders are not updated between steps",
            "parallelism": "ray-sharded x%d" % world,
            "timing": "GPU arm: sum of per-step CUDA-event pairs, max over ranks; reference arm: wall clock around the timed steps on the host"}


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def cpu_iteration_fn(sc, batch):
    """One tracking iteration of the reference algorithm on the host CPUs (oracle port = same torch ops as the reference)."""
    import scene_util as su
    from oracle import torch_port as tp
    grids, dec, bound = su.make_grids(sc, "soft"), su.load_decoders("soft"), su.scene_bound(sc)
    ro, rd, dirs, gd, gc = batch

    def step():
        # the reference's tracker leaves requires_grad on its deep-copied decoders (src/Tracker.py:138), so its backward
        # also computes their (unused) gradients -- kept here to time what the reference actually does
        out = tp.iteration("track", grids, dec, ro, rd, gd, gc, STAGE, bound, grad_rays=True, grad_decoders=("fine", "color", "middle"))
        d_c2w = torch.cat([out["d_rays_d"].double().t() @ dirs.double(), out["d_rays_o"].double().sum(0, keepdim=True).t()], 1)
        return float(out["loss"]), d_c2w
    return step


def pick_cpu_threads(sc, batch):
    """(seconds per iteration, threads): the faster of {1, all cores} by the MEDIAN of three timed iterations after one warm-up
    (CPU grid_sample is single-threaded for batch 1 and oversubscribed MKL can be slower than one thread; a single sample per setting
    made the choice flip between runs).  Leaves torch's thread count at the chosen setting."""
    best = None
    for threads in sorted({1, os.cpu_count() or 1}):
        torch.set_num_threads(threads)
        step = cpu_iteration_fn(sc, batch)
        step()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter(); step(); ts.append(time.perf_counter() - t0)
        dt = statistics.median(ts)
        if best is None or dt < best[0]:
            best = (dt, threads)
    torch.set_num_threads(best[1])
    return best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import scene_util as su
    sc = su.load_scenes()["room0"]
    batch = make_batch(sc, RAYS_PER_GPU, 0)
    best = pick_cpu_threads(sc, batch)
    # bounded sample: keep the whole run within ~2.5 minutes whatever --steps is
    n_rays = RAYS_PER_GPU
    budget = 150.0
    if (args.steps + args.warmup) * best[0] > budget:
        n_rays = max(8, int(RAYS_PER_GPU * budget / ((args.steps + args.warmup) * best[0])))
    sub = tuple(t[:n_rays] for t in batch)
    step = cpu_iteration_fn(sc, sub)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        loss, d_c2w = step()
    ms = (time.perf_counter() - t0) / args.steps * 1e3
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"loss": torch.tensor([loss], dtype=torch.float64), "d_c2w": d_c2w})
    value = n_rays / (ms * 1e-3)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args.gpus),
            "run": {"device": "host CPU", "rays_per_timed_step": n_rays},
            "cpu_baseline": {"value": value, "unit": "rays/s", "cores": best[1], "kind": "port",
                             "sample": "%d tracking iterations on %d of the 200 rays per step (oracle/torch_port.py, PyTorch CPU, %d threads of %d cores)"
                                       % (args.steps, n_rays, best[1], os.cpu_count() or 1)},
            "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def extra_workloads(sc, renderer, c, dec, dev, flush, peak):
    """Secondary measurements reported under `extra` (same timing rules: CUDA events per step, L2 flushed between steps):
    BASELINE configs[1] (mapping iteration, 996 rays = 6 frames x 166 px, stage color, voxel + colour-decoder gradients)
    and the ray-throughput sweep (tracking-style fwd+loss+bwd, 48 samples) at larger batches."""
    from nice_slam_b200.steps import IterationContext

    def time_steps(fn, steps, warmup=3):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in evs:
            flush.zero_(); a.record(); fn(); b.record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / steps

    def graphed(fn):
        """(callable, how): fn captured into a CUDA graph -- these iterations are 2-8 launches of 0.05-0.6 ms each, and with stream launches a slow
        or busy host makes them enqueue-bound (r02ae: 0.87 instead of 0.63 ms for the same mapping iteration) -- or fn itself if capture fails."""
        try:
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                fn(); fn()
            cur.wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            g.replay(); torch.cuda.synchronize()
            return g.replay, "CUDA graph replay"
        except Exception as e:                                     # noqa: BLE001
            torch.cuda.synchronize()
            return fn, "stream launches (graph capture failed: %s)" % type(e).__name__

    out = {}
    n = 996
    ro, rd, dirs, gd, gc = [t.to(dev) for t in make_batch(sc, n, 101)]
    ctx = IterationContext(renderer, n, "color", dev, kind="map", grad_grids=("grid_middle", "grid_fine", "grid_color"), grad_decoders=("color",))
    gcf = gc.float()
    step, how = graphed(lambda: ctx.run(c, dec, ro, rd, gd, gcf))
    ms = time_steps(step, 100)
    bpr = 48 * 3 * 1024 * 2
    out["mapping_configs1"] = {"workload": "room0 mapping iteration, 996 rays x 48, stage color, dense voxel grads (middle+fine+color) + colour-decoder grads",
                               "launch": how, "ms_per_step": ms, "rays_per_s": n / (ms * 1e-3), "algorithmic_bytes_per_ray": bpr,
                               "hbm_frac": n * bpr / (ms * 1e-3) / 1e9 / peak}
    # the same iteration inside the native mapper loop: frustum-selected voxels (on-GPU mask of a synthetic frame), compact gradients,
    # fused Adam in place on the grids + on the colour decoder (nice_slam_b200/mapping.py) -- what one joint_iter of Mapper.optimize_map costs
    import copy
    import scene_util as su
    from nice_slam_b200.mapping import FusedMappingLoop
    depth1, _ = su.make_frame(sc, 1)
    loop = FusedMappingLoop(renderer, {k: v.clone() for k, v in c.items()}, copy.deepcopy(dec), su.make_pose(sc, 1), depth1.to(dev))
    lr = dict(decoders=0.005, middle=0.005, fine=0.005, color=0.005)
    ms = time_steps(lambda: loop.iteration("color", ro, rd, gd, gcf, lr), 50)
    out["mapping_loop_step"] = {"workload": "one joint iteration of the native mapper loop, stage color, 996 rays: fused iteration (compact voxel grads of the "
                                            "frustum selection + colour-decoder grads) + fused Adam (3 grids in place + colour decoder)",
                                "selected_voxels": {k: m.count for k, m in loop.masked.items()}, "ms_per_step": ms, "rays_per_s": n / (ms * 1e-3)}
    del loop
    # the coarse mapper's joint iteration (Mapper.py:403-404,484: stage 'coarse', rendered WITHOUT the depth guide -- 32 uniform samples in the
    # enlarged bound -- and supervised with the sensor depth), native loop on the coarse grid only
    loopc = FusedMappingLoop(renderer, {k: v.clone() for k, v in c.items()}, copy.deepcopy(dec), su.make_pose(sc, 1), depth1.to(dev), keys=("grid_coarse",))
    lrc = dict(decoders=0.0, coarse=0.001)
    ms = time_steps(lambda: loopc.iteration("coarse", ro, rd, gd, gcf, lrc), 50)
    out["mapping_loop_step_coarse_mapper"] = {"workload": "one joint iteration of the coarse mapper in the native loop, stage coarse, 996 rays x 32 uniform samples "
                                                          "(no depth guide), compact coarse-voxel grads + fused Adam in place",
                                              "selected_voxels": {k: m.count for k, m in loopc.masked.items()}, "ms_per_step": ms, "rays_per_s": n / (ms * 1e-3)}
    del loopc
    # BASELINE configs[4]: ray-throughput sweep, tracking-style iteration (fwd + loss + bwd), stage color, N_surface = 16 fixed,
    # N_samples in {16, 32, 80} -> S in {32, 48, 96} samples per ray (SURVEY 8d config 5); one GPU here, --gpus N shards the 200-ray line
    from gpu_util import make_renderer
    sweep = []
    for n_uniform in (16, 32, 80):
        S = n_uniform + 16
        rr = renderer if n_uniform == 32 else make_renderer(sc, {k: v for k, v in c.items()}, su.load_decoders("soft"), dev, n_samples=n_uniform)[0]
        for nn, steps in ((256, 100), (1024, 100), (4096, 40), (16384, 12), (65536, 5)):
            ro, rd, dirs, gd, gc = [t.to(dev) for t in make_batch(sc, nn, 200 + nn)]
            cx = IterationContext(rr, nn, "color", dev, kind="track", host_staging=False)
            step, how = graphed(lambda: cx.run(c, dec, ro, rd, gd, gc))
            ms = time_steps(step, steps)
            sweep.append({"rays": nn, "samples": S, "launch": how, "ms_per_step": ms, "rays_per_s": nn / (ms * 1e-3),
                          "hbm_frac": nn * S * 3 * 1024 / (ms * 1e-3) / 1e9 / peak})
            del cx
    out["sweep_tracking_iteration"] = sweep
    out["dropin"] = dropin_iterations(sc, renderer, c, dec, dev, time_steps)
    # bulk no-grad paths of the same forward kernel (SURVEY.md 8f-3): Mesher-style eval_points and a full-image render
    pts = (torch.rand(1 << 22, 3, device=dev, dtype=torch.float64) - 0.5) * 4.0 + torch.tensor(su_center(sc), device=dev, dtype=torch.float64)
    ms = time_steps(lambda: renderer.eval_points(pts, dec, c, "fine", dev), 5, warmup=1)
    out["eval_points_fine"] = {"points": pts.shape[0], "ms_per_call": ms, "mpoints_per_s": pts.shape[0] / (ms * 1e-3) / 1e6}
    import scene_util as su
    depth, _ = su.make_frame(sc, 3)
    c2w = su.make_pose(sc, 3).to(dev)
    gtd = depth.to(dev)
    ms = time_steps(lambda: renderer.render_img(c, dec, c2w, dev, "color", gt_depth=gtd), 3, warmup=1)
    out["render_img_color"] = {"rays": int(gtd.numel()), "samples": 48, "ms_per_image": ms, "rays_per_s": gtd.numel() / (ms * 1e-3)}
    return out


def dropin_iterations(sc, renderer, c, dec, dev, time_steps):
    """The reference call surface, timed: an UNMODIFIED caller doing render_batch_ray + its own torch loss + loss.backward() (autograd) around
    FusedRenderer -- what Tracker.optimize_cam_in_batch (src/Tracker.py:106-125) and one joint_iter of Mapper.optimize_map (src/Mapper.py:482-503)
    cost when only `slam.renderer` is swapped (INTEGRATION.md), Adam step excluded as in the headline.  Same batches and timing rules as the fused
    numbers: the difference is the price of the torch glue (autograd graph, dense zero-filled grid gradients, separate loss kernels)."""
    import scene_util as su
    out = {}
    # tracking: camera tensor -> c2w -> rays (get_rays_from_uv) -> render -> tracking loss -> backward to the 7 pose numbers
    ro, rd, dirs, gd, gc = [t.to(dev) for t in make_batch(sc, RAYS_PER_GPU, 0)]
    from nice_slam_b200.mapping import tensor_from_c2w
    cam = tensor_from_c2w(su.make_pose(sc, 0)).to(dev).requires_grad_(True)

    def quad2rot(q):
        two_s = 2.0 / (q * q).sum()
        qr, qi, qj, qk = q[0], q[1], q[2], q[3]
        return torch.stack([1 - two_s * (qj ** 2 + qk ** 2), two_s * (qi * qj - qk * qr), two_s * (qi * qk + qj * qr),
                            two_s * (qi * qj + qk * qr), 1 - two_s * (qi ** 2 + qk ** 2), two_s * (qj * qk - qi * qr),
                            two_s * (qi * qk - qj * qr), two_s * (qj * qk + qi * qr), 1 - two_s * (qi ** 2 + qj ** 2)]).reshape(3, 3)

    def track():
        cam.grad = None
        R = quad2rot(cam[:4])
        rays_d = torch.sum(dirs.reshape(-1, 1, 3) * R, -1)
        rays_o = cam[4:].expand(rays_d.shape)
        depth, unc, color = renderer.render_batch_ray(c, dec, rays_d, rays_o, dev, "color", gt_depth=gd)
        unc = unc.detach()
        tmp = torch.abs(gd - depth) / torch.sqrt(unc + 1e-10)
        mask = (tmp < 10 * tmp.median()) & (gd > 0)
        loss = tmp[mask].sum() + 0.5 * torch.abs(gc - color)[mask].sum()
        loss.backward()
    out["tracking_iter_ms"] = time_steps(track, 100)
    # mapping: dense leaf grids + colour-decoder leaves (the reference's val[mask] = val_grad indexing is the caller's and not timed here)
    n = 996
    ro, rd, dirs, gd, gc = [t.to(dev) for t in make_batch(sc, n, 101)]
    gcf = gc.float()
    cm = {k: v.detach().clone().requires_grad_(k != "grid_coarse") for k, v in c.items()}
    import copy
    dm = copy.deepcopy(dec)
    for name, p in dm.named_parameters():
        p.requires_grad_(name.startswith("color_decoder"))

    def mapit():
        for v in cm.values():
            v.grad = None
        for p in dm.parameters():
            p.grad = None
        depth, unc, color = renderer.render_batch_ray(cm, dm, rd, ro, dev, "color", gt_depth=gd)
        m = gd > 0
        loss = torch.abs(gd[m] - depth[m]).sum() + 0.2 * torch.abs(gcf - color).sum()
        loss.backward()
    out["mapping_iter_ms"] = time_steps(mapit, 50)
    out["note"] = ("FusedRenderer.render_batch_ray + torch loss + autograd (the drop-in path of INTEGRATION.md); compare with ms_per_step (tracking) and "
                   "extra.mapping_configs1 (mapping) of the fused C-ABI iterations")
    return out


def su_center(sc):
    import scene_util as su
    b = su.scene_bound(sc)
    return [float((b[i][0] + b[i][1]) / 2) for i in range(3)]


def frustum_masks(renderer, c, sc, seed, dev, keys):
    """{key: MaskedVoxels}: the voxels the synthetic frame `seed` sees (nsb_frustum_mask = Mapper.get_mask_from_c2w, src/Mapper.py:93-164)."""
    import scene_util as su
    from nice_slam_b200.masked import MaskedVoxels, frustum_voxel_mask
    depth, _ = su.make_frame(sc, seed)
    pose = su.make_pose(sc, seed)
    return {k: MaskedVoxels(c[k], frustum_voxel_mask(renderer, pose, k, c[k], depth.to(dev))) for k in keys}


def timed_sharded(fn, steps, flush, dev, world):
    """ms per step: CUDA-event pairs around every step on this rank, L2 flushed between steps, max over ranks."""
    import torch.distributed as dist
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        flush.zero_(); a.record(); fn(); b.record()
    torch.cuda.synchronize()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs) / steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def scene_workloads(dev, flush, rank, world):
    """BASELINE configs[2], configs[3]: one mapping iteration (stage color, frustum-masked voxel parameterisation, compact voxel grads +
    colour-decoder grads in one packed block) on ScanNet scene0000 (5000 rays), Apartment as configured (0.98 M voxels, 10000 rays) and Apartment
    with the TUM grid lengths (8.0 M voxels, 1.0 GB of grids -- larger than L2, so the gather really comes from HBM).  STRONG scaling: the global
    batch is fixed and ray-sharded over the ranks (contiguous shards), the batch depth maxima come from the full batch on every rank and the
    packed gradient block is all-reduced ONCE per iteration (SURVEY.md 8e).  Runs on every rank; the report is returned on every rank."""
    import torch.nn.functional as F
    import scene_util as su
    from gpu_util import make_renderer
    from nice_slam_b200.dist import ShardedMappingIteration, shard_bounds
    from nice_slam_b200.steps import IterationContext
    out = []
    for name, n, variant in (("scene0000", 5000, None), ("apartment", 10000, None), ("apartment", 10000, "tum_grid_len")):
        sc = dict(su.load_scenes()[name])
        shapes = dict(sc["shapes"])
        if variant:
            shapes["grid_middle"] = list(shapes["grid_fine"])
            shapes["grid_fine"] = shapes["grid_color"] = [2 * d + 1 for d in sc["shapes"]["grid_fine"]]
        g = torch.Generator(device=dev).manual_seed(5)
        grids = {}
        for key in ("grid_coarse", "grid_middle", "grid_fine", "grid_color"):
            D, H, W = shapes[key]
            lo = torch.randn(1, 32, max(D // 4, 2), max(H // 4, 2), max(W // 4, 2), device=dev, generator=g)
            t = F.interpolate(lo, size=(D, H, W), mode="trilinear", align_corners=True) * 0.3
            t += torch.randn(t.shape, device=dev, generator=g) * (0.003 if key == "grid_fine" else 0.3)
            grids[key] = t
        renderer, c, dec = make_renderer(sc, grids, su.load_decoders("soft"), dev)
        del grids
        ro, rd, dirs, gd, gc = [t.to(dev) for t in make_batch(sc, n, 77)]          # the same global batch on every rank
        keys = ("grid_middle", "grid_fine", "grid_color")
        mv = frustum_masks(renderer, c, sc, 77, dev, keys)
        lo_, hi_ = shard_bounds(n, rank, world)
        ctx = IterationContext(renderer, hi_ - lo_, "color", dev, kind="map", grad_grids=keys, grad_decoders=("color",), masked=mv, host_staging=False)
        ctx.load_device_inputs(ro[lo_:hi_], rd[lo_:hi_], gd[lo_:hi_], gc[lo_:hi_].float())
        sh = ShardedMappingIteration(ctx)
        sh.prepare(c, dec, global_gt_depth=gd)
        ms = timed_sharded(sh.enqueue, 20, flush, dev, world)
        assert torch.isfinite(ctx.packed).all()
        vox = sum(int(c[k].shape[2] * c[k].shape[3] * c[k].shape[4]) for k in c)
        bpr = 48 * 3 * 1024 * 2
        out.append({"scene": name + ("+" + variant if variant else ""), "rays_global": n, "rays_per_gpu": hi_ - lo_, "voxels": vox, "grid_mbytes": vox * 128 / 1e6,
                    "selected_voxels": {k: m.count for k, m in mv.items()}, "allreduce_bytes": int(ctx.packed.numel() * 4),
                    "collectives_per_step": sh.collectives_per_step, "scaling": "strong", "ms_per_step": ms, "rays_per_s": n / (ms * 1e-3),
                    "algorithmic_gbytes_per_s": n * bpr / (ms * 1e-3) / 1e9})
        del ctx, sh, mv, c, renderer
        torch.cuda.empty_cache()
    return out


def mapping_sharded_workload(sc, renderer, c, dec, dev, flush, rank, world):
    """BASELINE configs[1]-style mapping iteration, ray-sharded (weak scaling: 996 rays = 6 keyframes x 166 px per GPU), with the
    frustum-masked voxel parameterisation (nsb_frustum_mask of the current frame): compact voxel gradients + colour-decoder gradients + keyframe
    pose gradients in one packed float32 block and ONE all-reduce per iteration -- the batch depth maxima are taken over the whole window batch,
    which every rank knows (replicated keyframes), before sharding (SURVEY.md 8e).  Runs on every rank; returns the report on every rank."""
    import torch.distributed as dist
    from nice_slam_b200.dist import ShardedMappingIteration
    from nice_slam_b200.steps import IterationContext
    n, n_frames = 996, 6
    batches = [make_batch(sc, n, 301 + r) for r in range(world)]
    ro, rd, dirs, gd, gc = [t.to(dev) for t in batches[rank]]
    gd_global = torch.cat([b[3] for b in batches]).to(dev)
    keys = ("grid_middle", "grid_fine", "grid_color")
    mv = frustum_masks(renderer, c, sc, 301, dev, keys)
    ctx = IterationContext(renderer, n, "color", dev, kind="map", grad_grids=keys, grad_decoders=("color",), masked=mv, n_frames=n_frames, host_staging=False)
    ctx.load_device_inputs(ro, rd, gd, gc.float())
    offs = torch.tensor([i * 166 for i in range(n_frames + 1)], dtype=torch.int32, device=dev)
    sh = ShardedMappingIteration(ctx)
    sh.prepare(c, dec, dirs, offs, global_gt_depth=gd_global)
    sh.enqueue(); torch.cuda.synchronize()
    g = sh.build_graph() if os.environ.get("NSB_DIST_GRAPH", "1") == "1" else None
    ok = torch.tensor([1.0 if g is not None else 0.0], device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    use_graph = bool(ok.item() > 0.5)
    ms = timed_sharded(g.replay if use_graph else sh.enqueue, 100, flush, dev, world)
    assert torch.isfinite(ctx.packed).all()
    return {"workload": "room0 mapping iteration, 996 rays x 48 per GPU (weak scaling), stage color, frustum-masked voxel parameterisation (on-GPU frustum mask of "
                        "the frame), compact voxel grads + colour-decoder grads + 6 keyframe pose grads",
            "selected_voxels": {k: m.count for k, m in mv.items()},
            "ms_per_step": ms, "rays_per_s": n * world / (ms * 1e-3), "allreduce_bytes": int(ctx.packed.numel() * 4),
            "collectives_per_step": sh.collectives_per_step, "launch": "CUDA graph" if use_graph else "stream launches"}


# ------------------------------------------------------------------------------------------------ native arm (GPU)
# dram__bytes_read.sum + dram__bytes_write.sum of one render_bwd_tile_kernel launch of THIS workload (200 rays x 48, room0), taken from the
# committed `ncu --set full` capture (never measured inside a timed run): the 48.5 MB of grids are L2-resident, so DRAM traffic is far
# below the 29.5 MB of algorithmic gather bytes.
NCU_DRAM_BYTES_PER_BWD_LAUNCH = 3777280
NCU_TRAFFIC_SOURCE = "profiles/ncu_full_r02o_render_kernels.txt (ncu --set full: render_bwd_tile_kernel, 3.78 MB read + 0 B written per launch)"


def dbg(msg):
    if os.environ.get("NSB_BENCH_DEBUG"):
        print("[bench rank %s] %s" % (os.environ.get("RANK", "0"), msg), file=sys.stderr, flush=True)


def run_native(args):
    import torch.distributed as dist
    if os.environ.get("NSB_BENCH_DEBUG"):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["NSB_BENCH_DEBUG"]), exit=True)      # where is every rank after N seconds?
    from nice_slam_b200.steps import IterationContext
    from nice_slam_b200.dist import ShardedTrackingIteration
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, "--gpus must equal the number of launched ranks"

    sc, renderer, c, dec = build_scene(dev)
    host = make_batch(sc, RAYS_PER_GPU, rank)
    ro, rd, dirs, gd, gc = [t.to(dev) for t in host]
    ctx = IterationContext(renderer, RAYS_PER_GPU, STAGE, dev, kind="track")
    ctx.stage_host_inputs(host[0], host[1], host[3], host[4])
    sharded = ShardedTrackingIteration(ctx) if world > 1 else None            # in-kernel peer-memory exchanges when available, else NCCL
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2

    use_graph = True
    if sharded is None:
        # single GPU: the whole iteration (and, for e2e, its host copies) is one CUDA-graph launch
        ctx.load_device_inputs(ro, rd, gd, gc)
        g_dev = ctx.build_graph(c, dec, dirs=dirs, host_io=False)
        g_e2e = ctx.build_graph(c, dec, dirs=dirs, host_io=True)
        g_e2e_sm = {m: ctx.build_graph(c, dec, dirs=dirs, host_io=m) for m in ("sm", "sm_push")}

        def step_dev():
            g_dev.replay()

        def step_e2e():
            g_e2e.replay()
            torch.cuda.current_stream().synchronize()      # the caller reads loss / pose gradient from pinned memory

        def step_e2e_sm(mode):
            g_e2e_sm[mode].replay()
            torch.cuda.current_stream().synchronize()
        # every end-to-end form delivers the same bits to the pinned result block
        ctx.h_res.zero_(); step_e2e(); want_res = ctx.h_res.clone()
        sm_ok = {}
        for m in g_e2e_sm:
            ctx.h_res.zero_(); step_e2e_sm(m)
            sm_ok[m] = torch.equal(ctx.h_res, want_res)
    else:
        # N > 1: split-phase iteration with the three NCCL exchanges; captured into one CUDA graph per rank when possible
        ctx.load_device_inputs(ro, rd, gd, gc)
        # every rank knows the whole batch (a sharded tracker splits one pixel list): the batch depth maxima are reduced locally over all ranks' depths
        # (one tiny launch) instead of being exchanged before sampling (SURVEY.md 8e: "gt_max_depth computed once on the full batch")
        gd_global = torch.cat([make_batch(sc, RAYS_PER_GPU, r)[3] for r in range(world)]).to(dev)
        sharded.prepare(c, dec, dirs, global_gt_depth=gd_global)
        sharded.enqueue(); torch.cuda.synchronize()
        exchange = ("NVLink peer memory inside the two render launches (median pool in the forward's tail, [loss | d c2w] sum in the backward's); depth maxima from "
                    "the full batch's depths, known on every rank") if sharded.peers is not None else "NCCL (all-reduce MAX, all-gather, all-reduce SUM)"
        if sharded.peers is not None:                              # cross-check the in-kernel exchanges against the NCCL collectives once
            ref = ShardedTrackingIteration(ctx, exchange="nccl")
            ref.prepare(c, dec, dirs)
            want = ref.enqueue().clone()
            got = sharded.enqueue().clone()
            torch.cuda.synchronize()
            assert torch.allclose(got, want, rtol=1e-9, atol=1e-12), (got, want)
            dbg("peer exchange == NCCL exchange")
        want_graph = os.environ.get("NSB_DIST_GRAPH", "1") == "1"
        dbg("capturing sharded graphs" if want_graph else "eager sharded path")
        g_dev = sharded.build_graph(host_io=False) if want_graph else None
        g_e2e = sharded.build_graph(host_io=True) if want_graph else None
        g_e2e_sm = {m: (sharded.build_graph(host_io=m) if want_graph else None) for m in ("sm", "sm_push")}
        dbg("graphs done")
        flag = torch.tensor([1.0 if (g_dev is not None and g_e2e is not None) else 0.0, 1.0 if all(g is not None for g in g_e2e_sm.values()) else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)                # all ranks must agree (collectives inside the graph)
        use_graph = bool(flag[0].item() > 0.5)
        sm_graph = bool(flag[1].item() > 0.5)

        def step_dev():
            if use_graph:
                g_dev.replay()
            else:
                sharded.enqueue()

        def step_e2e():      # host inputs -> device -> sharded iteration (NCCL exchanges) -> [loss | d_c2w] back to the host
            if use_graph:
                g_e2e.replay()
            else:
                ctx.d_in.copy_(ctx.h_in, non_blocking=True)
                sharded.enqueue()
                ctx.h_pose13.copy_(sharded.packed, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        def step_e2e_sm(mode):
            if use_graph and sm_graph:
                g_e2e_sm[mode].replay()
            else:
                ctx.copy_in_sm()
                sharded.enqueue()
                ctx.copy_out_sm(ctx.h_pose13, sharded.packed)
            torch.cuda.current_stream().synchronize()
        # every end-to-end form delivers the same [loss | d c2w] to pinned host memory
        ctx.h_pose13.zero_(); step_e2e(); want13 = ctx.h_pose13.clone()
        okf = torch.ones(2, device=dev)
        for i, m in enumerate(g_e2e_sm):
            ctx.h_pose13.zero_(); step_e2e_sm(m)
            okf[i] = 1.0 if torch.equal(ctx.h_pose13, want13) else 0.0
        dist.all_reduce(okf, op=dist.ReduceOp.MIN)                  # (a mismatch disqualifies the form instead of killing the multi-rank job)
        sm_ok = {m: bool(okf[i].item() > 0.5) for i, m in enumerate(g_e2e_sm)}

    def timed(fn, steps, warmup, flush_l2):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t0 = time.time()
        for a, b in evs:
            if flush_l2:
                flush.zero_()
            a.record(); fn(); b.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t1 = time.time()
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        if world > 1:
            t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t)
        return total_ms, t0, t1

    # correctness guard of the timed path (cheap): loss finite
    step_dev(); torch.cuda.synchronize()
    assert torch.isfinite(ctx.loss if sharded is None else sharded.packed).all()

    dbg("timing main loop")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, t0, t1 = timed(step_dev, args.steps, max(args.warmup, 3), True)
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    if args.dump_outputs and rank == 0:                            # before the loops below overwrite the context's buffers
        if sharded is None:
            dump_outputs(args.dump_outputs, {"loss": ctx.loss, "d_c2w": ctx.d_c2w, "depth": ctx.depth, "var": ctx.var, "rgb": ctx.rgb,
                                             "d_rays_o": ctx.d_rays_o, "d_rays_d": ctx.d_rays_d})
        else:
            dump_outputs(args.dump_outputs, {"loss": sharded.packed[:1], "d_c2w": sharded.packed[1:].view(3, 4)})
    # dominant kernel (render_bwd_kernel): events recorded by the library around its launch, averaged over a short loop
    bwd_ms = []
    ctx.time_backward(True)
    for _ in range(50):                                            # rank-local (the kernel has no collective inside)
        flush.zero_(); ctx.run(c, dec, ro, rd, gd, gc); torch.cuda.synchronize()
        bwd_ms.append(ctx.ev_bwd[0].elapsed_time(ctx.ev_bwd[1]))
    ctx.time_backward(False)
    dbg("warm + e2e loops")
    warm_ms, _, _ = timed(step_dev, args.steps, 3, False)                 # L2-warm (production steady state), reported as extra
    e2e_dma_ms, _, _ = timed(step_e2e, args.steps, 3, True)
    e2e_forms = {"dma": e2e_dma_ms}
    for m in ("sm", "sm_push"):
        ms_m, _, _ = timed(lambda: step_e2e_sm(m), args.steps, 3, True)
        if sm_ok[m]:
            e2e_forms[m] = ms_m
        else:
            print("[bench] WARNING: end-to-end form %r delivered a different result block than the copy-engine form; not used" % m, file=sys.stderr)
    # the public end-to-end call (IterationContext.build_graph(host_io=...)) offers three transports for its two host blocks; the line reports
    # the fastest and keeps all figures (every rank takes the same decision: the times are already max-reduced over the ranks)
    e2e_copies = min(e2e_forms, key=e2e_forms.get)
    e2e_ms = e2e_forms[e2e_copies]

    # opt-in forward arithmetic (option fwd_f16: FP16 hi|lo operands, tcgen05 kind::f16 -- half the MMAs of the 3xTF32 forward; DESIGN.md 4):
    # the same iteration re-captured with the option on, reported as an extra -- the headline above is the default 3xTF32 path
    f16_opt = None
    if sharded is None and os.environ.get("NSB_FWD_F16") is None:
        from nice_slam_b200 import _lib
        L = _lib.lib()
        if L.nsb_set_option(b"fwd_f16", 1) == 0:
            try:
                g_f16 = ctx.build_graph(c, dec, dirs=dirs, host_io=False)
                ms16, _, _ = timed(g_f16.replay, args.steps, 3, True)
                f16_opt = {"ms_per_step": ms16 / args.steps, "rays_per_s": RAYS_PER_GPU / (ms16 / args.steps * 1e-3),
                           "note": "nsb_set_option('fwd_f16', 1) / NSB_FWD_F16=1; default off: operands must stay inside the fp16 range and "
                                   "values below 2^-14 keep an absolute (2^-25) rather than relative accuracy"}
            finally:
                L.nsb_set_option(b"fwd_f16", 0)
    fast = os.environ.get("NSB_BENCH_FAST") == "1"              # development aid: headline numbers only (never used by the driver)
    dbg("mapping sharded workload")
    map_sharded = None if fast else mapping_sharded_workload(sc, renderer, c, dec, dev, flush, rank, world)
    dbg("strong-scaled scene workloads")
    scenes = None if fast else scene_workloads(dev, flush, rank, world)

    if rank != 0:
        shutdown(world)
        return
    ms = total_ms / args.steps
    rays = RAYS_PER_GPU * world
    value = rays / (ms * 1e-3)
    peak, peak_src = peaks()
    line = {"metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "run": {"launch": "CUDA graph replay (one graph per iteration)" if (sharded is None or use_graph) else "stream launches + NCCL",
                    "exchange": exchange if sharded is not None else "none (single GPU)"},
            "clocks": clocks,
            "e2e": {"value": rays / (e2e_ms / args.steps * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": ctx.h2d_bytes,
                    "d2h_bytes_per_step": ctx.d2h_bytes if sharded is None else 13 * 8, "ms_per_step": e2e_ms / args.steps,
                    "copies": ("one pinned input block -> device and one result block -> pinned host per step, inside the graph, moved by " +
                               {"dma": "copy-engine transfers (cudaMemcpyAsync nodes)",
                                "sm": "nsb_copy_block kernels (SM loads / stores over the mapped host views)",
                                "sm_push": "the SMs over the mapped host views (input block: one nsb_copy_block kernel; result block: stored by the "
                                           "backward's last CTA)"}[e2e_copies]),
                    "ms_per_step_by_transport": {k: v / args.steps for k, v in e2e_forms.items()}},
            "gpu_launches": (2 if sharded is None else (2 if sharded.fused else (5 if sharded.peers is not None else 6))) * args.steps,
            "extra": {"l2_warm_ms_per_step": warm_ms / args.steps, "l2_warm_rays_per_s": rays / (warm_ms / args.steps * 1e-3),
                      "mapping_sharded_masked": map_sharded, "mapping_other_scenes": scenes, "fwd_f16_option": f16_opt}}
    if bwd_ms:
        t_bwd = statistics.mean(bwd_ms) * 1e-3
        ach = BYTES_PER_RAY * RAYS_PER_GPU / t_bwd / 1e9
        it_ach = BYTES_PER_RAY * rays / (ms * 1e-3) / 1e9 / world          # per GPU
        line["roofline"] = {"bound": "hbm", "kernel": "render_bwd_tile_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                            "traffic": NCU_DRAM_BYTES_PER_BWD_LAUNCH, "traffic_source": NCU_TRAFFIC_SOURCE,
                            "peak_source": peak_src, "launch_ms": t_bwd * 1e3,
                            "algorithmic_bytes_per_launch": BYTES_PER_RAY * RAYS_PER_GPU,
                            # SURVEY 8d charges the gather ONCE per fused fwd+bwd iteration: the same bytes over the whole step time
                            "iteration_achieved": it_ach, "iteration_frac": it_ach / peak,
                            "note": "frac = the iteration's algorithmic gather bytes over the backward launch alone; iteration_frac = the same bytes over "
                                    "ms_per_step (the figure SURVEY 8d defines).  The 200-ray batch (225 tile x decoder CTAs) is latency bound, not HBM "
                                    "bound: the 48.5 MB of grids are L2-resident (see DESIGN.md)"}
        tpk, tpk_src = tensor_peak()
        tf = FLOPS_PER_RAY * rays / (ms * 1e-3) / 1e12 / world
        line["roofline_tensor"] = {"bound": "tensor", "dtype": "tf32 (3xTF32 split: every product is three tcgen05.mma.kind::tf32)", "unit": "TFLOP/s",
                                   "algorithmic": tf, "achieved": 3 * tf, "peak": tpk, "frac": 3 * tf / tpk, "peak_source": tpk_src,
                                   "flops_per_ray": FLOPS_PER_RAY,
                                   "note": "per GPU, whole iteration; algorithmic = fp32-equivalent flops of the decoders' forward + input-gradient backward "
                                           "(SURVEY 8a MAC counts), achieved = what the tensor cores execute for them; sm__pipe_tensor_cycles_active from the "
                                           "ncu capture is in profiles/"}
    if world == 1 and not fast:
        line["extra"].update(extra_workloads(sc, renderer, c, dec, dev, flush, peak))
        best = pick_cpu_threads(sc, host)
        step = cpu_iteration_fn(sc, host)
        t0c, k = time.perf_counter(), 0
        while k < 10 or time.perf_counter() - t0c < 10.0:
            step(); k += 1
        dtc = (time.perf_counter() - t0c) / k
        line["cpu_baseline"] = {"value": RAYS_PER_GPU / dtc, "unit": "rays/s", "cores": best[1], "kind": "port",
                                "sample": "%d iterations of the same 200-ray batch, oracle/torch_port.py on PyTorch CPU (%d threads of %d cores)"
                                          % (k, best[1], os.cpu_count() or 1),
                                "ms_per_step": dtc * 1e3}
    emit(line)
    shutdown(world)


def shutdown(world):
    """Leave the process group.  Communicators that were captured into CUDA graphs can make destroy_process_group block: bounded wait,
    then exit hard (everything has been printed and flushed by then)."""
    if world <= 1:
        return
    import torch.distributed as dist
    sys.stdout.flush(); sys.stderr.flush()
    torch.cuda.synchronize()
    t = threading.Thread(target=dist.destroy_process_group, daemon=True)
    t.start(); t.join(15.0)
    if t.is_alive():
        os._exit(0)


def dump_outputs(dirname, arrays):
    """{name: tensor} -> dirname/<name>.npy, float64 tensors as float64, everything else as float32."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(dirname, name + ".npy"), t.numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32))


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract goes to the real stdout; everything else this process (or a library: NCCL prints its version
    banner to stdout) writes to fd 1 has been redirected to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        args.steps = 30 if args.steps is None else args.steps
        args.warmup = 3 if args.warmup is None else args.warmup
        run_reference(args)
    else:
        args.steps = 1000 if args.steps is None else args.steps
        args.warmup = 20 if args.warmup is None else args.warmup
        run_native(args)


if __name__ == "__main__":
    main()
