#!/usr/bin/env python
"""Cycle breakdown of one CTA of the tile kernels (instrumented build: make -C nice_slam_b200/csrc ../libnsb_timing.so).
   NSB_LIB=nice_slam_b200/libnsb_timing.so python tools/phase_timing.py [n_rays]"""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ.setdefault("NSB_LIB", os.path.join(ROOT, "nice_slam_b200", "libnsb_timing.so"))
import torch  # noqa: E402
import scene_util as su  # noqa: E402
from gpu_util import make_renderer  # noqa: E402
from nice_slam_b200 import _lib  # noqa: E402
from nice_slam_b200.steps import IterationContext  # noqa: E402

NAMES = {40: "fwd: launch -> depth max done", 41: "fwd: ray table (bbox far, near)", 42: "fwd: sample z", 43: "fwd: rank sort", 44: "fwd: point geometry + syncs",
         1: "fwd: gather (per grid)", 2: "fwd: publish + issue fc_c", 6: "fwd: wait free buffer (E block)", 3: "fwd: embed block compute", 4: "fwd: publish + issue layer-0 block",
         7: "fwd: wait MMAs of the layer", 8: "fwd: layer epilogue (tmem ld, relu, operand write)", 9: "fwd: publish + issue hidden layer", 12: "fwd: output layer + syncs",
         14: "fwd: dealloc + sync", 15: "fwd: parts store + ray completion", 16: "fwd: compositing of completed rays",
         20: "bwd: launch -> ray prologue (weights, dL/docc)", 21: "bwd: point geometry + sync", 22: "bwd: G/DU operand write", 23: "bwd: publish + issue layer", 24: "bwd: wait MMAs",
         27: "bwd: dc rows + cos chain", 29: "bwd: scatter + dp", 30: "bwd: per-ray partial sums", 31: "bwd: ray completion", 32: "bwd: final ray reduce"}


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    dev = torch.device("cuda")
    sc = su.load_scenes()["room0"]
    renderer, c, dec = make_renderer(sc, su.make_grids(sc, "soft"), su.load_decoders("soft"), dev)
    ro, rd, gd, gc = [t.to(dev) for t in su.make_rays(sc, n, seed=3)]
    ctx = IterationContext(renderer, n, "color", dev, kind="track")
    _lib.lib()
    fn = C.CDLL(os.environ["NSB_LIB"]).nsb_debug_phases
    fn.argtypes = [C.c_void_p, C.c_int]
    buf = (C.c_longlong * 64)()
    iters = 50
    for it in range(3 + iters):
        if it == 3:
            torch.cuda.synchronize(); fn(buf, 1)
        ctx.run(c, dec, ro, rd, gd, gc.double())
    torch.cuda.synchronize()
    fn(buf, 0)
    tot_f = sum(buf[i] for i in range(0, 20)); tot_b = sum(buf[i] for i in range(20, 40))
    print("cycles per launch of CTA 0 (avg of %d iterations, %d rays): forward %.0f, backward %.0f" % (iters, n, tot_f / iters, tot_b / iters))
    for i in range(64):
        if buf[i]:
            tot = tot_f if i < 20 else tot_b
            print("  %2d %-46s %9.0f  %5.1f %%" % (i, NAMES.get(i, "?"), buf[i] / iters, 100.0 * buf[i] / tot))


if __name__ == "__main__":
    main()
