"""Trees for the same kernels: host median split (reference semantics), device LBVH, device PLOC and, with --sah, the
host binned SAH.  Per builder: build time, stack depth, SAH cost, traversal work and render time; pixels that differ
from the median-split tree.

    python tools/bvh_compare.py [grid] [--sah]      grid 707: 1 M triangles, 1581: 5 M
"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lens_trace_b200 import capi, host, layouts as L  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
grid = int(args[0]) if args else 707
with_sah = "--sah" in sys.argv
try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=60).stdout.strip().splitlines()[0]
except (OSError, IndexError, subprocess.SubprocessError):
    gpu = "unknown"
print("GPU 0: %s" % gpu, flush=True)

path = "/tmp/bvhcmp_%d_%d.obj" % (grid, os.getpid())
host.write_synthetic_scene(path, grid, 0x5EED)
t0 = time.perf_counter()
model = host.Model(path)
t_parse = time.perf_counter() - t0
t0 = time.perf_counter()
accel = host.AccelerationStructure(model)
t_host = time.perf_counter() - t0
median = accel.buffers()
print("triangles %d: OBJ parse %.2f s" % (len(median.prims), t_parse), flush=True)


def sah_cost(nodes):
    """sum of the inner nodes' half-areas over the root's"""
    inner = nodes[nodes["count"] == 0]
    half = lambda e: e[..., 0] * e[..., 1] + e[..., 1] * e[..., 2] + e[..., 2] * e[..., 0]
    return half((inner["max"] - inner["min"]).astype(np.float64)).sum() / half(
        (nodes["max"][0] - nodes["min"][0]).astype(np.float64))


ctx = capi.Context(0)
trees = []  # (name, scene, build text)
sc_m = ctx.upload(median)
trees.append(("median-split", sc_m, "host %.2f s" % t_host))
for name, build in (("LBVH", ctx.build_lbvh), ("PLOC", ctx.build_ploc)):
    dev, wall = [], []
    for _ in range(3):  # the first build also loads the module and sizes the cub temporaries
        t0 = time.perf_counter()
        sc = build(median.prims, median.materials)  # any order works; the builders re-sort
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(ctx.stats().upload_ms)
        if len(dev) < 3:
            sc.release()
    trees.append((name, sc, "device %.1f ms (H2D of primitives + build + re-flatten), wall %.1f ms (median of 3: %.1f / %.1f)"
                  % (min(dev), min(wall), sorted(dev)[1], sorted(wall)[1])))
if with_sah:
    t0 = time.perf_counter()
    sah = host.AccelerationStructure(model, host.AccelerationStructure.HOST_SAH).buffers()
    trees.append(("host SAH", ctx.upload(sah), "host %.2f s" % (time.perf_counter() - t0)))

cam = L.make_camera(0, 2.5, -50, 0.0, 1)
w, h = 1920, 1080
ref = ctx.render(sc_m, cam, capi.make_params(L.KERNEL_BASIC_CU, w, h))
for name, sc, build_text in trees:
    sb, depth = ctx.download(sc)
    print("%s: build %s; stack depth %d; SAH cost %.2f" % (name, build_text, depth, sah_cost(sb.nodes)), flush=True)
    for kernel, frames, label in ((L.KERNEL_BASIC_CU, 1, "primary"), (L.KERNEL_GI, 8, "GI 8 spp")):
        p = capi.make_params(kernel, w, h, max_ray_depth=4, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN)
        ts = []
        for _ in range(3):
            ctx.accum_reset()
            ctx.render(sc, cam, p, want_output=False)
            ts.append(ctx.stats().kernel_ms)
        ps = capi.make_params(kernel, w, h, max_ray_depth=4, frames=1, accum_mode=L.ACCUM_RUNNING_MEAN, flags=L.FLAG_STATS)
        ctx.render(sc, cam, ps, want_output=False)
        st = ctx.stats()
        print("  %-9s %8.3f ms   box tests/ray %.1f  triangle tests/ray %.2f" % (
            label, min(ts), st.node_tests / st.rays, st.tri_tests / st.rays), flush=True)
    if sc is not sc_m:
        img = ctx.render(sc, cam, capi.make_params(L.KERNEL_BASIC_CU, w, h))
        print("  pixels whose colour differs from the median-split tree's: %d of %d" % (
            (np.abs(img - ref).max(-1) > 0).sum(), w * h), flush=True)
for f in (path, path[:-4] + ".mtl"):
    os.remove(f)
