"""One bench workload's step (bench.py WORKLOADS: frames, running mean, L2 flushed before each step) timed on every
tree the library can build for it: host median split, device LBVH, device PLOC, host binned SAH.

    python tools/tree_frames.py [workload] [--steps K]      default: cornell_gi_1080p_64spp
"""
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from lens_trace_b200 import capi, host, layouts as L  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
workload = args[0] if args else bench.DEFAULT_WORKLOAD
steps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 3
model, kernel, w, h, frames, depth, _ = bench.WORKLOADS[workload]
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True, timeout=60).stdout.strip().splitlines()[0]
print("GPU 0: %s; workload %s, %d steps after one warm-up" % (gpu, workload, steps), flush=True)

median = bench.load_scene(model)
ctx = capi.Context(0)
stream = torch.cuda.Stream()
ctx.set_stream(stream.cuda_stream)
acc = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2
cam = L.make_camera(0, 2.5, -50, 0.0, 0)
params = lambda flags=0: capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames,
                                          accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)


def time_steps(scene):
    times = []
    for _ in range(steps + 1):
        with torch.cuda.stream(stream):
            flush.fill_(1.0)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        ctx.render_device(scene, cam, params(), acc.data_ptr(), sync=False)
        c1.record(stream)
        torch.cuda.synchronize()
        times.append(c0.elapsed_time(c1))
    ctx.render_device(scene, cam, params(L.FLAG_STATS), acc.data_ptr(), sync=True)
    s = ctx.stats()
    return times[1:], s.node_tests / max(1, s.rays)


trees = [("median-split", lambda: ctx.upload(median)),
         ("device LBVH", lambda: ctx.build_lbvh(median.prims, median.materials)),
         ("device PLOC", lambda: ctx.build_ploc(median.prims, median.materials)),
         ("host SAH", lambda: ctx.upload(bench.load_scene(model, host.AccelerationStructure.HOST_SAH)))]
for name, make in trees:
    t0 = time.perf_counter()
    sc = make()
    build_s = time.perf_counter() - t0
    ts, box = time_steps(sc)
    print("%-13s %9.2f ms per step (min %.2f, max %.2f); box tests per ray %.1f; load/build %.2f s" % (
        name, sum(ts) / len(ts), min(ts), max(ts), box, build_s), flush=True)
    sc.release()
