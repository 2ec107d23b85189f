"""Device time of the OpenCL C test kernels (tests/plugins/cl_*.cl) next to the built-in pipeline of the same workload.

    python tools/cl_plugin_timing.py [--size 1920 1080] [--reps 20] [--out FILE]

Rows: lt_stats.kernel_ms (CUDA events around the launches of one call), best and median of --reps calls after two
warm-up calls, Cornell box, default camera.  cl_barycentric.cl is set against the built-in custom_opencl.cl pipeline
(barycentric colour of the primary hit); cl_direct_light.cl (one light sample with a shadow ray) against the built-in
accumulator.cl pipeline, which also traces one camera ray and one shadow ray per pixel.  Also prints the translation +
NVRTC compile time of each test kernel and the card's name and power limit, read in the same run."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from lens_trace_b200 import capi, host, layouts as L  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, nargs=2, default=(1920, 1080))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out")
    a = ap.parse_args()
    w, h = a.size
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    say("card: %s" % (gpu[0] if gpu else "unknown"))
    plugins = os.path.join(ROOT, "tests", "plugins")
    for name in ("cl_barycentric.cl", "cl_direct_light.cl", "cl_tile_groups.cl"):
        t = time.perf_counter()
        ok, log = capi.compile_cl(os.path.join(plugins, name))
        say("%-20s translation + NVRTC compile %.1f ms%s" % (name, (time.perf_counter() - t) * 1e3,
                                                             "" if ok else " FAILED " + log))
    sb = host.load_scene_buffers(os.path.join(ROOT, "resources", "models", "cornell_box.obj"))
    ctx = capi.Context(0)
    sc = ctx.upload(sb)
    cam = L.make_camera(0, 2.5, -50, 0.0, 0)

    def timed(fn):
        for _ in range(2):
            fn()
        ms = []
        for _ in range(a.reps):
            fn()
            ms.append(ctx.stats().kernel_ms)
        return min(ms), float(np.median(ms))

    say("%dx%d, Cornell box, kernel_ms best / median of %d calls" % (w, h, a.reps))
    for name, builtin in (("cl_barycentric.cl", L.KERNEL_CUSTOM_BARY), ("cl_direct_light.cl", L.KERNEL_ACCUMULATOR)):
        pid = ctx.plugin_load(os.path.join(plugins, name))
        cb, cm = timed(lambda: ctx.render_plugin_cl(sc, cam, pid, w, h))
        params = capi.make_params(builtin, w, h)
        bb, bm = timed(lambda: ctx.render(sc, cam, params))
        say("  %-20s %8.3f / %8.3f ms   built-in %-16s %8.3f / %8.3f ms" % (
            name, cb, cm, capi.load().lt_kernel_name(builtin).decode(), bb, bm))
    sc.release()
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
