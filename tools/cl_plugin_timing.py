"""Device time of the OpenCL C test kernels (tests/plugins/cl_*.cl) next to the built-in pipeline of the same workload.

    python tools/cl_plugin_timing.py [--size 1920 1080] [--reps 20] [--out FILE] [--device-api]

Rows: lt_stats.kernel_ms (CUDA events around the launches of one call), best and median of --reps calls after two
warm-up calls, Cornell box, default camera.  cl_barycentric.cl is set against the built-in custom_opencl.cl pipeline
(barycentric colour of the primary hit); cl_direct_light.cl (one light sample with a shadow ray) against the built-in
accumulator.cl pipeline, which also traces one camera ray and one shadow ray per pixel.  Also prints the translation +
NVRTC compile time of each test kernel and the card's name and power limit, read in the same run.

--device-api times the global-illumination kernel on the plug-in device API instead, one frame of 4 bounces:
tests/plugins/gi_plugin.cl (the example's GI kernel ported to lens_trace_b200_device_cl.h, launched with
lt_render_plugin_cl's defaults), tests/plugins/gi_plugin.cu (8x8 blocks) and the built-in LT_KERNEL_GI pipeline; and,
when oracle/_ref is built, the reference's unmodified example GI text as a .cl plug-in.  That text walks its own
64-entry stack over the 32-byte nodes and keeps the example's cap of 16 bounces, so it is set against the built-in
pipeline at 16 bounces."""
import argparse
import os
import subprocess
import sys
import tempfile
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
    ap.add_argument("--device-api", action="store_true", help="time the GI kernel on the device API (see above)")
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
    names = ("gi_plugin.cl",) if a.device_api else ("cl_barycentric.cl", "cl_direct_light.cl", "cl_tile_groups.cl")
    for name in names:
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
    if a.device_api:
        def row(label, fn):
            b, m = timed(fn)
            say("  %-44s %8.3f / %8.3f ms" % (label, b, m))

        cl = ctx.plugin_load(os.path.join(plugins, "gi_plugin.cl"))
        cu = ctx.plugin_load(os.path.join(plugins, "gi_plugin.cu"))
        row("gi_plugin.cl (device API), 4 bounces", lambda: ctx.render_plugin_cl(sc, cam, cl, w, h))
        row("gi_plugin.cu (device API, 8x8), 4 bounces", lambda: ctx.render_plugin(sc, cam, cu, w, h, block=(8, 8)))
        row("built-in LT_KERNEL_GI, 4 bounces", lambda: ctx.render(
            sc, cam, capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4)))
        ref = os.path.join(ROOT, "oracle", "_ref", "cl", "global_illumination_example.inc")
        if os.path.exists(ref):
            with tempfile.TemporaryDirectory() as d:
                path = os.path.join(d, "global_illumination.cl")
                with open(path, "w") as f:
                    f.write(open(ref).read())
                own = ctx.plugin_load(path)
            row("reference example GI text (.cl), 16 bounces", lambda: ctx.render_plugin_cl(sc, cam, own, w, h))
            row("built-in LT_KERNEL_GI, 16 bounces", lambda: ctx.render(
                sc, cam, capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=16)))
        else:
            say("  reference example GI text: not measured (oracle/_ref is not built)")
    else:
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
