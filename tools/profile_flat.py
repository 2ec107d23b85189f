#!/usr/bin/env python3
"""Primary rays (basic.cu pipeline, k_flat) on a scene, timed; meant to be run plain and under ncu:

    python tools/profile_flat.py [synth:707|cornell_box] [W H] [reps]
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import bench  # noqa: E402
from lens_trace_b200 import capi, layouts as L  # noqa: E402


def main():
    model = sys.argv[1] if len(sys.argv) > 1 else "synth:707"
    w = int(sys.argv[2]) if len(sys.argv) > 2 else 1920
    h = int(sys.argv[3]) if len(sys.argv) > 3 else 1080
    reps = int(sys.argv[4]) if len(sys.argv) > 4 else 5
    flags = int(os.environ.get("LT_PROFILE_FLAGS", "0"))
    sb = bench.load_scene(model)
    ctx = capi.Context(0)
    scene = ctx.upload(sb)
    cam = L.make_camera(0, 2.5, -50)
    for kernel in (L.KERNEL_BASIC_CU, L.KERNEL_ACCUMULATOR):
        p = capi.make_params(kernel, w, h, flags=flags)
        ms = []
        for _ in range(reps):
            ctx.render(scene, cam, p, want_output=False)
            ms.append(ctx.stats().kernel_ms)
        knobs = " ".join("%s=%s" % (k, v) for k, v in sorted(os.environ.items()) if k.startswith(("LT_STREAM", "LT_THREADED", "LT_PROFILE_FLAGS")))
        print("%s kernel %d %dx%d [%s]: ms %s" % (model, kernel, w, h, knobs, " ".join("%.4f" % m for m in ms)), flush=True)
    if not os.environ.get("LT_PROFILE_NOREF"):
        ref = bench.reference_cuda_kernel_rate(sb, w, h)
        print("reference basic.cu:", ref, flush=True)
    scene.release()
    ctx.close()


if __name__ == "__main__":
    main()
