"""Times the wavefront pipeline with the stackless threaded traversal against the stack traversal, and two
overlapped batches against one stream (LT_FLAG_SERIAL); checks that the images are identical.
    python tools/tune_threaded.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import bench  # noqa: E402
from lens_trace_b200 import capi, layouts as L  # noqa: E402


def timed(ctx, sc, cam, p, n=4):
    ts, tr = [], []
    for _ in range(n):
        ctx.render(sc, cam, p, want_output=False)
        st = ctx.stats()
        ts.append(st.kernel_ms)
        tr.append(st.trace_ms)
    return min(ts[1:]), min(tr[1:])


def main():
    ctx = capi.Context(0)
    cam = L.make_camera(0, 2.5, -50)
    cases = [("cornell_box", L.KERNEL_GI, 1920, 1080, 64, 4), ("cornell_box", L.KERNEL_ACCUMULATOR, 1920, 1080, 64, 0),
             ("synth:96", L.KERNEL_GI, 1920, 1080, 16, 4), ("synth:707", L.KERNEL_GI, 1920, 1080, 16, 4)]
    for model, kernel, w, h, frames, depth in cases:
        sb = bench.load_scene(model)
        sc = ctx.upload(sb)
        base = capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN,
                                flags=L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED)
        thr = capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN,
                               flags=L.FLAG_WAVEFRONT)
        ctx.accum_reset()
        a = ctx.render(sc, cam, base).copy()
        ctx.accum_reset()
        b = ctx.render(sc, cam, thr).copy()
        same = bool((a.view(np.uint32) == b.view(np.uint32)).all())
        t0, tr0 = timed(ctx, sc, cam, base)
        t1, tr1 = timed(ctx, sc, cam, thr)
        print("%-12s k%d %d nodes frames %d: stack %.2f ms (trace %.2f)  threaded %.2f ms (trace %.2f)  x%.3f  identical=%s" % (
            model, kernel, len(sb.nodes), frames, t0, tr0, t1, tr1, t0 / t1, same), flush=True)
        ser = capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN,
                               flags=L.FLAG_WAVEFRONT | L.FLAG_SERIAL)
        ctx.accum_reset()
        c = ctx.render(sc, cam, ser)
        t2, tr2 = timed(ctx, sc, cam, ser)
        print("      one stream (LT_FLAG_SERIAL): threaded %.2f ms (trace %.2f)  identical=%s" % (
            t2, tr2, bool((c.view(np.uint32) == b.view(np.uint32)).all())), flush=True)
        sc.release()


if __name__ == "__main__":
    main()
