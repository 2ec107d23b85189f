"""Cost of moving an uploaded scene's triangles: lt_scene_refit and lt_scene_refit_device against a new lt_scene_upload
of the same buffers, and what a refit costs in tree quality.

    python tools/refit_timing.py [--reps 5] [--out FILE]

Scenes: the Cornell box, and the synthetic meshes of grid 122 (about 30 K triangles, about 60 K nodes: host-built
threaded copies near their 65 536-node limit), 707 (1 M triangles) and 1581 (5 M triangles).  The deformation is a
sine displacement of y.  Each call is timed on the host around the synchronous call (both entry points return when
the scene is ready), and its device time is lt_stats.upload_ms; the figures are the median of --reps repetitions after
one warm-up.  For refit_device the primitives are already in a torch CUDA tensor.  The upload row includes the
host-side checks and the host pass of small trees, as a caller replacing a scene would pay them.

Tree quality: one 16-spp 1080p GI frame (4 bounces) of the deformed 1 M mesh, rendered on the refitted tree (the
median split of the undeformed mesh) and on a fresh lt_scene_build_ploc of the deformed mesh; median of --reps
renders, device events on the context's stream.  The card's name and power limit are read in the same run."""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

from lens_trace_b200 import capi, host, layouts as L  # noqa: E402


def synthetic_scene(grid_n):
    path = os.path.join(tempfile.gettempdir(), "lt_refit_synth_%d_%d.obj" % (grid_n, os.getpid()))
    host.write_synthetic_scene(path, grid_n, 0x5EED)
    sb = host.load_scene_buffers(path)
    for p in (path, path[:-4] + ".mtl"):
        if os.path.exists(p):
            os.remove(p)
    return sb


def sine(prims, amp=0.02):
    out = prims.copy()
    for k in ("a", "b", "c"):
        v = out[k].astype(np.float64)
        v[:, 1] += amp * np.sin(3.0 * v[:, 0] + 2.0 * v[:, 2])
        out[k] = v.astype(np.float32)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    say("card: %s" % (gpu[0] if gpu else "unknown"))
    ctx = capi.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)

    def timed(fn):
        host_ms, dev_ms = [], []
        for rep in range(a.reps + 1):  # the first is the warm-up
            t0 = time.perf_counter()
            fn()
            t1 = time.perf_counter()
            if rep:
                host_ms.append((t1 - t0) * 1e3)
                dev_ms.append(ctx.stats().upload_ms)
        return float(np.median(host_ms)), float(np.median(dev_ms))

    say("rows: scene, triangles, nodes; call: host ms (synchronous call), device ms (lt_stats.upload_ms)")
    scenes = [("cornell_box", host.load_scene_buffers(os.path.join(ROOT, "resources", "models", "cornell_box.obj"))),
              ("synth122", synthetic_scene(122)), ("synth707", synthetic_scene(707)),
              ("synth1581", synthetic_scene(1581))]
    kept = {}
    for name, sb in scenes:
        moved = sine(sb.prims)
        sc = ctx.upload(sb)
        dev = torch.from_numpy(moved.view(np.uint8).copy()).to("cuda:0")
        torch.cuda.synchronize()
        rows = []
        for label, fn in (("refit", lambda: ctx.refit(sc, moved)),
                          ("refit_device", lambda: ctx.refit_device(sc, dev.data_ptr(), moved.nbytes))):
            rows.append((label,) + timed(fn))
        fresh = L.SceneBuffers(ctx.download(sc)[0].nodes, moved, sb.materials, sb.lights)

        host_ms, dev_ms = [], []
        for rep in range(a.reps + 1):
            t0 = time.perf_counter()
            s = ctx.upload(fresh)
            t1 = time.perf_counter()
            d = ctx.stats().upload_ms
            s.release()
            if rep:
                host_ms.append((t1 - t0) * 1e3)
                dev_ms.append(d)
        rows.append(("upload", float(np.median(host_ms)), float(np.median(dev_ms))))
        say("%-11s %8d tris %8d nodes   %s" % (name, len(sb.prims), len(sb.nodes), "   ".join(
            "%s %9.3f / %8.3f ms" % r for r in rows)))
        if name == "synth707":
            kept = {"sb": sb, "moved": moved, "scene": sc}
        else:
            sc.release()
        del dev
        torch.cuda.empty_cache()

    sb, moved, refitted = kept["sb"], kept["moved"], kept["scene"]
    ctx.refit(refitted, moved)
    rebuilt = ctx.build_ploc(moved, sb.materials)
    w, h = 1920, 1080
    p = capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, frames=16, accum_mode=L.ACCUM_RUNNING_MEAN)
    out = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda:0")
    cam = L.make_camera(0, 2.5, -50, 0.0, 0)

    def frame_ms(sc):
        times = []
        for rep in range(a.reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ctx.render_device(sc, cam, p, out.data_ptr(), sync=False)
            e1.record(stream)
            torch.cuda.synchronize()
            if rep:
                times.append(e0.elapsed_time(e1))
        return float(np.median(times))

    say("tree quality: synth707 after the sine deformation, GI 1080p 16 spp, 4 bounces, ms per call")
    say("  refitted median-split tree %9.3f ms   fresh lt_scene_build_ploc tree %9.3f ms" % (
        frame_ms(refitted), frame_ms(rebuilt)))
    refitted.release()
    rebuilt.release()
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
