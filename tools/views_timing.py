"""Cost per view of rendering V camera views in one call (lt_render_views_device) against V single calls
(lt_render_device), and the crossover of the view planner.

    python tools/views_timing.py [--reps 3] [--out FILE]

Workloads: GI, 4 bounces, 1080p, running mean from each view's frameCount; V views of the Cornell box with different
positions, yaws and frameCounts at V in {8, 64} x F in {1, 16}, and the synthetic 1 M-triangle mesh at V = 8, F = 1.
Each row times, on one stream with device events and one synchronise at the end of each repetition:
  - views: one lt_render_views_device call of V views (the planner's schedule);
  - singles: V lt_render_device calls, one per view (the planner's schedule for one view).
Crossover rows (Cornell box, F = 1, V in {1, 2, 4, 8, 16}): the views call forced onto the megakernel (one launch per
view) and onto the wavefront (the views' pairs in one launch).  Every configuration runs once as warm-up; the figures
are the median of --reps repetitions, in ms per view.  The card's name and power limit are read in the same run."""
import argparse
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

from lens_trace_b200 import capi, host, layouts as L  # noqa: E402

PIPES = {capi.PIPE_FLAT: "k_flat", capi.PIPE_FLAT_STREAM: "k_flat_stream", capi.PIPE_PATH: "k_path",
         capi.PIPE_WAVEFRONT: "wavefront"}


def cameras(n):
    rng = np.random.default_rng(n)
    cams = [L.make_camera(float(rng.uniform(-3, 3)), float(rng.uniform(1.5, 3.5)), float(rng.uniform(-55, -45)),
                          float(rng.uniform(-0.06, 0.06)), int(rng.integers(0, 32))) for _ in range(n)]
    return np.concatenate(cams)


def synthetic_scene(grid_n):
    path = os.path.join(tempfile.gettempdir(), "lt_views_synth_%d_%d.obj" % (grid_n, os.getpid()))
    host.write_synthetic_scene(path, grid_n, 0x5EED)
    sb = host.load_scene_buffers(path)
    for p in (path, path[:-4] + ".mtl"):
        if os.path.exists(p):
            os.remove(p)
    return sb


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
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
    w, h = 1920, 1080
    ctx = capi.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    scenes = {"cornell_box": host.load_scene_buffers(os.path.join(ROOT, "resources", "models", "cornell_box.obj")),
              "synth1m": synthetic_scene(707)}
    uploaded = {k: ctx.upload(v) for k, v in scenes.items()}

    def params(frames, flags=0):
        return capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN,
                                flags=flags)

    def timed(fn):
        times = []
        for rep in range(a.reps + 1):  # the first is the warm-up
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            torch.cuda.synchronize()
            if rep:
                times.append(e0.elapsed_time(e1))
        return float(np.median(times))

    def plan_name(p, v, sb):
        return PIPES[capi.plan_views(p, v, len(sb.nodes), 8, torch.cuda.get_device_properties(0).total_memory,
                                     torch.cuda.get_device_properties(0).multi_processor_count)["pipeline"]]

    say("rows: scene, V, F, views call ms/view (plan), V single calls ms/view (plan), singles / views")
    for name, V, F in (("cornell_box", 8, 1), ("cornell_box", 8, 16), ("cornell_box", 64, 1), ("cornell_box", 64, 16),
                       ("synth1m", 8, 1)):
        sc, sb = uploaded[name], scenes[name]
        cams = cameras(V)
        p = params(F)
        out = torch.zeros((V, h, w, 3), dtype=torch.float32, device="cuda")
        image = h * w * 3 * 4

        def views():
            ctx.render_views_device(sc, cams, p, out.data_ptr(), sync=False)

        def singles():
            for v in range(V):
                ctx.render_device(sc, cams[v:v + 1], p, out.data_ptr() + v * image, sync=False)

        tv, ts = timed(views), timed(singles)
        say("%-12s V=%-3d F=%-3d views %8.3f ms/view (%s)   singles %8.3f ms/view (%s)   %.3fx" % (
            name, V, F, tv / V, plan_name(p, V, sb), ts / V, plan_name(p, 1, sb), ts / tv))
        del out
        torch.cuda.empty_cache()

    say("crossover: cornell_box, F=1, views call per schedule, ms/view")
    for V in (1, 2, 4, 8, 16):
        sc = uploaded["cornell_box"]
        cams = cameras(V)
        out = torch.zeros((V, h, w, 3), dtype=torch.float32, device="cuda")
        row = []
        for label, flags in (("megakernel", L.FLAG_MEGAKERNEL), ("wavefront", L.FLAG_WAVEFRONT)):
            p = params(1, flags)
            t = timed(lambda: ctx.render_views_device(sc, cams, p, out.data_ptr(), sync=False))
            row.append("%s %8.3f" % (label, t / V))
        say("V=%-3d paths=%-9d %s   planner: %s" % (V, V * w * h, "   ".join(row),
                                                     plan_name(params(1), V, scenes["cornell_box"])))
        del out
        torch.cuda.empty_cache()
    for sc in uploaded.values():
        sc.release()
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
