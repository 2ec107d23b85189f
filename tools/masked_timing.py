"""Cost of masked continuation (lt_render_masked_device) against the unmasked call (lt_render_device), and an adaptive
loop against uniform sampling.

    python tools/masked_timing.py [--reps 3] [--out FILE]

Workloads: GI, 4 bounces, 1080p, running mean.  On the Cornell box and the synthetic 1 M-triangle mesh, a 16-frame
continuation from frameCount 16:
  - unmasked: lt_render_device;
  - NULL mask and full mask: lt_render_masked_device over every pixel;
  - mask fractions 0.5, 0.25 and 0.1: seeded random masks (the pixels scattered over the image), under the planner's
    schedule and with each schedule forced (LT_FLAG_MEGAKERNEL, LT_FLAG_WAVEFRONT).
Crossover rows (Cornell box): scattered masks of N = 2^12 .. 2^20 pixels, 1, 4 and 16 frames, each schedule forced.
Each call includes what the masked form adds: the compaction kernel and, with a mask, the readback of the list's length
(one 4-byte copy and a stream synchronisation).  Timed on one stream with device events and one synchronise per
repetition; every configuration runs once as warm-up; the figures are the median of --reps repetitions.
Adaptive loop on the Cornell box: 16 frames on every pixel with m2, then up to three rounds of 16 frames on the pixels
whose relative standard error (sqrt(m2 / (n (n - 1))) / mean, largest channel) is above the threshold, against 64
uniform frames; pixel-frames rendered, wall time (host clock around the whole loop, torch's error computation included)
and the fraction of pixels that stopped before 64 frames, under the planner's schedule and forced onto the wavefront.  The card's name and power limit are read in the same run."""
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
    path = os.path.join(tempfile.gettempdir(), "lt_masked_synth_%d_%d.obj" % (grid_n, os.getpid()))
    host.write_synthetic_scene(path, grid_n, 0x5EED)
    sb = host.load_scene_buffers(path)
    for p in (path, path[:-4] + ".mtl"):
        if os.path.exists(p):
            os.remove(p)
    return sb


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--threshold", type=float, default=0.05)
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
    cam16 = L.make_camera(0, 2.5, -50, 0.0, 16)

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

    props = torch.cuda.get_device_properties(0)
    say("rows: scene, what, ms per 16-frame 1080p GI continuation, against unmasked, planned pipeline")
    for name in ("cornell_box", "synth1m"):
        sc, sb = uploaded[name], scenes[name]
        p = params(16)
        out = torch.rand((h, w, 3), dtype=torch.float32, device="cuda")
        m2 = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        base = timed(lambda: ctx.render_device(sc, cam16, p, out.data_ptr()))
        plan = capi.plan(p, len(sb.nodes), 8, props.total_memory, props.multi_processor_count)["pipeline"]
        say("%-12s %-22s %9.3f ms   1.000x   pipeline %d" % (name, "unmasked", base, plan))
        t = timed(lambda: ctx.render_masked_device(sc, cam16, p, out.data_ptr()))
        say("%-12s %-22s %9.3f ms   %.3fx   pipeline %d" % (name, "NULL mask", t, t / base, plan))
        t = timed(lambda: ctx.render_masked_device(sc, cam16, p, out.data_ptr(), None, m2.data_ptr()))
        say("%-12s %-22s %9.3f ms   %.3fx   pipeline %d" % (name, "NULL mask + m2", t, t / base, plan))
        g = torch.Generator(device="cuda").manual_seed(1)
        for frac in (1.0, 0.5, 0.25, 0.1):
            mask = (torch.rand((h, w), generator=g, device="cuda") < frac).to(torch.uint8)
            n = int(mask.sum())
            pm = capi.plan_masked(p, n, len(sb.nodes), 8, props.total_memory, props.multi_processor_count)["pipeline"]
            torch.cuda.synchronize()
            t = timed(lambda: ctx.render_masked_device(sc, cam16, p, out.data_ptr(), mask.data_ptr()))
            say("%-12s %-22s %9.3f ms   %.3fx   pipeline %d   (%d pixels)" % (
                name, "mask %.2f" % frac, t, t / base, pm, n))
            if frac < 1.0:  # both schedules, whichever the planner takes
                for label, flags in (("megakernel", L.FLAG_MEGAKERNEL), ("wavefront", L.FLAG_WAVEFRONT)):
                    q = params(16, flags)
                    t = timed(lambda: ctx.render_masked_device(sc, cam16, q, out.data_ptr(), mask.data_ptr()))
                    say("%-12s %-22s %9.3f ms   %.3fx" % (name, "mask %.2f %s" % (frac, label), t, t / base))
        del out, m2
        torch.cuda.empty_cache()

    say("crossover: cornell_box, scattered random masks of N pixels, ms per call, megakernel against wavefront")
    sc = uploaded["cornell_box"]
    out = torch.rand((h, w, 3), dtype=torch.float32, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(2)
    for n in (1 << 12, 1 << 14, 1 << 16, 1 << 18, 1 << 20):
        idx = torch.randperm(h * w, generator=g, device="cuda")[:n]
        mask = torch.zeros(h * w, dtype=torch.uint8, device="cuda")
        mask[idx] = 1
        torch.cuda.synchronize()
        for frames in (1, 4, 16):
            row = []
            for label, flags in (("megakernel", L.FLAG_MEGAKERNEL), ("wavefront", L.FLAG_WAVEFRONT)):
                q = params(frames, flags)
                t = timed(lambda: ctx.render_masked_device(sc, cam16, q, out.data_ptr(), mask.data_ptr()))
                row.append("%s %8.3f" % (label, t))
            pm = capi.plan_masked(params(frames), n, len(scenes["cornell_box"].nodes), 8, props.total_memory,
                                  props.multi_processor_count)["pipeline"]
            say("N=%-8d F=%-3d paths=%-9d %s   planner: pipeline %d" % (n, frames, n * frames, "   ".join(row), pm))
    del out
    torch.cuda.empty_cache()

    say("adaptive loop, cornell_box, threshold %.3g on the relative standard error, against 64 uniform frames" %
        a.threshold)
    sc = uploaded["cornell_box"]
    cam = [L.make_camera(0, 2.5, -50, 0.0, k) for k in (0, 16, 32, 48)]
    for label, p in (("planner's schedule", params(16)), ("wavefront", params(16, L.FLAG_WAVEFRONT))):
        adaptive(a, ctx, stream, say, w, h, label, p, sc, cam)
    for sc in uploaded.values():
        sc.release()
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


def adaptive(a, ctx, stream, say, w, h, label, p, sc, cam):
    import torch
    for rep in range(2):  # the first is the warm-up
        out = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(4):
            ctx.render_device(sc, cam[k], p, out.data_ptr())
        torch.cuda.synchronize()
        uniform = (time.perf_counter() - t0) * 1e3
        with torch.cuda.stream(stream):
            out = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
            m2 = torch.zeros_like(out)
            n = torch.full((h, w), 16, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctx.render_masked_device(sc, cam[0], p, out.data_ptr(), None, m2.data_ptr())
            rounds = []
            for k in range(1, 4):
                nf = n.to(torch.float32)[..., None]
                err = (torch.sqrt(m2 / (nf * (nf - 1))) / out.clamp_min(1e-4)).amax(dim=2)
                mask = ((err > a.threshold) & (n == 16 * k)).to(torch.uint8)
                ctx.render_masked_device(sc, cam[k], p, out.data_ptr(), mask.data_ptr(), m2.data_ptr())
                n += 16 * mask.to(torch.int32)
                rounds.append(mask)
            torch.cuda.synchronize()
            t_adaptive = (time.perf_counter() - t0) * 1e3
    listed = [int(m.sum()) for m in rounds]
    frames = int(n.sum())
    early = float((n < 64).float().mean())
    say("%s: uniform 64 frames   %d pixel-frames   %9.3f ms" % (label, w * h * 64, uniform))
    say("%s: adaptive 16+3x16    %d pixel-frames   %9.3f ms   (%.3f of uniform)   pixels per round %s   "
        "stopped early %.3f" % (label, frames, t_adaptive, t_adaptive / uniform, listed, early))


if __name__ == "__main__":
    main()
