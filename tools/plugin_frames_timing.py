"""Cost of rendering a plug-in kernel many frames per call (lt_render_plugin_frames) against the reference's protocol
and the built-in pipeline of the same workload.

    python tools/plugin_frames_timing.py [--size 1920 1080] [--frames 64] [--reps 5] [--gpus 1 2 4 8] [--out FILE]

Workload: tests/plugins/gi_plugin.cu (the example's GI kernel on the device API, 4 bounces), Cornell box, default
camera, RUNNING_MEAN from frameCount 0.  Rows, best and median of --reps after one warm-up:
  - one lt_render_plugin_frames call;
  - the reference protocol: --frames lt_render_plugin calls, each copied to the host and folded into a host running
    mean (numpy, FP32);
  - the built-in LT_KERNEL_GI call of the same frames (lt_render).
kernel = lt_stats.kernel_ms (CUDA events around the call's launches; for the protocol the sum over its calls), wall =
host clock around the call(s) including the copy to a pageable host buffer.
k_plugin_accumulate: per-launch device time from torch.profiler (CUDA activities) over one call, against the bytes it
moves per frame (3 floats read from the sample, 3 read and 3 written in the accumulator per pixel).
Then the same plug-in call on 1, 2, 4, 8 GPUs of one multi-GPU context (sample split), as many as the machine has.
The card's name and power limit are read in the same run."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

from lens_trace_b200 import capi, host, layouts as L  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, nargs=2, default=(1920, 1080))
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--gpus", type=int, nargs="*", default=[1, 2, 4, 8])
    ap.add_argument("--out")
    a = ap.parse_args()
    w, h, F = a.size[0], a.size[1], a.frames
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    say("card: %s (%d visible)" % (gpu[0] if gpu else "unknown", len(gpu)))
    sb = host.load_scene_buffers(os.path.join(ROOT, "resources", "models", "cornell_box.obj"))
    gi = os.path.join(ROOT, "tests", "plugins", "gi_plugin.cu")
    cam = L.make_camera(0, 2.5, -50, 0.0, 0)

    def params(kernel=0, **kw):
        p = capi.make_params(kernel, w, h, frames=F, accum_mode=L.ACCUM_RUNNING_MEAN, **kw)
        p.block_x, p.block_y = 8, 8
        return p

    def timed(fn):
        fn()
        ks, ws = [], []
        for _ in range(a.reps):
            t = time.perf_counter()
            k = fn()
            ws.append((time.perf_counter() - t) * 1e3)
            ks.append(k)
        return "kernel %8.2f / %8.2f ms   wall %8.2f / %8.2f ms" % (min(ks), np.median(ks), min(ws), np.median(ws))

    ctx = capi.Context(0)
    sc = ctx.upload(sb)
    pid = ctx.plugin_load(gi)

    def one_call():
        ctx.render_plugin_frames(sc, cam, pid, params())
        return ctx.stats().kernel_ms

    def protocol():
        acc = np.zeros((h, w, 3), np.float32)
        k_ms = 0.0
        for k in range(F):
            s = ctx.render_plugin(sc, L.make_camera(0, 2.5, -50, 0.0, k), pid, w, h, block=(8, 8))
            k_ms += ctx.stats().kernel_ms
            acc = s if k == 0 else (s + acc * np.float32(k)) / np.float32(k + 1)
        return k_ms

    def builtin():
        ctx.render(sc, cam, params(L.KERNEL_GI, max_ray_depth=4))
        return ctx.stats().kernel_ms

    say("gi_plugin.cu, %dx%d, %d frames, 4 bounces, Cornell box; best / median of %d" % (w, h, F, a.reps))
    say("  lt_render_plugin_frames, one call       %s" % timed(one_call))
    say("  %d lt_render_plugin calls + host mean   %s" % (F, timed(protocol)))
    say("  built-in LT_KERNEL_GI, one lt_render    %s" % timed(builtin))

    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        one_call()
        torch.cuda.synchronize()
    fold = [e for e in prof.events() if e.name == "k_plugin_accumulate" or e.name.startswith("k_plugin_accumulate(")]
    if fold:
        us = np.array([e.device_time_total for e in fold], np.float64)
        moved = 36.0 * w * h
        say("k_plugin_accumulate: %d launches, %.1f us mean, %.1f us min per frame; %.1f MB per frame -> %.2f TB/s at "
            "the mean" % (len(us), us.mean(), us.min(), moved / 1e6, moved / (us.mean() * 1e-6) / 1e12))
    else:
        say("k_plugin_accumulate: not found in the profile (not measured)")
    sc.release()
    ctx.close()

    have = torch.cuda.device_count()
    for n in a.gpus:
        if n > have:
            say("%d GPUs: not measured (%d visible)" % (n, have))
            continue
        g = capi.Context(list(range(n)))
        gs = g.upload(sb)
        gp = g.plugin_load(gi)

        def group_call():
            g.render_plugin_frames(gs, cam, gp, params(split_mode=L.SPLIT_SAMPLES))
            return g.stats().kernel_ms

        say("%d GPU%s, sample split                    %s" % (n, "" if n == 1 else "s", timed(group_call)))
        gs.release()
        g.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
