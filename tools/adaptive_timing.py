"""Adaptive sampling inside the library (lt_render_adaptive_device, lt_render_adaptive) against the torch loop of
INTEGRATION section 5d and against uniform sampling.

    python tools/adaptive_timing.py [--reps 3] [--out FILE]

Workload: GI, 4 bounces, 1080p, running mean, on the Cornell box and on the synthetic 1 M-triangle mesh, with the
section 5d parameters: 16 frames on every pixel, then up to three rounds of 16 frames on the pixels whose relative
standard error is above 0.05.  Rows per scene:
  (a) lt_render_adaptive_device (mean, m2 and frame counts in torch tensors);
  (b) the section 5d torch loop on lt_render_masked_device (the rule in torch float32 ops, one masked call per round);
  (c) 64 uniform frames (lt_render_device);
  (d) the host form, lt_render_adaptive, with its download of the mean and the frame counts into pageable memory;
  and, when several GPUs are present, (d) on a multi-GPU context of 2, 4 and 8 devices, with the rounds of each device.
Each row: wall time of the whole call (host clock, the work ends in a synchronise; median of --reps after one warm-up),
rounds and pixel-frames.  (a) and (b) are compared bit for bit (mean, m2, frame counts).  The card's name and power
limit are read in the same run."""
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
    path = os.path.join(tempfile.gettempdir(), "lt_adaptive_synth_%d_%d.obj" % (grid_n, os.getpid()))
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
    say("card: %s (%d visible)" % (gpu[0] if gpu else "unknown", torch.cuda.device_count()))
    w, h, F, R, MAX, THR = 1920, 1080, 16, 16, 64, 0.05
    ctx = capi.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    scenes = {"cornell_box": host.load_scene_buffers(os.path.join(ROOT, "resources", "models", "cornell_box.obj")),
              "synth1m": synthetic_scene(707)}
    cam0 = L.make_camera(0, 2.5, -50, 0.0, 0)

    def params(frames):
        return capi.make_params(L.KERNEL_GI, w, h, max_ray_depth=4, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN)

    def timed(fn):
        times, ret = [], None
        for rep in range(a.reps + 1):  # the first is the warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ret = fn()
            torch.cuda.synchronize()
            if rep:
                times.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(times)), ret

    def f32(x):
        return torch.tensor(x, dtype=torch.float32, device="cuda")

    say("rows: scene, what, ms per call (median of %d), rounds, pixel-frames (fraction of 64 uniform frames)" % a.reps)
    for name, sb in scenes.items():
        sc = ctx.upload(sb)
        out = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
        m2 = torch.zeros_like(out)
        n = torch.zeros((h, w), dtype=torch.int32, device="cuda")

        def adaptive():
            with torch.cuda.stream(stream):
                return ctx.render_adaptive_device(sc, cam0, params(F), out.data_ptr(), m2.data_ptr(), n.data_ptr(),
                                                  target=THR, round_frames=R, max_frames=MAX, sync=True)

        def loop():
            with torch.cuda.stream(stream):
                ctx.render_masked_device(sc, cam0, params(F), out.data_ptr(), None, m2.data_ptr())
                n.fill_(F)
                active = torch.ones((h, w), dtype=torch.bool, device="cuda")
                done, rounds, pf = F, 1, F * w * h
                while True:
                    d = f32(float(done)) * f32(float(done - 1))
                    err = (torch.sqrt(m2 / d) / out.clamp_min(f32(1e-4))).amax(dim=2)
                    go = (err > f32(THR)) & active
                    if done == MAX:
                        break
                    k = int(go.sum())
                    if k == 0:
                        break
                    f = min(R, MAX - done)
                    ctx.render_masked_device(sc, L.make_camera(0, 2.5, -50, 0.0, done), params(f), out.data_ptr(),
                                             go.to(torch.uint8).data_ptr(), m2.data_ptr())
                    done += f
                    n[go] = done
                    active = go
                    rounds += 1
                    pf += k * f
            return rounds, pf

        t_a, res = timed(adaptive)
        a_out, a_m2, a_n = out.clone(), m2.clone(), n.clone()
        t_b, (rounds_b, pf_b) = timed(loop)
        same = torch.equal(a_out.view(torch.int32), out.view(torch.int32)) and \
            torch.equal(a_m2.view(torch.int32), m2.view(torch.int32)) and torch.equal(a_n, n)
        t_c, _ = timed(lambda: ctx.render_device(sc, cam0, params(MAX), out.data_ptr(), sync=True))
        host_mean = np.empty((h, w, 3), np.float32)
        host_n = np.empty((h, w), np.uint32)
        lib = ctx.lib
        ap_ = capi.make_adaptive(THR, MAX, R)
        r_d = capi.AdaptiveResult()
        t_d, _ = timed(lambda: ctx._check(lib.lt_render_adaptive(ctx.h, sc.h, cam0.ctypes.data, capi.C.byref(params(F)),
                                                                 capi.C.byref(ap_), host_mean.ctypes.data,
                                                                 host_n.ctypes.data, capi.C.byref(r_d)),
                                          "lt_render_adaptive"))
        total = MAX * w * h
        say("%-12s (a) adaptive_device      %9.2f ms  rounds %d  pixel-frames %d (%.3f)  unconverged %d" % (
            name, t_a, res.rounds, res.pixel_frames, res.pixel_frames / total, res.pixels_unconverged))
        say("%-12s (b) 5d torch loop        %9.2f ms  rounds %d  pixel-frames %d (%.3f)  (a) == (b) bit for bit: %s" % (
            name, t_b, rounds_b, pf_b, pf_b / total, same))
        say("%-12s (c) 64 uniform frames    %9.2f ms  rounds 1  pixel-frames %d (1.000)" % (name, t_c, total))
        say("%-12s (d) host form + download %9.2f ms  rounds %d  pixel-frames %d (%.3f)  frame counts equal (a): %s" % (
            name, t_d, r_d.rounds, r_d.pixel_frames, r_d.pixel_frames / total,
            bool((host_n == a_n.cpu().numpy().view(np.uint32)).all())))
        say("%-12s (a) / (b) = %.3f, (a) / (c) = %.3f" % (name, t_a / t_b, t_a / t_c))
        sc.release()
        del out, m2, n, a_out, a_m2, a_n
        torch.cuda.empty_cache()

    G = torch.cuda.device_count()
    if G < 2:
        say("multi-GPU host form: not measured (one GPU visible)")
    else:
        for g in (2, 4, 8):
            if g > G:
                say("multi-GPU host form on %d devices: not measured (%d visible)" % (g, G))
                continue
            with capi.Context(list(range(g))) as multi:
                for name, sb in scenes.items():
                    sc = multi.upload(sb)
                    t, (_, _, r) = timed(lambda: multi.render_adaptive(sc, cam0, params(F), THR, R, MAX))
                    say("%-12s (d) host form on %d GPUs %9.2f ms  rounds %d  pixel-frames %d" % (
                        name, g, t, r.rounds, r.pixel_frames))
                    sc.release()
    ctx.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
