#!/usr/bin/env python3
"""bench.py -- the measurement contract of this repo.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

Default workload = BASELINE.json configs[1]: Cornell box, the global_illumination example kernel
(one sample per frame, seed = frameCount), 1920x1080, 64 frames kept as a running mean on the device,
4 bounces, one B200.  A "step" is one such 64-spp frame.  metric = Mrays/s (every BVH traversal call is
one ray: primary + shadow + GI extension), ms_per_step = ms/frame 1080p 64spp.

N > 1 (torchrun, one rank per GPU): sample split -- rank r renders frames r, r+N, ... of the frame into
its own FP32 accumulator with weight 1/frames; one NCCL all-reduce(sum) per step combines them.  Default
--scaling strong: the workload's frames are divided among the GPUs (64/N spp each); --scaling weak: every
GPU renders all of them (64*N spp).  Time = CUDA events on the stream the kernels run on, max over ranks.

--impl reference: the reference has no CPU implementation of this path and its OpenCL kernels cannot
run here (no OpenCL ICD), so this arm times the CPU restatement of the same kernel (oracle/, "port")
on all host cores, on a bounded sample of the same workload.

--dump-outputs DIR: after the timed steps, the image the last timed step produced (what a caller of the timed
path receives) is written as DIR/image.npy, float32 [H, W, 3] (--impl reference: the CPU port's frames of its last
step, DIR/frames.npy [frames, H, W, 3]).  Output above 64 MB is written as a fixed, seeded sample of its pixels
instead (DIR/image_sample.npy [n, 3] and their flat pixel indices DIR/image_sample_pixels.npy).  Inputs depend
only on the arguments, so two builds of the project can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from lens_trace_b200 import layouts as L  # noqa: E402

WORKLOADS = {
    # name: (model, kernel, width, height, frames, max_ray_depth, description)
    "cornell_gi_1080p_64spp": ("cornell_box", L.KERNEL_GI, 1920, 1080, 64, 4,
                               "Cornell box, global_illumination example kernel, 1080p, 64 spp running mean, 4 bounces"),
    "cornell_primary_512": ("cornell_box", L.KERNEL_BASIC_CL, 512, 512, 1, 0,
                            "Cornell box, basic kernel, 512x512 primary rays 1 spp"),
    "cornell_custom_1080p_16": ("cornell_box", L.KERNEL_CUSTOM_BARY, 1920, 1080, 16, 0,
                                "custom_kernel (barycentric) on the Cornell OBJ, 1080p, 16 accumulated frames"),
    "synth1m_shadow_1080p": ("synth:707", L.KERNEL_ACCUMULATOR, 1920, 1080, 1, 0,
                             "synthetic 1M-triangle mesh, primary + shadow rays, 1080p 1 spp"),
    "synth1m_gi_1080p_16spp": ("synth:707", L.KERNEL_GI, 1920, 1080, 16, 4,
                               "synthetic 1M-triangle mesh, GI 4 bounces, 1080p 16 spp"),
    "synth5m_gi_4k_256spp": ("synth:1581", L.KERNEL_GI, 3840, 2160, 256, 4,
                             "synthetic 5M-triangle mesh, GI 4 bounces, 4K 256 spp"),
}
DEFAULT_WORKLOAD = "cornell_gi_1080p_64spp"
DUMP_MAX_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, name, image):
    """Writes the float32 [..., 3] image(s) of the last timed step as out_dir/<name>.npy, or, above DUMP_MAX_BYTES, a
    fixed sample of their pixels (seed 0) as <name>_sample.npy [n, 3] with the flat pixel indices in
    <name>_sample_pixels.npy (see --dump-outputs)."""
    os.makedirs(out_dir, exist_ok=True)
    image = np.ascontiguousarray(image, dtype=np.float32)
    if image.nbytes <= DUMP_MAX_BYTES:
        np.save(os.path.join(out_dir, name + ".npy"), image)
        return
    flat = image.reshape(-1, image.shape[-1])
    n = (DUMP_MAX_BYTES - 4096) // (flat.shape[1] * 4 + 8)  # a pixel row + its float64 index; 4 KB for the headers
    pixels = np.sort(np.random.default_rng(0).choice(len(flat), size=n, replace=False))
    np.save(os.path.join(out_dir, name + "_sample.npy"), flat[pixels])
    np.save(os.path.join(out_dir, name + "_sample_pixels.npy"), pixels.astype(np.float64))


def load_scene(model, kind=0):
    """kind: AccelerationStructureExplicitType (0 = the reference's median split, 101 = binned SAH, opt-in)"""
    from lens_trace_b200 import host
    if model.startswith("synth:"):
        n = int(model.split(":")[1])
        path = os.path.join(tempfile.gettempdir(), "lt_synth_%d_%d.obj" % (n, os.getpid()))
        host.write_synthetic_scene(path, n, 0x5EED)
        sb = host.load_scene_buffers(path, kind)
        for p in (path, path[:-4] + ".mtl"):
            try:
                os.remove(p)
            except OSError:
                pass
        return sb
    return host.load_scene_buffers(os.path.join(ROOT, "resources", "models", model + ".obj"), kind)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "sm_max_mhz": d.get("sm_max_mhz", 1965.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe): one
    nvidia-smi process streaming a sample every 50 ms between start() and summary()."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.15)  # let the first sample land before the timed region starts
        except Exception:
            self.proc = None

    def summary(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ""
        samples = []
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 6:
                try:
                    float(f[0])
                    samples.append(f)
                except ValueError:
                    pass
        if not samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi gave no samples"]}
        sm = sorted(float(s[0]) for s in samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": float(samples[0][1]), "reasons": reasons,
                "samples": len(sm)}


def cpu_oracle_rate(sb, kernel, w, h, depth, frame_list, threads=0, images=None):
    """Mrays/s of the CPU restatement on `frame_list` full frames; returns (mrays_s, rays, seconds, cores).
    The rendered frames are appended to `images` when it is a list."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lt_oracle as O
    cores = os.cpu_count() or 1
    rays, t = 0, 0.0
    for f in frame_list:
        cam = L.make_camera(0, 2.5, -50, 0.0, f)
        t0 = time.perf_counter()
        img, st = O.render(kernel, sb, cam, w, h, max_ray_depth=depth if depth else 16, threads=threads, with_stats=True)
        t += time.perf_counter() - t0
        rays += st.rays
        if images is not None:
            images.append(img)
    return rays / t / 1e6, rays, t, (threads if threads > 0 else cores)


def cpu_reference_text_seconds(sb, kernel, w, h, depth, frame_list):
    """Seconds the reference's OWN kernel file takes on the host cores for `frame_list` full frames: its OpenCL C
    text compiled for the CPU through oracle/cl_shim (oracle/_ref/libltref_cl.so, built where /root/reference
    exists and shipped with the repo snapshot) -- the stand-in for the north star's "OpenCL backend on a CPU
    device (POCL)", which cannot be installed here.  None when the library is absent or the kernel has no .cl file."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lt_ref_cl as R
    if not R.available() or not (1 <= kernel <= 6):
        return None
    t = 0.0
    for f in frame_list:
        cam = L.make_camera(0, 2.5, -50, 0.0, f)
        t0 = time.perf_counter()
        R.render(kernel, sb, cam, w, h, max_ray_depth=depth if depth else 16, threads=0)
        t += time.perf_counter() - t0
    return t


def shared_config(workload, total_frames):
    """The `config` object both arms print (identical keys and values, so the two lines can be matched)."""
    model, kernel, w, h, frames, depth, desc = WORKLOADS[workload]
    return {"workload": workload, "description": desc, "width": w, "height": h, "frames_per_step": total_frames,
            "max_ray_depth": depth}


def run_reference(args, rank, world):
    """--impl reference: the reference's kernel on the CPU, all host cores, bounded sample per step.  The reference's
    own kernel text (oracle/_ref/libltref_cl.so) when it is present, else the CPU port (oracle/lt_oracle.c); the ray
    count of a frame always comes from the port's counters.  A step here is a bounded SAMPLE of the workload's step
    (per_step of its frames at full size): value is a rate, ms_per_step is what one sample really took."""
    if rank != 0:
        return
    model, kernel, w, h, frames, depth, desc = WORKLOADS[args.workload]
    total_frames = frames if args.scaling == "strong" else frames * world
    sb = load_scene(model)
    per_step = max(1, min(frames, 2))
    cpu_oracle_rate(sb, kernel, w, h, depth, [0])  # warm-up (page in, build)
    use_text = cpu_reference_text_seconds(sb, kernel, w, h, depth, [0]) is not None
    for i in range(max(0, args.warmup - 1)):
        cpu_oracle_rate(sb, kernel, w, h, depth, [i])
    rays, secs, port_secs, cores = 0, 0.0, 0.0, 1
    frames_out = []
    for s in range(args.steps):
        fl = [s * per_step + k for k in range(per_step)]
        frames_out.clear()
        _, r, t, cores = cpu_oracle_rate(sb, kernel, w, h, depth, fl, images=frames_out)
        rays += r
        port_secs += t
        secs += cpu_reference_text_seconds(sb, kernel, w, h, depth, fl) if use_text else t
    if args.dump_outputs and frames_out:
        # the CPU port's frames of the last step, [per_step, H, W, 3]
        dump_outputs(args.dump_outputs, "frames", np.stack(frames_out))
    value = rays / secs / 1e6
    sample = "%d of the %d frames per step at full %dx%d (frameCount = step*%d + k)" % (per_step, frames, w, h, per_step)
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(args.workload, total_frames),
        "config_detail": {"sample_per_step": sample,
                          "whole_step_ms_extrapolated": secs / args.steps * 1e3 * (total_frames / per_step),
                          "bvh": "built by this repo's deterministic median-split builder (lens_trace_b200.host: "
                                 "Model + AccelerationStructureExplicit), because the reference's builder reads "
                                 "uninitialised memory and gives a different tree per run; no repo kernel runs in "
                                 "this arm, the timed compute is oracle/_ref/libltref_cl.so (the reference's kernel text)"},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": "reference" if use_text else "port",
                         "sample": sample, "port_value": rays / port_secs / 1e6,
                         "what": "the reference's own kernel file compiled for the CPU (oracle/cl_shim), std::thread over "
                                 "image rows; port_value = the C restatement (oracle/lt_oracle.c)" if use_text else
                                 "C restatement of the reference kernel (oracle/lt_oracle.c), pthreads over image rows"},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def reference_cuda_kernel_rate(sb, w, h):
    """The reference's own CUDA backend on this GPU, primary rays (its only CUDA kernel, basic.cu), same scene
    and size -- context for the north star's 10x target.  Two numbers, as SURVEY.md 8(d) asks:
      kernel only : NVRTC build of its basic.cu launched on resident buffers, CUDA events (ltref_time_kernel)
      as shipped  : wall time of RendererCUDA::render() -- per call it JIT-loads the module, allocates and
                    uploads five buffers, launches, synchronises and copies the frame back (pageable memory)
    None when oracle/_ref is absent."""
    import ctypes as C
    lib_path = os.path.join(ROOT, "oracle", "_ref", "libltref.so")
    kpath = os.path.join(ROOT, "oracle", "_ref", "resources", "kernels", "cuda", "basic.cu")
    if not (os.path.exists(lib_path) and os.path.exists(kpath)):
        return None
    try:
        lib = C.CDLL(lib_path)
        vp, u64 = C.c_void_p, C.c_uint64
        lib.ltref_renderer_cuda_create.restype = vp
        lib.ltref_time_kernel.restype = C.c_double
        lib.ltref_time_kernel.argtypes = [C.c_char_p, C.c_char_p, vp, u64, vp, u64, vp, u64, vp, u64, vp, u64, u64, u64,
                                          C.c_uint, C.c_uint, C.c_int, C.c_int, vp]
        renderer = lib.ltref_renderer_cuda_create()
        cam = L.make_camera(0, 2.5, -50)
        res = {}
        for bx, by in ((32, 1), (8, 8)):
            ms = lib.ltref_time_kernel(kpath.encode(), b"linearKernel", sb.nodes.ctypes.data, sb.nodes.nbytes,
                                       sb.prims.ctypes.data, sb.prims.nbytes, sb.materials.ctypes.data,
                                       sb.materials.nbytes, sb.lights.ctypes.data, sb.lights.nbytes, cam.ctypes.data,
                                       w, h, 3, bx, by, 3, 10, None)
            if ms > 0:
                res["block_%dx%d" % (bx, by)] = {"ms": ms, "mrays_s": w * h / ms / 1e3}
        # as shipped: the reference's own objects (its Model/AS of the Cornell box) through RendererCUDA::render
        obj = os.path.join(ROOT, "oracle", "_ref", "resources", "models", "cornell_box.obj")
        if os.path.exists(obj) and len(sb.prims) == 42:
            for n in ("ltref_model_create", "ltref_as_create", "ltref_camera_create"):
                getattr(lib, n).restype = vp
            lib.ltref_model_create.argtypes = [C.c_char_p]
            lib.ltref_as_create.argtypes = [vp]
            lib.ltref_camera_create.argtypes = [C.c_float] * 4
            lib.ltref_render_cuda.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, u64, u64, u64, u64, u64, vp, u64, vp, vp,
                                              vp]
            lib.ltref_render_cuda.restype = None
            model = lib.ltref_model_create(obj.encode())
            accel = lib.ltref_as_create(model)
            rcam = lib.ltref_camera_create(0, 2.5, -50, 0)
            out = np.zeros((h, w, 3), np.float32)
            times = []
            for i in range(6):
                t0 = time.perf_counter()
                lib.ltref_render_cuda(renderer, kpath.encode(), 0, 0, 0, 0, w, h, 3, out.ctypes.data, out.nbytes, accel,
                                      model, rcam)
                times.append((time.perf_counter() - t0) * 1e3)
            res["render_as_shipped_ms"] = sorted(times[1:])[len(times[1:]) // 2]
        return res or None
    except Exception as e:  # pragma: no cover
        return {"error": str(e)}


def this_repo_render_call_ms(w, h):
    """Wall time of this repo's RendererCUDA::render() for the same call (scene cached after the first call,
    kernel, D2H into a malloc'ed host buffer)."""
    from lens_trace_b200 import host
    cwd = os.getcwd()
    os.chdir(ROOT)
    try:
        cam = host.Camera(0, 2.5, -50, 0)
        model = host.Model("resources/models/cornell_box.obj")
        accel = host.AccelerationStructure(model)
        r = host.Renderer(host.PLATFORM_CUDA)
        out = np.zeros((h, w, 3), np.float32)
        times = []
        for i in range(6):
            t0 = time.perf_counter()
            r.render("resources/kernels/cuda/basic.cu", w, h, accel, model, cam, out=out)
            times.append((time.perf_counter() - t0) * 1e3)
        r.close(); accel.close(); model.close(); cam.close()
        return sorted(times[1:])[len(times[1:]) // 2]
    finally:
        os.chdir(cwd)


def gather_ceiling(ctx, traversal_bytes):
    """Measured ceilings of the node fetches (SURVEY.md 8(d), VERDICT r1 #3): the rate the device sustains for per-lane
    32-byte gathers (lt_debug_gather_peak, lens_trace_b200/csrc/lt_microbench.cu), measured live on (i) a 21 KB table
    -- L1-resident: the ceiling of ANY per-lane gather, whatever the size of the tree, and the level a small scene
    lives in -- and (ii) a table the size of this workload's traversal set (the level it lives in as a whole; a
    traversal beats that rate when its upper tree levels are served by L1/L2).  profiles/gather_peaks.json holds the
    same measurements from the profiling session.  Returns (natural level, L1 peak GB/s, natural-level peak GB/s, details)."""
    level = "l1" if traversal_bytes <= 192 * 1024 else ("l2" if traversal_bytes <= 126e6 else "hbm")
    table = max(4096, min(int(traversal_bytes), 2 * 1000 * 1000 * 1000))
    details = {"natural_level": level, "natural_table_bytes": table}

    def measure(nbytes):
        iters = 2000 if nbytes < 1e6 else 500
        ind, _ = ctx.gather_peak(nbytes, dependent=False, ilp=4, blocks_per_sm=8, iters=iters)
        dep, ns = ctx.gather_peak(nbytes, dependent=True, ilp=1, blocks_per_sm=8, iters=iters)
        return ind, dep, ns

    try:
        i1, d1, _ = measure(21 * 1024)
        l1_peak = max(i1, d1)
        details["l1_21KB"] = {"independent_gbs": i1, "dependent_gbs": d1}
        if level == "l1":
            nat_peak = l1_peak
        else:
            i2, d2, ns = measure(table)
            nat_peak = max(i2, d2)
            details["natural"] = {"independent_gbs": i2, "dependent_gbs": d2, "dependent_ns_per_gather": ns}
        details["source"] = ("measured live: lt_debug_gather_peak, 32-byte ld.global.nc.v8 per lane at random records, "
                             "8 persistent blocks per SM")
        return level, l1_peak, nat_peak, details
    except Exception as e:  # pragma: no cover
        details["error"] = str(e)
    path = os.path.join(ROOT, "profiles", "gather_peaks.json")
    if os.path.exists(path):
        tabs = json.load(open(path))["tables"]
        key = {"l1": "l1_21KB", "l2": "l2_112MB", "hbm": "hbm_0.9GB"}[level]
        details["source"] = "profiles/gather_peaks.json"
        return level, tabs["l1_21KB"]["peak_gbs"], tabs[key]["peak_gbs"], details
    return level, None, None, details


def image_parity(got, want):
    """got, want: float32 [H, W, 3] numpy.  Bitwise-equal pixels, largest relative difference (relative to the
    pixel's largest channel, floor 1e-3), PSNR (peak 1.0)."""
    gb, wb = got.view(np.uint32), want.view(np.uint32)
    equal = int((gb == wb).all(axis=-1).sum())
    scale = np.maximum(np.abs(want).max(axis=-1), 1e-3)
    rel = np.abs(got.astype(np.float64) - want).max(axis=-1) / scale
    mse = float(((got.astype(np.float64) - want) ** 2).mean())
    return {"pixels": int(got.shape[0] * got.shape[1]), "pixels_bitwise_equal": equal, "max_rel": float(rel.max()),
            "pixels_beyond_1e-4_rel": int((rel > 1e-4).sum()),
            "psnr_db": None if mse == 0 else 10.0 * np.log10(1.0 / mse)}


def cpu_frames_mean(sb, kernel, w, h, depth, frames, want_text):
    """Running mean (accumulator.frag:10-19, oracle/lt_oracle.c: lto_accumulate) of `frames` full frames rendered by
    the CPU port, timed; and, when the reference's own kernel text is available (oracle/_ref/libltref_cl.so), the
    same by that.  Returns dict with images, seconds and ray count."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lt_oracle as O
    import lt_ref_cl as R
    acc = np.zeros((h, w, 3), np.float32)
    rays, secs = 0, 0.0
    for f in range(frames):
        cam = L.make_camera(0, 2.5, -50, 0.0, f)
        t0 = time.perf_counter()
        img, st = O.render(kernel, sb, cam, w, h, max_ray_depth=depth if depth else 16, threads=0, with_stats=True)
        secs += time.perf_counter() - t0
        rays += st.rays
        O.accumulate(acc, img, f)
    out = {"port_mean": acc, "port_seconds": secs, "rays": rays, "frames": frames, "text_mean": None}
    if want_text and R.available() and 1 <= kernel <= 6:
        tacc = np.zeros((h, w, 3), np.float32)
        tsecs = 0.0
        for f in range(frames):
            cam = L.make_camera(0, 2.5, -50, 0.0, f)
            t0 = time.perf_counter()
            img = R.render(kernel, sb, cam, w, h, max_ray_depth=depth if depth else 16, threads=0)
            tsecs += time.perf_counter() - t0
            O.accumulate(tacc, img, f)
        out.update({"text_mean": tacc, "text_seconds": tsecs})
    return out


def reference_protocol_ms(kernel_path, w, h, frames, depth):
    """The reference example's own protocol (examples/global_illumination/src/main.cpp:296-325): one
    RendererOpenCL::render() per sample into a malloc'ed host buffer (pageable), frameCount incremented by the
    caller, running mean on the host.  Wall milliseconds per call and for the whole frame."""
    from lens_trace_b200 import host
    cwd = os.getcwd()
    os.chdir(ROOT)
    try:
        cam = host.Camera(0, 2.5, -50, 0)
        model = host.Model("resources/models/cornell_box.obj")
        accel = host.AccelerationStructure(model)
        r = host.Renderer(host.PLATFORM_OPENCL)
        ext = host.make_extension(frames=1, accumulate=False, max_ray_depth=depth)
        out = np.zeros((h, w, 3), np.float32)
        acc = np.zeros((h, w, 3), np.float32)
        r.render(kernel_path, w, h, accel, model, cam, ext=ext, out=out)  # upload + first launch
        calls = []
        t_all = time.perf_counter()
        for f in range(frames):
            cam.set_frame_count(f)
            t0 = time.perf_counter()
            r.render(kernel_path, w, h, accel, model, cam, ext=ext, out=out)
            calls.append((time.perf_counter() - t0) * 1e3)
            if f == 0:
                acc[...] = out
            else:
                acc *= np.float32(f)
                acc += out
                acc /= np.float32(f + 1)
        total = (time.perf_counter() - t_all) * 1e3
        # the same calls after the application page-locked its buffer once (lt_host_register, opt-in)
        from lens_trace_b200 import capi
        pinned_calls = []
        if capi.load().lt_host_register(out.ctypes.data, out.nbytes) == 0:
            for f in range(min(frames, 16)):
                cam.set_frame_count(f)
                t0 = time.perf_counter()
                r.render(kernel_path, w, h, accel, model, cam, ext=ext, out=out)
                pinned_calls.append((time.perf_counter() - t0) * 1e3)
            capi.load().lt_host_unregister(out.ctypes.data)
        r.close(); accel.close(); model.close(); cam.close()
        calls.sort()
        pinned_calls.sort()
        return {"render_call_ms_median": calls[len(calls) // 2], "render_call_ms_min": calls[0],
                "frame_ms_with_host_mean": total, "render_calls_ms_total": sum(calls), "calls": frames,
                "render_call_ms_median_registered_buffer": pinned_calls[len(pinned_calls) // 2] if pinned_calls else None}
    finally:
        os.chdir(cwd)


def reference_cuda_section(ctx, scene, sb, w, h, acc_ptr, label):
    """Reference CUDA kernel (basic.cu through NVRTC, its own launch shape) vs this repo's pipeline for the same file,
    primary rays, same buffers, same size, same GPU: kernel-only times by CUDA events."""
    from lens_trace_b200 import capi
    ref = reference_cuda_kernel_rate(sb, w, h)
    if not ref or "error" in ref:
        return {"scene": label, "reference_kernel": ref}
    pp = capi.make_params(L.KERNEL_BASIC_CU, w, h)
    cam = L.make_camera(0, 2.5, -50)
    for _ in range(3):
        ctx.render_device(scene, cam, pp, acc_ptr, sync=True)
    mine = []
    for _ in range(10):
        ctx.render_device(scene, cam, pp, acc_ptr, sync=True)
        mine.append(ctx.stats().kernel_ms)
    mine = sum(mine) / len(mine)
    best_ref = min(v["ms"] for k, v in ref.items() if k.startswith("block_"))
    out = {"scene": label, "what": "primary rays (basic.cu), %dx%d, same buffers, same GPU, kernel only" % (w, h),
           "reference_kernel": ref, "reference_kernel_ms": best_ref,
           "this_repo_kernel": {"ms": mine, "mrays_s": w * h / mine / 1e3},
           "kernel_ratio": best_ref / mine}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="strong (default): the workload's frames are divided among the GPUs (total work fixed); "
                         "weak: every GPU renders all of the workload's frames (N x the samples)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU baseline and the parity block it feeds")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-cull", action="store_true", help="skip the secondary opt-in culled measurement")
    ap.add_argument("--no-lbvh", action="store_true", help="skip the secondary opt-in GPU-built LBVH measurement")
    ap.add_argument("--no-protocol", action="store_true", help="skip the reference-protocol (one render() per frame) timing")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step to DIR as .npy files (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from lens_trace_b200 import capi

    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # keep stdout to the one JSON line: NCCL writes its version banner (and anything else it logs) to stdout
        # unless it is given a file, and it honours NCCL_DEBUG_FILE only above the VERSION level
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    model, kernel, w, h, total_frames, depth, desc = WORKLOADS[args.workload]
    if args.scaling == "strong":
        if total_frames % world:
            sys.exit("bench.py: --scaling strong needs the workload's %d frames to divide by %d GPUs" % (total_frames, world))
        frames = total_frames // world  # this rank's share; frame k of rank r has frameCount r + k*world
    else:
        frames = total_frames
        total_frames = frames * world
    sb = load_scene(model)
    ctx = capi.Context(local_rank)
    scene = ctx.upload(sb)
    upload_ms = ctx.stats().upload_ms
    # a non-default torch stream: lt_ctx_set_stream(NULL) would mean "the context's own stream", and
    # torch.cuda.Event only sees the stream it is recorded on
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    acc = torch.zeros((h, w, 3), dtype=torch.float32, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2
    pinned = torch.empty((h, w, 3), dtype=torch.float32).pin_memory()

    def make_step_params(flags=0):
        if world == 1:
            return capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames,
                                    accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags)
        return capi.make_params(kernel, w, h, max_ray_depth=depth, frames=frames, frame_stride=world,
                                accum_mode=L.ACCUM_WEIGHTED_SUM, accum_weight=1.0 / total_frames, flags=flags)

    cam = L.make_camera(0, 2.5, -50, 0.0, rank if world > 1 else 0)

    def step():
        """one frame of the workload: all samples of this rank, then the exchange step"""
        if world > 1:
            acc.zero_()
        ctx.render_device(scene, cam, make_step_params(), acc.data_ptr(), sync=False)
        if world > 1:
            dist.all_reduce(acc)

    # counters of one step (untimed): rays and the reference-order node/triangle tests
    ctx.render_device(scene, cam, make_step_params(L.FLAG_STATS), acc.data_ptr(), sync=True)
    st = ctx.stats()
    counts = torch.tensor([st.rays, st.node_tests, st.tri_tests], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(counts)
    rays, node_tests, tri_tests = [float(x) for x in counts.tolist()]
    # ... and of what the exact pipelines really trace: an extension ray that hits a light is traced once, its
    # remaining depths are accumulated without retracing (the reference retraces the identical ray per depth)
    ctx.render_device(scene, cam, make_step_params(L.FLAG_STATS | L.FLAG_STATS_TRACED), acc.data_ptr(), sync=True)
    stt = ctx.stats()
    counts_t = torch.tensor([stt.rays, stt.node_tests, stt.tri_tests], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(counts_t)
    rays_t, node_tests_t, tri_tests_t = [float(x) for x in counts_t.tolist()]
    # The camera ray of a pixel is the same in every frame (the reference has no sub-pixel jitter), so the wavefront
    # pipeline traces it once per pixel per step and starts all `frames` paths of the pixel from that hit record.
    # rays / node_tests / tri_tests above are the reference's counts (one primary ray per pixel per frame); the
    # traversal kernels actually execute (frames - 1) primary rays per pixel fewer.  Counted with the primary-only
    # kernel (basic.cl: one camera ray per pixel; the bench scenes have no lens material).
    ctx.render_device(scene, cam, capi.make_params(L.KERNEL_BASIC_CL, w, h, flags=L.FLAG_STATS), acc.data_ptr(), sync=True)
    sp = ctx.stats()
    primary_counts = (float(sp.rays), float(sp.node_tests), float(sp.tri_tests))

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    events = []
    for _ in range(args.steps):
        flush.fill_(1.0)  # L2 flush between timed iterations (untimed)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        if world > 1:
            acc.zero_()
        ctx.render_device(scene, cam, make_step_params(), acc.data_ptr(), sync=False)
        e1.record(stream)
        if world > 1:
            dist.all_reduce(acc)
        e2.record(stream)
        events.append((e0, e1, e2))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.summary()
    launches_per_step = ctx.stats().kernel_launches
    result_image = acc.clone()  # what the last timed step left: the image every parity check below is about
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "image", result_image.cpu().numpy())

    # The kernels timed in isolation, live, for the roofline: in the timed steps above consecutive batches of the
    # wavefront pipeline overlap on two streams (a trace kernel beside another batch's shade kernel), so a launch's
    # own duration is only defined with the overlap off (LT_FLAG_SERIAL: same kernels, same output, one stream).
    # Synchronous call: the library brackets every launch with CUDA events on this stream and sums them per kind
    # (lt_stats: trace_ms, shade_ms, primary_shade_ms, accumulate_ms).
    iso_steps = max(1, min(args.steps, 3))
    iso = {"pipeline": 0.0, "trace": 0.0, "trace_launches": 0, "shade": 0.0, "shade_launches": 0, "primary_shade": 0.0,
           "accumulate": 0.0}
    for _ in range(iso_steps):
        flush.fill_(1.0)
        if world > 1:
            acc.zero_()
        ctx.render_device(scene, cam, make_step_params(L.FLAG_SERIAL), acc.data_ptr(), sync=True)
        s1 = ctx.stats()
        iso["pipeline"] += s1.kernel_ms
        iso["trace"] += s1.trace_ms
        iso["trace_launches"] += s1.trace_launches
        iso["shade"] += s1.shade_ms
        iso["shade_launches"] += s1.shade_launches
        iso["primary_shade"] += s1.primary_shade_ms
        iso["accumulate"] += s1.accumulate_ms
    total_ms = sum(a.elapsed_time(c) for a, _, c in events)
    kernel_ms = sum(a.elapsed_time(b) for a, b, _ in events)
    exchange_ms = sum(b.elapsed_time(c) for _, b, c in events)
    t = torch.tensor([total_ms, kernel_ms, exchange_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kernel_ms, exchange_ms = t.tolist()
    ms_per_step = total_ms / args.steps
    value = rays / (ms_per_step * 1e-3) / 1e6

    # end to end through the public C-ABI with host buffers (lt_render: H2D of the camera, kernels, D2H).  With
    # several GPUs only rank 0 holds the caller's buffer: it alone copies the all-reduced frame to the host.
    e2e_times = []
    for i in range(max(2, min(args.steps, 3)) + 1):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if world == 1:
            ctx.render_into(scene, cam, make_step_params(), pinned.data_ptr())
        else:
            acc.zero_()
            ctx.render_device(scene, cam, make_step_params(), acc.data_ptr(), sync=False)
            dist.all_reduce(acc)
            if rank == 0:
                pinned.copy_(acc, non_blocking=False)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()  # the step is over when rank 0 has the frame
        dt = time.perf_counter() - t0
        if i > 0:
            e2e_times.append(dt)
    # the same call with the buffer the reference's callers really pass: malloc'ed, pageable memory (structures.h:62,76;
    # lt_render stages it through its own pinned buffer, DESIGN.md 2)
    pageable_ms = None
    if world == 1:
        pageable = np.empty((h, w, 3), dtype=np.float32)
        pageable.fill(0.0)  # touch the pages
        pt = []
        for i in range(max(2, min(args.steps, 3)) + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctx.render_into(scene, cam, make_step_params(), pageable.ctypes.data)
            torch.cuda.synchronize()
            if i > 0:
                pt.append((time.perf_counter() - t0) * 1e3)
        pageable_ms = sum(pt) / len(pt)
    e2e_t = torch.tensor([sum(e2e_times) / len(e2e_times)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_s = e2e_t.item()

    # N > 1: the all-reduced image against ONE GPU's running mean of the same frames (rank 0 renders all of them)
    multi_parity = None
    if world > 1:
        if rank == 0:
            single = torch.zeros_like(acc)
            ctx.render_device(scene, L.make_camera(0, 2.5, -50, 0.0, 0),
                              capi.make_params(kernel, w, h, max_ray_depth=depth, frames=total_frames,
                                               accum_mode=L.ACCUM_RUNNING_MEAN), single.data_ptr(), sync=True)
            multi_parity = image_parity(result_image.cpu().numpy(), single.cpu().numpy())
            multi_parity["what"] = ("all-reduced %d-GPU image vs one GPU's running mean of the same %d frames "
                                    "(differs by FP32 summation order only)" % (world, total_frames))
        dist.barrier()

    if rank == 0:
        pk = peaks()
        sm_count = st.sm_count or 148
        fp32_peak = sm_count * 128 * pk["sm_max_mhz"] * 1e6  # lane-instructions / s
        # roofline of ONE GPU's kernels: the counters were summed over ranks
        shared_primary = launches_per_step > 1 and frames > 1  # the wavefront pipeline (exact mode) does this
        skipped = (frames - 1) * world if shared_primary else 0
        rays_traced = rays_t - skipped * primary_counts[0]
        node_traced = node_tests_t - skipped * primary_counts[1]
        tri_traced = tri_tests_t - skipped * primary_counts[2]
        if kernel <= 2 and frames > 1:
            # deterministic kernels: every frame is the same image, k_flat traces once and applies the frame
            # combiner `frames` times in registers
            shared_primary = True
            rays_traced, node_traced, tri_traced = rays / frames, node_tests / frames, tri_tests / frames
        # algorithmic work of the rays the timed traversal launches actually trace (SURVEY 8(d): 32 B and 12
        # lane-instructions per box test, 36 B and 45 per triangle test, counted in the reference's traversal order)
        alg_instr = (12.0 * node_traced + 45.0 * tri_traced) / world
        alg_bytes = (32.0 * node_traced + 36.0 * tri_traced) / world
        ref_alg_bytes = (32.0 * node_tests + 36.0 * tri_tests) / world
        trace_s = iso["trace"] / iso_steps * 1e-3
        k_s = trace_s if trace_s > 0 else kernel_ms / args.steps * 1e-3
        step_s = kernel_ms / args.steps * 1e-3  # this GPU's kernels of one timed step (overlapped batches)
        scene_bytes = sb.nodes.nbytes + sb.prims.nbytes
        # what the traversal kernels read: 32 B per reference node (child-pair or threaded records; small trees hold
        # eight octant copies of the 32-byte records) + 48-byte triangles
        threaded = len(sb.nodes) <= 65536
        traversal_bytes = len(sb.nodes) * 32 * (8 if threaded else 1) + len(sb.prims) * 48
        ctx.set_stream(None)
        level, l1_gather, natural_gather, gather_details = gather_ceiling(ctx, traversal_bytes)
        ctx.set_stream(stream.cuda_stream)
        nominal_l1 = sm_count * 128 * pk["sm_max_mhz"] * 1e6 / 1e9  # GB/s, 128 B/clk/SM: what a coalesced stream reaches
        # The ceiling every traversal is rated against is the measured L1 gather rate: no per-lane 32-byte gather is
        # faster, wherever the tree lives.  The rate of the level the traversal set lives in as a whole is given
        # beside it; large trees exceed it because their upper levels are served by L1/L2.
        bw_peak = l1_gather if l1_gather else nominal_l1
        fp32 = {"achieved": alg_instr / k_s / 1e12, "peak": fp32_peak / 1e12, "unit": "T lane-instr/s",
                "frac": alg_instr / k_s / fp32_peak, "frac_step": alg_instr / step_s / fp32_peak}
        fetch = {"level": "l1", "achieved": alg_bytes / k_s / 1e9, "peak": bw_peak, "unit": "GB/s",
                 "frac": alg_bytes / k_s / 1e9 / bw_peak, "frac_step": alg_bytes / step_s / 1e9 / bw_peak,
                 "peak_source": "measured" if l1_gather else "nominal", "peak_details": gather_details,
                 "natural_level": level, "natural_level_gather_gbs": natural_gather,
                 "frac_of_natural_level_gather": (alg_bytes / k_s / 1e9 / natural_gather) if natural_gather else None,
                 "nominal_l1_gbs": nominal_l1, "frac_of_nominal_l1": alg_bytes / k_s / 1e9 / nominal_l1,
                 "hbm_copy_gbs": pk["hbm_gbs"], "frac_of_hbm_copy": alg_bytes / k_s / 1e9 / pk["hbm_gbs"]}
        t_fp32 = alg_instr / fp32_peak
        t_fetch = alg_bytes / (bw_peak * 1e9)
        if t_fetch >= t_fp32:
            roof = {"bound": "l1", "achieved": fetch["achieved"], "peak": fetch["peak"], "unit": "GB/s",
                    "frac": fetch["frac"], "frac_traversal": fetch["frac"], "frac_step": fetch["frac_step"],
                    "peak_source": fetch["peak_source"], "traffic": None,
                    "bound_note": "measured rate of per-lane 32-byte gathers from L1 (lt_debug_gather_peak): the ceiling of "
                                  "a node fetch; the traversal set as a whole lives in %s" % level}
        else:
            roof = {"bound": "fp32", "achieved": fp32["achieved"], "peak": fp32["peak"], "unit": "T lane-instr/s",
                    "frac": fp32["frac"], "frac_traversal": fp32["frac"], "frac_step": fp32["frac_step"],
                    "peak_source": "nominal issue rate at the measured sm_max_mhz", "traffic": None}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        ncu_kernels = {}
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            tr = tj.get(args.workload)
            if tr:
                roof["traffic"] = tr["bytes"]
                roof["traffic_source"] = tr["capture"]
            ncu_kernels = tj.get("kernels_" + args.workload, {})
        wavefront = launches_per_step > 1
        pipeline = "wavefront (k_wf_primary_trace once, then per batch k_wf_primary + (k_wf_trace, k_wf_shade) x rounds + k_wf_accumulate; two batches in flight on two streams)" \
            if wavefront else ("k_path" if kernel >= 3 else "k_flat / k_flat_stream")
        # per-kernel view of one (serialised) step: live CUDA-event times; DRAM bytes per step from the committed ncu
        # launch list of the same command (profiles/traffic.json: kernels_<workload>), rated against the measured
        # HBM copy bandwidth
        kernels = {}
        if wavefront:
            for name, key, launches in (("k_wf_trace+k_wf_primary_trace", "trace", iso["trace_launches"]),
                                        ("k_wf_shade", "shade", iso["shade_launches"]),
                                        ("k_wf_primary", "primary_shade", None), ("k_wf_accumulate", "accumulate", None)):
                ms = iso[key] / iso_steps
                ent = {"ms_per_step": ms, "share_of_serialised_step": iso[key] / max(1e-9, iso["pipeline"])}
                if launches is not None:
                    ent["launches_per_step"] = launches / iso_steps
                nk = ncu_kernels.get(name.split("+")[0])
                if nk and ms > 0:
                    ent["dram_bytes_per_step_ncu"] = nk["dram_bytes_per_step"]
                    ent["dram_gbs"] = nk["dram_bytes_per_step"] / (ms * 1e-3) / 1e9
                    ent["frac_hbm"] = ent["dram_gbs"] / pk["hbm_gbs"]
                kernels[name] = ent
        roof.update({"kernel": "k_wf_primary_trace + k_wf_trace (traversal kernels of the wavefront pipeline)"
                     if wavefront else pipeline,
                     "pipeline": pipeline,
                     "timing": "every launch timed live with CUDA events, kernels in isolation (LT_FLAG_SERIAL: one "
                               "stream, %d steps); the timed steps overlap consecutive batches on two streams; "
                               "frac_traversal = algorithmic bytes / traversal-kernel time / peak, frac_step = the "
                               "same bytes / whole step time / peak" % iso_steps,
                     "traversal_ms_per_step": iso["trace"] / iso_steps,
                     "traversal_launches_per_step": iso["trace_launches"] / iso_steps,
                     "traversal_avg_launch_ms": iso["trace"] / max(1, iso["trace_launches"]),
                     "traversal_share_of_step": iso["trace"] / max(1e-9, iso["pipeline"]),
                     "pipeline_ms_per_step_in_isolation": iso["pipeline"] / iso_steps,
                     "pipeline_ms_per_step": kernel_ms / args.steps,
                     "kernels_per_step": launches_per_step,
                     "kernels": kernels,
                     "algorithmic_units": "per step (all traversal launches of one step), per GPU; rays actually traced",
                     "algorithmic_bytes_per_step": alg_bytes, "algorithmic_fp32_instr_per_step": alg_instr,
                     "traversal_set_bytes": traversal_bytes,
                     "rays_traced_per_step": rays_traced / world,
                     "light_hit_retraces_folded_per_step": (rays - rays_t) / world,
                     "reference_rays_per_step": rays / world,
                     "reference_algorithmic_bytes_per_step": ref_alg_bytes,
                     "primary_rays": "traced once per pixel per step and shared by the step's %d frames "
                                     "(identical camera ray in every frame); value counts the reference's rays" % frames
                     if shared_primary else "one per pixel per frame",
                     "node_tests_per_ray": node_tests / rays, "tri_tests_per_ray": tri_tests / rays,
                     "fp32_issue": fp32, "node_fetch": fetch})
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(args.workload, total_frames),
            "config_detail": {"frames_per_step_per_gpu": frames, "rays_per_step": rays,
                              "parallelism": "spp-split x%d + 1 all-reduce/step" % world if world > 1 else "single GPU",
                              "l2": "flushed between timed steps (256 MB write); scene is %d bytes" % scene_bytes,
                              "scene_upload_ms": upload_ms,
                              "bvh": "this repo's deterministic median-split builder (reference semantics); both arms "
                                     "traverse the same node array"},
            "roofline": roof,
            "e2e": {"value": rays / e2e_s / 1e6, "unit": "Mrays/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": 28, "d2h_bytes_per_step": int(w * h * 3 * 4),
                    "api": "lt_render (C-ABI, pinned host output buffer)" if world == 1 else
                    "lt_render_device + NCCL all-reduce + D2H on rank 0",
                    "ms_per_step_pageable_buffer": pageable_ms},
            "gpu_launches": args.steps * launches_per_step,
            "clocks": clocks,
        }
        if world > 1:
            line["allreduce_ms"] = exchange_ms / args.steps
            line["render_ms_per_step"] = kernel_ms / args.steps
            line["parity"] = {"multi_gpu": multi_parity}
        if world == 1 and not args.no_cpu_baseline:
            # CPU baseline and parity from the same frames: the port (and the reference's own kernel text) render
            # frames 0..per-1 at full size; when that is the whole step the timed accumulator itself is compared
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            _, _, t1, _ = cpu_oracle_rate(sb, kernel, w, h, depth, [0])
            per = max(1, min(frames, int(20.0 / max(t1, 1e-3))))
            cpu = cpu_frames_mean(sb, kernel, w, h, depth, per, want_text=True)
            cores = os.cpu_count() or 1
            line["cpu_baseline"] = {"value": cpu["rays"] / cpu["port_seconds"] / 1e6, "unit": "Mrays/s", "cores": cores,
                                    "kind": "port", "sample": "frames 0..%d of the %d at full %dx%d (%.1f s of CPU work)" % (
                                        per - 1, frames, w, h, cpu["port_seconds"])}
            if cpu["text_mean"] is not None:
                line["cpu_baseline"] = {
                    "value": cpu["rays"] / cpu["text_seconds"] / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "reference",
                    "sample": "frames 0..%d of the %d at full %dx%d (%.1f s of CPU work)" % (per - 1, frames, w, h, cpu["text_seconds"]),
                    "what": "the reference's own kernel file (OpenCL C) compiled for the CPU through oracle/cl_shim, "
                            "std::thread over image rows -- stand-in for the OpenCL backend on a POCL CPU device",
                    "port_value": cpu["rays"] / cpu["port_seconds"] / 1e6,
                    "port_sample": "same frames (%.1f s), C restatement oracle/lt_oracle.c" % cpu["port_seconds"]}
            if per == frames:
                gpu_img = result_image.cpu().numpy()
                what = "the accumulator the last TIMED step left (%d frames, running mean)" % frames
            else:
                tmp = torch.zeros_like(acc)
                ctx.render_device(scene, L.make_camera(0, 2.5, -50, 0.0, 0),
                                  capi.make_params(kernel, w, h, max_ray_depth=depth, frames=per,
                                                   accum_mode=L.ACCUM_RUNNING_MEAN), tmp.data_ptr(), sync=True)
                gpu_img = tmp.cpu().numpy()
                what = "running mean of frames 0..%d by the timed kernels (the CPU cannot render all %d in the bench's time)" % (per - 1, frames)
            par = image_parity(gpu_img, cpu["port_mean"])
            par["what"] = what + " vs the CPU oracle's running mean of the same frames (oracle/lt_oracle.c, device FP flavour)"
            par["frames_compared"] = per
            if cpu["text_mean"] is not None:
                pt = image_parity(gpu_img, cpu["text_mean"])
                par["psnr_vs_reference_text"] = pt["psnr_db"]
                par["vs_reference_text"] = {k: pt[k] for k in ("pixels_bitwise_equal", "max_rel", "pixels_beyond_1e-4_rel")}
                par["vs_reference_text"]["note"] = ("the reference's kernel text executed on the CPU; the residue is FMA "
                                                    "contraction and sin/cos the OpenCL text leaves to the implementation")
            line["parity"] = par
        if world == 1 and not args.no_cull:
            # OPT-IN culled traversal (LT_FLAG_CULL): reported beside the headline, never instead of it.
            # It does less work than the reference's traversal; identity of the full-size output is checked here.
            ctx.set_stream(stream.cuda_stream)
            pc = make_step_params(L.FLAG_CULL)
            ctx.render_device(scene, cam, pc, acc.data_ptr(), sync=True)
            identical = bool(torch.equal(acc.view(torch.int32), result_image.view(torch.int32)))
            times = []
            for _ in range(max(2, min(args.steps, 3))):
                flush.fill_(1.0)
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record(stream)
                ctx.render_device(scene, cam, pc, acc.data_ptr(), sync=False)
                c1.record(stream)
                torch.cuda.synchronize()
                times.append(c0.elapsed_time(c1))
            ctx.render_device(scene, cam, make_step_params(L.FLAG_CULL | L.FLAG_STATS), acc.data_ptr(), sync=True)
            sc_ = ctx.stats()
            cms = sum(times) / len(times)
            line["culled_opt_in"] = {
                "flag": "LT_FLAG_CULL (off by default)", "ms_per_step": cms, "value": rays / (cms * 1e-3) / 1e6,
                "unit": "Mrays/s (same ray count as the exact run)", "output_bit_identical_to_exact": identical,
                "node_tests_per_ray_actual": sc_.node_tests / max(1, sc_.rays),
                "tri_tests_per_ray_actual": sc_.tri_tests / max(1, sc_.rays),
                "speedup_vs_exact": ms_per_step / cms}
        if world == 1 and not args.no_lbvh and len(sb.prims) >= 2:
            # OPT-IN device-built LBVH (lt_scene_build_lbvh): a different tree than the reference builder's, so it is
            # reported beside the headline only.  Same kernels, same workload; picture compared with the headline's.
            ctx.set_stream(stream.cuda_stream)
            t0 = time.perf_counter()
            lscene = ctx.build_lbvh(sb.prims, sb.materials)
            build_wall_ms = (time.perf_counter() - t0) * 1e3
            build_dev_ms = ctx.stats().upload_ms
            times = []
            for _ in range(max(2, min(args.steps, 3)) + 1):
                flush.fill_(1.0)
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record(stream)
                ctx.render_device(lscene, cam, make_step_params(), acc.data_ptr(), sync=False)
                c1.record(stream)
                torch.cuda.synchronize()
                times.append(c0.elapsed_time(c1))
            lms = sum(times[1:]) / len(times[1:])
            differing = int(((acc - result_image).abs().amax(dim=-1) >
                             1e-4 * result_image.abs().amax(dim=-1).clamp_min(1e-3)).sum().item())
            ctx.render_device(lscene, cam, make_step_params(L.FLAG_STATS), acc.data_ptr(), sync=True)
            sl = ctx.stats()
            line["lbvh_opt_in"] = {
                "what": "same workload on an LBVH built on the GPU (ACCELERATION_STRUCTURE_TYPE_LBVH_B200), not the "
                        "reference builder's tree",
                "build_ms_device": build_dev_ms, "build_ms_wall": build_wall_ms, "ms_per_step": lms,
                "value": sl.rays / (lms * 1e-3) / 1e6, "unit": "Mrays/s", "speedup_vs_reference_tree": ms_per_step / lms,
                "node_tests_per_ray": sl.node_tests / max(1, sl.rays), "tri_tests_per_ray": sl.tri_tests / max(1, sl.rays),
                "pixels_differing_beyond_1e-4_rel": differing, "pixels": w * h}
            lscene.release()
        if world == 1 and not args.no_lbvh:
            # OPT-IN host builder with binned SAH splits (ACCELERATION_STRUCTURE_TYPE_SAH_B200): again a different tree
            # in the same layout, same kernels, reported beside the headline only
            ctx.set_stream(stream.cuda_stream)
            t0 = time.perf_counter()
            sb_sah = load_scene(model, 101)
            sah_build_s = time.perf_counter() - t0
            sscene = ctx.upload(sb_sah)
            times = []
            for _ in range(max(2, min(args.steps, 3)) + 1):
                flush.fill_(1.0)
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record(stream)
                ctx.render_device(sscene, cam, make_step_params(), acc.data_ptr(), sync=False)
                c1.record(stream)
                torch.cuda.synchronize()
                times.append(c0.elapsed_time(c1))
            sms = sum(times[1:]) / len(times[1:])
            differing = int(((acc - result_image).abs().amax(dim=-1) >
                             1e-4 * result_image.abs().amax(dim=-1).clamp_min(1e-3)).sum().item())
            ctx.render_device(sscene, cam, make_step_params(L.FLAG_STATS), acc.data_ptr(), sync=True)
            ss = ctx.stats()
            line["sah_opt_in"] = {
                "what": "same workload on a binned-SAH tree built on the host (ACCELERATION_STRUCTURE_TYPE_SAH_B200), "
                        "not the reference builder's tree",
                "load_and_build_s_host": sah_build_s, "ms_per_step": sms, "value": ss.rays / (sms * 1e-3) / 1e6,
                "unit": "Mrays/s", "speedup_vs_reference_tree": ms_per_step / sms,
                "node_tests_per_ray": ss.node_tests / max(1, ss.rays), "tri_tests_per_ray": ss.tri_tests / max(1, ss.rays),
                "pixels_differing_beyond_1e-4_rel": differing, "pixels": w * h}
            sscene.release()
        if world == 1 and not args.no_ref_cuda:
            # the reference's CUDA kernel only exists for primary rays (basic.cu): the workload's scene, and -- because
            # a 42-triangle box says little about traversal -- the synthetic 1 M-triangle mesh (BASELINE configs[2])
            ctx.set_stream(None)
            sections = [reference_cuda_section(ctx, scene, sb, w, h, acc.data_ptr(), model)]
            if "render_as_shipped_ms" in (sections[0].get("reference_kernel") or {}):
                sections[0]["this_repo_render_call_ms"] = this_repo_render_call_ms(w, h)
            if model != "synth:707" and args.workload == DEFAULT_WORKLOAD:
                sb2 = load_scene("synth:707")
                scene2 = ctx.upload(sb2)
                sections.append(reference_cuda_section(ctx, scene2, sb2, 1920, 1080, acc.data_ptr(), "synth:707"))
                scene2.release()
            line["reference_cuda_backend"] = {
                "note": "the reference's only CUDA kernel; kernel_ratio = reference kernel ms / this repo's kernel ms "
                        "(north star: >= 10x -- not met, see DESIGN.md)",
                "scenes": sections}
        if world == 1 and not args.no_protocol and args.workload == DEFAULT_WORKLOAD:
            line["e2e_reference_protocol"] = reference_protocol_ms(
                "examples/global_illumination/resources/kernels/global_illumination.cl", w, h, frames, depth)
            line["e2e_reference_protocol"]["what"] = (
                "%d x RendererOpenCL::render() of ONE frame each into a malloc'ed buffer + host running mean "
                "(examples/global_illumination/src/main.cpp:296-325), wall clock" % frames)
        print(json.dumps(line), flush=True)

    scene.release()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
