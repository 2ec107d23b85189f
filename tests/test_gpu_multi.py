"""Multi-GPU contexts of the C-ABI (lt_ctx_create_multi) and of the C++ surface (RenderExtensionB200::deviceCount):
the sample split with one all-reduce per call (NCCL, and this repo's own peer-memory kernel) and the tile split,
against one GPU rendering the same call.  On a machine with one GPU the groups are shared groups (util.device_group:
every member on device 0), which run all of it but the NCCL and peer-mapping transport; the tests that need real
device ordinals (the renderer classes, the example program) and the nccl cases skip there.

Tolerance: the sample split sums per-device partial sums, the single GPU keeps a sequential running mean -- the
two differ by FP32 rounding order only; bound 1e-5 relative (measured ~2e-7).  The tile split is bit-exact."""
import os
import subprocess

import numpy as np
import pytest

import util
from lens_trace_b200 import capi, host, layouts as L

pytestmark = pytest.mark.gpu


def device_count():
    import torch
    return torch.cuda.device_count()


needs_two = pytest.mark.skipif("device_count() < 2", reason="needs two or more GPUs")


def rel_diff(a, b):
    return float((np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b), 1e-3)).max())


@pytest.mark.parametrize("exchange", ["nccl", "p2p"])
def test_sample_split_equals_one_gpu(exchange, monkeypatch):
    util.skip_nccl_without_two_gpus(exchange)
    monkeypatch.setenv("LT_MULTI_EXCHANGE", exchange)
    sb = util.scene("cornell_box")
    with capi.Context(0) as one:
        s1 = one.upload(sb)
        for n in util.group_sizes():
            with util.device_group(n) as many:
                assert many.device_count() == n
                sm = many.upload(sb)
                sample_split_equals_one_gpu(exchange, one, s1, many, sm)
                sm.release()
        s1.release()


def sample_split_equals_one_gpu(exchange, one, s1, many, sm):
    cam = util.default_camera(0.0, 0)
    for kernel, depth, w, h, frames in ((L.KERNEL_GI, 4, 640, 360, 16), (L.KERNEL_ACCUMULATOR, 0, 333, 111, 5),
                                        (L.KERNEL_GI, 3, 1920, 1080, 8)):
        p = dict(max_ray_depth=depth, frames=frames, accum_mode=L.ACCUM_RUNNING_MEAN)
        one.accum_reset()
        want = one.render(s1, cam, capi.make_params(kernel, w, h, **p))
        many.accum_reset()
        got = many.render(sm, cam, capi.make_params(kernel, w, h, split_mode=L.SPLIT_SAMPLES, **p))
        assert rel_diff(got, want) <= 1e-5, (exchange, kernel, rel_diff(got, want))
        # progressive: the same frames in two calls (the second continues the accumulator at frameCount = half)
        half = frames // 2
        many.accum_reset()
        many.render(sm, cam, capi.make_params(kernel, w, h, split_mode=L.SPLIT_SAMPLES, max_ray_depth=depth, frames=half,
                                             accum_mode=L.ACCUM_RUNNING_MEAN))
        got2 = many.render(sm, util.default_camera(0.0, half),
                           capi.make_params(kernel, w, h, split_mode=L.SPLIT_SAMPLES, max_ray_depth=depth,
                                            frames=frames - half, accum_mode=L.ACCUM_RUNNING_MEAN))
        assert rel_diff(got2, want) <= 1e-5
    # a sample split of a non-accumulating call is refused; AUTO picks tiles for it
    with pytest.raises(capi.LtError):
        many.render(sm, cam, capi.make_params(L.KERNEL_GI, 64, 64, split_mode=L.SPLIT_SAMPLES))
    auto = many.render(sm, cam, capi.make_params(L.KERNEL_GI, 64, 48, max_ray_depth=2))
    util.assert_bit_equal(auto, one.render(s1, cam, capi.make_params(L.KERNEL_GI, 64, 48, max_ray_depth=2)))


def test_tile_split_is_bit_exact():
    with capi.Context(0) as one:
        for n in util.group_sizes():
            with util.device_group(n) as many:
                tile_split_is_bit_exact(one, many, n)


def tile_split_is_bit_exact(one, many, n):
    for name in ("cornell_box", "cornell_box_lens"):
        sb = util.scene(name)
        s1, sm = one.upload(sb), many.upload(sb)
        for w, h in ((1920, 1080), (101, 75), (64, 5), (33, 8 * n + 3)):
            for kernel, depth, frames in ((L.KERNEL_BASIC_CU, 0, 1), (L.KERNEL_CUSTOM_BARY, 0, 3), (L.KERNEL_GI, 3, 4),
                                          (L.KERNEL_GI25, 2, 1)):
                if kernel == L.KERNEL_GI25 and w * h > 20000:
                    continue
                cam = util.default_camera(0.03, 1)
                acc = L.ACCUM_RUNNING_MEAN if frames > 1 else L.ACCUM_NONE
                p = dict(max_ray_depth=depth, frames=frames, accum_mode=acc)
                one.accum_reset()
                want = one.render(s1, cam, capi.make_params(kernel, w, h, **p))
                many.accum_reset()
                got = many.render(sm, cam, capi.make_params(kernel, w, h, split_mode=L.SPLIT_TILES, **p))
                util.assert_bit_equal(got, want, "%s kernel %d %dx%d tiles over %d GPUs" % (name, kernel, w, h, n))
        s1.release(); sm.release()


@needs_two
def test_multi_gpu_through_the_renderer_classes(root):
    """RendererOpenCL::render with RenderExtensionB200{deviceCount, splitMode}: same picture as one device."""
    os.chdir(root)
    n = min(device_count(), 8)
    cam = host.Camera(0, 2.5, -50, 0)
    model = host.Model("resources/models/cornell_box.obj")
    accel = host.AccelerationStructure(model)
    r = host.Renderer(host.PLATFORM_OPENCL)
    K = "examples/global_illumination/resources/kernels/global_illumination.cl"
    w, h = 320, 200
    want = r.render(K, w, h, accel, model, cam, ext=host.make_extension(frames=8, accumulate=True, max_ray_depth=4))
    for split in (1, 2, 0):
        cam.set_frame_count(0)
        got = r.render(K, w, h, accel, model, cam,
                       ext=host.make_extension(frames=8, accumulate=True, max_ray_depth=4, devices=n, split=split))
        if split == 2:
            util.assert_bit_equal(got, want, "tile split through RendererOpenCL")
        else:
            assert rel_diff(got, want) <= 1e-5
    r.close(); accel.close(); model.close(); cam.close()


@needs_two
def test_multi_gpu_example_program(root, tmp_path):
    subprocess.check_call(["make", "-C", os.path.join(root, "examples"), "-s"])
    n = min(device_count(), 8)
    for split in ("samples", "tiles"):
        r = subprocess.run([os.path.join(root, "examples", "bin", "multi_gpu"), "--devices", str(n), "--size", "640", "360",
                            "--frames", "16", "--split", split], cwd=root, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "GPUs:" in r.stdout


def test_one_device_group_is_a_plain_context():
    c = capi.Context([0])
    assert c.device_count() == 1
    sb = util.scene("green_wall")
    sc = c.upload(sb)
    img = c.render(sc, util.default_camera(), capi.make_params(L.KERNEL_BASIC_CU, 32, 32))
    assert img[16, 16].tolist() == [0.0, 1.0, 0.0]
    sc.release(); c.close()
    with pytest.raises(capi.LtError):
        capi.Context([0, 0])
    for members in (0, 1, 17):  # a shared group has 2..16 members
        with pytest.raises(capi.LtError, match="2..16"):
            capi.Context.shared(0, members)


# ---------------------------------------------------------------- the sample split, restated exactly
#
# lt_multi_render's sample split of F frames at camera frameCount fc over G devices: device k < F renders frames
# k, k + G, ... as a weighted sum into its own accumulator, device 0 carrying the previous image scaled by keep; the
# p2p exchange (k_sum_peers) then adds the G accumulators in device order.  One single-GPU context restates every
# device's share with lt_render_device, so the p2p result is checked bit for bit.

U = 2.0 ** -24  # unit roundoff of FP32


def gamma(n):
    return n * U / (1.0 - n * U)


def gpu_props():
    import torch
    p = torch.cuda.get_device_properties(0)
    return p.total_memory, p.multi_processor_count


def split_weights(fc, F, accum_mode, accum_weight):
    """(w, keep) as lt_multi_render computes them: for a running mean both divided in double, then rounded to FP32"""
    total = float(fc) + float(F)
    if accum_mode == L.ACCUM_RUNNING_MEAN:
        return np.float32(1.0 / total), np.float32(fc / total)
    return np.float32(accum_weight), np.float32(1.0)


def render_device_from(one, s1, cam, params, start):
    """lt_render_device of `params` into a device buffer holding `start`: the accumulator a call continues"""
    import torch
    buf = torch.from_numpy(np.ascontiguousarray(start, np.float32)).cuda()
    torch.cuda.synchronize()
    one.render_device(s1, cam, params, buf.data_ptr(), sync=True)
    return buf.cpu().numpy()


def restate_sample_split(one, s1, G, kernel, w, h, depth, max_ray_depth, F, fc, accum_mode, accum_weight=0.0,
                         stride=1, old=None):
    """The image a p2p sample split of G devices returns, from one single-GPU context: device k's share rendered as
    lt_multi_render renders it, the shares added left to right in FP32.  old: the group's previous output."""
    old = np.zeros((h, w, depth), np.float32) if old is None else old
    wt, keep = split_weights(fc, F, accum_mode, accum_weight)
    total = None
    for k in range(G):
        if k >= F:
            part = np.zeros_like(old)
        else:
            if k > 0 or keep == 0:
                start = np.zeros_like(old)
            elif keep == 1:
                start = old
            else:
                start = old * keep  # one FP32 rounding, as k_scale
            p = capi.make_params(kernel, w, h, depth=depth, max_ray_depth=max_ray_depth, frames=-(-(F - k) // G),
                                 frame_stride=stride * G, accum_mode=L.ACCUM_WEIGHTED_SUM, accum_weight=float(wt))
            part = render_device_from(one, s1, util.default_camera(0.0, fc + k * stride), p, start)
        total = part if total is None else total + part  # FP32, device order
    return total


def split_params(kernel, w, h, depth, max_ray_depth, F, accum_mode, accum_weight=0.0, stride=1):
    return capi.make_params(kernel, w, h, depth=depth, max_ray_depth=max_ray_depth, frames=F, frame_stride=stride,
                            accum_mode=accum_mode, accum_weight=accum_weight, split_mode=L.SPLIT_SAMPLES)


# G, (W, H, depth), kernel, max_ray_depth, F: every group size, image shape (the float4 body and the scalar tail of
# k_sum_peers, and at 1080p several grid-stride passes), kernel and frame count (1, G - 1, G, 2G + 1, 16) at least once
SPLIT_CASES = [
    (2, (1, 1, 3), L.KERNEL_GI, 4, 1),
    (3, (1, 2, 3), L.KERNEL_ACCUMULATOR, 0, 2),
    (8, (3, 1, 3), L.KERNEL_GI25, 2, 8),
    (16, (333, 111, 3), L.KERNEL_CUSTOM_BARY, 0, 33),
    (3, (72, 40, 4), L.KERNEL_GI, 4, 16),
    (8, (1920, 1080, 3), L.KERNEL_GI, 4, 7),
    (2, (72, 40, 4), L.KERNEL_GI25, 2, 5),
    (16, (1, 1, 3), L.KERNEL_CUSTOM_BARY, 0, 16),
    (16, (3, 1, 3), L.KERNEL_ACCUMULATOR, 0, 1),
    (3, (333, 111, 3), L.KERNEL_GI, 4, 7),
]


@pytest.mark.parametrize("case", SPLIT_CASES, ids=lambda c: "G%d-%dx%dx%d-k%d-F%d" % (c[0], *c[1], c[2], c[4]))
def test_sample_split_restated_bit_for_bit(case, monkeypatch):
    """Every float of the p2p sample split (the fourth channel at depth 4 included) equals its restatement: a running
    mean from frameCount 0, its continuation, a continuation at frameCount 100 000 (keep close to 1), then weighted sums
    (weight 0.25, frame_stride 1 or 3) as a first call and continuing."""
    monkeypatch.setenv("LT_MULTI_EXCHANGE", "p2p")
    G, (w, h, depth), kernel, mrd, F = case
    stride = 3 if G % 2 else 1
    sb = util.scene("cornell_box")
    with capi.Context(0) as one, util.device_group(G) as many:
        s1, sm = one.upload(sb), many.upload(sb)
        old = None
        for fc in (0, F, 100000):
            got = many.render(sm, util.default_camera(0.0, fc), split_params(kernel, w, h, depth, mrd, F,
                                                                              L.ACCUM_RUNNING_MEAN))
            want = restate_sample_split(one, s1, G, kernel, w, h, depth, mrd, F, fc, L.ACCUM_RUNNING_MEAN, old=old)
            util.assert_bit_equal(got, want, "G %d: running mean at frameCount %d" % (G, fc))
            old = got
        many.accum_reset()
        old = None
        for call in range(2):
            fc = 5 + call * F * stride
            got = many.render(sm, util.default_camera(0.0, fc), split_params(kernel, w, h, depth, mrd, F,
                                                                              L.ACCUM_WEIGHTED_SUM, 0.25, stride))
            want = restate_sample_split(one, s1, G, kernel, w, h, depth, mrd, F, fc, L.ACCUM_WEIGHTED_SUM, 0.25,
                                        stride, old=old)
            util.assert_bit_equal(got, want, "G %d: weighted sum, stride %d, call %d" % (G, stride, call))
            old = got
        s1.release(); sm.release()


def frame_samples(one, s1, kernel, w, h, depth, mrd, fc, F, stride):
    """The F frames of a call, one per single-GPU call (LT_ACCUM_NONE), in float64: [F, H, W, 3]"""
    return np.stack([one.render(s1, util.default_camera(0.0, fc + f * stride),
                                capi.make_params(kernel, w, h, depth=depth, max_ray_depth=mrd))[..., :3]
                     for f in range(F)]).astype(np.float64)


def check_against_exact(got, exact, scale, n, what):
    got = got[..., :3].astype(np.float64)
    bound = gamma(n) * scale
    err = np.abs(got - exact)
    bad = err > bound
    assert not bad.any(), "%s: %d values beyond gamma_%d; worst excess %s" % (
        what, bad.sum(), n, (err - bound).max())


@pytest.mark.parametrize("exchange", ["nccl", "p2p"])
def test_sample_split_against_the_exact_mean(exchange, monkeypatch):
    """The sample split and the single-GPU running mean against the exact result in FP64, with bounds derived from the
    operation count (u = 2^-24, gamma_n = n u / (1 - n u), and prod (1 + d_i) over n roundings |d_i| <= u lies in
    [1 - gamma_n, 1 + gamma_n]).  The exact result of F frames s_f at frameCount fc onto the previous image `old` is
    (fc old + sum s_f) / (fc + F) for a running mean, old + w sum s_f for a weighted sum of weight w.

    Sample split over G devices: a term w s_f passes the rounding of w (1/(fc+F) to FP32), the product w s_f, at most
    ceil(F/G) + 1 additions in its device's accumulator and G - 1 additions of the exchange, in whatever order the
    exchange adds (so NCCL's too); the term keep old passes the rounding of keep, the product of k_scale and the same
    additions.  With n = ceil(F/G) + G + 4 covering every path, |got - exact| <= gamma_n (w sum |s_f| + keep |old|)
    with the exact w = 1/(fc+F), keep = fc/(fc+F) (for a weighted sum, w as given and keep = 1).

    Single GPU (accumulator.frag): a_{j+1} = fl(fl(s_j + fl(a_j n_j)) / (n_j + 1)), n_j = fc + j, so A_j = a_j n_j obeys
    A_{j+1} = s_j (1+d2)(1+d3) + A_j (1+d1)(1+d2)(1+d3): three roundings per frame, at most 3F on any term, and
    |got - exact| <= gamma_{3F} (sum |s_f| + fc |old|) / (fc + F)."""
    util.skip_nccl_without_two_gpus(exchange)
    monkeypatch.setenv("LT_MULTI_EXCHANGE", exchange)
    import math
    sb = util.scene("cornell_box")
    w, h, depth, mrd = 160, 96, 3, 4
    kernel = L.KERNEL_GI
    with capi.Context(0) as one:
        s1 = one.upload(sb)
        for G in sorted(set(util.group_sizes()) | {2}):
            with util.device_group(G) as many:
                sm = many.upload(sb)
                old = np.zeros((h, w, depth), np.float32)
                calls = ((0, 2 * G + 1, L.ACCUM_RUNNING_MEAN, 0.0, 1), (2 * G + 1, G - 1 or 1, L.ACCUM_RUNNING_MEAN, 0.0, 1),
                         (3 * G, G, L.ACCUM_WEIGHTED_SUM, 0.25, 3))
                for fc, F, mode, aw, stride in calls:
                    s = frame_samples(one, s1, kernel, w, h, depth, mrd, fc, F, stride)
                    o = old[..., :3].astype(np.float64)
                    if mode == L.ACCUM_RUNNING_MEAN:
                        exact = (fc * o + s.sum(axis=0)) / (fc + F)
                        wt, keep = 1.0 / (fc + F), fc / (fc + F)
                    else:
                        exact = o + aw * s.sum(axis=0)
                        wt, keep = aw, 1.0
                    scale = wt * np.abs(s).sum(axis=0) + keep * np.abs(o)
                    got = many.render(sm, util.default_camera(0.0, fc),
                                      split_params(kernel, w, h, depth, mrd, F, mode, aw, stride))
                    check_against_exact(got, exact, scale, math.ceil(F / G) + G + 4,
                                        "%s, G %d, frameCount %d, %d frames" % (exchange, G, fc, F))
                    if mode == L.ACCUM_RUNNING_MEAN:  # the single GPU's running mean from the same image
                        single = render_device_from(one, s1, util.default_camera(0.0, fc),
                                                    capi.make_params(kernel, w, h, depth=depth, max_ray_depth=mrd,
                                                                     frames=F, accum_mode=mode), old)
                        check_against_exact(single, exact, scale, 3 * F, "one GPU, frameCount %d, %d frames" % (fc, F))
                    old = got
                sm.release()
        s1.release()


# ---------------------------------------------------------------- the tile split at its edges

def synthetic_scene(tmp_path_factory):
    p = str(tmp_path_factory.mktemp("synth") / "synth160.obj")
    host.write_synthetic_scene(p, 160, 0x5EED)  # about 102 000 nodes: above the default stream_min_nodes
    return host.load_scene_buffers(p)


# name, scene, kernel, max_ray_depth, flags: k_flat, k_path, the wavefront on the threaded and the child-pair tree, the
# culled traversal, and k_flat_stream on a scene large enough for it
TILE_PIPELINES = [
    ("flat", "cornell_box", L.KERNEL_BASIC_CU, 0, 0),
    ("path", "cornell_box", L.KERNEL_GI, 3, L.FLAG_MEGAKERNEL),
    ("wavefront", "cornell_box", L.KERNEL_GI, 3, L.FLAG_WAVEFRONT),
    ("wavefront_no_threaded", "cornell_box", L.KERNEL_GI, 3, L.FLAG_WAVEFRONT | L.FLAG_NO_THREADED),
    ("cull_flat", "cornell_box", L.KERNEL_BASIC_CU, 0, L.FLAG_CULL),
    ("cull_gi", "cornell_box", L.KERNEL_GI, 3, L.FLAG_CULL),
    ("flat_stream", "synthetic", L.KERNEL_BASIC_CU, 0, 0),
]


@pytest.mark.parametrize("G", [2, 3, 8, 16])
def test_tile_split_at_its_edges(G, tmp_path_factory):
    """Heights that leave members without rows (1, 7, 8, 9), end inside a block on the last member and on member 0
    (8G - 1, 8G + 1, 3 * 8G + 5) or exactly on a block (8G); widths 1, 17 and 1920; depth 4; a running mean over two
    tile calls.  Each call bit for bit against the single-GPU call."""
    scenes = {"cornell_box": util.scene("cornell_box"), "synthetic": synthetic_scene(tmp_path_factory)}
    heights = (1, 7, 8, 9, 8 * G - 1, 8 * G, 8 * G + 1, 3 * 8 * G + 5)
    shapes = [(wd, ht) for wd in (1, 17) for ht in heights] + [(1920, 8 * G + 1)]
    total_mem, sm_count = gpu_props()
    with capi.Context(0) as one, util.device_group(G) as many:
        up1 = {k: one.upload(v) for k, v in scenes.items()}
        upm = {k: many.upload(v) for k, v in scenes.items()}
        stack = one.download(up1["synthetic"])[1]
        for name, scene, kernel, mrd, flags in TILE_PIPELINES:
            for w, h in shapes:
                def p(**kw):
                    return capi.make_params(kernel, w, h, depth=4, max_ray_depth=mrd, frames=2,
                                            accum_mode=L.ACCUM_RUNNING_MEAN, flags=flags, **kw)
                if name == "flat_stream":  # a member's share really runs k_flat_stream
                    rows = len(capi.tile_rows(h, G, 0))
                    plan = capi.plan(capi.make_params(kernel, w, rows, depth=4, frames=2,
                                                      accum_mode=L.ACCUM_RUNNING_MEAN),
                                     len(scenes[scene].nodes), stack, total_mem, sm_count)
                    assert plan["pipeline"] == capi.PIPE_FLAT_STREAM, (w, rows, plan)
                one.accum_reset()
                many.accum_reset()
                for fc in (0, 2):
                    cam = util.default_camera(0.03, fc)
                    want = one.render(up1[scene], cam, p())
                    got = many.render(upm[scene], cam, p(split_mode=L.SPLIT_TILES))
                    util.assert_bit_equal(got, want, "%s %dx%d over %d members, frameCount %d" % (name, w, h, G, fc))
        for s in up1.values():
            s.release()
        for s in upm.values():
            s.release()


# ---------------------------------------------------------------- one group across calls

def test_one_group_across_calls(monkeypatch):
    """Tiles, then samples, then tiles again at another image size: each result is that of a fresh single-GPU sequence
    (the accumulators reset when the split or the size changes).  A views call and an adaptive call between two
    accumulating tile calls leave the second tile call's result unchanged."""
    monkeypatch.setenv("LT_MULTI_EXCHANGE", "p2p")
    sb = util.scene("cornell_box")
    G = 3

    def tiles(w, h, depth=3):
        return capi.make_params(L.KERNEL_GI, w, h, depth=depth, max_ray_depth=3, frames=2,
                                accum_mode=L.ACCUM_RUNNING_MEAN, split_mode=L.SPLIT_TILES)

    with capi.Context(0) as one, util.device_group(G) as many:
        s1, sm = one.upload(sb), many.upload(sb)
        # tiles at frameCount 0 and 2
        one.accum_reset()
        for fc in (0, 2):
            want = one.render(s1, util.default_camera(0.0, fc), tiles(64, 48))
            util.assert_bit_equal(many.render(sm, util.default_camera(0.0, fc), tiles(64, 48)), want, "tiles %d" % fc)
        # a weighted-sum sample split: device 0's accumulator starts from zero, not from its tile rows
        sp = split_params(L.KERNEL_GI, 64, 48, 3, 3, 5, L.ACCUM_WEIGHTED_SUM, 0.25)
        got = many.render(sm, util.default_camera(0.0, 4), sp)
        want = restate_sample_split(one, s1, G, L.KERNEL_GI, 64, 48, 3, 3, 5, 4, L.ACCUM_WEIGHTED_SUM, 0.25)
        util.assert_bit_equal(got, want, "samples after tiles")
        # tiles again, another size: frameCount 4 folds into a reset accumulator, as on a fresh single GPU
        one.accum_reset()
        for fc in (4, 6):
            want = one.render(s1, util.default_camera(0.0, fc), tiles(40, 29, 4))
            util.assert_bit_equal(many.render(sm, util.default_camera(0.0, fc), tiles(40, 29, 4)), want,
                                  "tiles at another size, frameCount %d" % fc)
        # a views call and an adaptive call between two accumulating tile calls
        one.accum_reset()
        one.render(s1, util.default_camera(0.0, 0), tiles(64, 48))
        want = one.render(s1, util.default_camera(0.0, 2), tiles(64, 48))
        many.accum_reset()
        many.render(sm, util.default_camera(0.0, 0), tiles(64, 48))
        many.render_views(sm, np.concatenate([util.default_camera(0.01 * v, v) for v in range(4)]),
                          capi.make_params(L.KERNEL_GI, 64, 48, max_ray_depth=3, frames=2,
                                           accum_mode=L.ACCUM_RUNNING_MEAN))
        many.render_adaptive(sm, util.default_camera(0.0, 0),
                             capi.make_params(L.KERNEL_GI, 64, 48, max_ray_depth=3, frames=2,
                                              accum_mode=L.ACCUM_RUNNING_MEAN), 0.1, round_frames=2, max_frames=6)
        got = many.render(sm, util.default_camera(0.0, 2), tiles(64, 48))
        util.assert_bit_equal(got, want, "tile call after views and adaptive calls")
        s1.release(); sm.release()


# ---------------------------------------------------------------- more members than work

@pytest.mark.parametrize("G", [2, 3, 8, 16])
def test_views_with_more_members_than_views(G):
    """V views over G members, V in {2, G - 1, G + 1, 2G + 3}: bit for bit the single-GPU lt_render_views; with V < G
    the idle members add no launches to the call's statistics."""
    sb = util.scene("cornell_box")
    p = capi.make_params(L.KERNEL_GI, 37, 21, max_ray_depth=3, frames=2, accum_mode=L.ACCUM_RUNNING_MEAN)
    with capi.Context(0) as one, util.device_group(G) as many:
        s1, sm = one.upload(sb), many.upload(sb)
        for V in sorted({2, max(G - 1, 1), G + 1, 2 * G + 3}):
            cams = np.concatenate([util.default_camera(0.01 * v, v % 3) for v in range(V)])
            want = one.render_views(s1, cams, p)
            got = many.render_views(sm, cams, p)
            util.assert_bit_equal(got, want, "%d views over %d members" % (V, G))
            if V < G:  # the same call after one that kept every member busy
                launches = many.stats().kernel_launches
                busy = np.concatenate([util.default_camera(0.01 * v, 0) for v in range(2 * G)])
                many.render_views(sm, busy, p)
                assert many.stats().kernel_launches > launches
                util.assert_bit_equal(many.render_views(sm, cams, p), want, "%d views again" % V)
                assert many.stats().kernel_launches == launches, (V, G)
        s1.release(); sm.release()


def test_adaptive_with_members_without_rows():
    """G = 8 at height 20: three blocks of rows, five members without any; the mean, the frame counts and the pixel
    frames equal one GPU's."""
    sb = util.scene("cornell_box_lens")
    p = capi.make_params(L.KERNEL_GI, 45, 20, max_ray_depth=4, frames=4, accum_mode=L.ACCUM_RUNNING_MEAN)
    cam = util.default_camera(0.03, 0)
    with capi.Context(0) as one, util.device_group(8) as many:
        s1, sm = one.upload(sb), many.upload(sb)
        want, want_n, want_res = one.render_adaptive(s1, cam, p, 0.08, round_frames=4, max_frames=16)
        got, got_n, res = many.render_adaptive(sm, cam, p, 0.08, round_frames=4, max_frames=16)
        util.assert_bit_equal(got, want, "adaptive mean, 8 members, height 20")
        np.testing.assert_array_equal(got_n, want_n)
        assert (res.pixel_frames, res.pixels_unconverged) == (want_res.pixel_frames, want_res.pixels_unconverged)
        s1.release(); sm.release()


# ---------------------------------------------------------------- host threads on one device

def test_deep_culled_tile_split_in_a_fresh_process():
    """Eight members of a shared group launch the culled traversal of a 61-level tree, which needs more than 48 KB of
    dynamic shared memory, from eight host threads at once, in a process where no kernel has been opted in yet: none
    may launch before the opt-in is complete.  Bit for bit against one GPU."""
    import sys
    script = r'''
import numpy as np
import util
from lens_trace_b200 import capi, layouts as L
from test_gpu_round2 import chain_scene
sb = chain_scene(62)
cam = L.make_camera(0.0, 2.5, -20.0, 0.0, 1)
p = dict(max_ray_depth=3, flags=L.FLAG_CULL)
with capi.Context.shared(0, 8) as many:
    sm = many.upload(sb)
    got = [many.render(sm, cam, capi.make_params(k, 160, 120, split_mode=L.SPLIT_TILES, **p))
           for k in (L.KERNEL_BASIC_CU, L.KERNEL_GI)]
    sm.release()
with capi.Context(0) as one:
    s1 = one.upload(sb)
    for k, g in zip((L.KERNEL_BASIC_CU, L.KERNEL_GI), got):
        util.assert_bit_equal(g, one.render(s1, cam, capi.make_params(k, 160, 120, **p)), "kernel %d" % k)
    s1.release()
print("ok")
'''
    tests = os.path.dirname(os.path.abspath(__file__))
    path = [util.ROOT, os.path.join(util.ROOT, "oracle"), tests] + [x for x in [os.environ.get("PYTHONPATH")] if x]
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(path))
    r = subprocess.run([sys.executable, "-s", "-c", script], cwd=tests, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr
