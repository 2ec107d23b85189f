#!/usr/bin/env python3
"""Box tests per ray on the full and the pruned threaded copies (lt_debug_build_threaded / _pruned), counted on the
CPU by walking the records in float32 the way trav_threaded_nodes does, root excluded (it comes from the kernel
parameters).  Rays: the camera rays of the default camera at W x H and, from every camera hit, one bounce ray in a
uniformly sampled direction of the hemisphere around the shading normal (seeded) -- a stand-in for the GI kernel's
ray stream, which the library does not expose.  For the real stream, the oracle's own count of the reference's box
tests (full sequences, root included) is printed beside it.  Rays with a zero or non-finite reciprocal walk the full
copies on the device and are counted there.
    python tools/threaded_prune_counts.py [model] [W H]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import lt_oracle as O  # noqa: E402
import util  # noqa: E402
from lens_trace_b200 import capi, layouts as L  # noqa: E402
from test_threaded_prune import _walk  # noqa: E402

model = sys.argv[1] if len(sys.argv) > 1 else "cornell_box"
w = int(sys.argv[2]) if len(sys.argv) > 2 else 480
h = int(sys.argv[3]) if len(sys.argv) > 3 else 270
f32 = np.float32
sb = util.scene(model)
cam = util.default_camera(0.0, 0)

# camera rays (basic.cu:350-358 at yaw 0)
py, px = np.mgrid[0:h, 0:w]
fx = (px.astype(f32) / f32(w) - f32(0.5)).astype(f32).reshape(-1)
fy = (py.astype(f32) / f32(h) - f32(0.5)).astype(f32).reshape(-1)
pos = cam["pos"][0]
O3 = np.stack([fx + pos[0], fy + pos[1], np.full_like(fx, pos[2])], axis=1).astype(f32)
D = np.stack([-fx, -fy, np.full_like(fx, 5.0)], axis=1).astype(f32)

# bounce rays from the camera hits
ids, hit, tuv, _ = O.primary_hits(2, sb, cam, w, h)
m = hit.reshape(-1) == 1
t, u, v = (tuv.reshape(-1, 3)[m, k].astype(np.float64)[:, None] for k in range(3))
p = sb.prims[ids.reshape(-1)[m]]
nrm = (1 - u - v) * p["na"] + u * p["nb"] + v * p["nc"]
nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
rng = np.random.default_rng(1)
d = rng.normal(size=nrm.shape)
d /= np.linalg.norm(d, axis=1, keepdims=True)
d *= np.sign((d * nrm).sum(axis=1, keepdims=True))
hp = O3[m] + t * D[m]
O3 = np.concatenate([O3, (hp + 1e-4 * nrm).astype(f32)])
D = np.concatenate([D, d.astype(f32)])

with np.errstate(all="ignore"):
    INV = f32(1.0) / D
pruned_ok = np.isfinite(INV).all(axis=1) & (INV != 0).all(axis=1) & np.isfinite(O3).all(axis=1)
full = capi.build_threaded(sb.nodes)
pruned = capi.build_threaded_pruned(sb.nodes)
_, _, tf = _walk(full, O3, INV)
tp = tf.copy()
_, _, tp[pruned_ok] = _walk(pruned, O3[pruned_ok], INV[pruned_ok])
print("%s: %d nodes, %d records per pruned copy; %d rays (%d camera, %d bounce), %d on the full copies" % (
    model, len(sb.nodes), pruned.shape[1], len(O3), w * h, int(m.sum()), int((~pruned_ok).sum())))
print("box tests per ray, root excluded: full copies %.2f, pruned copies %.2f (%+.1f %%)" % (
    tf.mean() - 1, tp.mean() - 1, 100.0 * (tp.mean() - tf.mean()) / (tf.mean() - 1)))
_, st = O.render(L.KERNEL_GI, sb, util.default_camera(0.0, 0), w, h, max_ray_depth=4, with_stats=True, threads=0)
print("GI kernel, frame 0, depth 4 (oracle): %d rays, %.2f box tests per ray on the full sequences, root included" % (
    st.rays, st.nodeTests / st.rays))
