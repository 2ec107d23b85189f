#!/usr/bin/env python3
"""Box tests per ray on the full and the pruned threaded copies (lt_debug_build_threaded / _pruned), counted on the
CPU by walking the records in float32 the way trav_threaded_nodes does, root excluded (it comes from the kernel
parameters).  Rays: the camera rays of the default camera at W x H and, from every camera hit, one bounce ray in a
uniformly sampled direction of the hemisphere around the shading normal (seeded) -- a stand-in for the GI kernel's
ray stream, which the library does not expose.  For the real stream, the oracle's own count of the reference's box
tests (full sequences, root included) is printed beside it.  Rays with a zero or non-finite reciprocal walk the full
copies on the device and are counted there.  Beside them: the pruned copies of the traversal tree lt_scene_upload
builds over the reference's leaves (lt_debug_build_traversal_tree), and those of a PLOC tree over the primitives
(the NumPy restatement of tests/test_ploc_builder.py), which reach the same triangles.  Each row also gives the cost
model the traversal tree is chosen by (lt_debug_traversal_tree: expected box tests per root-hitting ray, by surface
area), and the costs of the traversal tree's candidates are listed.
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
from test_ploc_builder import emit, ploc_tree  # noqa: E402
from test_traversal_tree_cost import box_tests_per_ray, stand_in_rays  # noqa: E402

model = sys.argv[1] if len(sys.argv) > 1 else "cornell_box"
w = int(sys.argv[2]) if len(sys.argv) > 2 else 480
h = int(sys.argv[3]) if len(sys.argv) > 3 else 270
sb = util.scene(model)
O3, INV, pruned_ok = stand_in_rays(sb, w, h)
full = capi.build_threaded(sb.nodes)
pruned = capi.build_threaded_pruned(sb.nodes)
_, _, tf = _walk(full, O3, INV)
tp = box_tests_per_ray(pruned, tf, O3, INV, pruned_ok)
costs = capi.traversal_tree(sb.nodes, len(sb.prims))
print("%s: %d nodes, %d records per pruned copy; %d rays (%d camera, %d bounce), %d on the full copies" % (
    model, len(sb.nodes), pruned.shape[1], len(O3), w * h, len(O3) - w * h, int((~pruned_ok).sum())))
print("box tests per ray, root excluded: full copies %.2f, pruned copies %.2f (%+.1f %%); cost model %.2f" % (
    tf.mean() - 1, tp, 100.0 * (tp - (tf.mean() - 1)) / (tf.mean() - 1), costs["reference"]))
trav = capi.build_traversal_tree(sb.nodes, len(sb.prims))
assert trav["traversal"]
ploc_sb, _ = emit(ploc_tree(sb.prims), sb.prims, sb.materials)
ploc = capi.build_threaded_pruned(ploc_sb.nodes)
ploc_cost = capi.traversal_tree(ploc_sb.nodes, len(ploc_sb.prims))["reference"]
for name, T, c in (("traversal tree (over the leaves, by the pruned walk's cost)", trav["pruned"],
                    min(costs["sah"], costs["ploc"], costs["restructured"])),
                   ("PLOC tree over the primitives", ploc, ploc_cost)):
    tt = box_tests_per_ray(T, tf, O3, INV, pruned_ok)
    print("  %s: %d records per pruned copy, cost model %.2f, %.2f box tests per ray (%+.1f %% against the "
          "reference's pruned copies)" % (name, T.shape[1], c, tt, 100.0 * (tt - tp) / tp))
print("  traversal tree candidates, cost model: SAH sweep %.2f, PLOC %.2f, restructured %.2f" % (
    costs["sah"], costs["ploc"], costs["restructured"]))
_, st = O.render(L.KERNEL_GI, sb, util.default_camera(0.0, 0), w, h, max_ray_depth=4, with_stats=True, threads=0)
print("GI kernel, frame 0, depth 4 (oracle): %d rays, %.2f box tests per ray on the full sequences, root included" % (
    st.rays, st.nodeTests / st.rays))
