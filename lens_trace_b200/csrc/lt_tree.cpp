// lt_tree.cpp -- host algorithms over the reference's node array (no CUDA call): validation, the threaded copies of a
// small tree (full, then pruned, possibly of the traversal tree over the reference's leaves, with its rank table), and
// the host-only test hooks that show them.
#include "lens_trace_b200.h"
#include "lt_internal.h"

#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

int lt_validate_tree(const RefNode* nodes, int nodeCount, int primCount, int* stackDepth, std::string* why) {
  std::vector<std::pair<int, int>> todo;  // (node, number of inner ancestors)
  todo.reserve(128);
  todo.push_back({0, 0});
  long long visited = 0;
  int maxInner = 0;
  while (!todo.empty()) {
    std::pair<int, int> cur = todo.back();
    todo.pop_back();
    int i = cur.first, d = cur.second;
    if (++visited > nodeCount) { *why = "node array is not a tree (cycle or shared child)"; return -1; }
    const RefNode& n = nodes[i];
    if (n.primitiveCount > 0) {
      if (n.offset < 0 || n.offset >= primCount) { *why = "leaf primitivesOffset out of range"; return -1; }
    } else {
      if (i + 1 >= nodeCount || n.offset <= i + 1 || n.offset >= nodeCount) {
        *why = "inner node child index out of range";
        return -1;
      }
      if (n.axis > 2) { *why = "inner node axis > 2"; return -1; }
      if (d + 1 > maxInner) maxInner = d + 1;
      todo.push_back({n.offset, d + 1});
      todo.push_back({i + 1, d + 1});
    }
  }
  // every array entry must belong to the tree: the re-flatten kernels process all nodeCount entries and size their
  // output from the full-binary-tree count, so an unreachable entry would be followed unvalidated
  if (visited != nodeCount) { *why = "node array has entries that are not reachable from the root"; return -1; }
  *stackDepth = maxInner;
  return 0;
}

// Threaded form of the tree (LtThreadNode, lens_trace_b200_device.cuh): eight copies of the node array, copy o in
// the order the reference's traversal visits the nodes for rays of sign octant o, then eight pruned copies.  Built
// on the host, for small trees only (lt_plan_threaded_copies).

// The order in which the reference's traversal visits the nodes for rays of sign octant o (bit k: negative direction
// on axis k), whole tree, no culling.
static void visit_order(const RefNode* nodes, int o, std::vector<int>& order) {
  std::vector<int> stack(1, 0);
  order.clear();
  while (!stack.empty()) {
    int i = stack.back();
    stack.pop_back();
    order.push_back(i);
    const RefNode& r = nodes[i];
    if (r.primitiveCount == 0) {
      bool neg = (o >> r.axis) & 1;  // basic.cu:180-186: second child first when the direction is negative
      int nearC = neg ? r.offset : i + 1, farC = neg ? i + 1 : r.offset;
      stack.push_back(farC);
      stack.push_back(nearC);
    }
  }
}

// Appends eight copies of the threaded form to `out`, each in the visit order of its sign octant, leaving out the
// nodes with keep[i] == 0.  Copy o is records [base + o * stride, base + (o + 1) * stride), base = out.size() on
// entry, stride = the number of kept nodes; skip links are absolute record indices.  A link to a left-out node goes
// to the first kept record after it in the visit order (its first child, or that child's first child ...).
// Returns the stride.
static int append_threaded(const RefNode* nodes, int n, const std::vector<char>& keep, std::vector<LtThreadNode>& out) {
  const int base = (int)out.size();
  int stride = 0;
  for (char k : keep) stride += k ? 1 : 0;
  out.resize((size_t)base + 8 * (size_t)stride);
  std::vector<int> size(n), order, before(n + 1);
  for (int i = n - 1; i >= 0; i--)  // children follow their parent in the depth-first array
    size[i] = nodes[i].primitiveCount > 0 ? 1 : 1 + size[i + 1] + size[nodes[i].offset];
  auto bitsf = [](int v) { float f; memcpy(&f, &v, 4); return f; };
  for (int o = 0; o < 8; o++) {
    visit_order(nodes, o, order);
    // before[p]: kept nodes among the first p of the visit order = copy index of the first kept record at or after p
    // (every position has one: leaves are always kept, and a left-out node is followed by its subtree)
    for (int p = 0; p < n; p++) before[p + 1] = before[p] + (keep[order[p]] ? 1 : 0);
    const int copy = base + o * stride;
    for (int p = 0; p < n; p++) {
      const int i = order[p];
      if (!keep[i]) continue;
      const RefNode& r = nodes[i];
      const bool leaf = r.primitiveCount > 0;
      const float* lo[3];
      const float* hi[3];
      for (int k = 0; k < 3; k++) {
        bool neg = (o >> k) & 1;
        lo[k] = neg ? r.boundsMax : r.boundsMin;
        hi[k] = neg ? r.boundsMin : r.boundsMax;
      }
      const int end = p + size[i];
      const int skip = end >= n ? LT_DONE : copy + before[end];
      LtThreadNode& t = out[(size_t)copy + before[p]];
      t.a = make_float4(lo[0][0], lo[1][1], lo[2][2], hi[0][0]);
      t.b = make_float4(hi[1][1], hi[2][2], bitsf(leaf ? ~r.offset : 0), bitsf(skip));
    }
  }
  return stride;
}

// Nodes of the pruned copies.  Every builder here makes an inner box the exact min/max of its primitives, so a child
// box lies inside its parent box.  For a ray with finite, nonzero direction reciprocals and a finite origin,
// (b - o) * inv in round-to-nearest is monotonic in the bound b, so a contained child's entry is at least its
// parent's and its exit at most the parent's: a child is hit only if its parent is.  An inner node m whose two
// children lie inside its box can therefore be left out of the visit sequence.  If m would be hit, the walk goes on
// to its first child anyway.  If m would be missed, every record below it misses until a kept one misses, through the
// chain of left-out nodes, and the walk reaches m's old skip target.  Either way the same leaves are recorded in the
// same order.
// Leaving m out saves 2 p(m) - p(a) box tests per ray, p = probability that a box is hit and a = the nearest kept
// ancestor, so m goes when a ray that enters a usually enters m as well: surface area SA(m) > SA(a) / 2.  Box tests
// per ray (reference traversal order, no any-hit early exit, root excluded) for the GI kernel on the Cornell box
// (480x270, frames 0-1, depth 4, the 766 767 rays of an instrumented oracle): 26.70 with the full copies, 19.57 with
// this rule, 18.13 with per-node hit counts measured on those rays in place of the areas (an upper bound: it needs
// ray statistics); tools/threaded_prune_counts.py recounts the rule on a stand-in stream.  Leaves stay: a leaf box
// gates a triangle test, and a triangle can be hit a rounding step outside its box.  The rule does not depend on the
// octant, so all eight pruned copies have one length.  A tree that breaks containment (or has NaN or inverted
// bounds) keeps the records where it does; the comparisons below are false for NaN.
//
// Cost of the pruned walk: a kept record is tested exactly when the ray hits its nearest kept ancestor's box (the
// left-out nodes between them decide nothing), so the expected box tests per ray that hits the root are
// sum over kept records r != root of SA(keptAncestor(r)) / SA(root) -- the root's own test comes from the kernel
// parameters.  *cost receives it.  The octant changes neither the records nor the stride.
static double half_area(const float* mn, const float* mx) {
  double dx = (double)mx[0] - mn[0], dy = (double)mx[1] - mn[1], dz = (double)mx[2] - mn[2];
  return dx * dy + dy * dz + dz * dx;
}

// The rule above for a node m whose children lie inside its box, a = its nearest kept ancestor: leave m out.
static bool prune_contained(double areaM, double areaA) { return areaM > 0.5 * areaA; }

static std::vector<char> pruned_keep(const RefNode* nodes, int n, double* cost = nullptr) {
  std::vector<char> keep(n, 1);
  std::vector<int> anc(n, 0);  // nearest kept ancestor
  auto inside = [](const RefNode& c, const RefNode& m) {
    for (int k = 0; k < 3; k++)
      if (!(m.boundsMin[k] <= c.boundsMin[k] && c.boundsMin[k] <= c.boundsMax[k] && c.boundsMax[k] <= m.boundsMax[k]))
        return false;
    return true;
  };
  auto area = [](const RefNode& r) { return half_area(r.boundsMin, r.boundsMax); };
  for (int i = 0; i < n; i++) {  // parents precede their children in the depth-first array
    const RefNode& m = nodes[i];
    if (m.primitiveCount > 0) continue;
    if (i > 0)
      keep[i] = !(inside(nodes[i + 1], m) && inside(nodes[m.offset], m) &&
                  prune_contained(area(m), area(nodes[anc[i]])));
    anc[i + 1] = anc[m.offset] = keep[i] ? i : anc[i];
  }
  if (cost) {
    double sum = 0.0;
    for (int i = 1; i < n; i++)
      if (keep[i]) sum += area(nodes[anc[i]]);
    const double root = area(nodes[0]);
    *cost = root > 0.0 ? sum / root : sum;
  }
  return keep;
}

// Traversal tree (LtThreadNode).  By the argument above, applied to every ancestor of a leaf L, the reference reaches
// L exactly when L's own box is hit, provided L's box lies inside all its ancestors' boxes: which leaves a ray reaches
// is a property of the leaf boxes alone.  Any tree over the same leaves with containing inner boxes reaches the same
// ones and changes only the order of the triangle tests; the reference's result is the least (t, rank), rank = the
// leaf's position in the reference's visit order of the ray's octant (tri_test).  NaN t is never accepted, t == tInit
// without a hit stays rejected, and an any-hit ray only asks whether some reached triangle is accepted.
//
// Whether the reference's leaves allow one: every leaf box inside each of its ancestors' boxes, all bounds finite
// with lo <= hi (the builder below sorts centroids and sums areas), no primitive linked by two leaves (a rank per
// primitive), an inner root.  The tie-break table (8 ints per primitive) may take at most as much memory as the
// threaded copies (16 records per node): a small tree over a huge primitive array keeps the reference's copies.
static bool leaves_decide_reach(const RefNode* nodes, int n, int primCount) {
  if (n < 3 || nodes[0].primitiveCount > 0 || (long long)primCount > 16ll * n) return false;
  // lo, hi of node i: the intersection of its ancestors' boxes
  std::vector<float> lo((size_t)n * 3, -INFINITY), hi((size_t)n * 3, INFINITY);
  std::vector<char> linked((size_t)primCount, 0);
  for (int i = 0; i < n; i++) {  // parents precede their children in the depth-first array
    const RefNode& r = nodes[i];
    for (int k = 0; k < 3; k++)
      if (!(std::isfinite(r.boundsMin[k]) && std::isfinite(r.boundsMax[k]) && r.boundsMin[k] <= r.boundsMax[k]))
        return false;
    if (r.primitiveCount > 0) {
      for (int k = 0; k < 3; k++)
        if (r.boundsMin[k] < lo[(size_t)i * 3 + k] || r.boundsMax[k] > hi[(size_t)i * 3 + k]) return false;
      if (linked[r.offset]) return false;
      linked[r.offset] = 1;
      continue;
    }
    for (int c : {i + 1, r.offset})
      for (int k = 0; k < 3; k++) {
        lo[(size_t)c * 3 + k] = std::max(lo[(size_t)i * 3 + k], r.boundsMin[k]);
        hi[(size_t)c * 3 + k] = std::min(hi[(size_t)i * 3 + k], r.boundsMax[k]);
      }
  }
  return true;
}

// The traversal tree's builders share one form: a binary tree over the reference's leaf records.  Node j < m is leaf
// ordinal j (the j-th leaf of the reference's array), inner nodes follow, kid[0] = -1 for a leaf.  A leaf's box is its
// record's; an inner node's box is the exact float min/max of its children's, so every child lies inside its parent.
struct LeafTree {
  struct Node {
    int kid[2];
    float mn[3], mx[3];
  };
  std::vector<Node> node;
  int root = 0;

  LeafTree(const RefNode* nodes, const std::vector<int>& leaf) : node(leaf.size()) {
    node.reserve(2 * leaf.size() - 1);
    for (size_t j = 0; j < leaf.size(); j++) {
      node[j].kid[0] = node[j].kid[1] = -1;
      memcpy(node[j].mn, nodes[leaf[j]].boundsMin, sizeof node[j].mn);
      memcpy(node[j].mx, nodes[leaf[j]].boundsMax, sizeof node[j].mx);
    }
  }
  void fit(int i) {
    const Node &a = node[node[i].kid[0]], &b = node[node[i].kid[1]];
    for (int k = 0; k < 3; k++) {
      node[i].mn[k] = std::min(a.mn[k], b.mn[k]);
      node[i].mx[k] = std::max(a.mx[k], b.mx[k]);
    }
  }
  int join(int a, int b) {
    node.push_back(Node{{a, b}, {}, {}});
    fit((int)node.size() - 1);
    return (int)node.size() - 1;
  }
  double area(int i) const { return half_area(node[i].mn, node[i].mx); }
  // every node, children before their parent
  std::vector<int> postorder() const {
    std::vector<int> order, stack(1, root);
    while (!stack.empty()) {
      const int i = stack.back();
      stack.pop_back();
      order.push_back(i);
      if (node[i].kid[0] >= 0) {
        stack.push_back(node[i].kid[0]);
        stack.push_back(node[i].kid[1]);
      }
    }
    std::reverse(order.begin(), order.end());
    return order;
  }
};

// (a) SAH sweep: every split is a full sweep over the leaf-box centroids on each axis, minimising
// SA(first) * leaves(first) + SA(second) * leaves(second).
static LeafTree sah_leaf_tree(const RefNode* nodes, const std::vector<int>& leaf) {
  LeafTree t(nodes, leaf);
  const int m = (int)leaf.size();
  std::vector<double> cen((size_t)m * 3);
  for (int j = 0; j < m; j++)
    for (int k = 0; k < 3; k++) cen[(size_t)j * 3 + k] = (double)t.node[j].mn[k] + t.node[j].mx[k];
  std::vector<int> item(m);
  for (int j = 0; j < m; j++) item[j] = j;
  std::vector<double> secondCost(m);
  struct Box {
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    void grow(const LeafTree::Node& r) {
      for (int k = 0; k < 3; k++) {
        mn[k] = std::min(mn[k], r.mn[k]);
        mx[k] = std::max(mx[k], r.mx[k]);
      }
    }
    double area() const { return half_area(mn, mx); }
  };
  struct Task { int begin, end, parent, side; };
  std::vector<Task> todo = {{0, m, -1, 0}};
  while (!todo.empty()) {
    const Task tk = todo.back();
    todo.pop_back();
    const int b = tk.begin, e = tk.end;
    int id = item[b];
    if (e - b > 1) {
      int bestAxis = 0, bestCut = b + 1;
      double bestCost = INFINITY;
      for (int k = 0; k < 3; k++) {
        std::sort(item.begin() + b, item.begin() + e, [&](int x, int y) {
          double cx = cen[(size_t)x * 3 + k], cy = cen[(size_t)y * 3 + k];
          return cx < cy || (cx == cy && x < y);
        });
        Box second, first;
        for (int j = e - 1; j > b; j--) {
          second.grow(t.node[item[j]]);
          secondCost[j] = second.area() * (e - j);
        }
        for (int j = b + 1; j < e; j++) {  // cut j: first child [b, j), second [j, e)
          first.grow(t.node[item[j - 1]]);
          const double cost = first.area() * (j - b) + secondCost[j];
          if (cost < bestCost) {
            bestCost = cost;
            bestAxis = k;
            bestCut = j;
          }
        }
      }
      if (bestAxis != 2)
        std::sort(item.begin() + b, item.begin() + e, [&](int x, int y) {
          double cx = cen[(size_t)x * 3 + bestAxis], cy = cen[(size_t)y * 3 + bestAxis];
          return cx < cy || (cx == cy && x < y);
        });
      id = (int)t.node.size();
      t.node.push_back(LeafTree::Node{{-1, -1}, {}, {}});
      todo.push_back({bestCut, e, id, 1});
      todo.push_back({b, bestCut, id, 0});
    }
    if (tk.parent >= 0)
      t.node[tk.parent].kid[tk.side] = id;
    else
      t.root = id;
  }
  for (int i = (int)t.node.size() - 1; i >= m; i--) t.fit(i);  // inner children come after their parent
  return t;
}

// (b) PLOC over the leaf boxes, as lt_bvh.cu builds it over primitive boxes: clusters in the Morton order of their
// centroids (21 bits per axis over the centroids' bounds, stable), each one's nearest neighbour within kPlocRadius
// positions by the float half-area of the union, ties by (pair hash, lower position, higher position); mutual
// nearest neighbours merge into the lower position.  The smallest pair key is always mutual, so every round merges.
static LeafTree ploc_leaf_tree(const RefNode* nodes, const std::vector<int>& leaf) {
  constexpr int kPlocRadius = 8;
  LeafTree t(nodes, leaf);
  const int m = (int)leaf.size();
  std::vector<float> c((size_t)m * 3);
  float cmn[3] = {INFINITY, INFINITY, INFINITY}, cmx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int j = 0; j < m; j++)
    for (int k = 0; k < 3; k++) {
      const float v = 0.5f * t.node[j].mn[k] + 0.5f * t.node[j].mx[k];
      c[(size_t)j * 3 + k] = v;
      cmn[k] = std::min(cmn[k], v);
      cmx[k] = std::max(cmx[k], v);
    }
  auto spread21 = [](uint64_t x) {
    x &= 0x1FFFFF;
    x = (x | x << 32) & 0x1F00000000FFFFull;
    x = (x | x << 16) & 0x1F0000FF0000FFull;
    x = (x | x << 8) & 0x100F00F00F00F00Full;
    x = (x | x << 4) & 0x10C30C30C30C30C3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
  };
  std::vector<uint64_t> key(m);
  for (int j = 0; j < m; j++) {
    uint64_t q[3];
    for (int k = 0; k < 3; k++) {
      const float ext = cmx[k] - cmn[k];
      const float u = ext > 0.0f ? (c[(size_t)j * 3 + k] - cmn[k]) / ext : 0.0f;
      q[k] = (uint64_t)std::min(std::max(u * 2097152.0f, 0.0f), 2097151.0f);
    }
    key[j] = spread21(q[0]) << 2 | spread21(q[1]) << 1 | spread21(q[2]);
  }
  std::vector<int> cl(m);  // cluster at each position -> tree node
  for (int j = 0; j < m; j++) cl[j] = j;
  std::stable_sort(cl.begin(), cl.end(), [&](int x, int y) { return key[x] < key[y]; });
  auto pair_hash = [](uint32_t a, uint32_t b) {
    uint32_t h = a ^ (b * 0x9E3779B9u);
    h ^= h >> 16;
    h *= 0x85EBCA6Bu;
    h ^= h >> 13;
    h *= 0xC2B2AE35u;
    h ^= h >> 16;
    return h;
  };
  std::vector<int> nn(m), next;
  while (cl.size() > 1) {
    const int cnt = (int)cl.size();
    for (int i = 0; i < cnt; i++) {
      uint32_t bd = 0, bh = 0;
      int ba = 0, bb = 0, best = -1;
      for (int j = std::max(0, i - kPlocRadius); j <= std::min(cnt - 1, i + kPlocRadius); j++) {
        if (j == i) continue;
        const LeafTree::Node &p = t.node[cl[i]], &q = t.node[cl[j]];
        float e[3];
        for (int k = 0; k < 3; k++) e[k] = std::max(p.mx[k], q.mx[k]) - std::min(p.mn[k], q.mn[k]);
        const float area = (e[0] * e[1] + e[1] * e[2]) + e[2] * e[0];
        uint32_t d;
        memcpy(&d, &area, 4);
        const int a = std::min(i, j), b = std::max(i, j);
        const uint32_t h = pair_hash((uint32_t)a, (uint32_t)b);
        if (best < 0 || d < bd || (d == bd && (h < bh || (h == bh && (a < ba || (a == ba && b < bb)))))) {
          best = j;
          bd = d;
          bh = h;
          ba = a;
          bb = b;
        }
      }
      nn[i] = best;
    }
    next.clear();
    for (int i = 0; i < cnt; i++) {
      const int j = nn[i];
      if (nn[j] != i)
        next.push_back(cl[i]);
      else if (i < j)
        next.push_back(t.join(cl[i], cl[j]));
    }
    cl.swap(next);
  }
  t.root = cl[0];
  return t;
}

// (c) Treelet restructuring (Karras & Aila, "Fast Parallel Construction of High-Quality Bounding Volume
// Hierarchies", HPG 2013) with the pruned walk's cost as the objective.  One pass visits every inner node x, children
// before parents, grows a treelet below x to kTreeletLeaves leaves by expanding its largest inner leaf, and replaces
// the treelet by the topology over the same leaves with the least cost, found exhaustively by dynamic programming
// over leaf sets.  The cost is not a plain SAH: a node's keep decision and test probability depend on the area of its
// nearest kept ancestor, so a leaf set's optimum is taken per ancestor (x's own nearest kept ancestor, or any larger
// leaf set of the treelet), and the subtrees hanging below the treelet are costed by walking them down to their kept
// nodes, whose subtree costs `g` are kept up to date.  The box of x, and so everything outside the treelet, does not
// change, and every accepted treelet lowers the cost, so the build may stop after any treelet: at the end of a pass
// that improved none, or once its work (node walks and split evaluations) exceeds the budget it is given.
class TreeletRestructure {
 public:
  static constexpr int kTreeletLeaves = 7, kSets = 1 << kTreeletLeaves;

  TreeletRestructure(LeafTree& t, long long budget)
      : t_(t), area_(t.node.size()), g_(t.node.size()), budget_(budget),
        memo_((size_t)kSets * kSets), choice_((size_t)kSets * kSets), stamp_((size_t)kSets * kSets, 0),
        leafMemo_((size_t)kTreeletLeaves * kSets), leafStamp_((size_t)kTreeletLeaves * kSets, 0) {
    for (size_t i = 0; i < t.node.size(); i++) area_[i] = t.area((int)i);
    for (int x : t.postorder())
      if (t.node[x].kid[0] >= 0) regain(x);
  }

  // One bottom-up pass; whether some treelet improved.
  bool pass() {
    bool improved = false;
    struct Frame { int x; double a; bool down; };  // a: area of x's nearest kept ancestor
    std::vector<Frame> st = {{t_.root, 0.0, true}};
    while (!st.empty() && work_ <= budget_) {
      const Frame f = st.back();
      if (!f.down) {
        st.pop_back();
        improved |= treelet(f.x, f.a);
        continue;
      }
      const int k0 = t_.node[f.x].kid[0], k1 = t_.node[f.x].kid[1];
      if (k0 < 0) {
        st.pop_back();
        continue;
      }
      st.back().down = false;
      const double a = kept_area(f.x, f.a);
      st.push_back({k1, a, true});
      st.push_back({k0, a, true});
    }
    return improved;
  }
  bool exhausted() const { return work_ > budget_; }

 private:
  // the area that x's children see as their nearest kept ancestor's, when x's own is `a` (the root is always kept)
  double kept_area(int x, double a) const {
    return x == t_.root || !prune_contained(area_[x], a) ? area_[x] : a;
  }

  // cost of the records of x's subtree, x included, when x's nearest kept ancestor has area a
  double below(int x, double a) {
    double s = 0.0;
    walk_.assign(1, x);
    while (!walk_.empty()) {
      const int y = walk_.back();
      walk_.pop_back();
      work_++;
      const LeafTree::Node& nd = t_.node[y];
      if (nd.kid[0] >= 0 && prune_contained(area_[y], a)) {
        walk_.push_back(nd.kid[1]);
        walk_.push_back(nd.kid[0]);
      } else {
        s += a + (nd.kid[0] >= 0 ? g_[y] : 0.0);
      }
    }
    return s;
  }
  // g: cost of x's subtree below x when x is kept
  void regain(int x) { g_[x] = below(t_.node[x].kid[0], area_[x]) + below(t_.node[x].kid[1], area_[x]); }

  double set_area(int s) const { return s == full_ ? rootA_ : sarea_[s]; }  // full_: x's children's kept ancestor

  double leaf_cost(int s, int a) {
    const int j = __builtin_ctz(s);
    const size_t i = (size_t)j * kSets + a;
    if (leafStamp_[i] != gen_) {
      leafStamp_[i] = gen_;
      leafMemo_[i] = below(lv_[j], set_area(a));
    }
    return leafMemo_[i];
  }

  // least cost of a subtree over leaf set s (two or more leaves) below the children of the best split, given the
  // kept ancestor set a; *part receives that split's part holding s's lowest leaf
  double split(int s, int a, int* part) {
    const int low = s & -s;
    double best = INFINITY;
    for (int p = (s - 1) & s; p; p = (p - 1) & s) {
      if (!(p & low)) continue;
      work_++;
      const double c = opt(p, a) + opt(s ^ p, a);
      if (c < best) {
        best = c;
        *part = p;
      }
    }
    return best;
  }

  // least cost of a subtree over leaf set s whose nearest kept ancestor is set a
  double opt(int s, int a) {
    if (!(s & (s - 1))) return leaf_cost(s, a);
    const size_t i = (size_t)s * kSets + a;
    if (stamp_[i] != gen_) {
      const bool pruned = prune_contained(sarea_[s], set_area(a));
      stamp_[i] = gen_;
      memo_[i] = (pruned ? 0.0 : set_area(a)) + split(s, pruned ? a : s, &choice_[i]);
    }
    return memo_[i];
  }

  int mask_of(int x) const {
    for (int j = 0; j < nl_; j++)
      if (lv_[j] == x) return 1 << j;
    return mask_of(t_.node[x].kid[0]) | mask_of(t_.node[x].kid[1]);
  }

  // the same cost for the treelet's current topology below node x (leaf set s)
  double current(int x, int s, int a) {
    if (!(s & (s - 1))) return leaf_cost(s, a);
    const bool pruned = prune_contained(sarea_[s], set_area(a));
    return (pruned ? 0.0 : set_area(a)) + current_split(x, s, pruned ? a : s);
  }
  double current_split(int x, int s, int a) {
    const int k0 = t_.node[x].kid[0], k1 = t_.node[x].kid[1], s0 = mask_of(k0);
    const bool first0 = (s0 & s & -s) != 0;
    const double c0 = current(k0, s0, a), c1 = current(k1, s ^ s0, a);
    return first0 ? c0 + c1 : c1 + c0;
  }

  // rebuilds leaf set s with the optimum's splits on the treelet's inner nodes; returns its node
  int rebuild(int s, int a, int* next) {
    if (!(s & (s - 1))) return lv_[__builtin_ctz(s)];
    const size_t i = (size_t)s * kSets + a;
    const int cs = prune_contained(sarea_[s], set_area(a)) ? a : s;
    const int x = in_[(*next)++];
    const int k0 = rebuild(choice_[i], cs, next), k1 = rebuild(s ^ choice_[i], cs, next);
    t_.node[x].kid[0] = k0;
    t_.node[x].kid[1] = k1;
    t_.fit(x);
    area_[x] = t_.area(x);
    regain(x);
    return x;
  }

  bool treelet(int x, double a) {
    in_[0] = x;
    lv_[0] = t_.node[x].kid[0];
    lv_[1] = t_.node[x].kid[1];
    int ni = 1;
    nl_ = 2;
    while (nl_ < kTreeletLeaves) {
      int k = -1;
      for (int j = 0; j < nl_; j++)
        if (t_.node[lv_[j]].kid[0] >= 0 && (k < 0 || area_[lv_[j]] > area_[lv_[k]])) k = j;
      if (k < 0) break;
      in_[ni++] = lv_[k];
      lv_[nl_++] = t_.node[lv_[k]].kid[1];
      lv_[k] = t_.node[lv_[k]].kid[0];
    }
    bool improved = false;
    if (nl_ >= 3) {
      full_ = (1 << nl_) - 1;
      rootA_ = kept_area(x, a);
      gen_++;
      for (int s = 1; s <= full_; s++) {
        const int low = s & -s;
        if (s == low) {
          const LeafTree::Node& nd = t_.node[lv_[__builtin_ctz(s)]];
          memcpy(smn_[s], nd.mn, sizeof smn_[s]);
          memcpy(smx_[s], nd.mx, sizeof smx_[s]);
        } else {
          for (int k = 0; k < 3; k++) {
            smn_[s][k] = std::min(smn_[low][k], smn_[s ^ low][k]);
            smx_[s][k] = std::max(smx_[low][k], smx_[s ^ low][k]);
          }
        }
        sarea_[s] = half_area(smn_[s], smx_[s]);
      }
      const double now = current_split(x, full_, full_);
      int p = 0;
      const double best = split(full_, full_, &p);
      if (best < now - 1e-9 * now) {
        int next = 1;
        const int k0 = rebuild(p, full_, &next), k1 = rebuild(full_ ^ p, full_, &next);
        t_.node[x].kid[0] = k0;
        t_.node[x].kid[1] = k1;
        improved = true;
      }
    }
    regain(x);  // the subtrees below may have changed since x's g was last computed
    return improved;
  }

  LeafTree& t_;
  std::vector<double> area_, g_;
  long long work_ = 0, budget_;
  std::vector<int> walk_;
  // the current treelet: leaves, inner nodes (in_[0] = its root), leaf sets' boxes and areas
  int lv_[kTreeletLeaves], in_[kTreeletLeaves - 1], nl_ = 0, full_ = 0;
  double rootA_ = 0.0, sarea_[kSets];
  float smn_[kSets][3], smx_[kSets][3];
  // opt() per (leaf set, kept ancestor set), valid when stamp_ == gen_
  std::vector<double> memo_;
  std::vector<int> choice_, stamp_;
  std::vector<double> leafMemo_;
  std::vector<int> leafStamp_;
  int gen_ = 0;
};

// A leaf tree in the reference's depth-first layout, each leaf record copied as it is: its box gates its triangle
// test, and a multi-primitive leaf's box may be larger than the one triangle it tests.  `axis` is the axis on which
// the two children's box centroids lie farthest apart, the child with the lower centroid on it first (the child with
// the lower leaf ordinal when they are equal), as lt_bvh.cu orders PLOC's merges.  n = 2 m - 1 nodes again.
static std::vector<RefNode> emit_leaf_tree(const RefNode* nodes, const std::vector<int>& leaf, const LeafTree& t) {
  const int m = (int)leaf.size();
  std::vector<int> low(t.node.size());  // lowest leaf ordinal below each node
  for (int i : t.postorder())
    low[i] = t.node[i].kid[0] < 0 ? i : std::min(low[t.node[i].kid[0]], low[t.node[i].kid[1]]);
  std::vector<RefNode> out((size_t)(2 * m - 1));
  struct Task { int node, parent; };  // parent >= 0: this node is the second child of out[parent]
  std::vector<Task> todo = {{t.root, -1}};
  int next = 0;
  while (!todo.empty()) {
    const Task tk = todo.back();
    todo.pop_back();
    const int idx = next++;
    if (tk.parent >= 0) out[tk.parent].offset = idx;
    const LeafTree::Node& nd = t.node[tk.node];
    if (nd.kid[0] < 0) {
      out[idx] = nodes[leaf[tk.node]];
      continue;
    }
    const LeafTree::Node &a = t.node[nd.kid[0]], &b = t.node[nd.kid[1]];
    double d[3];
    int axis = 0;
    for (int k = 0; k < 3; k++) {
      d[k] = ((double)b.mn[k] + b.mx[k]) - ((double)a.mn[k] + a.mx[k]);
      if (std::fabs(d[k]) > std::fabs(d[axis])) axis = k;
    }
    const bool swap = d[axis] < 0.0 || (d[axis] == 0.0 && low[nd.kid[1]] < low[nd.kid[0]]);
    RefNode& r = out[idx];
    memset(&r, 0, sizeof r);
    memcpy(r.boundsMin, nd.mn, sizeof r.boundsMin);
    memcpy(r.boundsMax, nd.mx, sizeof r.boundsMax);
    r.axis = (uint8_t)axis;
    todo.push_back({nd.kid[swap ? 0 : 1], idx});  // second child, placed after the whole first subtree
    todo.push_back({nd.kid[swap ? 1 : 0], -1});   // first child: the next node, idx + 1
  }
  return out;
}

// The traversal tree: of (a) the SAH sweep tree, (b) the PLOC tree and (c) the better of the two after treelet
// restructuring, the one whose pruned copies cost the least (pruned_keep), the earlier one on equal cost.  costs
// (optional) receives the three costs.  Cornell box: 16.77 / 15.95 / 15.70 (box tests per ray on the stand-in stream of
// tools/threaded_prune_counts.py: SAH sweep 7.30, this tree 6.86); lens scene: 22.73 / 21.57 / 21.34 (11.52, 10.51).
// A pass costs about 330 work units per leaf on ordinary trees, and two or three passes reach the local optimum
// (passes after the third gained less than 0.05 % on a 64 539-node tree), hence at most kMaxPasses passes within
// kRestructureWork units per leaf: on that tree the build takes 0.63 s instead of the SAH tree's 0.19 s (one core of
// an x86-64 server CPU), and the budget bounds it where walks grow long (leaves with equal boxes).
static std::vector<RefNode> build_traversal_tree(const RefNode* nodes, int n, double* costs = nullptr) {
  constexpr int kMaxPasses = 3;
  constexpr long long kRestructureWork = 1024;
  std::vector<int> leaf;  // leaf ordinal -> reference node
  for (int i = 0; i < n; i++)
    if (nodes[i].primitiveCount > 0) leaf.push_back(i);
  auto cost_of = [](const std::vector<RefNode>& r) {
    double c = 0.0;
    pruned_keep(r.data(), (int)r.size(), &c);
    return c;
  };
  const LeafTree sah = sah_leaf_tree(nodes, leaf), ploc = ploc_leaf_tree(nodes, leaf);
  std::vector<RefNode> best = emit_leaf_tree(nodes, leaf, sah), other = emit_leaf_tree(nodes, leaf, ploc);
  const double costSah = cost_of(best), costPloc = cost_of(other);
  LeafTree tuned = costPloc < costSah ? ploc : sah;
  if (costPloc < costSah) best.swap(other);
  TreeletRestructure rs(tuned, kRestructureWork * (long long)leaf.size());
  for (int p = 0; p < kMaxPasses && !rs.exhausted(); p++)
    if (!rs.pass()) break;
  other = emit_leaf_tree(nodes, leaf, tuned);
  const double costTuned = cost_of(other);
  if (costs) {
    costs[0] = costSah;
    costs[1] = costPloc;
    costs[2] = costTuned;
  }
  if (costTuned < std::min(costSah, costPloc)) best.swap(other);
  return best;
}

// rank[o * primCount + p]: the position of the leaf linking primitive p among the leaves of octant o's reference visit
// order (the sequence of append_threaded's copy o).  Primitives no leaf links keep 0: they are never tested.
static std::vector<int> leaf_ranks(const RefNode* nodes, int primCount) {
  std::vector<int> rank((size_t)8 * primCount, 0), order;
  for (int o = 0; o < 8; o++) {
    visit_order(nodes, o, order);
    int pos = 0;
    for (int i : order)
      if (nodes[i].primitiveCount > 0) rank[(size_t)o * primCount + nodes[i].offset] = pos++;
  }
  return rank;
}

// Full copies of the reference tree (records [0, 8 n)), then the pruned copies (from record 8 n): of the traversal
// tree when the reference's leaves decide reach, with its tie-break table in `rank`; otherwise of the reference tree,
// and `rank` empty.  Returns the pruned stride.
int lt_build_threaded(const RefNode* nodes, int n, int primCount, std::vector<LtThreadNode>& out,
                      std::vector<int>& rank) {
  out.clear();
  rank.clear();
  append_threaded(nodes, n, std::vector<char>(n, 1), out);
  if (!leaves_decide_reach(nodes, n, primCount)) return append_threaded(nodes, n, pruned_keep(nodes, n), out);
  const std::vector<RefNode> trav = build_traversal_tree(nodes, n);
  rank = leaf_ranks(nodes, primCount);
  return append_threaded(trav.data(), (int)trav.size(), pruned_keep(trav.data(), (int)trav.size()), out);
}

// The node array of a host-only hook: a valid tree whose leaves link primitives below primCount.  *n: its node count.
static int debug_tree_arg(const void* nodes, uint64_t node_bytes, int primCount, const char* who, int* n) {
  if (!nodes || node_bytes == 0 || node_bytes % sizeof(RefNode) || node_bytes / sizeof(RefNode) > 0x0fffffffull)
    return lt_internal_fail(nullptr, LT_ERR_INVALID, std::string(who) + ": bad arguments");
  int depth = 0;
  *n = (int)(node_bytes / sizeof(RefNode));
  std::string why;
  const RefNode* r = (const RefNode*)nodes;
  if (lt_validate_tree(r, *n, 0x7fffffff, &depth, &why) != 0)
    return lt_internal_fail(nullptr, LT_ERR_INVALID, std::string(who) + ": " + why);
  for (int i = 0; i < *n; i++)
    if (r[i].primitiveCount > 0 && r[i].offset >= primCount)
      return lt_internal_fail(nullptr, LT_ERR_INVALID, std::string(who) + ": leaf primitivesOffset out of range");
  return LT_OK;
}

extern "C" int lt_debug_build_threaded(const void* nodes, uint64_t node_bytes, void* out_records) {
  int n = 0;
  if (!out_records) return lt_internal_fail(nullptr, LT_ERR_INVALID, "lt_debug_build_threaded: bad arguments");
  if (int rc = debug_tree_arg(nodes, node_bytes, 0x7fffffff, "lt_debug_build_threaded", &n)) return rc;
  std::vector<LtThreadNode> out;
  append_threaded((const RefNode*)nodes, n, std::vector<char>(n, 1), out);
  memcpy(out_records, out.data(), out.size() * sizeof(LtThreadNode));
  return LT_OK;
}

extern "C" int lt_debug_build_threaded_pruned(const void* nodes, uint64_t node_bytes, void* out_records,
                                              int32_t* out_stride) {
  int n = 0;
  if (!out_stride) return lt_internal_fail(nullptr, LT_ERR_INVALID, "lt_debug_build_threaded_pruned: bad arguments");
  if (int rc = debug_tree_arg(nodes, node_bytes, 0x7fffffff, "lt_debug_build_threaded_pruned", &n)) return rc;
  std::vector<LtThreadNode> out;
  *out_stride = append_threaded((const RefNode*)nodes, n, pruned_keep((const RefNode*)nodes, n), out);
  if (out_records) memcpy(out_records, out.data(), out.size() * sizeof(LtThreadNode));
  return LT_OK;
}

// What lt_scene_upload builds for a small tree: out_records (16 n records of room) receives the full copies and then the
// pruned ones, skip links as uploaded (absolute, from record 8 n); out_rank (8 x prim_count ints of room) the
// tie-break table when *out_traversal == 1, i.e. when the pruned copies are a traversal tree.
extern "C" int lt_debug_build_traversal_tree(const void* nodes, uint64_t node_bytes, int32_t prim_count,
                                             void* out_records, int32_t* out_stride, int32_t* out_rank,
                                             int32_t* out_traversal) {
  const char* who = "lt_debug_build_traversal_tree";
  int n = 0;
  if (!out_records || !out_stride || !out_rank || !out_traversal || prim_count < 1)
    return lt_internal_fail(nullptr, LT_ERR_INVALID, std::string(who) + ": bad arguments");
  if (int rc = debug_tree_arg(nodes, node_bytes, prim_count, who, &n)) return rc;
  std::vector<LtThreadNode> out;
  std::vector<int> rank;
  *out_stride = lt_build_threaded((const RefNode*)nodes, n, prim_count, out, rank);
  *out_traversal = rank.empty() ? 0 : 1;
  memcpy(out_records, out.data(), out.size() * sizeof(LtThreadNode));
  if (!rank.empty()) memcpy(out_rank, rank.data(), rank.size() * sizeof(int));
  return LT_OK;
}

// The traversal tree lt_scene_upload builds for a small tree, in the reference layout, and the costs it is chosen by.
extern "C" int lt_debug_traversal_tree(const void* nodes, uint64_t node_bytes, int32_t prim_count, void* out_nodes,
                                       double* out_costs) {
  const char* who = "lt_debug_traversal_tree";
  int n = 0;
  if (!out_nodes || !out_costs || prim_count < 1)
    return lt_internal_fail(nullptr, LT_ERR_INVALID, std::string(who) + ": bad arguments");
  if (int rc = debug_tree_arg(nodes, node_bytes, prim_count, who, &n)) return rc;
  const RefNode* r = (const RefNode*)nodes;
  pruned_keep(r, n, &out_costs[0]);
  out_costs[1] = out_costs[2] = out_costs[3] = NAN;
  if (leaves_decide_reach(r, n, prim_count)) {
    const std::vector<RefNode> trav = build_traversal_tree(r, n, out_costs + 1);
    memcpy(out_nodes, trav.data(), trav.size() * sizeof(RefNode));
  }
  return LT_OK;
}
