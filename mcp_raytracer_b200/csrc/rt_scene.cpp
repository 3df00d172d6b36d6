// rt_scene.cpp — host scene compiler.
//
// Turns the flattened SceneData of include/rt_b200.h into the device layout of rt_types.h:
// camera block (src/camera.ts:107-166), primitive records with the constructor-time products
// the reference caches (src/entities/plane.ts:33-42, quad.ts:37, sphere.ts:25-30), material
// node table with precomputed emission (src/materials/*.ts), light list
// (src/scenes/scenes.ts:74-79) and one of three acceleration structures:
//   REFERENCE  the reference's median-split topology (src/geometry/bvh.ts:34-102), flattened;
//   SAH        binned surface-area-heuristic BVH2 over the bounded primitives, unbounded ones
//              (infinite planes) kept in an always-tested prefix;
//   LIST       no hierarchy, object order (tiny scenes: the reference's Cornell BVH degenerates
//              to "all 8 primitives behind 3 box tests", SURVEY.md App. C.2).
//
// Host arithmetic follows the reference's numeric model where values are handed to the
// device as data: vectors are rounded to FP32 after every vector op, scalars stay FP64.
#include "rt_scene.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <limits>
#include <atomic>
#include <numeric>
#include <thread>

namespace rt {
namespace {

const double kInfD = std::numeric_limits<double>::infinity();
const double kPiD = 3.141592653589793;

// FP32-stored 3-vector with FP64 evaluation (gl-matrix Float32Array semantics).
struct H3 {
  float v[3];
  float& operator[](int i) { return v[i]; }
  float operator[](int i) const { return v[i]; }
};
template <class F>
H3 map3(F f) {
  H3 r;
  for (int i = 0; i < 3; ++i) r.v[i] = (float)f(i);
  return r;
}
H3 from_d(const double* p) { return map3([&](int i) { return p[i]; }); }
H3 vsum(const H3& a, const H3& b) { return map3([&](int i) { return (double)a[i] + (double)b[i]; }); }
H3 vdiff(const H3& a, const H3& b) { return map3([&](int i) { return (double)a[i] - (double)b[i]; }); }
H3 vtimes(const H3& a, double s) { return map3([&](int i) { return (double)a[i] * s; }); }
H3 vover(const H3& a, double t) { return vtimes(a, 1.0 / t); }
double vdot(const H3& a, const H3& b) { return (double)a[0] * b[0] + (double)a[1] * b[1] + (double)a[2] * b[2]; }
H3 vcross(const H3& a, const H3& b) {
  return map3([&](int i) {
    int j = (i + 1) % 3, k = (i + 2) % 3;
    return (double)a[j] * b[k] - (double)a[k] * b[j];
  });
}
H3 vnormalize(const H3& a) {
  double l = vdot(a, a);
  if (l > 0) l = 1.0 / std::sqrt(l);
  return vtimes(a, l);
}
H3 vnegate(const H3& a) {
  return map3([&](int i) { double x = -(double)a[i]; return x == 0 ? 0.0 : x; });
}
void put3(float* dst, const H3& a) { dst[0] = a[0]; dst[1] = a[1]; dst[2] = a[2]; }

struct Box {
  float mn[3], mx[3];
};
Box empty_box() {
  Box b;
  for (int i = 0; i < 3; ++i) { b.mn[i] = (float)kInfD; b.mx[i] = (float)-kInfD; }
  return b;
}
Box merge(const Box& a, const Box& b) { // aabb.ts:68-80 (min/max of FP32 values is exact)
  Box r;
  for (int i = 0; i < 3; ++i) { r.mn[i] = std::min(a.mn[i], b.mn[i]); r.mx[i] = std::max(a.mx[i], b.mx[i]); }
  return r;
}
bool finite_box(const Box& b) {
  for (int i = 0; i < 3; ++i)
    if (!std::isfinite(b.mn[i]) || !std::isfinite(b.mx[i])) return false;
  return true;
}

// One object with everything its reference constructor computes.
struct Prim {
  int type = 0, obj = 0, mat = 0;
  H3 q{}, u{}, v{}, n{}, w{};
  double r = 0, D = 0, area = 0;
  Box ref_box; // exactly the reference's boundingBox()
  Box sah_box; // finite and non-inverted where possible
  bool bounded = true;
  F4 rec0{}, rec1{}, rec2{}, rec3{};
  // axis-aligned quad specialisation (device type OBJ_AAQUAD): plane x_K = c, box test on the other two axes
  bool aa = false;
  F4 aa1{}, aa2{};
};

// u and v each along one (different) coordinate axis?
void detect_axis_aligned(Prim& p) {
  auto single_axis = [](const H3& a) {
    int ax = -1;
    for (int i = 0; i < 3; ++i)
      if (a[i] != 0.f) { if (ax >= 0) return -1; ax = i; }
    return ax;
  };
  const int iu = single_axis(p.u), iv = single_axis(p.v);
  if (iu < 0 || iv < 0 || iu == iv) return;
  const int K = 3 - iu - iv, I = (K + 1) % 3, J = (K + 2) % 3;
  auto range = [&](int ax, float& lo, float& hi) { // the quad's extent along in-plane axis ax: q .. q+u (or q+v), FP32 like q.add(u)
    const H3& e = ax == iu ? p.u : p.v;
    const float a = p.q[ax], b = (float)((double)p.q[ax] + (double)e[ax]);
    lo = std::min(a, b);
    hi = std::max(a, b);
  };
  float loI, hiI, loJ, hiJ;
  range(I, loI, hiI);
  range(J, loJ, hiJ);
  p.aa = true;
  p.aa1 = F4{p.q[K], loI, loJ, hiI};
  float axis_bits;
  std::memcpy(&axis_bits, &K, sizeof(float));
  p.aa2 = F4{hiJ, axis_bits, 0.f, 0.f};
}

void make_sphere(Prim& p) {
  H3 rv = map3([&](int) { return p.r; }); // Vec3.create(r,r,r), sphere.ts:26
  H3 lo = vdiff(p.q, rv), hi = vsum(p.q, rv);
  for (int i = 0; i < 3; ++i) {
    p.ref_box.mn[i] = lo[i];
    p.ref_box.mx[i] = hi[i];
    p.sah_box.mn[i] = std::min(lo[i], hi[i]);
    p.sah_box.mx[i] = std::max(lo[i], hi[i]);
  }
  p.bounded = finite_box(p.sah_box);
  p.rec0 = F4{p.q[0], p.q[1], p.q[2], (float)p.r};
}

void make_planar(Prim& p) {
  H3 cp = vcross(p.u, p.v); // plane.ts:33-42
  p.n = vnormalize(cp);
  p.D = vdot(p.n, p.q);
  p.w = vover(cp, vdot(cp, cp));
  const double eps = 1e-4;
  if (p.type == OBJ_PLANE) { // plane.ts:122-154
    Box b;
    for (int i = 0; i < 3; ++i) { b.mn[i] = (float)-kInfD; b.mx[i] = (float)kInfD; }
    for (int ax = 0; ax < 3; ++ax) {
      if (std::fabs((double)p.n[ax]) > 0.9999) {
        double c = p.D / (double)p.n[ax];
        b.mn[ax] = (float)(c - eps);
        b.mx[ax] = (float)(c + eps);
        break;
      }
    }
    p.ref_box = b;
    p.sah_box = b;
    p.bounded = false;
  } else { // quad.ts:92-114
    p.area = std::hypot((double)cp[0], (double)cp[1], (double)cp[2]);
    H3 c1 = p.q, c2 = vsum(p.q, p.u), c3 = vsum(p.q, p.v), c4 = vsum(vsum(p.q, p.u), p.v);
    for (int i = 0; i < 3; ++i) {
      double lo = std::min(std::min((double)c1[i], (double)c2[i]), std::min((double)c3[i], (double)c4[i]));
      double hi = std::max(std::max((double)c1[i], (double)c2[i]), std::max((double)c3[i], (double)c4[i]));
      p.ref_box.mn[i] = (float)(lo - eps);
      p.ref_box.mx[i] = (float)(hi + eps);
    }
    p.sah_box = p.ref_box;
    p.bounded = finite_box(p.sah_box);
  }
  // alpha = w.(hp x v) = hp.(v x w); beta = w.(u x hp) = hp.(w x u)   (plane.ts:71-74)
  double nn[3] = {p.n[0], p.n[1], p.n[2]};
  double A[3], B[3];
  double vv[3] = {p.v[0], p.v[1], p.v[2]}, uu[3] = {p.u[0], p.u[1], p.u[2]}, ww[3] = {p.w[0], p.w[1], p.w[2]},
         qq[3] = {p.q[0], p.q[1], p.q[2]};
  for (int i = 0; i < 3; ++i) {
    int j = (i + 1) % 3, k = (i + 2) % 3;
    A[i] = vv[j] * ww[k] - vv[k] * ww[j];
    B[i] = ww[j] * uu[k] - ww[k] * uu[j];
  }
  double a0 = qq[0] * A[0] + qq[1] * A[1] + qq[2] * A[2];
  double b0 = qq[0] * B[0] + qq[1] * B[1] + qq[2] * B[2];
  p.rec0 = F4{(float)nn[0], (float)nn[1], (float)nn[2], (float)p.D};
  p.rec1 = F4{(float)A[0], (float)A[1], (float)A[2], (float)a0};
  p.rec2 = F4{(float)B[0], (float)B[1], (float)B[2], (float)b0};
  const double eps4 = 4.0 / 16777216.0; // 4 * 2^-24
  p.rec3 = F4{(float)(std::fabs(A[0]) + std::fabs(A[1]) + std::fabs(A[2])), (float)(std::fabs(B[0]) + std::fabs(B[1]) + std::fabs(B[2])),
              (float)(eps4 * std::fabs(a0)), (float)(eps4 * std::fabs(b0))};
  if (p.type == OBJ_QUAD) detect_axis_aligned(p);
}

// ---- build tree (shared by both builders) ----
struct BNode {
  Box box;
  int left = -1, right = -1; // indices into the BNode pool; -1 = none
  std::vector<int> prims;    // leaf: ordered primitive indices
  bool leaf = false;
};

struct RefBuilder { // src/geometry/bvh.ts:34-102
  const std::vector<Prim>& P;
  std::vector<BNode>& pool;
  int build(const std::vector<int>& objects, size_t start, size_t end) {
    std::vector<int> list(objects.begin() + start, objects.begin() + end);
    Box nb = P[list[0]].ref_box;
    for (size_t i = 1; i < list.size(); ++i) nb = merge(nb, P[list[i]].ref_box);
    double ex = (double)nb.mx[0] - (double)nb.mn[0];
    double ey = (double)nb.mx[1] - (double)nb.mn[1];
    double ez = (double)nb.mx[2] - (double)nb.mn[2];
    int axis = 0;
    if (ey > ex && ey > ez) axis = 1;
    else if (ez > ex && ez > ey) axis = 2;
    size_t span = end - start;
    BNode node;
    auto less_on_axis = [&](int a, int b) { return P[a].ref_box.mn[axis] < P[b].ref_box.mn[axis]; };
    if (span <= 4) {
      node.leaf = true;
      if (span == 2 && !less_on_axis(list[0], list[1])) std::swap(list[0], list[1]);
      node.prims = list;
      // box = surroundingBox(left.box, right.box): fold of the members (empty box is the identity)
      Box b = empty_box();
      for (int pi : list) b = merge(b, P[pi].ref_box);
      node.box = b;
      pool.push_back(node);
      return (int)pool.size() - 1;
    }
    // Array.prototype.sort with a comparator that only ever says "<0" or ">0": V8's TimSort
    // consults nothing but `order < 0`, which makes it a stable sort on `<`.
    std::stable_sort(list.begin(), list.end(), less_on_axis);
    size_t mid = span / 2;
    int l = build(list, 0, mid);
    int r = build(list, mid, span);
    node.left = l;
    node.right = r;
    node.box = merge(pool[l].box, pool[r].box);
    pool.push_back(node);
    return (int)pool.size() - 1;
  }
};

// Binned-SAH builder (16 bins, leaves <= 4) over compact records that are partitioned in place, so every
// pass streams through memory.  The top of the tree is split serially into up to 16 subtrees that are
// built by std::thread workers into private node pools and spliced in afterwards; split decisions do not
// depend on the thread count, so the tree (and the image) is the same on every machine.
struct SahRec {
  float mn[3], mx[3], c[3];
  int pi;
};

struct SahBuilder {
  static constexpr int NB = 16;
  static double area(const Box& b) {
    double dx = (double)b.mx[0] - b.mn[0], dy = (double)b.mx[1] - b.mn[1], dz = (double)b.mx[2] - b.mn[2];
    if (dx < 0 || dy < 0 || dz < 0) return 0;
    return 2 * (dx * dy + dy * dz + dz * dx);
  }
  static Box box_of(const SahRec& r) {
    Box b;
    for (int a = 0; a < 3; ++a) { b.mn[a] = r.mn[a]; b.mx[a] = r.mx[a]; }
    return b;
  }
  static int make_leaf(const SahRec* r, size_t n, std::vector<BNode>& out) {
    BNode nd;
    nd.leaf = true;
    nd.box = empty_box();
    nd.prims.reserve(n);
    for (size_t i = 0; i < n; ++i) { nd.prims.push_back(r[i].pi); nd.box = merge(nd.box, box_of(r[i])); }
    out.push_back(std::move(nd));
    return (int)out.size() - 1;
  }
  // One split decision.  Returns 0 for "make a leaf", else the size of the left part (records partitioned).
  static size_t split(SahRec* r, size_t n, int depth, Box& bounds) {
    bounds = empty_box();
    Box cb = empty_box();
    for (size_t i = 0; i < n; ++i) {
      for (int ax = 0; ax < 3; ++ax) {
        bounds.mn[ax] = std::min(bounds.mn[ax], r[i].mn[ax]);
        bounds.mx[ax] = std::max(bounds.mx[ax], r[i].mx[ax]);
        cb.mn[ax] = std::min(cb.mn[ax], r[i].c[ax]);
        cb.mx[ax] = std::max(cb.mx[ax], r[i].c[ax]);
      }
    }
    // Leaves: a single primitive always is one; 2-4 primitives stay together only when splitting them does not
    // pay (cost of a split = leaf_ct + SAH).  With 4-wide nodes a child box per primitive is nearly free and
    // saves the primitive tests of a shared leaf box: swept on the 100 k-sphere / 480-sphere scenes (ms at
    // 8 / 64 spp): always-leaf <= 2, ct 1.2: 116.4 / 40.6; <= 1, ct 1.2: 109.6 / 40.0; <= 1, ct 0.5: 108.8 / 39.8.
    static const int leaf_always = std::getenv("RT_B200_SAH_LEAF") ? std::atoi(std::getenv("RT_B200_SAH_LEAF")) : 1; // development override
    static const double leaf_ct = std::getenv("RT_B200_SAH_CT") ? std::atof(std::getenv("RT_B200_SAH_CT")) : 0.5;
    if (n <= (size_t)leaf_always) return 0;
    Box bb[3][NB];
    int cnt[3][NB];
    float lo[3], scale[3];
    bool use[3];
    for (int ax = 0; ax < 3; ++ax) {
      lo[ax] = cb.mn[ax];
      use[ax] = cb.mx[ax] > cb.mn[ax];
      scale[ax] = use[ax] ? NB / (cb.mx[ax] - cb.mn[ax]) : 0.f;
      for (int k = 0; k < NB; ++k) { bb[ax][k] = empty_box(); cnt[ax][k] = 0; }
    }
    for (size_t i = 0; i < n; ++i) {
      const Box b = box_of(r[i]);
      for (int ax = 0; ax < 3; ++ax) {
        if (!use[ax]) continue;
        int k = std::min(NB - 1, std::max(0, (int)((r[i].c[ax] - lo[ax]) * scale[ax])));
        cnt[ax][k]++;
        bb[ax][k] = merge(bb[ax][k], b);
      }
    }
    double best_cost = std::numeric_limits<double>::infinity();
    int best_axis = -1, best_split = -1;
    for (int ax = 0; ax < 3; ++ax) {
      if (!use[ax]) continue;
      double ra[NB];
      int rc[NB];
      Box acc = empty_box();
      int c = 0;
      for (int k = NB - 1; k >= 1; --k) { acc = merge(acc, bb[ax][k]); c += cnt[ax][k]; ra[k] = area(acc); rc[k] = c; }
      acc = empty_box();
      c = 0;
      for (int k = 0; k < NB - 1; ++k) {
        acc = merge(acc, bb[ax][k]);
        c += cnt[ax][k];
        if (c == 0 || rc[k + 1] == 0) continue;
        double cost = area(acc) * c + ra[k + 1] * rc[k + 1];
        if (cost < best_cost) { best_cost = cost; best_axis = ax; best_split = k; }
      }
    }
    size_t mid;
    if (best_axis < 0 || depth > 56) {
      if (n <= 4) return 0;
      // degenerate centroids (or a runaway depth): median split on the widest axis
      int ax = 0;
      float w = -1;
      for (int a = 0; a < 3; ++a) { float d = bounds.mx[a] - bounds.mn[a]; if (d > w) { w = d; ax = a; } }
      mid = n / 2;
      std::nth_element(r, r + mid, r + n, [ax](const SahRec& x, const SahRec& y) { return x.c[ax] < y.c[ax]; });
    } else {
      if (n <= 4) {
        // leaf cost (n prim tests) vs split cost (2 box tests + expected prim tests)
        double leaf_cost = (double)n;
        double split_cost = leaf_ct + best_cost / std::max(area(bounds), 1e-30);
        if (leaf_cost <= split_cost) return 0;
      }
      const float l = lo[best_axis], sc = scale[best_axis];
      const int ax = best_axis, bs = best_split;
      SahRec* it = std::partition(r, r + n, [=](const SahRec& x) {
        int k = std::min(NB - 1, std::max(0, (int)((x.c[ax] - l) * sc)));
        return k <= bs;
      });
      mid = (size_t)(it - r);
      if (mid == 0 || mid == n) mid = n / 2;
    }
    return mid;
  }
  static int build(SahRec* r, size_t n, int depth, std::vector<BNode>& out) {
    Box bounds;
    const size_t mid = split(r, n, depth, bounds);
    if (mid == 0) return make_leaf(r, n, out);
    const int l = build(r, mid, depth + 1, out);
    const int rr = build(r + mid, n - mid, depth + 1, out);
    BNode node;
    node.left = l;
    node.right = rr;
    node.box = bounds; // = merge of the children's boxes (every box is the bounds of its records)
    out.push_back(std::move(node));
    return (int)out.size() - 1;
  }

  struct Task {
    SahRec* r;
    size_t n;
    int depth;
    std::vector<BNode> local;
    int root = -1;
  };
  // top of the tree: children that became tasks are recorded as -(task + 2)
  static int build_top(SahRec* r, size_t n, int depth, int levels, std::vector<BNode>& out, std::vector<Task>& tasks) {
    if (levels == 0 || n < 4096) {
      tasks.push_back(Task{r, n, depth, {}, -1});
      return -((int)tasks.size() - 1 + 2);
    }
    Box bounds;
    const size_t mid = split(r, n, depth, bounds);
    if (mid == 0) return make_leaf(r, n, out);
    const int l = build_top(r, mid, depth + 1, levels - 1, out, tasks);
    const int rr = build_top(r + mid, n - mid, depth + 1, levels - 1, out, tasks);
    BNode node;
    node.left = l;
    node.right = rr;
    node.box = bounds;
    out.push_back(std::move(node));
    return (int)out.size() - 1;
  }
  static int build_all(const std::vector<Prim>& P, const std::vector<int>& prims, std::vector<BNode>& pool) {
    std::vector<SahRec> recs(prims.size());
    for (size_t i = 0; i < prims.size(); ++i) {
      const Box& b = P[prims[i]].sah_box;
      SahRec& r = recs[i];
      for (int a = 0; a < 3; ++a) { r.mn[a] = b.mn[a]; r.mx[a] = b.mx[a]; r.c[a] = 0.5f * (b.mn[a] + b.mx[a]); }
      r.pi = prims[i];
    }
    const unsigned hw = std::thread::hardware_concurrency();
    if (recs.size() < 32768 || hw < 2) return build(recs.data(), recs.size(), 0, pool);
    std::vector<Task> tasks;
    tasks.reserve(16);
    int root = build_top(recs.data(), recs.size(), 0, 4, pool, tasks);
    {
      std::atomic<size_t> next{0};
      auto work = [&]() {
        for (size_t k; (k = next.fetch_add(1)) < tasks.size();) {
          Task& t = tasks[k];
          t.local.reserve(t.n);
          t.root = build(t.r, t.n, t.depth, t.local);
        }
      };
      const unsigned nthreads = std::min<unsigned>(std::min<unsigned>(hw, 8u), (unsigned)tasks.size());
      std::vector<std::thread> th;
      for (unsigned k = 1; k < nthreads; ++k) th.emplace_back(work);
      work();
      for (auto& t : th) t.join();
    }
    // splice the private pools in and patch the placeholders
    std::vector<int> task_root(tasks.size());
    for (size_t k = 0; k < tasks.size(); ++k) {
      const int off = (int)pool.size();
      for (BNode& nd : tasks[k].local) {
        if (!nd.leaf) { nd.left += off; nd.right += off; }
        pool.push_back(std::move(nd));
      }
      task_root[k] = tasks[k].root + off;
    }
    auto fix = [&](int& ref) { if (ref <= -2) ref = task_root[(size_t)(-ref - 2)]; };
    for (BNode& nd : pool) if (!nd.leaf) { fix(nd.left); fix(nd.right); }
    fix(root);
    return root;
  }
};

struct Flattener {
  const std::vector<Prim>& P;
  const std::vector<BNode>& pool;
  HostScene& S;
  const std::vector<int>& rank; // per object: position in the reference's visiting order
  int max_depth = 0;
  std::vector<signed char> inv_memo; // per build node: -1 unknown, 0/1
  bool has_inverted(int bi) { // does the subtree hold a primitive whose reference box is inverted?
    if (inv_memo.size() != pool.size()) inv_memo.assign(pool.size(), -1);
    if (inv_memo[bi] >= 0) return inv_memo[bi] != 0;
    const BNode& n = pool[bi];
    bool inv = false;
    if (n.leaf) {
      for (int pi : n.prims)
        for (int a = 0; a < 3; ++a)
          if (P[pi].ref_box.mn[a] > P[pi].ref_box.mx[a]) inv = true;
    } else {
      const bool l = has_inverted(n.left), r = has_inverted(n.right); // both: every node of the subtree gets its memo
      inv = l || r;
    }
    inv_memo[bi] = inv ? 1 : 0;
    return inv;
  }
  void push_slot(int pi, bool prefix = false) {
    const Prim& p = P[pi];
    S.p0.push_back(p.rec0);
    // The axis-aligned specialisation pays in the LIST kernel, where the kind is warp-uniform, and in the
    // always-tested prefix of a SAH tree (every lane tests the same slot); inside tree leaves the per-lane
    // axis dispatch costs more than it saves (measured), so leaves keep general quads.
    const bool aa = p.aa && (S.bvh_kind == BVH_LIST || prefix);
    S.p1.push_back(aa ? p.aa1 : p.rec1);
    S.p2.push_back(aa ? p.aa2 : p.rec2);
    S.p3.push_back(p.rec3);
    const unsigned dev_type = aa ? (unsigned)OBJ_AAQUAD : (unsigned)p.type;
    S.slot_info.push_back(I2{p.mat, (int)((unsigned)p.obj | (dev_type << 30))});
    ExactPrim e;
    std::memset(&e, 0, sizeof(e));
    put3(e.q, p.q); put3(e.u, p.u); put3(e.v, p.v); put3(e.n, p.n); put3(e.w, p.w);
    e.type = p.type; e.rank = rank[pi]; e.D = p.D; e.r = p.r; e.area = p.area;
    S.exact.push_back(e);
  }
  int leaf_ref(const BNode& n) {
    int first = (int)S.p0.size();
    int mask = 0;
    for (size_t k = 0; k < n.prims.size(); ++k) {
      if (P[n.prims[k]].type != OBJ_SPHERE) mask |= 1 << k;
      push_slot(n.prims[k]);
    }
    return make_leaf_ref(first, (int)n.prims.size(), mask);
  }
  int emit(int bi, int depth) { // returns the child ref for build node bi
    const BNode& n = pool[bi];
    max_depth = std::max(max_depth, depth);
    if (n.leaf) return leaf_ref(n);
    int idx = (int)S.nodes.size();
    S.nodes.emplace_back();
    fill_pair(idx, n.left, n.right, depth);
    return idx;
  }
  void fill_pair(int idx, int l, int r, int depth) {
    Node nd;
    std::memset(&nd, 0, sizeof(nd));
    Box lb = l >= 0 ? pool[l].box : empty_box();
    Box rb = r >= 0 ? pool[r].box : empty_box();
    std::memcpy(nd.lmin, lb.mn, 12); std::memcpy(nd.lmax, lb.mx, 12);
    std::memcpy(nd.rmin, rb.mn, 12); std::memcpy(nd.rmax, rb.mx, 12);
    nd.flags = ((l >= 0 && has_inverted(l)) ? 1 : 0) | ((r >= 0 && has_inverted(r)) ? 2 : 0);
    nd.left = l >= 0 ? emit(l, depth + 1) : kEmptyRef;
    nd.right = r >= 0 ? emit(r, depth + 1) : kEmptyRef;
    S.nodes[idx] = nd;
  }

  // SAH trees are flattened 4 wide (WideNode, 128 B = two Node slots): the binary tree is collapsed by
  // replacing the internal child with the largest box by its two children until a node has four children or
  // only leaves.  Half the dependent node fetches per ray; the deep-tree kernels wait on those fetches.
  // Returns the wide-node index (in units of WideNode) of build node bi (internal), or emits a single-leaf root.
  int emit_wide(int bi, int depth) {
    max_depth = std::max(max_depth, depth);
    int c[4], nc = 0;
    if (pool[bi].leaf) c[nc++] = bi; // a tree that is one leaf: root with a single leaf child
    else { c[nc++] = pool[bi].left; c[nc++] = pool[bi].right; }
    while (nc < 4) {
      int pick = -1;
      double best = -1;
      for (int k = 0; k < nc; ++k) {
        if (pool[c[k]].leaf) continue;
        const double a = SahBuilder::area(pool[c[k]].box);
        if (a > best) { best = a; pick = k; }
      }
      if (pick < 0) break;
      const int l = pool[c[pick]].left, r = pool[c[pick]].right;
      for (int k = nc; k > pick + 1; --k) c[k] = c[k - 1]; // keep the order: the two children take the parent's place
      c[pick] = l;
      c[pick + 1] = r;
      ++nc;
    }
    const int idx = (int)S.nodes.size() / 2;
    S.nodes.emplace_back();
    S.nodes.emplace_back();
    WideNode w;
    for (int k = 0; k < 4; ++k) {
      for (int a = 0; a < 3; ++a) { // (centre, half-extent), half-extent rounded up: the stored box contains the builder's
        float ctr = 0.f, half = -INFINITY; // unused child: never hit
        if (k < nc) {
          const double mn = pool[c[k]].box.mn[a], mx = pool[c[k]].box.mx[a];
          if (!std::isfinite(mn) || !std::isfinite(mx)) half = INFINITY; // unbounded on this axis
          else {
            ctr = (float)(0.5 * (mn + mx));
            // an inverted box (negative-radius sphere) keeps its extent: the min / max slab test never cared about the order
            const double hd = std::max(std::fabs(mx - (double)ctr), std::fabs((double)ctr - mn));
            half = (float)hd;
            if ((double)half < hd) half = std::nextafter(half, INFINITY);
          }
        }
        w.box[k][a] = ctr;
        w.box[k][3 + a] = half;
      }
      w.ref[k] = kEmptyRef;
      w.pad[k] = 0;
    }
    for (int k = 0; k < nc; ++k) w.ref[k] = pool[c[k]].leaf ? leaf_ref(pool[c[k]]) : emit_wide(c[k], depth + 1);
    std::memcpy(&S.nodes[2 * (size_t)idx], &w, sizeof(w));
    return idx;
  }
};

} // namespace

rt_status compile_scene(const rt_scene_desc* sd, const rt_render_opts* o, HostScene& S, std::string& err) {
  if (!sd || !o) { err = "null scene or options"; return RT_ERR_INVALID_ARGUMENT; }
  if (sd->n_objects == 0 || !sd->obj_type || !sd->obj_pos || !sd->obj_material) {
    err = "scene has no objects";
    return RT_ERR_INVALID_ARGUMENT;
  }
  if (sd->n_objects > (1u << 24)) { err = "too many objects (max 2^24)"; return RT_ERR_UNSUPPORTED; }
  if (o->width <= 0 || !(o->aspect > 0) || o->samples < 0 || o->depth < 0 || o->a_batch <= 0) {
    err = "invalid render options (width/aspect/samples/depth/aBatch)";
    return RT_ERR_INVALID_ARGUMENT;
  }
  // RT_B200_BUILD_TRACE=1: stage times of the scene compiler on stderr (development aid)
  static const bool trace = std::getenv("RT_B200_BUILD_TRACE") != nullptr;
  auto t_last = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!trace) return;
    auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[rt_b200 build] %-12s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
    t_last = now;
  };
  // ---- materials (createMaterial, scenes.ts:144-199) ----
  const uint32_t nm = sd->n_materials;
  if (nm && (!sd->mat_type || !sd->mat_color || !sd->mat_param)) { err = "material arrays missing"; return RT_ERR_INVALID_ARGUMENT; }
  S.matA.resize(nm); S.matB.resize(nm); S.matE.resize(nm); S.matF.resize(nm);
  for (uint32_t i = 0; i < nm; ++i) {
    int ty = sd->mat_type[i];
    const double* c = sd->mat_color + 3 * (size_t)i;
    double prm = sd->mat_param[i];
    int c0 = sd->mat_child ? sd->mat_child[2 * i] : -1, c1 = sd->mat_child ? sd->mat_child[2 * i + 1] : -1;
    H3 col = from_d(c);
    H3 emit = map3([](int) { return 0.0; });
    // feature albedo (the denoiser's demodulation): the colour of Lambert / Metal, 1 for Glass and Light (emission passes
    // through unchanged), folded through Mixed / Layered exactly like the emission
    H3 alb = ty == MAT_LAMBERT || ty == MAT_METAL ? col : map3([](int) { return 1.0; });
    auto f3 = [&](int k) { return H3{{S.matF[k].x, S.matF[k].y, S.matF[k].z}}; };
    auto child_ok = [&](int ci) { return ci >= 0 && (uint32_t)ci < i; }; // children precede parents => acyclic
    switch (ty) {
      case MAT_LAMBERT: break;
      case MAT_METAL: prm = prm < 1 ? std::max(0.0, prm) : 1; break; // metal.ts:20
      case MAT_GLASS: break;
      case MAT_LIGHT: emit = col; break; // diffuseLight.ts:29-31
      case MAT_MIXED: {
        if (!child_ok(c0) || !child_ok(c1)) { err = "Material not found: " + std::to_string(!child_ok(c0) ? c0 : c1); return RT_ERR_MATERIAL_NOT_FOUND; }
        prm = std::max(0.0, std::min(1.0, prm)); // mixedMaterial.ts:29
        H3 e1{{S.matE[c0].x, S.matE[c0].y, S.matE[c0].z}}, e2{{S.matE[c1].x, S.matE[c1].y, S.matE[c1].z}};
        emit = vsum(vtimes(e1, prm), vtimes(e2, 1.0 - prm)); // mixedMaterial.ts:52-57
        alb = vsum(vtimes(f3(c0), prm), vtimes(f3(c1), 1.0 - prm));
        break;
      }
      case MAT_LAYERED: {
        if (!child_ok(c1)) { err = "Material not found: " + std::to_string(c1); return RT_ERR_MATERIAL_NOT_FOUND; }
        if (sd->mat_type[c1] != MAT_GLASS) { err = "Material is not a dielectric: " + std::to_string(c1); return RT_ERR_NOT_DIELECTRIC; }
        if (!child_ok(c0)) { err = "Material not found: " + std::to_string(c0); return RT_ERR_MATERIAL_NOT_FOUND; }
        prm = sd->mat_param[c1];                                        // outer ior
        emit = H3{{S.matE[c0].x, S.matE[c0].y, S.matE[c0].z}};          // layeredMaterial.ts:61-63
        alb = f3(c0);
        break;
      }
      default: err = "Unknown material type: " + std::to_string(ty); return RT_ERR_UNKNOWN_MATERIAL_TYPE;
    }
    bool has_e = emit[0] != 0 || emit[1] != 0 || emit[2] != 0;
    S.matA[i] = F4{col[0], col[1], col[2], (float)prm};
    S.matB[i] = I4{ty, c0, c1, has_e ? 1 : 0};
    S.matE[i] = F4{emit[0], emit[1], emit[2], has_e ? 1.f : 0.f};
    S.matF[i] = F4{alb[0], alb[1], alb[2], 0.f};
  }
  lap("materials");
  // ---- objects (createSceneObject, scenes.ts:109-139) ----
  const uint32_t n = sd->n_objects;
  std::vector<Prim> P(n);
  bool any_negative = false, any_unbounded = false;
  S.planar_any = 0;
  // Geometry that is not finite in FP32 (the reference's Float32Array storage) renders NaN in the reference and
  // has no meaningful box for any tree: refuse it here instead of building on it.
  auto finite3 = [](const H3& a) { return std::isfinite(a[0]) && std::isfinite(a[1]) && std::isfinite(a[2]); };
  auto not_finite = [&](uint32_t i) { err = "object " + std::to_string(i) + " has non-finite geometry"; return RT_ERR_INVALID_ARGUMENT; };
  for (uint32_t i = 0; i < n; ++i) {
    Prim& p = P[i];
    int mi = sd->obj_material[i];
    if (mi < 0 || (uint32_t)mi >= nm) { err = "Material not found: " + std::to_string(mi); return RT_ERR_MATERIAL_NOT_FOUND; }
    p.obj = (int)i;
    p.mat = mi;
    p.type = sd->obj_type[i];
    p.q = from_d(sd->obj_pos + 3 * (size_t)i);
    if (!finite3(p.q)) return not_finite(i);
    if (p.type == OBJ_SPHERE) {
      p.r = sd->obj_r ? sd->obj_r[i] : 0;
      if (!std::isfinite((float)p.r)) return not_finite(i);
      if (p.r < 0) any_negative = true;
      make_sphere(p);
    } else if (p.type == OBJ_PLANE || p.type == OBJ_QUAD) {
      if (!sd->obj_u || !sd->obj_v) { err = "plane/quad without u/v"; return RT_ERR_INVALID_ARGUMENT; }
      p.u = from_d(sd->obj_u + 3 * (size_t)i);
      p.v = from_d(sd->obj_v + 3 * (size_t)i);
      if (!finite3(p.u) || !finite3(p.v)) return not_finite(i);
      make_planar(p);
      S.planar_any = 1;
    } else {
      err = "Unknown object type: " + std::to_string(p.type);
      return RT_ERR_UNKNOWN_OBJECT_TYPE;
    }
    if (!p.bounded) any_unbounded = true;
  }
  S.n_objects = (int)n;
  // ---- lights (scenes.ts:74-79): light:true AND has a `pdf` method (Sphere, Quad) ----
  for (uint32_t i = 0; i < n; ++i) {
    if (!(sd->obj_light && sd->obj_light[i])) continue;
    const Prim& p = P[i];
    if (p.type != OBJ_SPHERE && p.type != OBJ_QUAD) continue;
    DevLight L;
    std::memset(&L, 0, sizeof(L));
    L.p0 = p.rec0; L.p1 = p.rec1; L.p2 = p.rec2; L.p3 = p.rec3;
    put3(L.q, p.q); put3(L.u, p.u); put3(L.v, p.v);
    L.area = (float)p.area;
    L.radius = (float)p.r;
    L.type = p.type;
    L.slot = (int)i; // object index; resolved to a slot below
    S.lights.push_back(L);
  }
  lap("objects");
  // ---- acceleration structure ----
  int kind = o->bvh;
  if (kind == RT_BVH_AUTO) {
    if (any_negative) kind = BVH_REFERENCE;      // inverted boxes are only meaningful in the reference topology
    // Measured with the 4-wide while-while tree walk.  Open scene (scripts/gpu_list_vs_sah.py, spheres over a
    // ground; LIST / SAH ms): 13 objects 2.8 / 2.9, 17: 3.35 / 3.40, 25: 4.3 / 3.6, 33: 5.4 / 4.1, 49: 7.5 / 5.0.
    // Room (the 55-object layered/mixed box: walls everywhere, every ray hits, and only the LIST kernel has the
    // axis-aligned quad test): LIST 370 / 416 ms vs SAH 418 / 591 ms (fixed spp with the sorted integrator /
    // adaptive).  Cornell (8 objects) is the LIST kernel's case.
    else {
      uint32_t n_planar = 0;
      for (uint32_t i = 0; i < n; ++i) n_planar += P[i].type != OBJ_SPHERE;
      const bool room = n_planar >= 5;
      kind = n <= (room ? 64u : 16u) ? BVH_LIST : BVH_SAH;
    }
  }
  if (kind != BVH_REFERENCE && kind != BVH_SAH && kind != BVH_LIST) { err = "invalid bvh kind"; return RT_ERR_INVALID_ARGUMENT; }
  if (kind == BVH_LIST && n > 128) { err = "RT_BVH_LIST supports at most 128 objects"; return RT_ERR_UNSUPPORTED; }
  S.bvh_kind = kind;
  S.n_unbounded = 0;
  std::vector<BNode> pool;
  // Visiting order of the reference's own tree: decides which primitive keeps a hit when two
  // distances are exactly equal (first visited wins, hittableList.ts:76-84 / bvh.ts:139-145).
  // Ties need coincident surfaces, so large procedural scenes skip the O(n log^2 n) build.
  std::vector<int> rank(n);
  std::iota(rank.begin(), rank.end(), 0);
  std::vector<BNode> ref_pool;
  int ref_root = -1;
  if (kind != BVH_SAH || n <= 4096) {
    ref_pool.reserve(n);
    std::vector<int> all(n);
    std::iota(all.begin(), all.end(), 0);
    RefBuilder rb{P, ref_pool};
    ref_root = rb.build(all, 0, n);
    int next = 0;
    std::function<void(int)> walk = [&](int bi) {
      const BNode& b = ref_pool[bi];
      if (b.leaf) { for (int pi : b.prims) rank[pi] = next++; return; }
      walk(b.left);
      walk(b.right);
    };
    walk(ref_root);
  }
  S.p0.reserve(n); S.p1.reserve(n); S.p2.reserve(n); S.p3.reserve(n); S.slot_info.reserve(n); S.exact.reserve(n);
  S.nodes.reserve(n);
  Flattener fl{P, kind == BVH_SAH ? pool : ref_pool, S, rank};
  if (kind == BVH_LIST) {
    // Slots in the reference's visiting order; only the box tests are dropped, which cannot
    // change a nearest hit when no box is inverted.
    // Grouped by primitive kind (spheres, axis-aligned quads per axis, general quads, planes) so the
    // kernel runs one tight converged loop per kind; within a kind in the reference's visiting order.
    // The order cannot change a result: a closer hit is accepted only when it is closer by more than the
    // FP32 error bound, and anything nearer to a tie is decided in FP64 with the reference's
    // first-visited-wins rule on the stored rank.
    std::vector<int> by_rank(n);
    for (uint32_t i = 0; i < n; ++i) by_rank[rank[i]] = (int)i;
    auto group_of = [&](int pi) {
      const Prim& p = P[pi];
      if (p.type == OBJ_SPHERE) return 0;
      if (p.aa) { int K; std::memcpy(&K, &p.aa2.y, sizeof(int)); return 1 + K; }
      return p.type == OBJ_QUAD ? 4 : 5;
    };
    for (int g = 0; g < 6; ++g) {
      S.list_n[g] = 0;
      for (int pi : by_rank)
        if (group_of(pi) == g) { fl.push_slot(pi); S.list_n[g]++; }
    }
    S.n_unbounded = (int)n; // every slot is "always tested"
    for (uint32_t i = 0; i < n; ++i) // constants of the sphere loop's cheap miss test (rt_device.cuh)
      if (P[i].type == OBJ_SPHERE) {
        for (int a = 0; a < 3; ++a) S.sph_cmax = std::max(S.sph_cmax, std::fabs(P[i].q[a]));
        S.sph_r2max = std::max(S.sph_r2max, (float)(P[i].r * P[i].r));
      }
  } else if (kind == BVH_REFERENCE) {
    // node 0 = super-root: the reference tests the root's own box first (bvh.ts:130)
    S.nodes.emplace_back();
    fl.fill_pair(0, ref_root, -1, 0);
  } else {
    // Always-tested prefix: unbounded primitives (infinite planes), plus the few bounded ones whose box is a
    // large part of the scene's (room walls, a ground sphere): in the tree they would sit in a leaf next to the
    // root that nearly every ray visits anyway, while their boxes blow up every box above them; out of the tree
    // they cost one converged test per ray (axis-aligned quads with the cheap test) and the tree over the rest
    // is tight.  At most 8, each >= 20 % of the scene box's surface area.  Measured: 480 spheres on a ground
    // sphere 45.0 -> 40.9 ms; the 100 k-sphere scene loses 9 % (k_render_trav tests the prefix in its divergent
    // bounce-start phase), so big scenes keep everything in the tree.
    std::vector<int> bounded;
    std::vector<char> in_prefix(n, 0);
    {
      Box all = empty_box();
      uint32_t nb = 0;
      for (uint32_t i = 0; i < n; ++i)
        if (P[i].bounded) { all = merge(all, P[i].sah_box); ++nb; }
      const double scene_area = SahBuilder::area(all);
      if (nb > 8 && nb <= 8192 && scene_area > 0) {
        std::vector<std::pair<double, int>> big;
        for (uint32_t i = 0; i < n; ++i)
          if (P[i].bounded) {
            const double a = SahBuilder::area(P[i].sah_box);
            if (a >= 0.2 * scene_area) big.push_back({-a, (int)i});
          }
        std::sort(big.begin(), big.end());
        for (size_t k = 0; k < big.size() && k < 8; ++k) in_prefix[big[k].second] = 1;
      }
    }
    for (uint32_t i = 0; i < n; ++i) {
      if (!P[i].bounded) fl.push_slot((int)i, true);
      else if (in_prefix[i]) fl.push_slot((int)i, true);
      else bounded.push_back((int)i);
    }
    S.n_unbounded = (int)S.p0.size();
    (void)any_unbounded;
    if (!bounded.empty()) {
      pool.reserve(bounded.size());
      int root = SahBuilder::build_all(P, bounded, pool);
      lap("sah build");
      fl.emit_wide(root, 0); // wide node 0 = the root
    }
  }
  lap("flatten");
  S.max_depth = fl.max_depth;
  // device stacks: 64 entries for the binary REFERENCE walk (one push per level), 128 for the 4-wide SAH walk
  // (up to three pushes per level)
  if (S.max_depth > (kind == BVH_SAH ? 42 : 60)) { err = "BVH too deep"; return RT_ERR_UNSUPPORTED; }
  // resolve light slots
  {
    std::vector<int> obj_to_slot(n, -1);
    for (size_t s = 0; s < S.slot_info.size(); ++s) obj_to_slot[S.slot_info[s].y & 0x3fffffff] = (int)s;
    for (auto& L : S.lights) L.slot = obj_to_slot[L.slot];
  }
  // ---- camera (camera.ts:107-166) ----
  const rt_camera_desc& c = sd->camera;
  DevCamera& cam = S.cam;
  std::memset(&cam, 0, sizeof(cam));
  S.image_width = o->width;
  S.image_height = (int)std::ceil((double)o->width / o->aspect);
  if (S.image_height <= 0 || (double)S.image_width * S.image_height > 2147483647.0) { err = "image too large"; return RT_ERR_INVALID_ARGUMENT; }
  H3 from = from_d(c.from), at = from_d(c.at), up = from_d(c.up);
  double focus = (c.focus != 0 && !std::isnan(c.focus)) ? c.focus : [&] { H3 d = vdiff(from, at); return std::hypot((double)d[0], (double)d[1], (double)d[2]); }();
  double theta = c.vfov * (kPiD / 180);
  double h = std::tan(theta / 2);
  double vh = 2 * h * focus;
  double ar = (double)S.image_width / S.image_height;
  double vw = vh * ar;
  H3 w = vnormalize(vdiff(from, at));
  H3 u = vnormalize(vcross(up, w));
  H3 v = vcross(w, u);
  H3 viewportU = vtimes(u, vw), viewportV = vtimes(v, -vh);
  H3 du = vover(viewportU, S.image_width), dv = vover(viewportV, S.image_height);
  H3 ul = vdiff(vdiff(vdiff(from, vtimes(w, focus)), vover(viewportU, 2)), vover(viewportV, 2));
  H3 p00 = vsum(ul, vtimes(vsum(du, dv), 0.5));
  H3 ddu = vtimes(u, c.aperture / 2), ddv = vtimes(v, c.aperture / 2);
  put3(cam.center, from); put3(cam.p00, p00); put3(cam.du, du); put3(cam.dv, dv); put3(cam.ddu, ddu); put3(cam.ddv, ddv);
  put3(cam.bg_top, from_d(c.background_top)); put3(cam.bg_bottom, from_d(c.background_bottom));
  put3(S.cam_u, u); put3(S.cam_v, v); put3(S.cam_w, w);
  S.focus_distance = focus;
  cam.width = S.image_width; cam.height = S.image_height;
  cam.samples = o->samples; cam.depth = o->depth; cam.rr_depth = o->roulette_depth; cam.a_batch = o->a_batch;
  cam.mode = o->mode; cam.a_tol = (float)o->a_tolerance;
  cam.roulette = o->roulette != 0;
  cam.adaptive = (o->a_tolerance > 0 && o->samples > 1) ? 1 : 0; // camera.ts:165
  cam.shadow_rays = o->light_sampling == RT_LIGHTS_SHADOW_RAYS ? 1 : 0;
  cam.jitter = o->samples > 1;                                    // camera.ts:184
  cam.defocus = c.aperture > 0;                                   // camera.ts:197
  return RT_OK;
}

} // namespace rt
