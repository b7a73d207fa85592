// vad_tree.h -- a fitted sklearn DecisionTreeClassifier in the device layout (host code, no CUDA: the library and
// the CPU emulation tests/emul/emul_tree.cpp compile the same conversion).
//
// Input: exactly the arrays clf.tree_ and clf.classes_ expose -- children_left / children_right (-1 at a leaf),
// feature, threshold (float64), value [n_nodes][n_classes] (float64) and classes_.  sklearn routes x to the left
// child when float64(float32 x) <= threshold; for float32 x that is x <= t32 with t32 the largest float32 <= threshold
// (round toward -inf; >= FLT_MAX -> +inf), and the kernels test x > t32 to take the right child.
// Layout: nodes renumbered breadth first, so the children of node i are left(i) and left(i) + 1; a leaf is a node
// whose left child is itself with threshold +inf, so a walk of `depth` steps ends on the leaf whatever the row (a
// NaN never takes the right child).  Each node has a leaf entry (used at leaves only): the argmax decision, the float32
// probabilities by class id and predict_proba's class-1 column in float64 for the threshold rule.
#pragma once

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <string>
#include <utility>
#include <vector>

namespace vadb {

constexpr int kTreeFeatures = 39;                 // vadb200_vad_windows' feature rows
constexpr int kTreeLeftBits = 26;
constexpr long long kTreeMaxNodes = 1ll << kTreeLeftBits;  // the left field indexes every node

struct TreeNode {
  float t;       // t32; +inf at a leaf
  uint32_t fl;   // feature | left << 6
};
struct TreeLeaf {
  double p1;     // predict_proba's class-1 column (0 without class 1): speech <=> p1 >= (double)threshold
  float p[3];    // float32(predict_proba) in the columns of class ids 0, 1, 2 (0 for a class the tree lacks)
  uint32_t speech;  // classes_[argmax(value)] == 1, ties to the first maximum
};
static_assert(sizeof(TreeNode) == 8 && sizeof(TreeLeaf) == 24, "tree layout");

struct TreeLayout {
  std::vector<TreeNode> nodes;
  std::vector<TreeLeaf> leaves;  // one per node
  int depth = 0;                 // internal nodes on the longest root-to-leaf path
};

// The largest float32 <= t (round toward -inf); t >= FLT_MAX gives +inf.
inline float tree_threshold_f32(double t) {
  if (t >= static_cast<double>(FLT_MAX)) return INFINITY;
  float f = static_cast<float>(t);
  if (static_cast<double>(f) > t) f = std::nextafter(f, -INFINITY);
  return f;
}

// Checks the arrays and builds the layout; false (with *why) leaves *out untouched.
inline bool tree_convert(long long n, const int64_t* left, const int64_t* right, const int64_t* feature,
                         const double* threshold, const double* value, const int64_t* classes, int n_classes,
                         TreeLayout* out, std::string* why) {
  auto bad = [&](const std::string& m) {
    *why = m;
    return false;
  };
  if (n < 1) return bad("a tree needs at least one node");
  if (n > kTreeMaxNodes) return bad("more nodes than the device layout can index (2^26)");
  if (!left || !right || !feature || !threshold || !value || !classes) return bad("null argument");
  if (n_classes < 1 || n_classes > 3) return bad("n_classes must lie in [1, 3]");
  int cls1 = -1;
  for (int k = 0; k < n_classes; ++k) {
    if (classes[k] < 0 || classes[k] > 2) return bad("class ids must lie in {0, 1, 2}");
    if (k > 0 && classes[k] <= classes[k - 1]) return bad("class ids must be distinct and ascending");
    if (classes[k] == 1) cls1 = k;
  }
  std::vector<unsigned char> parents(static_cast<size_t>(n), 0);
  for (long long i = 0; i < n; ++i) {
    const int64_t l = left[i], r = right[i];
    if ((l == -1) != (r == -1)) return bad("node " + std::to_string(i) + " has only one child");
    for (long long k = 0; k < n_classes; ++k) {
      const double v = value[i * n_classes + k];
      if (!(v >= 0.0) || !std::isfinite(v)) return bad("node values must be finite and >= 0");
    }
    if (l == -1) continue;
    if (l <= i || r <= i || l >= n || r >= n || l == r)
      return bad("node " + std::to_string(i) + ": child index out of range or not greater than its parent's");
    if (parents[l]++ || parents[r]++) return bad("a node with two parents");
    if (feature[i] < 0 || feature[i] >= kTreeFeatures) return bad("feature index outside [0, 39)");
    if (std::isnan(threshold[i])) return bad("NaN threshold");
  }
  for (long long i = 1; i < n; ++i)
    if (!parents[i]) return bad("node " + std::to_string(i) + " is not reachable from the root");
  // breadth-first renumbering: children of each internal node get consecutive ids
  std::vector<long long> order(1, 0), id(static_cast<size_t>(n), -1), lvl(static_cast<size_t>(n), 0);
  order.reserve(static_cast<size_t>(n));
  id[0] = 0;
  int depth = 0;
  for (size_t q = 0; q < order.size(); ++q) {
    const long long o = order[q];
    if (left[o] == -1) continue;
    for (const int64_t c : {left[o], right[o]}) {
      id[c] = static_cast<long long>(order.size());
      lvl[c] = lvl[o] + 1;
      depth = std::max<int>(depth, static_cast<int>(lvl[c]));
      order.push_back(c);
    }
  }
  TreeLayout L;
  L.nodes.resize(static_cast<size_t>(n));
  L.leaves.assign(static_cast<size_t>(n), TreeLeaf{0.0, {0.0f, 0.0f, 0.0f}, 0u});
  L.depth = depth;
  for (long long o = 0; o < n; ++o) {
    const long long i = id[o];
    TreeNode& nd = L.nodes[i];
    if (left[o] != -1) {
      nd.t = tree_threshold_f32(threshold[o]);
      nd.fl = static_cast<uint32_t>(feature[o]) | static_cast<uint32_t>(id[left[o]]) << 6;
      continue;
    }
    nd.t = INFINITY;
    nd.fl = static_cast<uint32_t>(i) << 6;
    TreeLeaf& lf = L.leaves[i];
    const double* v = value + o * n_classes;
    int best = 0;
    for (int k = 1; k < n_classes; ++k)
      if (v[k] > v[best]) best = k;  // np.argmax: the first maximum
    lf.speech = classes[best] == 1 ? 1u : 0u;
    lf.p1 = cls1 >= 0 ? v[cls1] : 0.0;
    for (int k = 0; k < n_classes; ++k) lf.p[classes[k]] = static_cast<float>(v[k]);
  }
  *out = std::move(L);
  return true;
}

}  // namespace vadb
