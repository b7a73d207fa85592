// vad_tree.cuh -- the decision-tree classifier on the device (layout and semantics: vad_tree.h).
#pragma once

#include "vad_tree.h"

namespace vadb {

// The tree a kernel runs: its nodes and leaf entries (one vadb200_handle allocation) and the handle's threshold
// (<= 0: argmax).  A launch parameter, like the FFN weights.
struct TreeArg {
  const TreeNode* nodes;
  const TreeLeaf* leaves;
  int depth;
  float thresh;
};

// The leaf of the row whose feature f is x(f): `depth` steps, leaves step to themselves.
template <class X>
__device__ __forceinline__ const TreeLeaf& tree_walk(const TreeArg& tr, X&& x) {
  uint32_t i = 0;
  for (int d = 0; d < tr.depth; ++d) {
    const uint2 nd = __ldg(reinterpret_cast<const uint2*>(tr.nodes) + i);
    i = (nd.y >> 6) + (x(nd.y & 63u) > __uint_as_float(nd.x) ? 1u : 0u);
  }
  return tr.leaves[i];
}

// The leaf's decision (argmax, or p1 >= th in float64 for th > 0) and its probabilities.
__device__ __forceinline__ uint8_t tree_decide(const TreeLeaf& lf, float th, float (&p)[3]) {
  p[0] = lf.p[0];
  p[1] = lf.p[1];
  p[2] = lf.p[2];
  return th > 0.0f ? (lf.p1 >= static_cast<double>(th) ? 1 : 0) : static_cast<uint8_t>(lf.speech);
}

}  // namespace vadb
