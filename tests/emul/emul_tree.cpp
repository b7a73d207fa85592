// Host emulation of the tree path: the library's own conversion (vad_tree.h) and a walk of the converted layout with
// the kernels' arithmetic (vad_tree.cuh tree_walk / tree_decide), for the CPU tests.
#include <cstring>

#include "../../vad_b200/csrc/vad_tree.h"

using namespace vadb;

extern "C" {

// Converts; returns 0 and fills nodes [n] (t32, feature | left << 6), leaves [n][6] (p1, p0, p1f, p2, speech as
// doubles) and *depth, or -1 with the error message in err.
int emul_tree_convert(long long n, const int64_t* l, const int64_t* r, const int64_t* f, const double* t,
                      const double* v, const int64_t* c, int nc, float* node_t, uint32_t* node_fl, double* leaves,
                      int* depth, char* err, int err_len) {
  TreeLayout L;
  std::string why;
  if (!tree_convert(n, l, r, f, t, v, c, nc, &L, &why)) {
    std::strncpy(err, why.c_str(), err_len - 1);
    err[err_len - 1] = 0;
    return -1;
  }
  for (long long i = 0; i < n; ++i) {
    node_t[i] = L.nodes[i].t;
    node_fl[i] = L.nodes[i].fl;
    const TreeLeaf& lf = L.leaves[i];
    double* o = leaves + 5 * i;
    o[0] = lf.p1; o[1] = lf.p[0]; o[2] = lf.p[1]; o[3] = lf.p[2]; o[4] = lf.speech;
  }
  *depth = L.depth;
  return 0;
}

// Converts and walks rows x [m][39]: labels (decision at threshold th) and probabilities [m][3]; -1 when malformed.
int emul_tree_predict(long long n, const int64_t* l, const int64_t* r, const int64_t* f, const double* t,
                      const double* v, const int64_t* c, int nc, const float* x, long long m, float th,
                      uint8_t* labels, float* proba) {
  TreeLayout L;
  std::string why;
  if (!tree_convert(n, l, r, f, t, v, c, nc, &L, &why)) return -1;
  for (long long k = 0; k < m; ++k) {
    const float* row = x + k * kTreeFeatures;
    uint32_t i = 0;
    for (int d = 0; d < L.depth; ++d) {
      const TreeNode nd = L.nodes[i];
      i = (nd.fl >> 6) + (row[nd.fl & 63u] > nd.t ? 1u : 0u);
    }
    const TreeLeaf& lf = L.leaves[i];
    labels[k] = th > 0.0f ? (lf.p1 >= static_cast<double>(th) ? 1 : 0) : static_cast<uint8_t>(lf.speech);
    for (int j = 0; j < 3; ++j) proba[3 * k + j] = lf.p[j];
  }
  return 0;
}

}  // extern "C"
