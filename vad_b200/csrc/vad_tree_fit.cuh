// vad_tree_fit.cuh -- device fit of a Gini decision tree (vadb200_tree_fit), level by level over presorted columns.
//
// Contract (include/vadb200.h): the tree sklearn 1.9's DecisionTreeClassifier(criterion="gini", splitter="best",
// max_features=None) builds, array for array and bit for bit, at every node where sklearn's choice does not depend on
// its random feature order.  Where two features reach the same float64 best proxy, this fit takes the lower feature
// index and counts the node in tied_nodes; tied_nodes == 0 => sklearn builds this same tree for every random_state.
//
// Layout.  Every column f of the 39 holds the active rows sorted by x[:, f] as two arrays: the float32 value and
// `rl` = row << 2 | label.  Every open node owns the same position range [s, e) in every column, so a node's class
// counts before a position are a column-wide prefix minus the node's base (the counts of the open nodes before it),
// which is the same in every column.  The element kernels below all take one CTA per (chunk of kTfChunk positions,
// column): a count pass packs four 16-bit bucket counts per chunk, tf_chunk_scan turns them into exclusive prefixes
// per column, and the consumer recomputes its in-chunk prefix with a block scan.
//
// The launchers only enqueue; vadb200.cu validates arguments, counts the launches and runs the level loop.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace vadb {

constexpr int kTfFeat = 39;
constexpr int kTfThreads = 256;
constexpr int kTfItems = 8;
constexpr int kTfChunk = kTfThreads * kTfItems;  // positions per CTA; bucket counts per chunk fit 16 bits
constexpr int kTfSlots = kTfChunk / 2 + 1;       // open nodes one chunk can touch: each holds >= 2 rows
constexpr int kTfScanItems = 8;                  // ints per node in tf_level_scan
constexpr long long kTfMaxRows = 1ll << 30;      // row << 2 | label fits 32 bits
constexpr int kTfMaxNodes = 1 << 26;             // vadb200_set_tree's limit

// An open node: searched at this level.  base = class counts of the open nodes before it (column-wide prefix).
struct TfOpen {
  int s, e, depth, id;
  int c[3], base[3];
  double imp;
};

// A node record in creation (breadth-first) order; the host renumbers to preorder.  Leaves: left = right = -1.
struct TfRec {
  int left, right, feature, n;
  int c[3], pad;
  double thr, imp;
};

// Per open node: the decision and the partition offsets of its rows.
struct TfDec {
  int f, pos, split, tie;
  int cl[3], open_l, open_r;
  int dst1, dst2;        // new position of a row = dst + its column-wide prefix among rows of the same side
  double imp_l, imp_r;
};

struct TfParams {
  int max_depth;         // <= 0: unbounded
  int min_split;         // max(min_samples_split, 2 min_samples_leaf)
  int min_leaf;
  double min_decrease;
  double n_total;        // weighted_n_samples
};

// Per-fit counters on the device: [0] bad-feature flag, [1] bad-label flag, [2..4] class histogram, [5] tied nodes,
// [6..13] the last level's scan totals (tf_level_scan).
constexpr int kTfStats = 16;

enum TfCountMode { kTfByLabel = 0, kTfBySide = 1, kTfByDigit = 2 };

void tf_validate(const float* x, const uint8_t* y, long long n, int stride, float* val, uint32_t* rl, int* stats,
                 cudaStream_t st);
void tf_count(int mode, int shift, const float* val, const uint32_t* rl, const uint8_t* side, int n_act, int stride,
              int n_chunks, unsigned long long* chunk_cnt, cudaStream_t st);
void tf_chunk_scan(const unsigned long long* chunk_cnt, int n_chunks, int4* chunk_pre, cudaStream_t st);
void tf_radix_scatter(int shift, const float* val, const uint32_t* rl, int n, int stride, int n_chunks,
                      const int4* chunk_pre, float* val_out, uint32_t* rl_out, cudaStream_t st);
void tf_node_map(const TfOpen* open, int n_open, int n_act, int* pos_node, cudaStream_t st);
void tf_search(int phase, const float* val, const uint32_t* rl, int n_act, int stride, int n_chunks,
               const int4* chunk_pre, const int* pos_node, const TfOpen* open, int min_leaf,
               unsigned long long* best_key, int* best_pos, cudaStream_t st);
void tf_decide(const uint32_t* rl, int stride, const int4* chunk_pre, int n_chunks,
               const TfOpen* open, int n_open, const unsigned long long* best_key, const int* best_pos, TfParams p,
               TfDec* dec, int* scan, cudaStream_t st);
void tf_level_scan(int* scan, int n_open, int* totals, cudaStream_t st);
void tf_emit(const float* val, int stride, const TfOpen* open, int n_open, TfDec* dec, const int* scan, int next_id,
             int node_cap, TfRec* rec, TfOpen* open_next, int* stats, cudaStream_t st);
void tf_flag(const uint32_t* rl, int n_act, int stride, const int* pos_node, const TfDec* dec, uint8_t* side,
             cudaStream_t st);
void tf_partition(const float* val, const uint32_t* rl, int n_act, int stride, int n_chunks, const int4* chunk_pre,
                  const int* pos_node, const TfDec* dec, const uint8_t* side, float* val_out, uint32_t* rl_out,
                  cudaStream_t st);

}  // namespace vadb
