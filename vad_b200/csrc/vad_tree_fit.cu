// vad_tree_fit.cu -- the kernels of vadb200_tree_fit (vad_tree_fit.cuh), in a translation unit of their own so that
// the kernels of vadb200.cu compile exactly as they do without them.
//
// Arithmetic order.  sklearn's Gini proxy, child impurities and improvement are restated with __dmul_rn / __ddiv_rn /
// __dadd_rn / __dsub_rn, so no product is fused into a following sum: sklearn's wheels never fuse them, and a fused
// DFMA rounds once where sklearn rounds twice.  Class counts are integers, so their sums of squares are exact.
#include "vad_tree_fit.cuh"

#include <algorithm>
#include <cfloat>

namespace vadb {

static constexpr float kFeatureThreshold = 1e-7f;  // sklearn's FEATURE_THRESHOLD (float32)

__device__ __forceinline__ uint32_t tf_key(float v) {  // order-preserving uint32 image of a float32
  const uint32_t b = __float_as_uint(v);
  return b ^ ((b & 0x80000000u) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ unsigned long long tf_dkey(double d) {  // order-preserving uint64 image; never 0
  const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(d));
  return b ^ ((b >> 63) ? ~0ull : 0x8000000000000000ull);
}
__device__ __forceinline__ int tf_field(unsigned long long v, int b) { return static_cast<int>((v >> (16 * b)) & 0xffff); }

// sklearn Gini::children_impurity for one side: 1.0 - sq_count / (w * w), sq_count summed class by class from 0.0.
__device__ __forceinline__ double tf_gini(int c0, int c1, int c2, int n) {
  const double a = c0, b = c1, c = c2, w = n;
  const double sq = __dadd_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)), __dmul_rn(c, c));
  return __dsub_rn(1.0, __ddiv_rn(sq, __dmul_rn(w, w)));
}

// Exclusive block scan of packed 16-bit bucket counts over kTfThreads threads.  sh: kTfThreads / 32 entries.
__device__ unsigned long long tf_block_excl(unsigned long long v, unsigned long long* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned long long inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += o;
  }
  if (lane == 31) sh[w] = inc;
  __syncthreads();
  unsigned long long off = 0;
  for (int i = 0; i < w; ++i) off += sh[i];
  return off + inc - v;
}

// Exclusive block scan of one int over blockDim.x (a multiple of 32, <= 1024) threads.  sh: 32 entries.
__device__ int tf_block_excl_int(int v, int* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int o = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += o;
  }
  if (lane == 31) sh[w] = inc;
  __syncthreads();
  if (w == 0) {
    const int t = lane < static_cast<int>(blockDim.x >> 5) ? sh[lane] : 0;
    int x = t;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, x, d);
      if (lane >= d) x += o;
    }
    sh[lane] = x - t;
  }
  __syncthreads();
  const int r = sh[w] + inc - v;
  __syncthreads();
  return r;
}

template <int MODE>
__device__ __forceinline__ int tf_bucket(int shift, float v, uint32_t r, const uint8_t* side) {
  if (MODE == kTfByLabel) return static_cast<int>(r & 3u);
  if (MODE == kTfBySide) return side[r >> 2];
  return static_cast<int>((tf_key(v) >> shift) & 3u);
}

// ---- validation, transpose, class histogram ----------------------------------------------------------------------
__global__ void __launch_bounds__(256) tf_validate_kernel(const float* __restrict__ x, const uint8_t* __restrict__ y,
                                                          long long n, int stride, float* val, uint32_t* rl,
                                                          int* stats) {
  __shared__ int hist[3];
  if (threadIdx.x < 3) hist[threadIdx.x] = 0;
  __syncthreads();
  const long long total = n * kTfFeat;
  for (long long j = blockIdx.x * 256ll + threadIdx.x; j < total; j += static_cast<long long>(gridDim.x) * 256) {
    const long long i = j / kTfFeat;
    const int f = static_cast<int>(j - i * kTfFeat);
    const float v = x[j];
    if (!isfinite(v)) atomicOr(&stats[0], 1);
    const int lab = y[i];
    if (f == 0) {
      if (lab > 2) atomicOr(&stats[1], 1);
      else atomicAdd(&hist[lab], 1);
    }
    val[static_cast<long long>(f) * stride + i] = v;
    rl[static_cast<long long>(f) * stride + i] = static_cast<uint32_t>(i) << 2 | static_cast<uint32_t>(lab & 3);
  }
  __syncthreads();
  if (threadIdx.x < 3 && hist[threadIdx.x]) atomicAdd(&stats[2 + threadIdx.x], hist[threadIdx.x]);
}

// ---- bucket counts per (chunk, column) -----------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(kTfThreads) tf_count_kernel(int shift, const float* __restrict__ val,
                                                              const uint32_t* __restrict__ rl,
                                                              const uint8_t* __restrict__ side, int n_act, int stride,
                                                              int n_chunks, unsigned long long* chunk_cnt) {
  __shared__ unsigned long long sh[kTfThreads / 32];
  const int f = blockIdx.y, c = blockIdx.x;
  const float* v = val + static_cast<long long>(f) * stride;
  const uint32_t* r = rl + static_cast<long long>(f) * stride;
  const int p0 = c * kTfChunk + threadIdx.x * kTfItems;
  unsigned long long cnt = 0;
#pragma unroll
  for (int i = 0; i < kTfItems; ++i) {
    const int p = p0 + i;
    if (p < n_act) cnt += 1ull << (16 * tf_bucket<MODE>(shift, MODE == kTfByDigit ? v[p] : 0.0f, r[p], side));
  }
  const unsigned long long ex = tf_block_excl(cnt, sh);
  if (threadIdx.x == kTfThreads - 1) chunk_cnt[static_cast<long long>(f) * n_chunks + c] = ex + cnt;
}

// Exclusive prefixes of the chunk counts, one CTA per column: chunk_pre[f][c] (int4, one int per bucket), and
// chunk_pre[f][n_chunks] = the column's totals.
__global__ void __launch_bounds__(1024) tf_chunk_scan_kernel(const unsigned long long* __restrict__ chunk_cnt,
                                                             int n_chunks, int4* chunk_pre) {
  __shared__ int sh[32];
  const int f = blockIdx.x;
  const unsigned long long* in = chunk_cnt + static_cast<long long>(f) * n_chunks;
  int4* out = chunk_pre + static_cast<long long>(f) * (n_chunks + 1);
  const int per = (n_chunks + blockDim.x - 1) / blockDim.x;
  const int lo = min(n_chunks, static_cast<int>(threadIdx.x) * per), hi = min(n_chunks, lo + per);
  int s[4] = {0, 0, 0, 0};
  for (int i = lo; i < hi; ++i)
    for (int b = 0; b < 4; ++b) s[b] += tf_field(in[i], b);
  int run[4];
  for (int b = 0; b < 4; ++b) run[b] = tf_block_excl_int(s[b], sh);
  for (int i = lo; i < hi; ++i) {
    out[i] = make_int4(run[0], run[1], run[2], run[3]);
    for (int b = 0; b < 4; ++b) run[b] += tf_field(in[i], b);
  }
  if (threadIdx.x == blockDim.x - 1) out[n_chunks] = make_int4(run[0], run[1], run[2], run[3]);
}

// ---- presort: one stable 2-bit LSD radix pass over every column -------------------------------------------------
__global__ void __launch_bounds__(kTfThreads) tf_radix_kernel(int shift, const float* __restrict__ val,
                                                              const uint32_t* __restrict__ rl, int n, int stride,
                                                              int n_chunks, const int4* __restrict__ chunk_pre,
                                                              float* val_out, uint32_t* rl_out) {
  __shared__ unsigned long long sh[kTfThreads / 32];
  const int f = blockIdx.y, c = blockIdx.x;
  const long long col = static_cast<long long>(f) * stride;
  const int p0 = c * kTfChunk + threadIdx.x * kTfItems;
  float v[kTfItems];
  uint32_t r[kTfItems];
  unsigned long long cnt = 0;
#pragma unroll
  for (int i = 0; i < kTfItems; ++i) {
    const int p = p0 + i;
    if (p < n) {
      v[i] = val[col + p];
      r[i] = rl[col + p];
      cnt += 1ull << (16 * tf_bucket<kTfByDigit>(shift, v[i], 0, nullptr));
    }
  }
  unsigned long long run = tf_block_excl(cnt, sh);
  const int4* pre = chunk_pre + static_cast<long long>(f) * (n_chunks + 1);
  const int4 tot = pre[n_chunks], cp = pre[c];
  const int base[4] = {cp.x, tot.x + cp.y, tot.x + tot.y + cp.z, tot.x + tot.y + tot.z + cp.w};
#pragma unroll
  for (int i = 0; i < kTfItems; ++i) {
    if (p0 + i < n) {
      const int b = tf_bucket<kTfByDigit>(shift, v[i], 0, nullptr);
      const int q = base[b] + tf_field(run, b);
      run += 1ull << (16 * b);
      val_out[col + q] = v[i];
      rl_out[col + q] = r[i];
    }
  }
}

// ---- per level -------------------------------------------------------------------------------------------------------
__global__ void tf_node_map_kernel(const TfOpen* __restrict__ open, int n_open, int n_act, int* pos_node) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_act) return;
  int lo = 0, hi = n_open - 1;  // the last node with s <= p
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (open[mid].s <= p) lo = mid;
    else hi = mid - 1;
  }
  pos_node[p] = lo;
}

// PHASE 0: best_key[k][f] = max over candidates of the proxy's key.  PHASE 1: best_pos[k][f] = the earliest candidate
// position reaching it (sklearn's strict '>' within a feature).  A candidate is a position p of node k's range with
// x[p] > x[p - 1] + FEATURE_THRESHOLD in float32 and min_leaf rows on either side.
template <int PHASE>
__global__ void __launch_bounds__(kTfThreads) tf_search_kernel(const float* __restrict__ val,
                                                               const uint32_t* __restrict__ rl, int n_act, int stride,
                                                               int n_chunks, const int4* __restrict__ chunk_pre,
                                                               const int* __restrict__ pos_node,
                                                               const TfOpen* __restrict__ open, int min_leaf,
                                                               unsigned long long* best_key, int* best_pos) {
  constexpr unsigned long long kInit = PHASE ? ~0ull : 0ull;
  __shared__ unsigned long long slot[kTfSlots];
  __shared__ unsigned long long sh[kTfThreads / 32];
  const int f = blockIdx.y, c = blockIdx.x;
  const long long col = static_cast<long long>(f) * stride;
  const int lo = c * kTfChunk, hi = min(lo + kTfChunk, n_act);
  const int k0 = pos_node[lo], n_slots = pos_node[hi - 1] - k0 + 1;
  for (int i = threadIdx.x; i < n_slots; i += kTfThreads) slot[i] = kInit;
  const int p0 = lo + threadIdx.x * kTfItems;
  float v[kTfItems];
  uint32_t r[kTfItems];
  unsigned long long cnt = 0;
#pragma unroll
  for (int i = 0; i < kTfItems; ++i) {
    const int p = p0 + i;
    if (p < n_act) {
      v[i] = val[col + p];
      r[i] = rl[col + p];
      cnt += 1ull << (16 * (r[i] & 3u));
    }
  }
  unsigned long long run = tf_block_excl(cnt, sh);  // also orders the slot initialisation before its use
  const int4 cp = chunk_pre[static_cast<long long>(f) * (n_chunks + 1) + c];
  int run_k = -1;
  unsigned long long run_v = kInit;
  for (int i = 0; i < kTfItems; ++i) {
    const int p = p0 + i;
    if (p >= n_act) break;
    const int k = pos_node[p];
    const TfOpen& o = open[k];
    unsigned long long mine = kInit;
    const int nl = p - o.s, nr = o.e - p;
    if (nl >= min_leaf && nr >= min_leaf) {
      const float prev = i > 0 ? v[i - 1] : val[col + p - 1];
      if (v[i] > __fadd_rn(prev, kFeatureThreshold)) {
        const int l0 = cp.x + tf_field(run, 0) - o.base[0];
        const int l1 = cp.y + tf_field(run, 1) - o.base[1];
        const int l2 = cp.z + tf_field(run, 2) - o.base[2];
        const double gl = tf_gini(l0, l1, l2, nl), gr = tf_gini(o.c[0] - l0, o.c[1] - l1, o.c[2] - l2, nr);
        // sklearn: - weighted_n_right * impurity_right - weighted_n_left * impurity_left
        const double proxy = __dsub_rn(-__dmul_rn(static_cast<double>(nr), gr), __dmul_rn(static_cast<double>(nl), gl));
        const unsigned long long key = tf_dkey(proxy);
        if (PHASE == 0) mine = key;
        else if (key == best_key[static_cast<long long>(k) * kTfFeat + f]) mine = static_cast<unsigned long long>(p);
      }
    }
    run += 1ull << (16 * (r[i] & 3u));
    if (k != run_k) {
      if (run_k >= 0 && run_v != kInit) {
        if (PHASE == 0) atomicMax(&slot[run_k - k0], run_v);
        else atomicMin(&slot[run_k - k0], run_v);
      }
      run_k = k;
      run_v = kInit;
    }
    run_v = PHASE == 0 ? max(run_v, mine) : min(run_v, mine);
  }
  // Lanes are in position order, so equal final nodes are adjacent: a segmented reduction leaves each run's result in
  // its first lane, and one shared atomic per node and warp remains.
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int ok = __shfl_down_sync(0xffffffffu, run_k, d);
    const unsigned long long ov = __shfl_down_sync(0xffffffffu, run_v, d);
    if (lane + d < 32 && ok == run_k) run_v = PHASE == 0 ? max(run_v, ov) : min(run_v, ov);
  }
  const int prev_k = __shfl_up_sync(0xffffffffu, run_k, 1);
  if (run_k >= 0 && (lane == 0 || prev_k != run_k) && run_v != kInit) {
    if (PHASE == 0) atomicMax(&slot[run_k - k0], run_v);
    else atomicMin(&slot[run_k - k0], run_v);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n_slots; i += kTfThreads) {
    const unsigned long long s = slot[i];
    if (s == kInit) continue;
    const long long at = static_cast<long long>(k0 + i) * kTfFeat + f;
    if (PHASE == 0) atomicMax(&best_key[at], s);
    else atomicMin(&best_pos[at], static_cast<int>(s));
  }
}

// One warp per open node: the best feature (lowest index among equal keys), the tie flag, the left class counts at the
// chosen position, sklearn's stopping rules, and the node's entries of tf_level_scan.
__global__ void __launch_bounds__(256) tf_decide_kernel(const uint32_t* __restrict__ rl, int stride,
                                                        const int4* __restrict__ chunk_pre, int n_chunks,
                                                        const TfOpen* __restrict__ open, int n_open,
                                                        const unsigned long long* __restrict__ best_key,
                                                        const int* __restrict__ best_pos, TfParams prm, TfDec* dec,
                                                        int* scan) {
  const int lane = threadIdx.x & 31;
  const int k = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (k >= n_open) return;
  const TfOpen o = open[k];
  const unsigned long long* bk = best_key + static_cast<long long>(k) * kTfFeat;
  const unsigned long long a = bk[lane], b = lane + 32 < kTfFeat ? bk[lane + 32] : 0ull;
  unsigned long long m = max(a, b);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, d));
  const unsigned ba = __ballot_sync(0xffffffffu, m != 0 && a == m), bb = __ballot_sync(0xffffffffu, m != 0 && b == m);
  const int f = ba ? __ffs(ba) - 1 : bb ? __ffs(bb) + 31 : -1;
  int l[3] = {0, 0, 0};
  int pos = -1;
  if (f >= 0) {
    pos = best_pos[static_cast<long long>(k) * kTfFeat + f];
    const int c = pos / kTfChunk, cs = c * kTfChunk;
    const int from = max(cs, o.s);
    const uint32_t* r = rl + static_cast<long long>(f) * stride;
    for (int q = from + lane; q < pos; q += 32) ++l[r[q] & 3u];
#pragma unroll
    for (int j = 0; j < 3; ++j)
      for (int d = 16; d > 0; d >>= 1) l[j] += __shfl_xor_sync(0xffffffffu, l[j], d);
    if (cs > o.s) {
      const int4 cp = chunk_pre[static_cast<long long>(f) * (n_chunks + 1) + c];
      l[0] += cp.x - o.base[0];
      l[1] += cp.y - o.base[1];
      l[2] += cp.z - o.base[2];
    }
  }
  if (lane) return;
  TfDec dd;
  dd.f = f;
  dd.pos = pos;
  dd.tie = f >= 0 && __popc(ba) + __popc(bb) > 1;
  dd.split = 0;
  dd.open_l = dd.open_r = 0;
  dd.dst1 = dd.dst2 = 0;
  dd.imp_l = dd.imp_r = 0.0;
  const int nl = pos - o.s, nr = o.e - pos, n = o.e - o.s;
  const int r0 = o.c[0] - l[0], r1 = o.c[1] - l[1], r2 = o.c[2] - l[2];
  for (int j = 0; j < 3; ++j) dd.cl[j] = l[j];
  if (f >= 0) {
    dd.imp_l = tf_gini(l[0], l[1], l[2], nl);
    dd.imp_r = tf_gini(r0, r1, r2, nr);
    const double wn = n, wl = nl, wr = nr;
    // sklearn ClassificationCriterion.impurity_improvement, operation for operation
    const double impr = __dmul_rn(__ddiv_rn(wn, prm.n_total),
                                  __dsub_rn(__dsub_rn(o.imp, __dmul_rn(__ddiv_rn(wr, wn), dd.imp_r)),
                                            __dmul_rn(__ddiv_rn(wl, wn), dd.imp_l)));
    dd.split = !(__dadd_rn(impr, DBL_EPSILON) < prm.min_decrease);
  }
  if (dd.split) {
    const bool deep = prm.max_depth > 0 && o.depth + 1 >= prm.max_depth;
    dd.open_l = !(deep || nl < prm.min_split || nl < 2 * prm.min_leaf || dd.imp_l <= DBL_EPSILON);
    dd.open_r = !(deep || nr < prm.min_split || nr < 2 * prm.min_leaf || dd.imp_r <= DBL_EPSILON);
  }
  dec[k] = dd;
  int* s = scan + static_cast<long long>(k) * kTfScanItems;
  s[0] = dd.split;
  s[1] = dd.open_l + dd.open_r;
  s[2] = dd.open_l ? nl : 0;
  s[3] = dd.open_r ? nr : 0;
  s[4] = (dd.open_l ? l[0] : 0) + (dd.open_r ? r0 : 0);
  s[5] = (dd.open_l ? l[1] : 0) + (dd.open_r ? r1 : 0);
  s[6] = (dd.open_l ? l[2] : 0) + (dd.open_r ? r2 : 0);
  s[7] = 0;
}

// Exclusive prefixes of the per-node entries, in place; totals[0..7] = the sums.  One CTA.
__global__ void __launch_bounds__(1024) tf_level_scan_kernel(int* scan, int n, int* totals) {
  __shared__ int sh[32];
  const int per = (n + blockDim.x - 1) / blockDim.x;
  const int lo = min(n, static_cast<int>(threadIdx.x) * per), hi = min(n, lo + per);
  int s[kTfScanItems] = {};
  for (int k = lo; k < hi; ++k)
    for (int j = 0; j < kTfScanItems; ++j) s[j] += scan[k * kTfScanItems + j];
  int run[kTfScanItems];
  for (int j = 0; j < kTfScanItems; ++j) run[j] = tf_block_excl_int(s[j], sh);
  for (int k = lo; k < hi; ++k)
    for (int j = 0; j < kTfScanItems; ++j) {
      const int t = scan[k * kTfScanItems + j];
      scan[k * kTfScanItems + j] = run[j];
      run[j] += t;
    }
  if (threadIdx.x == blockDim.x - 1)
    for (int j = 0; j < kTfScanItems; ++j) totals[j] = run[j];
}

// One thread per open node: the node's split record, its children's records (leaves until they are split), the next
// level's open nodes, and the partition offsets.  Children are numbered next_id + 2 * (splits before this node).
__global__ void tf_emit_kernel(const float* __restrict__ val, int stride, const TfOpen* __restrict__ open, int n_open,
                               TfDec* dec, const int* __restrict__ scan, int next_id, int node_cap, TfRec* rec,
                               TfOpen* open_next, int* stats) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_open) return;
  TfDec d = dec[k];
  if (d.tie) atomicAdd(&stats[5], 1);
  if (!d.split) return;
  const TfOpen o = open[k];
  const int* sc = scan + static_cast<long long>(k) * kTfScanItems;
  const int id_l = next_id + 2 * sc[0], id_r = id_l + 1;
  const int nl = d.pos - o.s, nr = o.e - d.pos;
  const int cr[3] = {o.c[0] - d.cl[0], o.c[1] - d.cl[1], o.c[2] - d.cl[2]};
  if (id_r < node_cap) {
    const float* v = val + static_cast<long long>(d.f) * stride;
    TfRec& me = rec[o.id];
    me.left = id_l;
    me.right = id_r;
    me.feature = d.f;
    // sklearn: feature_values[p_prev] / 2.0 + feature_values[p] / 2.0
    me.thr = __dadd_rn(__ddiv_rn(static_cast<double>(v[d.pos - 1]), 2.0), __ddiv_rn(static_cast<double>(v[d.pos]), 2.0));
    TfRec cl, cr_rec;
    cl.left = cl.right = cr_rec.left = cr_rec.right = -1;
    cl.feature = cr_rec.feature = -2;
    cl.thr = cr_rec.thr = -2.0;
    cl.pad = cr_rec.pad = 0;
    cl.n = nl;
    cr_rec.n = nr;
    for (int j = 0; j < 3; ++j) {
      cl.c[j] = d.cl[j];
      cr_rec.c[j] = cr[j];
    }
    cl.imp = d.imp_l;
    cr_rec.imp = d.imp_r;
    rec[id_l] = cl;
    rec[id_r] = cr_rec;
  }
  const int rows = sc[2] + sc[3];
  const int L = d.open_l ? nl : 0;
  int oi = sc[1];
  if (d.open_l) {
    TfOpen c;
    c.s = rows;
    c.e = rows + nl;
    c.depth = o.depth + 1;
    c.id = id_l;
    for (int j = 0; j < 3; ++j) {
      c.c[j] = d.cl[j];
      c.base[j] = sc[4 + j];
    }
    c.imp = d.imp_l;
    open_next[oi++] = c;
  }
  if (d.open_r) {
    TfOpen c;
    c.s = rows + L;
    c.e = rows + L + nr;
    c.depth = o.depth + 1;
    c.id = id_r;
    for (int j = 0; j < 3; ++j) {
      c.c[j] = cr[j];
      c.base[j] = sc[4 + j] + (d.open_l ? d.cl[j] : 0);
    }
    c.imp = d.imp_r;
    open_next[oi] = c;
  }
  // A side-1 row at column prefix q1 (side-1 rows before it in its column) lands at rows + q1 - sc[2]; a side-2 row at
  // rows + L + q2 - sc[3].
  d.dst1 = sc[3];
  d.dst2 = sc[2] + L;
  dec[k] = d;
}

// side[row]: 1 = into the open left child, 2 = into the open right child, 0 = leaves the active arrays.
__global__ void tf_flag_kernel(const uint32_t* __restrict__ rl, int n_act, int stride, const int* __restrict__ pos_node,
                               const TfDec* __restrict__ dec, uint8_t* side) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_act) return;
  const TfDec& d = dec[pos_node[p]];
  if (d.split) {
    const uint32_t r = rl[static_cast<long long>(d.f) * stride + p];
    side[r >> 2] = p < d.pos ? (d.open_l ? 1 : 0) : (d.open_r ? 2 : 0);
  } else {
    side[rl[p] >> 2] = 0;
  }
}

// Stable partition of every column by side into the next level's layout.
__global__ void __launch_bounds__(kTfThreads) tf_partition_kernel(const float* __restrict__ val,
                                                                  const uint32_t* __restrict__ rl, int n_act,
                                                                  int stride, int n_chunks,
                                                                  const int4* __restrict__ chunk_pre,
                                                                  const int* __restrict__ pos_node,
                                                                  const TfDec* __restrict__ dec,
                                                                  const uint8_t* __restrict__ side, float* val_out,
                                                                  uint32_t* rl_out) {
  __shared__ unsigned long long sh[kTfThreads / 32];
  const int f = blockIdx.y, c = blockIdx.x;
  const long long col = static_cast<long long>(f) * stride;
  const int p0 = c * kTfChunk + threadIdx.x * kTfItems;
  float v[kTfItems];
  uint32_t r[kTfItems];
  int b[kTfItems];
  unsigned long long cnt = 0;
#pragma unroll
  for (int i = 0; i < kTfItems; ++i) {
    const int p = p0 + i;
    b[i] = 0;
    if (p < n_act) {
      v[i] = val[col + p];
      r[i] = rl[col + p];
      b[i] = side[r[i] >> 2];
      cnt += 1ull << (16 * b[i]);
    }
  }
  unsigned long long run = tf_block_excl(cnt, sh);
  const int4 cp = chunk_pre[static_cast<long long>(f) * (n_chunks + 1) + c];
#pragma unroll
  for (int i = 0; i < kTfItems; ++i) {
    if (b[i]) {
      const TfDec& d = dec[pos_node[p0 + i]];
      const int q = b[i] == 1 ? d.dst1 + cp.y + tf_field(run, 1) : d.dst2 + cp.z + tf_field(run, 2);
      val_out[col + q] = v[i];
      rl_out[col + q] = r[i];
    }
    run += 1ull << (16 * b[i]);
  }
}

static unsigned grid1(long long n, int threads) { return static_cast<unsigned>((n + threads - 1) / threads); }

void tf_validate(const float* x, const uint8_t* y, long long n, int stride, float* val, uint32_t* rl, int* stats,
                 cudaStream_t st) {
  const long long blocks = std::min<long long>((n * kTfFeat + 255) / 256, 148ll * 16);
  tf_validate_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(x, y, n, stride, val, rl, stats);
}

void tf_count(int mode, int shift, const float* val, const uint32_t* rl, const uint8_t* side, int n_act, int stride,
              int n_chunks, unsigned long long* chunk_cnt, cudaStream_t st) {
  const dim3 grid(n_chunks, kTfFeat);
  if (mode == kTfByLabel)
    tf_count_kernel<kTfByLabel><<<grid, kTfThreads, 0, st>>>(shift, val, rl, side, n_act, stride, n_chunks, chunk_cnt);
  else if (mode == kTfBySide)
    tf_count_kernel<kTfBySide><<<grid, kTfThreads, 0, st>>>(shift, val, rl, side, n_act, stride, n_chunks, chunk_cnt);
  else
    tf_count_kernel<kTfByDigit><<<grid, kTfThreads, 0, st>>>(shift, val, rl, side, n_act, stride, n_chunks, chunk_cnt);
}

void tf_chunk_scan(const unsigned long long* chunk_cnt, int n_chunks, int4* chunk_pre, cudaStream_t st) {
  tf_chunk_scan_kernel<<<kTfFeat, 1024, 0, st>>>(chunk_cnt, n_chunks, chunk_pre);
}

void tf_radix_scatter(int shift, const float* val, const uint32_t* rl, int n, int stride, int n_chunks,
                      const int4* chunk_pre, float* val_out, uint32_t* rl_out, cudaStream_t st) {
  tf_radix_kernel<<<dim3(n_chunks, kTfFeat), kTfThreads, 0, st>>>(shift, val, rl, n, stride, n_chunks, chunk_pre,
                                                                  val_out, rl_out);
}

void tf_node_map(const TfOpen* open, int n_open, int n_act, int* pos_node, cudaStream_t st) {
  tf_node_map_kernel<<<grid1(n_act, 256), 256, 0, st>>>(open, n_open, n_act, pos_node);
}

void tf_search(int phase, const float* val, const uint32_t* rl, int n_act, int stride, int n_chunks,
               const int4* chunk_pre, const int* pos_node, const TfOpen* open, int min_leaf,
               unsigned long long* best_key, int* best_pos, cudaStream_t st) {
  const dim3 grid(n_chunks, kTfFeat);
  if (phase == 0)
    tf_search_kernel<0><<<grid, kTfThreads, 0, st>>>(val, rl, n_act, stride, n_chunks, chunk_pre, pos_node, open,
                                                     min_leaf, best_key, best_pos);
  else
    tf_search_kernel<1><<<grid, kTfThreads, 0, st>>>(val, rl, n_act, stride, n_chunks, chunk_pre, pos_node, open,
                                                     min_leaf, best_key, best_pos);
}

void tf_decide(const uint32_t* rl, int stride, const int4* chunk_pre, int n_chunks,
               const TfOpen* open, int n_open, const unsigned long long* best_key, const int* best_pos, TfParams p,
               TfDec* dec, int* scan, cudaStream_t st) {
  tf_decide_kernel<<<grid1(n_open, 8), 256, 0, st>>>(rl, stride, chunk_pre, n_chunks, open, n_open, best_key,
                                                     best_pos, p, dec, scan);
}

void tf_level_scan(int* scan, int n_open, int* totals, cudaStream_t st) {
  tf_level_scan_kernel<<<1, 1024, 0, st>>>(scan, n_open, totals);
}

void tf_emit(const float* val, int stride, const TfOpen* open, int n_open, TfDec* dec, const int* scan, int next_id,
             int node_cap, TfRec* rec, TfOpen* open_next, int* stats, cudaStream_t st) {
  tf_emit_kernel<<<grid1(n_open, 256), 256, 0, st>>>(val, stride, open, n_open, dec, scan, next_id, node_cap, rec,
                                                     open_next, stats);
}

void tf_flag(const uint32_t* rl, int n_act, int stride, const int* pos_node, const TfDec* dec, uint8_t* side,
             cudaStream_t st) {
  tf_flag_kernel<<<grid1(n_act, 256), 256, 0, st>>>(rl, n_act, stride, pos_node, dec, side);
}

void tf_partition(const float* val, const uint32_t* rl, int n_act, int stride, int n_chunks, const int4* chunk_pre,
                  const int* pos_node, const TfDec* dec, const uint8_t* side, float* val_out, uint32_t* rl_out,
                  cudaStream_t st) {
  tf_partition_kernel<<<dim3(n_chunks, kTfFeat), kTfThreads, 0, st>>>(val, rl, n_act, stride, n_chunks, chunk_pre,
                                                                      pos_node, dec, side, val_out, rl_out);
}

}  // namespace vadb
