// ffn_train.cuh -- one optimisation step of the 39-64-32-16-3 FFN on the device (SURVEY.md 8f, f4).
//
// Reference: learning/ffn_trainer.py:104-120,139-148 -- Keras-1 Sequential(Dense64 relu relu Dense32 relu
// Dense16 relu Dense3 softmax), loss categorical_crossentropy, optimizer 'adadelta' (Keras-1 defaults lr 1.0,
// rho 0.95, epsilon 1e-8), model.train_on_batch(batch_x, batch_y).  Restated semantics:
//   p = softmax(logits);  loss = -mean_i sum_c y_ic log(clip(p_ic, 1e-7, 1 - 1e-7))
//   g = dloss/dtheta: dlogits = (p - y) / B, and 0 for a row whose p_true lies outside [1e-7, 1 - 1e-7] (the clip
//       passes no gradient there, in Theano's T.clip and TF's clip_by_value alike)
//   a <- rho a + (1 - rho) g^2;  u = g sqrt(d + eps) / sqrt(a + eps);  theta <- theta - lr u;  d <- rho d + (1 - rho) u^2
//
// Two kernels per step, both deterministic (no floating-point atomics):
//   ffn_train_grad_kernel  persistent CTAs (512 threads) walk tiles of 128 batch rows: forward, deltas and weight
//                           gradients as register-tiled products over transposed shared-memory tiles (below); weight
//                           gradients stay in registers across a CTA's tiles -> one partial gradient + partial loss per CTA.
//   ffn_train_update_kernel thread = parameter: sums the partials in CTA order, applies Adadelta in place.
#pragma once

#include <cuda_runtime.h>

#include "vad_core.cuh"

namespace vadb {

constexpr int kTrainRows = 128;                        // batch rows per CTA
constexpr int kNParams = kNFeat * kH1 + kH1 + kH1 * kH2 + kH2 + kH2 * kH3 + kH3 + kH3 * kNCls + kNCls;  // 5219
// parameter vector layout == FfnParams: W1 b1 W2 b2 W3 b3 W4 b4
constexpr int kOffW1 = 0, kOffB1 = kOffW1 + kNFeat * kH1, kOffW2 = kOffB1 + kH1, kOffB2 = kOffW2 + kH1 * kH2,
              kOffW3 = kOffB2 + kH2, kOffB3 = kOffW3 + kH2 * kH3, kOffW4 = kOffB3 + kH3, kOffB4 = kOffW4 + kH3 * kNCls;
static_assert(kOffB4 + kNCls == kNParams, "layout");
// ---- gradient kernel: register-tiled, persistent --------------------------------------------------------------------
// One CTA (512 threads) walks tiles of 128 batch rows.  Activations and deltas live in shared memory TRANSPOSED
// ([feature][128 rows]), so every product A^T B, D W^T and A^T D of the step is the same register-tiled loop: a thread
// owns 4 rows x 1-4 columns (or 4 x 4 weight-gradient entries), reads its operands with up to 128-bit loads and does
// 4-8 FMAs per load instead of one FMA per two loads; sixteen warps per SM cover the load latency.  Each activation buffer carries a row of ones after its
// features, so the bias gradients fall out of the weight-gradient tiles.  Weight gradients stay in registers across
// the CTA's tiles and are written once as this CTA's partial (summed by ffn_train_update_kernel in CTA order):
// deterministic for a given grid, no floating-point atomics.
constexpr int kTr2Threads = 512;
constexpr int kTr2KX = 40, kTr2KH1 = 68, kTr2KH2 = 36, kTr2KH3 = 20;     // rows of X^T / H^T incl. the ones row, padded to 4
constexpr int kTr2OffWT2 = ((kNParams + 3) / 4) * 4;                      // WT2[n][k] = W2[k][n]: [32][64]
constexpr int kTr2OffWT3 = kTr2OffWT2 + kH2 * kH1;                        // [16][32]
constexpr int kTr2OffWT4 = kTr2OffWT3 + kH3 * kH2;                        // [4][16], row 3 zero
constexpr int kTr2OffX = kTr2OffWT4 + 4 * kH3;
constexpr int kTr2OffH1 = kTr2OffX + kTr2KX * kTrainRows;
constexpr int kTr2OffH2 = kTr2OffH1 + kTr2KH1 * kTrainRows;
constexpr int kTr2OffH3 = kTr2OffH2 + kTr2KH2 * kTrainRows;
constexpr int kTr2OffD1 = kTr2OffH3 + kTr2KH3 * kTrainRows;               // deltas [N][128]; D1 doubles as the load staging
constexpr int kTr2OffD2 = kTr2OffD1 + kH1 * kTrainRows;
constexpr int kTr2OffD3 = kTr2OffD2 + kH2 * kTrainRows;
constexpr int kTr2OffD4 = kTr2OffD3 + kH3 * kTrainRows;                   // [4][128], row 3 zero
constexpr int kTr2OffLoss = kTr2OffD4 + 4 * kTrainRows;
constexpr int kTrain2SmemBytes = (kTr2OffLoss + 8) * 4;
static_assert(kTrain2SmemBytes <= 227 * 1024, "training tiles must fit one CTA's shared memory");
static_assert(kTrainRows * 41 <= kH1 * kTrainRows, "row-major staging of an input tile fits the D1 buffer");

// C^T[n][r] = sum_k At[k][r] B[k][n] over one 128-row tile; thread tile RM rows x CN columns; epi(row0, col0, acc).
template <int K, int N, int RM, int CN, class EPI>
__device__ __forceinline__ void tr2_gemm(const float* __restrict__ At, const float* __restrict__ B, EPI&& epi) {
  constexpr int CG = N / CN;
  static_assert((kTrainRows / RM) * CG == kTr2Threads && RM % 4 == 0 && (CN == 1 || CN == 2 || CN == 4), "thread tiling");
  const int tc = threadIdx.x % CG, tr = threadIdx.x / CG;
  float acc[RM][CN];
#pragma unroll
  for (int i = 0; i < RM; ++i)
#pragma unroll
    for (int j = 0; j < CN; ++j) acc[i][j] = 0.0f;
  const float* ap = At + tr * RM;
  const float* bp = B + tc * CN;
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    float a[RM], b[CN];
#pragma unroll
    for (int i = 0; i < RM; i += 4) {
      const float4 v = *reinterpret_cast<const float4*>(ap + k * kTrainRows + i);
      a[i] = v.x; a[i + 1] = v.y; a[i + 2] = v.z; a[i + 3] = v.w;
    }
    if constexpr (CN == 4) {
      const float4 v = *reinterpret_cast<const float4*>(bp + k * N);
      b[0] = v.x; b[1] = v.y; b[2] = v.z; b[3] = v.w;
    } else if constexpr (CN == 2) {
      const float2 v = *reinterpret_cast<const float2*>(bp + k * N);
      b[0] = v.x; b[1] = v.y;
    } else {
      b[0] = bp[k * N];
    }
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < CN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
  }
  epi(tr * RM, tc * CN, acc);
}
// forward epilogue: + bias, ReLU -> H^T[col][row0 ..]
template <int RM, int CN>
__device__ __forceinline__ void tr2_store_relu(float* Ht, const float* bias, int row0, int col0, float (&acc)[RM][CN]) {
#pragma unroll
  for (int j = 0; j < CN; ++j) {
    const float b = bias[col0 + j];
#pragma unroll
    for (int i = 0; i < RM; i += 4)
      *reinterpret_cast<float4*>(Ht + (col0 + j) * kTrainRows + row0 + i) =
          make_float4(fmaxf(acc[i][j] + b, 0.0f), fmaxf(acc[i + 1][j] + b, 0.0f), fmaxf(acc[i + 2][j] + b, 0.0f),
                      fmaxf(acc[i + 3][j] + b, 0.0f));
  }
}
// backward epilogue: delta = activation > 0 ? acc : 0 -> D^T[col][row0 ..]
template <int RM, int CN>
__device__ __forceinline__ void tr2_store_delta(float* Dt, const float* Ht, int row0, int col0, float (&acc)[RM][CN]) {
#pragma unroll
  for (int j = 0; j < CN; ++j)
#pragma unroll
    for (int i = 0; i < RM; i += 4) {
      const float4 hh = *reinterpret_cast<const float4*>(Ht + (col0 + j) * kTrainRows + row0 + i);
      *reinterpret_cast<float4*>(Dt + (col0 + j) * kTrainRows + row0 + i) =
          make_float4(hh.x > 0.0f ? acc[i][j] : 0.0f, hh.y > 0.0f ? acc[i + 1][j] : 0.0f,
                      hh.z > 0.0f ? acc[i + 2][j] : 0.0f, hh.w > 0.0f ? acc[i + 3][j] : 0.0f);
    }
}

// A weight-gradient tile: 4 rows of an activation buffer (k0 ..) x 4 rows of a delta buffer (n0 ..), summed over rows.
// 337 tiles, one per thread of the 512 (66 % of the threads busy in this stage; 4 x 2 tiles balance better and were
// measured 8 % slower: 50 % more shared-memory loads per FMA).
struct Tr2GradTile {
  int a_off, d_off;   // shared-memory offsets (floats) of the 4 activation rows / 4 delta rows
  int layer, k0, n0;  // where the 16 sums go; layer < 0: no tile
};
__device__ __forceinline__ Tr2GradTile tr2_grad_tile(int t) {
  // layer 1: 10 x 16 tiles, layer 2: 17 x 8, layer 3: 9 x 4, layer 4: 5 x 1
  Tr2GradTile g{0, 0, -1, 0, 0};
  if (t < 160) { g.layer = 0; g.k0 = 4 * (t / 16); g.n0 = 4 * (t % 16); g.a_off = kTr2OffX; g.d_off = kTr2OffD1; }
  else if (t < 296) { t -= 160; g.layer = 1; g.k0 = 4 * (t / 8); g.n0 = 4 * (t % 8); g.a_off = kTr2OffH1; g.d_off = kTr2OffD2; }
  else if (t < 332) { t -= 296; g.layer = 2; g.k0 = 4 * (t / 4); g.n0 = 4 * (t % 4); g.a_off = kTr2OffH2; g.d_off = kTr2OffD3; }
  else if (t < 337) { t -= 332; g.layer = 3; g.k0 = 4 * t; g.n0 = 0; g.a_off = kTr2OffH3; g.d_off = kTr2OffD4; }
  g.a_off += g.k0 * kTrainRows;
  g.d_off += g.n0 * kTrainRows;
  return g;
}
__device__ __forceinline__ void tr2_grad_accumulate(const float* sm, const Tr2GradTile& g, float (&acc)[4][4]) {
  const float* a = sm + g.a_off;
  const float* d = sm + g.d_off;
  // the eight lanes of a quarter-warp own tiles whose rows start a multiple of 128 floats apart (the same banks), so
  // each lane walks the 128 batch rows from its own starting group of four: conflict-free 128-bit loads
  const int rot = 4 * (threadIdx.x & 7);
#pragma unroll 2
  for (int rr = 0; rr < kTrainRows; rr += 4) {
    const int r = (rr + rot) & (kTrainRows - 1);
    float4 av[4], dv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      av[i] = *reinterpret_cast<const float4*>(a + i * kTrainRows + r);
      dv[i] = *reinterpret_cast<const float4*>(d + i * kTrainRows + r);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        acc[i][j] = fmaf(av[i].w, dv[j].w, fmaf(av[i].z, dv[j].z, fmaf(av[i].y, dv[j].y, fmaf(av[i].x, dv[j].x, acc[i][j]))));
  }
}
__device__ __forceinline__ void tr2_grad_write(float* g, const Tr2GradTile& t, const float (&acc)[4][4]) {
  if (t.layer < 0) return;
  const int K = t.layer == 0 ? kNFeat : t.layer == 1 ? kH1 : t.layer == 2 ? kH2 : kH3;
  const int N = t.layer == 0 ? kH1 : t.layer == 1 ? kH2 : t.layer == 2 ? kH3 : kNCls;
  const int ow = t.layer == 0 ? kOffW1 : t.layer == 1 ? kOffW2 : t.layer == 2 ? kOffW3 : kOffW4;
  const int ob = t.layer == 0 ? kOffB1 : t.layer == 1 ? kOffB2 : t.layer == 2 ? kOffB3 : kOffB4;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = t.k0 + i, n = t.n0 + j;
      if (n < N) {
        if (k < K) g[ow + k * N + n] = acc[i][j];
        else if (k == K) g[ob + n] = acc[i][j];   // the row of ones: bias gradient
      }
    }
}

__global__ void __launch_bounds__(kTr2Threads, 1) ffn_train_grad_kernel(const float* __restrict__ params,
                                                                         const float* __restrict__ x,
                                                                         const uint8_t* __restrict__ y, long long n_rows,
                                                                         float inv_b, float* partial /*[grid][kNParams + 1]*/) {
  extern __shared__ __align__(16) float sm[];
  float* w = sm;
  const int tid = threadIdx.x;
  // parameters, transposed copies for the delta products, constant rows (ones / zero padding)
  for (int i = tid; i < kNParams; i += kTr2Threads) w[i] = params[i];
  for (int i = tid; i < kH2 * kH1; i += kTr2Threads) sm[kTr2OffWT2 + i] = params[kOffW2 + (i % kH1) * kH2 + i / kH1];
  for (int i = tid; i < kH3 * kH2; i += kTr2Threads) sm[kTr2OffWT3 + i] = params[kOffW3 + (i % kH2) * kH3 + i / kH2];
  for (int i = tid; i < 4 * kH3; i += kTr2Threads)
    sm[kTr2OffWT4 + i] = i / kH3 < kNCls ? params[kOffW4 + (i % kH3) * kNCls + i / kH3] : 0.0f;
  for (int i = tid; i < kTrainRows; i += kTr2Threads) {
    sm[kTr2OffX + kNFeat * kTrainRows + i] = 1.0f;                      // X^T row 39
    for (int k = kH1; k < kTr2KH1; ++k) sm[kTr2OffH1 + k * kTrainRows + i] = k == kH1 ? 1.0f : 0.0f;
    for (int k = kH2; k < kTr2KH2; ++k) sm[kTr2OffH2 + k * kTrainRows + i] = k == kH2 ? 1.0f : 0.0f;
    for (int k = kH3; k < kTr2KH3; ++k) sm[kTr2OffH3 + k * kTrainRows + i] = k == kH3 ? 1.0f : 0.0f;
    sm[kTr2OffD4 + 3 * kTrainRows + i] = 0.0f;
  }
  const Tr2GradTile g0 = tr2_grad_tile(tid);   // 337 tiles: threads 337 .. 511 own none
  float acc0[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc0[i][j] = 0.0f;
  float loss_acc = 0.0f;   // thread 0 only: tile losses in tile order
  float* X = sm + kTr2OffX;
  float* H1 = sm + kTr2OffH1;
  float* H2 = sm + kTr2OffH2;
  float* H3 = sm + kTr2OffH3;
  float* D1 = sm + kTr2OffD1;
  float* D2 = sm + kTr2OffD2;
  float* D3 = sm + kTr2OffD3;
  float* D4 = sm + kTr2OffD4;
  float* sloss = sm + kTr2OffLoss;
  const long long n_tiles = (n_rows + kTrainRows - 1) / kTrainRows;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long row0 = tile * kTrainRows;
    const int rows = static_cast<int>(min(static_cast<long long>(kTrainRows), n_rows - row0));
    __syncthreads();   // previous tile's gradient pass is done with every buffer (also orders the set-up above)
    // coalesced load into a row-major staging tile (pitch 41: odd), then transpose into X^T; rows >= rows are zero
    float* stage = D1;
    for (int i = tid; i < kTrainRows * kNFeat; i += kTr2Threads) {
      const int r = i / kNFeat, k = i - r * kNFeat;
      stage[r * 41 + k] = r < rows ? x[row0 * kNFeat + i] : 0.0f;
    }
    __syncthreads();
    for (int i = tid; i < kTrainRows * kNFeat; i += kTr2Threads) {
      const int k = i / kTrainRows, r = i - k * kTrainRows;
      X[k * kTrainRows + r] = stage[r * 41 + k];
    }
    __syncthreads();
    // ---- forward (learning/ffn_trainer.py:106-116) ----
    tr2_gemm<kNFeat, kH1, 4, 4>(X, w + kOffW1, [&](int r0, int c0, float (&a)[4][4]) { tr2_store_relu<4, 4>(H1, w + kOffB1, r0, c0, a); });
    __syncthreads();
    tr2_gemm<kH1, kH2, 4, 2>(H1, w + kOffW2, [&](int r0, int c0, float (&a)[4][2]) { tr2_store_relu<4, 2>(H2, w + kOffB2, r0, c0, a); });
    __syncthreads();
    tr2_gemm<kH2, kH3, 4, 1>(H2, w + kOffW3, [&](int r0, int c0, float (&a)[4][1]) { tr2_store_relu<4, 1>(H3, w + kOffB3, r0, c0, a); });
    __syncthreads();
    // ---- layer 4, softmax, categorical cross-entropy, dlogits: thread = row ----
    float loss = 0.0f;
    if (tid < kTrainRows) {
      const int r = tid;
      float lg[kNCls];
#pragma unroll
      for (int o = 0; o < kNCls; ++o) lg[o] = w[kOffB4 + o];
#pragma unroll
      for (int i = 0; i < kH3; ++i) {
        const float hv = H3[i * kTrainRows + r];
#pragma unroll
        for (int o = 0; o < kNCls; ++o) lg[o] = fmaf(hv, w[kOffW4 + i * kNCls + o], lg[o]);
      }
      const float mx = fmaxf(lg[0], fmaxf(lg[1], lg[2]));
      const float e0 = expf(lg[0] - mx), e1 = expf(lg[1] - mx), e2 = expf(lg[2] - mx);
      const float inv = 1.0f / (e0 + e1 + e2);
      const float p[kNCls] = {e0 * inv, e1 * inv, e2 * inv};
      const bool live = r < rows;
      const int cls = live ? y[row0 + r] : 0;
      const float py = cls == 0 ? p[0] : cls == 1 ? p[1] : p[2];
      // the high end as "the other two sum below 1e-7": float32 cannot resolve p_y > 1 - 1e-7 directly
      const float rest = cls == 0 ? p[1] + p[2] : cls == 1 ? p[0] + p[2] : p[0] + p[1];
      const bool clipped = py < 1e-7f || rest < 1e-7f;
      loss = live ? -logf(fminf(fmaxf(py, 1e-7f), 1.0f - 1e-7f)) : 0.0f;
#pragma unroll
      for (int o = 0; o < kNCls; ++o)
        D4[o * kTrainRows + r] = live && !clipped ? (p[o] - (o == cls ? 1.0f : 0.0f)) * inv_b : 0.0f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) loss += __shfl_down_sync(0xffffffffu, loss, o);
    if ((tid & 31) == 0) sloss[tid >> 5] = loss;
    __syncthreads();
    if (tid == 0) loss_acc += (sloss[0] + sloss[1]) + (sloss[2] + sloss[3]);
    // ---- backward: deltas ----
    tr2_gemm<4, kH3, 4, 1>(D4, sm + kTr2OffWT4, [&](int r0, int c0, float (&a)[4][1]) { tr2_store_delta<4, 1>(D3, H3, r0, c0, a); });
    __syncthreads();
    tr2_gemm<kH3, kH2, 4, 2>(D3, sm + kTr2OffWT3, [&](int r0, int c0, float (&a)[4][2]) { tr2_store_delta<4, 2>(D2, H2, r0, c0, a); });
    __syncthreads();
    tr2_gemm<kH2, kH1, 4, 4>(D2, sm + kTr2OffWT2, [&](int r0, int c0, float (&a)[4][4]) { tr2_store_delta<4, 4>(D1, H1, r0, c0, a); });
    __syncthreads();
    // ---- weight (and, through the rows of ones, bias) gradients, accumulated over this CTA's tiles ----
    if (g0.layer >= 0) tr2_grad_accumulate(sm, g0, acc0);
  }
  float* g = partial + static_cast<long long>(blockIdx.x) * (kNParams + 1);
  tr2_grad_write(g, g0, acc0);
  if (tid == 0) g[kNParams] = loss_acc * inv_b;
}

// state: [0] parameters, [1] accumulated squared gradients a, [2] accumulated squared updates d (kNParams each)
__global__ void ffn_train_update_kernel(float* params, float* acc_g, float* acc_u, const float* partial, int n_part,
                                        float lr, float rho, float eps, float* loss_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > kNParams) return;
  float g = 0.0f;
  for (int c = 0; c < n_part; ++c) g += partial[static_cast<long long>(c) * (kNParams + 1) + i];
  if (i == kNParams) {
    if (loss_out) *loss_out = g;
    return;
  }
  const float a = rho * acc_g[i] + (1.0f - rho) * g * g;
  const float u = g * sqrtf(acc_u[i] + eps) / sqrtf(a + eps);
  params[i] -= lr * u;
  acc_g[i] = a;
  acc_u[i] = rho * acc_u[i] + (1.0f - rho) * u * u;
}

}  // namespace vadb
