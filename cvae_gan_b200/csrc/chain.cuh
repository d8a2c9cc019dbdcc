// cvaegan_b200 - the critic's and the classifier's forward + input-gradient chains of a D / C training step, one row-tile
// kernel each.
//
// Neither network has BatchNorm, so every batch row of their chains is independent of every other: a CTA that owns CH_TM
// rows of one pass runs all layers with the tile's activations in shared memory, reading the weights (< 200 KB per network)
// from L2 in chunks.  That replaces 8 (critic) or 10 (classifier) dependent layer launches of a step by one.
//
// The chains write every buffer the layer kernels write (activations, masks applied, scores, logits, gradients w.r.t. the
// pre-activations), with the same values bit for bit: each output element is produced by the operation sequence of
// gemm_mn_kernel (k-group g = (k % TBK) / 4 accumulates its k in ascending order with fmaf from +0, zero-padded k included,
// the four groups are added as ((p0 + p1) + p2) + p3) and the epilogue, LayerNorm and cross-entropy expressions are the
// device functions the layer kernels call.  The weight-gradient kernels (gemm_dw_kernel) then read these buffers.
#pragma once
#include "gemm.cuh"
#include "misc_kernels.cuh"

namespace cvg {

constexpr int CH_TM = 32;            // batch rows per CTA: one LayerNorm / cross-entropy warp tile
constexpr int CH_THREADS = 256;
constexpr int CH_NB = 64;            // output features per sweep over the row tile
constexpr int CH_KC = 64;            // reduction indices per staged weight chunk (four TBK chunks)
constexpr int CH_H0 = 256, CH_H1 = 128, CH_H2 = 64;   // the hidden widths the chains are built for (the reference's)
constexpr int CH_MAX_IN = 256;       // input features
constexpr int CH_MAX_K = 32;         // classes
constexpr int CH_WBUF = 2 * CH_KC * CH_NB;   // double-buffered weight chunk; also the [4][CH_NB][CH_TM] k-group partials

struct CriticChainArgs {
  int M = 0, ld = 0, F = 0;
  const float* x = nullptr;          // [F][ld], pass p at x + p * sx
  long long sx = 0;
  const float* W[4] = {};            // [out][ldw[l]]
  int ldw[4] = {};
  const float* b[4] = {};
  const float* wlabel = nullptr;     // layer 0 one-hot column (null: unconditional critic)
  int ldwl = 0;
  const float* inv_sigma = nullptr;  // [layer][pass]
  const uint8_t* m1 = nullptr;       // [2][H0][ld]
  const uint8_t* m2 = nullptr;       // [2][H1][ld]
  float keep_inv = 1.f, slope = 0.2f;
  float* a[3] = {};                  // d_a: [2][Hl][ld]
  float* s = nullptr;                // d_s: [2][1][ld]
  float* g[3] = {};                  // d_g: [2][Hl][ld]
  double* osum = nullptr;            // [pass] score sums
  float seed[2] = {0.f, 0.f};        // dL/dscore per pass
};

struct ClassifierChainArgs {
  int M = 0, ld = 0, F = 0, K = 0, label = 0;
  const float* x = nullptr;
  long long sx = 0;
  const float* W[4] = {};
  const float* b[4] = {};
  const float* gamma = nullptr;      // LayerNorm of layer 1
  const float* beta = nullptr;
  float ln_eps = 1e-5f;
  const uint8_t* m1 = nullptr;       // [2][H0][ld]
  const uint8_t* m2 = nullptr;       // [2][H1][ld]
  float keep_inv = 1.f;
  float *a1 = nullptr, *h2 = nullptr, *a2 = nullptr, *rs = nullptr, *a3 = nullptr, *logit = nullptr, *dlogit = nullptr;
  float* g[3] = {};
  float coef = 1.f;                  // 1 / Bg
  double* loss = nullptr;            // [pass] cross-entropy sums
  float* dgamma = nullptr;           // LayerNorm affine gradients
  float* dbeta = nullptr;
  unsigned long long* acc = nullptr; // [2 * H1] fixed-point affine sums (Workspace::det_acc of the launch stream)
  unsigned* cnt = nullptr;           // ticket counter
};

// Y[n][m] = sum_k X[k][m] * W(k, n) for the CH_TM rows of the tile, n < N, k < R.  WT: W(k, n) = W[n * ldw + k] (forward),
// otherwise W[k * ldw + n] (input gradient).  X: shared [roundup(R, TBK)][CH_TM], rows >= R zero.  Per output element the
// sequence of gemm_mn_kernel; ep(n, m, y) gets rows m..m+3 of column n.  Ends with a CTA barrier.
template <bool WT, class Ep>
__device__ __forceinline__ void chain_layer(const float* X, const float* __restrict__ W, int ldw, int R, int N, float* wbuf,
                                            Ep ep) {
  const int tid = threadIdx.x;
  const int grp = tid >> 6, t64 = tid & 63;
  const int tm = (t64 & 7) * 4, tn = (t64 >> 3) * 8;   // this thread: rows tm..tm+3 x columns tn..tn+7 of k-group grp
  const int Rp = (R + TBK - 1) / TBK * TBK;
  const int nkc = (Rp + CH_KC - 1) / CH_KC;
  const bool wvec = (ldw & 3) == 0;
  for (int n0 = 0; n0 < N; n0 += CH_NB) {
    float4 pre[4];
    auto gload = [&](int kc) {
#pragma unroll
      for (int j = 0; j < 4; ++j) pre[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (WT) {                      // W[n][kc + 16 q .. +16] -> rows of the chunk, transposed on the store
        const int n = n0 + (tid & 63);
        if (n >= N) return;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = kc + (tid >> 6) * 16 + 4 * j;
          const float* src = W + (size_t)n * ldw + k;
          if (wvec && k + 3 < R) {
            pre[j] = ld4(src);
          } else {
            if (k < R) pre[j].x = src[0];
            if (k + 1 < R) pre[j].y = src[1];
            if (k + 2 < R) pre[j].z = src[2];
            if (k + 3 < R) pre[j].w = src[3];
          }
        }
      } else {                       // W[kc + k][n0 + 16 q .. +16]
        const int k = kc + (tid >> 2);
        if (k >= R) return;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int n = n0 + (tid & 3) * 16 + 4 * j;
          const float* src = W + (size_t)k * ldw + n;
          if (wvec && n + 3 < N) {
            pre[j] = ld4(src);
          } else {
            if (n < N) pre[j].x = src[0];
            if (n + 1 < N) pre[j].y = src[1];
            if (n + 2 < N) pre[j].z = src[2];
            if (n + 3 < N) pre[j].w = src[3];
          }
        }
      }
    };
    auto sstore = [&](float* buf) {   // buf[k][n]
      if (WT) {
        const int kq = (tid >> 6) * 16, n = tid & 63;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          buf[(kq + 4 * j + 0) * CH_NB + n] = pre[j].x;
          buf[(kq + 4 * j + 1) * CH_NB + n] = pre[j].y;
          buf[(kq + 4 * j + 2) * CH_NB + n] = pre[j].z;
          buf[(kq + 4 * j + 3) * CH_NB + n] = pre[j].w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) st4(buf + (tid >> 2) * CH_NB + (tid & 3) * 16 + 4 * j, pre[j]);
      }
    };
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    gload(0);
    sstore(wbuf);
    __syncthreads();
    for (int c = 0; c < nkc; ++c) {
      const float* cur = wbuf + (c & 1) * CH_KC * CH_NB;
      const int kc = c * CH_KC;
      if (c + 1 < nkc) gload(kc + CH_KC);          // in flight across the FFMA block
      const int nt = min(CH_KC, Rp - kc) / TBK;
      for (int t = 0; t < nt; ++t) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int kl = t * TBK + grp * 4 + q;
          const float4 a = ld4(X + (size_t)(kc + kl) * CH_TM + tm);
          const float4 w0 = ld4(cur + kl * CH_NB + tn), w1 = ld4(cur + kl * CH_NB + tn + 4);
          const float av[4] = {a.x, a.y, a.z, a.w};
          const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
        }
      }
      if (c + 1 < nkc) sstore(wbuf + ((c + 1) & 1) * CH_KC * CH_NB);
      __syncthreads();
    }
    // k-group partials meet in shared memory (over the weight chunks, which every thread is done reading)
    float* red = wbuf;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      st4(red + ((size_t)grp * CH_NB + tn + j) * CH_TM + tm, make_float4(acc[0][j], acc[1][j], acc[2][j], acc[3][j]));
    __syncthreads();
    {
      const int n = tid >> 2;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int m = (tid & 3) * 8 + 4 * h;
        const float4 y = ksum4(ld4(red + ((size_t)0 * CH_NB + n) * CH_TM + m), ld4(red + ((size_t)1 * CH_NB + n) * CH_TM + m),
                               ld4(red + ((size_t)2 * CH_NB + n) * CH_TM + m), ld4(red + ((size_t)3 * CH_NB + n) * CH_TM + m));
        if (n0 + n < N) ep(n0 + n, m, y);
      }
    }
    __syncthreads();
  }
}

// Forward epilogue (EP_LINEAR of gemm_mn_kernel): act(fma(acc, scale, bias')) then dropout, stored to Y (global, every row
// of the tile, as the layer kernel does) and to S (shared operand of the next layer, rows >= M zero).  Returns the sum of
// the valid rows' outputs (critic score).
struct FwdEp {
  const float* bias;
  const float* wlabel;
  int ldwl;
  float scale;
  int act;
  float slope;
  const uint8_t* mask;               // [N][ld] of this pass, or null
  float keep_inv;
  float* Y;                          // [N][ld] of this pass
  float* S;                          // [N][CH_TM] or null
  int ld, m0, M;
  __device__ __forceinline__ double operator()(int n, int m, float4 v) const {
    float y[4] = {v.x, v.y, v.z, v.w};
    const float b = ep_bias(bias, wlabel, ldwl, n, scale);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = ep_act(ep_linear(y[i], scale, b), act, slope);
    const size_t off = (size_t)n * ld + m0 + m;
    if (mask) {
      const uchar4 mk = *reinterpret_cast<const uchar4*>(mask + off);
      y[0] = ep_dropout(y[0], mk.x, keep_inv);
      y[1] = ep_dropout(y[1], mk.y, keep_inv);
      y[2] = ep_dropout(y[2], mk.z, keep_inv);
      y[3] = ep_dropout(y[3], mk.w, keep_inv);
    }
    st4(Y + off, make_float4(y[0], y[1], y[2], y[3]));
    double tot = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const bool valid = m0 + m + i < M;
      if (S) S[n * CH_TM + m + i] = valid ? y[i] : 0.f;
      if (valid) tot += (double)y[i];
    }
    return tot;
  }
};

// Input-gradient epilogue (EP_DACT): dropout and activation derivative of the layer below, whose output A (shared, the
// same values the layer kernel reads from memory) may be overwritten in place by S.  Rows >= M come out as +0 whatever A
// holds there, as in the layer kernel (their operand rows are zero).
struct DactEp {
  float scale;
  const uint8_t* mask;
  float keep_inv;
  float neg;
  const float* A;                    // [N][CH_TM]
  float* Y;                          // [N][ld] of this pass
  float* S;                          // [N][CH_TM] or null
  int ld, m0, M;
  __device__ __forceinline__ void operator()(int n, int m, float4 v) const {
    float y[4] = {v.x, v.y, v.z, v.w};
    const size_t off = (size_t)n * ld + m0 + m;
    float keep[4] = {1.f, 1.f, 1.f, 1.f};
    if (mask) {
      const uchar4 mk = *reinterpret_cast<const uchar4*>(mask + off);
      keep[0] = ep_keep(mk.x, keep_inv);
      keep[1] = ep_keep(mk.y, keep_inv);
      keep[2] = ep_keep(mk.z, keep_inv);
      keep[3] = ep_keep(mk.w, keep_inv);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = ep_dact(y[i], scale, keep[i], A[n * CH_TM + m + i], neg);
    st4(Y + off, make_float4(y[0], y[1], y[2], y[3]));
    if (S)
#pragma unroll
      for (int i = 0; i < 4; ++i) S[n * CH_TM + m + i] = m0 + m + i < M ? y[i] : 0.f;
  }
};

// rows [0, rows) of a [rows][CH_TM] shared operand from feature-major memory; rows >= nvalid and batch rows >= M read 0
__device__ __forceinline__ void chain_stage(float* S, int rows, const float* src, int nvalid, int ld, int m0, int M) {
  for (int i = threadIdx.x; i < rows * CH_TM; i += CH_THREADS) {
    const int k = i / CH_TM, m = i % CH_TM;
    S[i] = (k < nvalid && m0 + m < M) ? src[(size_t)k * ld + m0 + m] : 0.f;
  }
}

__host__ __device__ inline int chain_x_rows(int F, int K) {
  const int fp = (F + TBK - 1) / TBK * TBK;
  const int kp = 2 * ((K + TBK - 1) / TBK * TBK);
  return fp > kp ? fp : kp;
}
inline size_t critic_chain_smem(int F) {
  return sizeof(float) * ((size_t)CH_WBUF + (size_t)(CH_H0 + CH_H1 + CH_H2) * CH_TM + (size_t)chain_x_rows(F, 1) * CH_TM);
}
inline size_t classifier_chain_smem(int F, int K) {
  return sizeof(float) * ((size_t)CH_WBUF + (size_t)(CH_H0 + 2 * CH_H1 + CH_H2) * CH_TM + (size_t)chain_x_rows(F, K) * CH_TM);
}

// grid (2 * ceil(M / 64), 2 passes): the 64-row tiles the layer kernels cover, in halves
__global__ void __launch_bounds__(CH_THREADS, 2) critic_chain_kernel(const CriticChainArgs g) {
  extern __shared__ __align__(16) float ch_smem[];
  float* wbuf = ch_smem;
  float* A0 = wbuf + CH_WBUF;                      // layer outputs; the input gradients overwrite A2 and A1 in place
  float* A1 = A0 + CH_H0 * CH_TM;
  float* A2 = A1 + CH_H1 * CH_TM;
  float* X = A2 + CH_H2 * CH_TM;                   // input rows, later the constant score seed
  const int pass = blockIdx.y, m0 = blockIdx.x * CH_TM;
  const int M = g.M, ld = g.ld;
  const size_t ps0 = (size_t)pass * CH_H0 * ld, ps1 = (size_t)pass * CH_H1 * ld, ps2 = (size_t)pass * CH_H2 * ld;

  chain_stage(X, (g.F + TBK - 1) / TBK * TBK, g.x + (long long)pass * g.sx, g.F, ld, m0, M);
  __syncthreads();
  // ---- forward: Linear (1/sigma, label column) -> LeakyReLU -> dropout, x3, then the score ----
  chain_layer<true>(X, g.W[0], g.ldw[0], g.F, CH_H0, wbuf,
                    FwdEp{g.b[0], g.wlabel, g.ldwl, g.inv_sigma[0 + pass], ACT_LRELU, g.slope, g.m1 + ps0, g.keep_inv,
                          g.a[0] + ps0, A0, ld, m0, M});
  chain_layer<true>(A0, g.W[1], g.ldw[1], CH_H0, CH_H1, wbuf,
                    FwdEp{g.b[1], nullptr, 0, g.inv_sigma[2 + pass], ACT_LRELU, g.slope, g.m2 + ps1, g.keep_inv,
                          g.a[1] + ps1, A1, ld, m0, M});
  chain_layer<true>(A1, g.W[2], g.ldw[2], CH_H1, CH_H2, wbuf,
                    FwdEp{g.b[2], nullptr, 0, g.inv_sigma[4 + pass], ACT_LRELU, g.slope, nullptr, 1.f,
                          g.a[2] + ps2, A2, ld, m0, M});
  double tot = 0.0;
  const FwdEp score{g.b[3], nullptr, 0, g.inv_sigma[6 + pass], ACT_NONE, g.slope, nullptr, 1.f,
                    g.s + (size_t)pass * ld, nullptr, ld, m0, M};
  chain_layer<true>(A2, g.W[3], g.ldw[3], CH_H2, 1, wbuf, [&](int n, int m, float4 y) { tot += score(n, m, y); });
  tot = warp_sum_d(tot);
  if (threadIdx.x == 0) atomicAdd(g.osum + pass, tot);   // only threads 0..3 hold score columns
  // ---- input gradients from the constant seed down to the first hidden layer (no dx: the D step has none) ----
  for (int i = threadIdx.x; i < TBK * CH_TM; i += CH_THREADS)
    X[i] = (i < CH_TM && m0 + i < M) ? g.seed[pass] : 0.f;
  __syncthreads();
  chain_layer<false>(X, g.W[3], g.ldw[3], 1, CH_H2, wbuf,
                     DactEp{g.inv_sigma[6 + pass], nullptr, 1.f, g.slope, A2, g.g[2] + ps2, A2, ld, m0, M});
  chain_layer<false>(A2, g.W[2], g.ldw[2], CH_H2, CH_H1, wbuf,
                     DactEp{g.inv_sigma[4 + pass], g.m2 + ps1, g.keep_inv, g.slope, A1, g.g[1] + ps1, A1, ld, m0, M});
  chain_layer<false>(A1, g.W[1], g.ldw[1], CH_H1, CH_H0, wbuf,
                     DactEp{g.inv_sigma[2 + pass], g.m1 + ps0, g.keep_inv, g.slope, A0, g.g[0] + ps0, nullptr, ld, m0, M});
}

__global__ void __launch_bounds__(CH_THREADS, 2) classifier_chain_kernel(const ClassifierChainArgs g) {
  extern __shared__ __align__(16) float ch_smem[];
  __shared__ float red1[8][LN_ROWS], red2[8][LN_ROWS];
  __shared__ unsigned s_last;
  float* wbuf = ch_smem;
  float* A1 = wbuf + CH_WBUF;
  float* H2 = A1 + CH_H0 * CH_TM;
  float* A2 = H2 + CH_H1 * CH_TM;                  // LayerNorm output, later dL/dn and dL/dh in place
  float* A3 = A2 + CH_H1 * CH_TM;                  // later dL/d(layer-2 pre-activation) in place
  float* X = A3 + CH_H2 * CH_TM;                   // input rows; later logits (K rows) and dlogits (Kp rows)
  const int Kp = (g.K + TBK - 1) / TBK * TBK;
  float* L = X;
  float* D = X + Kp * CH_TM;
  const int pass = blockIdx.y, m0 = blockIdx.x * CH_TM;
  const int M = g.M, ld = g.ld;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const bool valid = m0 + lane < M;                // LayerNorm / cross-entropy row of this lane
  const size_t ps0 = (size_t)pass * CH_H0 * ld, ps1 = (size_t)pass * CH_H1 * ld, ps2 = (size_t)pass * CH_H2 * ld;
  const size_t psk = (size_t)pass * g.K * ld;

  chain_stage(X, (g.F + TBK - 1) / TBK * TBK, g.x + (long long)pass * g.sx, g.F, ld, m0, M);
  for (int i = threadIdx.x; i < CH_H1 * CH_TM; i += CH_THREADS) A2[i] = 0.f;   // LayerNorm writes valid rows only
  __syncthreads();
  // ---- forward: Linear -> ReLU -> dropout -> Linear -> LayerNorm + ReLU + dropout -> Linear -> ReLU -> Linear ----
  chain_layer<true>(X, g.W[0], g.F, g.F, CH_H0, wbuf,
                    FwdEp{g.b[0], nullptr, 0, 1.0f, ACT_RELU, 0.f, g.m1 + ps0, g.keep_inv, g.a1 + ps0, A1, ld, m0, M});
  chain_layer<true>(A1, g.W[1], CH_H0, CH_H0, CH_H1, wbuf,
                    FwdEp{g.b[1], nullptr, 0, 1.0f, ACT_NONE, 0.f, nullptr, 1.f, g.h2 + ps1, H2, ld, m0, M});
  float mean, rstd;
  {
    const uint8_t* mk = g.m2 + ps1 + m0 + lane;
    float* a2g = g.a2 + ps1 + m0 + lane;
    ln_fwd_row<LN_MAXF>(
        CH_H1, valid, g.ln_eps, g.gamma, g.beta, mk, ld, g.keep_inv, red1, [&](int c) { return H2[c * CH_TM + lane]; },
        [&](int c, float n) {
          a2g[(size_t)c * ld] = n;
          A2[c * CH_TM + lane] = n;
        },
        mean, rstd);
    if (valid && w == 0) {
      float* rs = g.rs + (size_t)pass * 2 * ld;
      rs[m0 + lane] = mean;
      rs[ld + m0 + lane] = rstd;
    }
  }
  for (int i = threadIdx.x; i < Kp * CH_TM; i += CH_THREADS) D[i] = 0.f;   // cross-entropy writes valid rows only
  __syncthreads();
  chain_layer<true>(A2, g.W[2], CH_H1, CH_H1, CH_H2, wbuf,
                    FwdEp{g.b[2], nullptr, 0, 1.0f, ACT_RELU, 0.f, nullptr, 1.f, g.a3 + ps2, A3, ld, m0, M});
  chain_layer<true>(A3, g.W[3], CH_H2, CH_H2, g.K, wbuf,
                    FwdEp{g.b[3], nullptr, 0, 1.0f, ACT_NONE, 0.f, nullptr, 1.f, g.logit + psk, L, ld, m0, M});
  // ---- cross-entropy with the step's label: loss sum and dlogits ----
  if (w == 0) {
    double nll = 0.0;
    if (valid) {
      nll = ce_row(L + lane, CH_TM, D + lane, CH_TM, g.K, g.label, g.coef);
      float* dg = g.dlogit + psk + m0 + lane;
      for (int k = 0; k < g.K; ++k) dg[(size_t)k * ld] = D[k * CH_TM + lane];
    }
    nll = warp_sum_d(nll);
    if (lane == 0 && nll != 0.0) atomicAdd(g.loss + pass, nll);
  }
  __syncthreads();
  // ---- input gradients ----
  chain_layer<false>(D, g.W[3], CH_H2, g.K, CH_H2, wbuf,
                     DactEp{1.0f, nullptr, 1.f, 0.f, A3, g.g[2] + ps2, A3, ld, m0, M});
  chain_layer<false>(A3, g.W[2], CH_H1, CH_H2, CH_H1, wbuf,
                     DactEp{1.0f, g.m2 + ps1, g.keep_inv, 0.f, A2, g.g[1] + ps1, A2, ld, m0, M});
  {   // LayerNorm backward in place: dL/dn -> dL/dh, affine gradients in fixed point
    float* dhg = g.g[1] + ps1 + m0 + lane;
    ln_bwd_row<LN_MAXF>(
        CH_H1, valid, mean, rstd, g.gamma, red1, red2, [&](int c) { return A2[c * CH_TM + lane]; },
        [&](int c) { return H2[c * CH_TM + lane]; },
        [&](int c, float v) {
          dhg[(size_t)c * ld] = v;
          A2[c * CH_TM + lane] = v;
        },
        g.dgamma ? g.acc : nullptr);
  }
  if (g.dgamma) {   // the last CTA converts the sums, adds them to the gradients and clears the slot (as ln_bwd_kernel)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(g.cnt, 1u) == gridDim.x * gridDim.y - 1 ? 1u : 0u;
    __syncthreads();
    if (s_last) {
      __threadfence();
      for (int e = threadIdx.x; e < 2 * CH_H1; e += CH_THREADS) {
        const float v = det_unfix(__ldcg(g.acc + e));
        g.acc[e] = 0ull;
        atomicAdd(e < CH_H1 ? g.dgamma + e : g.dbeta + (e - CH_H1), v);
      }
      if (threadIdx.x == 0) *g.cnt = 0u;
    }
  }
  __syncthreads();
  chain_layer<false>(A2, g.W[1], CH_H0, CH_H1, CH_H0, wbuf,
                     DactEp{1.0f, g.m1 + ps0, g.keep_inv, 0.f, A1, g.g[0] + ps0, nullptr, ld, m0, M});
}

}  // namespace cvg
