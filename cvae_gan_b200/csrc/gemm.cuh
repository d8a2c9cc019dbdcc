// cvaegan_b200 - tiled FP32 GEMM kernels with fused prologues / epilogues.
//
// Data layout in HBM: every activation / gradient matrix is FEATURE-MAJOR, [features][ld] with the
// batch row index contiguous (ld = rows rounded up to 64).  With that layout all three GEMMs of a
// layer read both operands with 16-byte coalesced loads and no transposition:
//   forward   Y[n][m]  = sum_r A[r][m] * W[n][r]          (gemm_mn_kernel<true>)
//   backward  dA[j][m] = sum_r dY[r][m] * W[r][j]         (gemm_mn_kernel<false>)
//   weight    dW[n][k] = sum_m dY[n][m] * A[k][m]         (gemm_dw_kernel)
// Operand transforms (BatchNorm+LeakyReLU of the producing layer, reparameterisation, BatchNorm
// backward) are applied while the tile is staged into shared memory, so normalised activations are
// never written to memory; epilogues fuse bias / one-hot column / 1/sigma / activation / dropout /
// batch-moment accumulation / KL / activation derivatives.
#pragma once
#include <cstddef>
#include "common.cuh"
#include "comm_nvl.cuh"

namespace cvg {

constexpr int TBM = 64;   // tile rows (batch)
constexpr int TBN = 64;   // tile cols (features)
constexpr int TBK = 16;   // reduction chunk
constexpr int GEMM_THREADS = 256;
constexpr int RED_LD = TBM + 4;   // padded row of the split-K partial tiles

enum { OP_PLAIN = 0, OP_BN_ACT = 1, OP_REPARAM = 2, OP_BN_BWD = 3, OP_CONST = 4 };
enum { ACT_NONE = 0, ACT_LRELU = 1, ACT_RELU = 2, ACT_SIGMOID = 3 };
enum { EP_LINEAR = 0, EP_DBN = 1, EP_DACT = 2, EP_STORE = 3, EP_REPARAM_BWD = 4 };

// Reference to one BatchNorm layer's statistics (SURVEY appendix A.2).
struct BnRef {
  const double* fstats = nullptr;  // [pass][2][C]  sum h, sum h^2 over the (global) batch   (train)
  long long sf = 0;
  const double* bstats = nullptr;  // [pass][2][C]  sum dy, sum dy*xhat                       (backward)
  long long sb = 0;
  const float* gamma = nullptr;
  const float* beta = nullptr;
  float* rmean = nullptr;          // running stats: source in eval mode, update target in train mode
  float* rvar = nullptr;
  int C = 0;
  int eval = 0;
  int update_running = 0;          // CTA (0,0,0) applies the momentum update for all passes, in order
  // data parallel, exchange folded into the kernels (comm_nvl.cuh): the sums named by `poll_which` (1 fstats, 2 bstats)
  // are still in flight as `poll_npass` passes of LL packets; this kernel is their first reader
  int poll = 0;                    // which | passes << 4 | first pass << 12 | via_lead << 20  (NvlDev pointer: GemmArgs / DwArgs ::nvl)
};

struct Operand {
  int kind = OP_PLAIN;
  int rows = 0;                    // feature rows available (reduction length)
  const float* p = nullptr;        // [rows][ld] (+ pass * sp)
  long long sp = 0;
  const float* h = nullptr;        // OP_BN_BWD: pre-BN activations of the same layer
  long long sh = 0;
  const float* mu = nullptr;       // OP_REPARAM (pass == reparam_pass): mu + eps * exp(0.5 * logvar)
  const float* lv = nullptr;
  const float* eps = nullptr;
  int reparam_pass = -1;
  float cst = 0.f;                 // OP_CONST
  BnRef bn;
};

// number of float constants an operand keeps in shared memory
__host__ __device__ inline int operand_const_floats(const Operand& o) {
  if (o.kind == OP_BN_ACT) return 3 * o.bn.C;
  if (o.kind == OP_BN_BWD) return 5 * o.bn.C;
  return 0;
}

struct GemmArgs {
  int M = 0, ld = 0, npass = 1;
  float Bg = 1.f;                  // global batch rows (M * world)
  int R = 0;                       // reduction length
  int N = 0;                       // output features
  Operand a;
  const float* W = nullptr;        // <true>: W[n*ldw + wcol0 + r]   <false>: W[r*ldw + wcol0 + n]
  int ldw = 0, wcol0 = 0;
  float bn_eps = 1e-5f, momentum = 0.1f, slope = 0.2f;
  // ---- epilogue ----
  int ekind = EP_LINEAR;
  const float* bias = nullptr;     // [N]
  const float* wlabel = nullptr;   // one-hot column: bias'[n] = bias[n] + scale * wlabel[n*ldwl]
  int ldwl = 0;
  const float* scale = nullptr;    // per-pass device scalar (1/sigma) or null
  int act = ACT_NONE;
  const uint8_t* mask = nullptr;   // [N][ld] keep mask (+ pass * smask)
  long long smask = 0;
  float keep_inv = 1.f;
  float* Y = nullptr;              // [N][ld] (+ pass * sY)
  long long sY = 0;
  int accumulate = 0;
  double* ostats = nullptr;        // [pass][2][N]
  long long sostats = 0;
  double* osum = nullptr;          // [pass] sum of all outputs
  double* kl_acc = nullptr;        // KL accumulation over the (mu | logvar) head outputs
  int kl_split = 0;
  const float* prev = nullptr;     // EP_DBN: h_prev ; EP_DACT: a_prev   [N][ld] (+ pass * sprev)
  long long sprev = 0;
  BnRef prev_bn;                   // EP_DBN
  const float* mu = nullptr;       // EP_REPARAM_BWD
  const float* lv = nullptr;
  const float* eps = nullptr;
  float kl_coef = 0.f;
  int only_pass = -1;              // if >= 0 the grid has one pass slot mapped to this pass index
  const NvlDev* nvl = nullptr;     // data parallel with the exchange folded in: polling (a.bn.poll) and / or ...
  int push = 0;                    // ... the last CTA sends ostats to every peer (nvl_push_stats_tail)
};
// what a step-program op record carries of it (mega.cuh): everything before the folded-exchange fields
constexpr size_t GEMM_ARGS_OP_BYTES = offsetof(GemmArgs, nvl);

struct DwArgs {
  int M = 0, ld = 0, npass = 1;
  float Bg = 1.f;
  int N = 0, K = 0;                // dW is [N][K] inside a [N][ldw] matrix at column wcol0
  Operand p;                       // dY operand, rows = N
  Operand q;                       // activation operand, rows = K
  float* dW = nullptr;
  long long sdW = 0;               // per-pass stride (spectral-norm layers keep per-pass gradients)
  int ldw = 0, wcol0 = 0;
  float* db = nullptr;             // [N] or null
  int label_col = -1;              // one-hot column receives the bias gradient as well
  float* dgamma = nullptr;         // BatchNorm affine grads come straight from p.bn.bstats
  float* dbeta = nullptr;
  int add_affine = 0;
  int rows_per_cta = 256;
  float bn_eps = 1e-5f, slope = 0.2f;
  const NvlDev* nvl = nullptr;     // set when p.bn.poll / q.bn.poll is
};

// ------------------------------------------------------------------------------------------------
// per-CTA BatchNorm constants
// ------------------------------------------------------------------------------------------------
// A feature's pair of batch sums, [sum (C) | second sum (C)] of `which` (1 forward, 2 backward).
// nvl != null: this CTA takes in-flight sums from the LL packets instead of the buffer.
__device__ __forceinline__ void bn_stat2(const BnRef& bn, int which, int pass, int c, const NvlDev* nvl, double& s1,
                                         double& s2) {
  const double* base = which == 1 ? bn.fstats : bn.bstats;
  const long long stride = which == 1 ? bn.sf : bn.sb;
  if (nvl == nullptr || (bn.poll & 15) != which) {
    s1 = __ldcg(base + (long long)pass * stride + c);        // L2: another CTA of this launch may have just written them
    s2 = __ldcg(base + (long long)pass * stride + bn.C + c);
    return;
  }
  const int p0 = (bn.poll >> 12) & 255;           // the pushed group's first pass: its slot holds the exchange number
  const unsigned long long ep = (unsigned long long)base[(long long)p0 * stride + stride - 1];
  const long long e = (long long)(pass - p0) * 2 * bn.C + c;
  nvl_poll_f64x2(*nvl, (unsigned int)ep, (int)(ep & 1ull), e, e + bn.C, s1, s2);
}

// The CTA that owns the write-back: global sums of passes [p0, p0 + np) from the packets into the buffer.
__device__ __forceinline__ void bn_poll_writeback(const BnRef& bn, int p0, int np, const NvlDev* nvl) {
  const int which = bn.poll & 15;
  double* base = const_cast<double*>(which == 1 ? bn.fstats : bn.bstats);
  const long long stride = which == 1 ? bn.sf : bn.sb;
  for (int i = threadIdx.x; i < np * bn.C; i += blockDim.x) {
    const int ps = p0 + i / bn.C, c = i % bn.C;
    double s1, s2;
    bn_stat2(bn, which, ps, c, nvl, s1, s2);
    base[(long long)ps * stride + c] = s1;
    base[(long long)ps * stride + bn.C + c] = s2;
  }
}

// With many ranks every CTA polling world x 2 C packets itself costs more L2 bandwidth than the exchange is worth
// (8 ranks, 512 CTAs, C = 256: 33 MB per launch).  via_lead: only the write-back CTA polls; it then publishes the exchange
// number next to the sums (slot[stride - 2]) and the other CTAs of that pass wait for it and read the 4 KB of global sums.
// A waiting CTA always has a higher linear index than its write-back CTA, which therefore was dispatched before it.
__device__ __forceinline__ void bn_publish(const BnRef& bn, int p0, int np) {
  const int which = bn.poll & 15;
  double* base = const_cast<double*>(which == 1 ? bn.fstats : bn.bstats);
  const long long stride = which == 1 ? bn.sf : bn.sb;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const double ep = base[(long long)((bn.poll >> 12) & 255) * stride + stride - 1];
    for (int p = p0; p < p0 + np; ++p) *reinterpret_cast<volatile double*>(base + (long long)p * stride + stride - 2) = ep;
  }
}
__device__ __forceinline__ void bn_wait_published(const BnRef& bn, int pass) {
  const int which = bn.poll & 15;
  const double* base = which == 1 ? bn.fstats : bn.bstats;
  const long long stride = which == 1 ? bn.sf : bn.sb;
  if (threadIdx.x == 0) {
    const double ep = base[(long long)((bn.poll >> 12) & 255) * stride + stride - 1];
    const long long t0 = clock64();
    while (*reinterpret_cast<const volatile double*>(base + (long long)pass * stride + stride - 2) != ep)
      if (clock64() - t0 > 120000000000ll) __trap();
    __threadfence();
  }
  __syncthreads();
}

__device__ __forceinline__ void bn_mean_rstd(const BnRef& bn, int pass, int c, float Bg, float eps, float& mean,
                                             float& rstd, float& var_biased, const NvlDev* poll = nullptr) {
  if (bn.eval) {
    mean = bn.rmean[c];
    var_biased = bn.rvar[c];
  } else {
    const double inv = 1.0 / (double)Bg;
    double s1, s2;
    bn_stat2(bn, 1, pass, c, poll, s1, s2);
    double m = s1 * inv;
    double v = s2 * inv - m * m;
    if (v < 0.0) v = 0.0;
    mean = (float)m;
    var_biased = (float)v;
  }
  rstd = 1.0f / sqrtf(var_biased + eps);
}

// fills cs[] for an operand; all threads of the CTA participate; caller syncs afterwards
template <int KIND>
__device__ __forceinline__ void operand_consts(const Operand& o, int pass, float Bg, float eps, float* cs,
                                               const NvlDev* poll = nullptr) {
  if (KIND == OP_BN_ACT) {
    const int C = o.bn.C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float mean, rstd, var;
      bn_mean_rstd(o.bn, pass, c, Bg, eps, mean, rstd, var, poll);
      // y = (h - mean) * (gamma * rstd) + beta : the subtraction is exact-ish even when |mean| >> std
      cs[c] = o.bn.gamma[c] * rstd;
      cs[C + c] = o.bn.beta[c];
      cs[2 * C + c] = mean;
    }
  } else if (KIND == OP_BN_BWD) {
    const int C = o.bn.C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float mean, rstd, var;
      double b1, b2;
      bn_stat2(o.bn, 2, pass, c, poll, b1, b2);     // first: the sums that may still be in flight
      bn_mean_rstd(o.bn, pass, c, Bg, eps, mean, rstd, var, poll);
      cs[c] = o.bn.gamma[c] * rstd;                 // c1
      cs[C + c] = (float)(b1 / (double)Bg);         // c2 = dbeta / B
      cs[2 * C + c] = (float)(b2 / (double)Bg);     // c3 = dgamma / B
      cs[3 * C + c] = mean;
      cs[4 * C + c] = rstd;
    }
  }
}

// BatchNorm running-stat momentum update, done once (CTA 0) by the kernel that consumes the layer.
__device__ __forceinline__ void bn_update_running(const BnRef& bn, int npass, float Bg, float momentum) {
  for (int c = threadIdx.x; c < bn.C; c += blockDim.x) {
    float rm = bn.rmean[c], rv = bn.rvar[c];
    for (int p = 0; p < npass; ++p) {
      const double* s = bn.fstats + (long long)p * bn.sf;
      double m = s[c] / (double)Bg;
      double v = s[bn.C + c] / (double)Bg - m * m;
      if (v < 0.0) v = 0.0;
      double unb = v * ((double)Bg / ((double)Bg - 1.0));
      rm = (1.0f - momentum) * rm + momentum * (float)m;
      rv = (1.0f - momentum) * rv + momentum * (float)unb;
    }
    bn.rmean[c] = rm;
    bn.rvar[c] = rv;
  }
}

__device__ __forceinline__ float act_lrelu(float x, float slope) { return x > 0.f ? x : x * slope; }

// Epilogue pieces shared by gemm_mn_kernel and the fused row-tile chains (chain.cuh), which must reproduce its results bit
// for bit: one definition of each expression, so the two cannot drift apart.
// EP_LINEAR: bias of output feature n with the one-hot label column folded in (scale = 1/sigma or 1)
__device__ __forceinline__ float ep_bias(const float* bias, const float* wlabel, int ldwl, int n, float scale) {
  float b = bias ? bias[n] : 0.f;
  if (wlabel) b += scale * wlabel[(size_t)n * ldwl];
  return b;
}
__device__ __forceinline__ float ep_linear(float acc, float scale, float b) { return fmaf(acc, scale, b); }
__device__ __forceinline__ float ep_act(float y, int act, float slope) {
  if (act == ACT_LRELU) return act_lrelu(y, slope);
  if (act == ACT_RELU) return fmaxf(y, 0.f);
  if (act == ACT_SIGMOID) return 1.0f / (1.0f + expf(-y));
  return y;
}
__device__ __forceinline__ float ep_dropout(float y, unsigned char keep, float keep_inv) { return keep ? y * keep_inv : 0.f; }
// EP_DACT: input gradient of a Linear -> gradient w.r.t. the pre-activation of the layer below (dropout, then activation)
__device__ __forceinline__ float ep_keep(unsigned char keep, float keep_inv) { return keep ? keep_inv : 0.f; }
__device__ __forceinline__ float ep_dact(float acc, float scale, float keep, float a_prev, float neg) {
  const float d = acc * scale * keep;
  return a_prev > 0.f ? d : d * neg;
}
// ((p0 + p1) + p2) + p3: the four k-group partials of one output element, in this order
__device__ __forceinline__ float4 ksum4(float4 v, float4 w1, float4 w2, float4 w3) {
  v.x += w1.x; v.y += w1.y; v.z += w1.z; v.w += w1.w;
  v.x += w2.x; v.y += w2.y; v.z += w2.z; v.w += w2.w;
  v.x += w3.x; v.y += w3.y; v.z += w3.z; v.w += w3.w;
  return v;
}

// Loads 4 consecutive batch rows (m..m+3) of feature row r of an operand, transformed; rows >= M and
// feature rows >= o.rows read as 0.
// Operand staging is split in two so that global loads stay in flight across the FFMA block: load_raw only
// ISSUES the loads (no dependent arithmetic), finish_operand applies the transform right before the value is
// stored to shared memory one chunk later.  Rows >= M and feature rows >= o.rows read as 0.
struct Raw {
  float4 a, b, c;
};

template <int KIND>
__device__ __forceinline__ void load_raw(const Operand& o, int pass, int r, int m, int M, int ld, Raw& w) {
  if (r >= o.rows || m >= M) return;
  const size_t off = (size_t)r * ld + m;
  switch (KIND) {
    case OP_PLAIN:
    case OP_BN_ACT:
      w.a = ld4(o.p + (long long)pass * o.sp + off);
      break;
    case OP_REPARAM:
      if (pass == o.reparam_pass) {
        w.a = ld4(o.mu + off);
        w.b = ld4(o.lv + off);
        w.c = ld4(o.eps + off);
      } else {
        w.a = ld4(o.p + (long long)pass * o.sp + off);
      }
      break;
    case OP_BN_BWD:
      w.a = ld4(o.p + (long long)pass * o.sp + off);
      w.b = ld4(o.h + (long long)pass * o.sh + off);
      break;
    case OP_CONST:
      break;
  }
}

template <int KIND>
__device__ __forceinline__ float4 finish_operand(const Operand& o, const float* cs, int pass, int r, int m, int M,
                                                 float slope, const Raw& w) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (r >= o.rows || m >= M) return v;
  switch (KIND) {
    case OP_PLAIN:
      v = w.a;
      break;
    case OP_BN_ACT: {
      const float sc = cs[r], sh = cs[o.bn.C + r], mean = cs[2 * o.bn.C + r];
      v.x = act_lrelu(fmaf(w.a.x - mean, sc, sh), slope);
      v.y = act_lrelu(fmaf(w.a.y - mean, sc, sh), slope);
      v.z = act_lrelu(fmaf(w.a.z - mean, sc, sh), slope);
      v.w = act_lrelu(fmaf(w.a.w - mean, sc, sh), slope);
    } break;
    case OP_REPARAM:
      if (pass == o.reparam_pass) {
        v.x = w.a.x + w.c.x * expf(0.5f * w.b.x);
        v.y = w.a.y + w.c.y * expf(0.5f * w.b.y);
        v.z = w.a.z + w.c.z * expf(0.5f * w.b.z);
        v.w = w.a.w + w.c.w * expf(0.5f * w.b.w);
      } else {
        v = w.a;
      }
      break;
    case OP_BN_BWD: {
      const int C = o.bn.C;
      const float c1 = cs[r], c2 = cs[C + r], c3 = cs[2 * C + r], mean = cs[3 * C + r], rstd = cs[4 * C + r];
      v.x = c1 * (w.a.x - c2 - (w.b.x - mean) * rstd * c3);
      v.y = c1 * (w.a.y - c2 - (w.b.y - mean) * rstd * c3);
      v.z = c1 * (w.a.z - c2 - (w.b.z - mean) * rstd * c3);
      v.w = c1 * (w.a.w - c2 - (w.b.w - mean) * rstd * c3);
    } break;
    case OP_CONST:
      v = make_float4(o.cst, o.cst, o.cst, o.cst);
      break;
  }
  if (m + 3 >= M) {
    if (m + 1 >= M) v.y = 0.f;
    if (m + 2 >= M) v.z = 0.f;
    if (m + 3 >= M) v.w = 0.f;
  }
  return v;
}

// ------------------------------------------------------------------------------------------------
// C[m][n] = sum_r A[r][m] * B[r][n]   (64 x 64 tile, 256 threads, 4 x 4 per thread)
// ------------------------------------------------------------------------------------------------
template <bool WT, int AK, int EK>
__global__ void __launch_bounds__(GEMM_THREADS, 2) gemm_mn_kernel(const GemmArgs g) {
  extern __shared__ __align__(16) float dyn_smem[];
  __shared__ __align__(16) float As[2][TBK][TBM];
  __shared__ __align__(16) float Bs[2][TBK][TBN];

  const int tid = threadIdx.x;
  const int pass = g.only_pass >= 0 ? g.only_pass : (int)blockIdx.z;
  const int m0 = blockIdx.x * TBM, n0 = blockIdx.y * TBN;
  float* cs_a = dyn_smem;                                  // operand constants
  float* cs_e = dyn_smem + operand_const_floats(g.a);      // epilogue constants (EP_DBN: 4 * C)

  // ---- preamble: per-feature constants ---------------------------------------------------------
  // in-flight batch sums (data parallel): CTA (0,0,0) lands every pass in the buffer, the others read the packets
  const NvlDev* poll_a = ((AK == OP_BN_ACT || AK == OP_BN_BWD) && g.a.bn.poll) ? g.nvl : nullptr;
  if (poll_a && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) {
    bn_poll_writeback(g.a.bn, (g.a.bn.poll >> 12) & 255, (g.a.bn.poll >> 4) & 255, poll_a);
    if (g.a.bn.poll >> 20) bn_publish(g.a.bn, (g.a.bn.poll >> 12) & 255, (g.a.bn.poll >> 4) & 255);
    __syncthreads();
    poll_a = nullptr;
  } else if (poll_a && (g.a.bn.poll >> 20)) {
    bn_wait_published(g.a.bn, pass);
    poll_a = nullptr;
  }
  operand_consts<AK>(g.a, pass, g.Bg, g.bn_eps, cs_a, poll_a);
  if (EK == EP_DBN) {
    const int C = g.prev_bn.C;
    for (int c = tid; c < C; c += GEMM_THREADS) {
      float mean, rstd, var;
      bn_mean_rstd(g.prev_bn, pass, c, g.Bg, g.bn_eps, mean, rstd, var);
      cs_e[c] = g.prev_bn.gamma[c] * rstd;
      cs_e[C + c] = g.prev_bn.beta[c];
      cs_e[2 * C + c] = mean;
      cs_e[3 * C + c] = rstd;
    }
  }
  if (AK == OP_BN_ACT && g.a.bn.update_running && !g.a.bn.eval && blockIdx.x == 0 && blockIdx.y == 0 &&
      blockIdx.z == 0) {
    bn_update_running(g.a.bn, g.npass, g.Bg, g.momentum);
  }
  __syncthreads();

  // ---- staging maps ------------------------------------------------------------------------------
  const int a_r = tid >> 4, a_m = (tid & 15) * 4;
  const bool wvec = ((g.ldw | g.wcol0) & 3) == 0;
  const int bt_n = tid & 63, bt_kg = tid >> 6;        // WT:  W[n][r..r+3] -> Bs[r..r+3][n]
  const int bn_r = tid >> 4, bn_n = (tid & 15) * 4;   // !WT: W[r][n..n+3] -> Bs[r][n..n+3]

  auto load_b = [&](int r0) -> float4 {
    float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
    if (WT) {
      const int n = n0 + bt_n, r = r0 + bt_kg * 4;
      if (n < g.N) {
        const float* src = g.W + (size_t)n * g.ldw + g.wcol0 + r;
        if (wvec && r + 3 < g.R) {
          w = ld4(src);
        } else {
          if (r < g.R) w.x = src[0];
          if (r + 1 < g.R) w.y = src[1];
          if (r + 2 < g.R) w.z = src[2];
          if (r + 3 < g.R) w.w = src[3];
        }
      }
    } else {
      const int r = r0 + bn_r, n = n0 + bn_n;
      if (r < g.R) {
        const float* src = g.W + (size_t)r * g.ldw + g.wcol0 + n;
        if (wvec && n + 3 < g.N) {
          w = ld4(src);
        } else {
          if (n < g.N) w.x = src[0];
          if (n + 1 < g.N) w.y = src[1];
          if (n + 2 < g.N) w.z = src[2];
          if (n + 3 < g.N) w.w = src[3];
        }
      }
    }
    return w;
  };
  auto store_b = [&](int buf, float4 w) {
    if (WT) {
      Bs[buf][bt_kg * 4 + 0][bt_n] = w.x;
      Bs[buf][bt_kg * 4 + 1][bt_n] = w.y;
      Bs[buf][bt_kg * 4 + 2][bt_n] = w.z;
      Bs[buf][bt_kg * 4 + 3][bt_n] = w.w;
    } else {
      st4(&Bs[buf][bn_r][bn_n], w);
    }
  };

  // Split-K inside the CTA: four 64-thread groups each take 4 of the 16 k-steps of a chunk with an 8 x 8
  // register tile (64 independent FFMAs per 4 LDS.128), which hides the shared-memory round trip that a
  // 4 x 4 tile with two warps per scheduler cannot.  Partials meet in shared memory before the epilogue.
  float acc8[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc8[i][j] = 0.f;
  const int grp = tid >> 6, t64 = tid & 63;
  const int tm8 = (t64 & 7) * 4, tn8 = (t64 >> 3) * 4;

  const int tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
  const int nchunks = (g.R + TBK - 1) / TBK;

  // Register prefetch runs TWO chunks ahead of the FFMA block (an L2 round trip is longer than one
  // chunk of math when only one or two CTAs are resident per SM).
  auto compute = [&](int cur) {
#pragma unroll
    for (int q = 0; q < TBK / 4; ++q) {
      const int kk = grp * (TBK / 4) + q;
      const float4 a0 = ld4(&As[cur][kk][tm8]), a1 = ld4(&As[cur][kk][32 + tm8]);
      const float4 b0 = ld4(&Bs[cur][kk][tn8]), b1 = ld4(&Bs[cur][kk][32 + tn8]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc8[i][j] = fmaf(av[i], bv[j], acc8[i][j]);
    }
  };
  auto gload = [&](int c, Raw& xa, float4& xb) {
    load_raw<AK>(g.a, pass, c * TBK + a_r, m0 + a_m, g.M, g.ld, xa);
    xb = load_b(c * TBK);
  };
  auto sstore = [&](int buf, int c, const Raw& xa, const float4& xb) {
    st4(&As[buf][a_r][a_m], finish_operand<AK>(g.a, cs_a, pass, c * TBK + a_r, m0 + a_m, g.M, g.slope, xa));
    store_b(buf, xb);
  };
  Raw ra;
  float4 rb;
  gload(0, ra, rb);
  sstore(0, 0, ra, rb);
  __syncthreads();
  for (int c = 0; c < nchunks; ++c) {
    const int cur = c & 1;
    if (c + 1 < nchunks) gload(c + 1, ra, rb);     // loads stay in flight across the FFMA block
    compute(cur);
    if (c + 1 < nchunks) sstore(cur ^ 1, c + 1, ra, rb);
    __syncthreads();
  }

  // ---- reduce the four K-slices: part[g][n][m] (m contiguous, row padded to RED_LD) ----------------------
  float* part = dyn_smem + ((operand_const_floats(g.a) + ((EK == EP_DBN) ? 4 * g.prev_bn.C : 0) + 3) & ~3);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int n = (j < 4) ? tn8 + j : 32 + tn8 + (j - 4);
    float* row = part + ((size_t)grp * TBN + n) * RED_LD;
    st4(row + tm8, make_float4(acc8[0][j], acc8[1][j], acc8[2][j], acc8[3][j]));
    st4(row + 32 + tm8, make_float4(acc8[4][j], acc8[5][j], acc8[6][j], acc8[7][j]));
  }
  __syncthreads();
  float acc[4][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 v = ksum4(ld4(part + (size_t)(tn + j) * RED_LD + tm), ld4(part + ((size_t)1 * TBN + tn + j) * RED_LD + tm),
                           ld4(part + ((size_t)2 * TBN + tn + j) * RED_LD + tm), ld4(part + ((size_t)3 * TBN + tn + j) * RED_LD + tm));
    acc[0][j] = v.x; acc[1][j] = v.y; acc[2][j] = v.z; acc[3][j] = v.w;
  }

  // ---- epilogue ------------------------------------------------------------------------------------
  const int m = m0 + tm;
  const float scale = g.scale ? g.scale[pass] : 1.0f;
  const bool rowv[4] = {m < g.M, m + 1 < g.M, m + 2 < g.M, m + 3 < g.M};
  double tot = 0.0, klsum = 0.0;

#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = n0 + tn + j;
    const bool nvalid = n < g.N;   // warp-uniform per half-warp (tn shared by 16 lanes)
    float y[4] = {acc[0][j], acc[1][j], acc[2][j], acc[3][j]};
    // batch moments are accumulated in double from the first addition: for a single-class batch the
    // pre-activations have |mean| >> std, and E[x^2] - mean^2 cancels ~mean^2/var digits
    double s1 = 0.0, s2 = 0.0;
    if (nvalid) {
      const size_t off = (size_t)n * g.ld + m;
      if (EK == EP_LINEAR) {
        const float b = ep_bias(g.bias, g.wlabel, g.ldwl, n, scale);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = ep_linear(y[i], scale, b);
        if (g.kl_acc) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (rowv[i]) klsum += (n < g.kl_split) ? 0.5 * (double)y[i] * (double)y[i]
                                                   : -0.5 * (1.0 + (double)y[i] - (double)expf(y[i]));
        }
        if (g.ostats) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (rowv[i]) { s1 += (double)y[i]; s2 += (double)y[i] * (double)y[i]; }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = ep_act(y[i], g.act, g.slope);
        if (g.mask) {
          const uchar4 mk = *reinterpret_cast<const uchar4*>(g.mask + (long long)pass * g.smask + off);
          y[0] = ep_dropout(y[0], mk.x, g.keep_inv);
          y[1] = ep_dropout(y[1], mk.y, g.keep_inv);
          y[2] = ep_dropout(y[2], mk.z, g.keep_inv);
          y[3] = ep_dropout(y[3], mk.w, g.keep_inv);
        }
        if (g.osum) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (rowv[i]) tot += (double)y[i];
        }
        st4(g.Y + (long long)pass * g.sY + off, make_float4(y[0], y[1], y[2], y[3]));
      } else if (EK == EP_DBN) {
        const int C = g.prev_bn.C;
        const float4 h = ld4(g.prev + (long long)pass * g.sprev + off);
        const float hh[4] = {h.x, h.y, h.z, h.w};
        const float sc = cs_e[n], sh = cs_e[C + n], mean = cs_e[2 * C + n], rstd = cs_e[3 * C + n];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float pre = fmaf(hh[i] - mean, sc, sh);
          const float dy = rowv[i] ? (pre > 0.f ? y[i] : y[i] * g.slope) : 0.f;
          y[i] = dy;
          s1 += (double)dy;
          s2 += (double)(dy * ((hh[i] - mean) * rstd));
        }
        st4(g.Y + (long long)pass * g.sY + off, make_float4(y[0], y[1], y[2], y[3]));
      } else if (EK == EP_DACT) {
        const float4 ap = ld4(g.prev + (long long)pass * g.sprev + off);
        const float aa[4] = {ap.x, ap.y, ap.z, ap.w};
        float keep[4] = {1.f, 1.f, 1.f, 1.f};
        if (g.mask) {
          const uchar4 mk = *reinterpret_cast<const uchar4*>(g.mask + (long long)pass * g.smask + off);
          keep[0] = ep_keep(mk.x, g.keep_inv);
          keep[1] = ep_keep(mk.y, g.keep_inv);
          keep[2] = ep_keep(mk.z, g.keep_inv);
          keep[3] = ep_keep(mk.w, g.keep_inv);
        }
        const float neg = (g.act == ACT_LRELU) ? g.slope : 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = ep_dact(y[i], scale, keep[i], aa[i], neg);
        st4(g.Y + (long long)pass * g.sY + off, make_float4(y[0], y[1], y[2], y[3]));
      } else if (EK == EP_STORE) {
        float* dst = g.Y + (long long)pass * g.sY + off;
        float4 o = make_float4(y[0] * scale, y[1] * scale, y[2] * scale, y[3] * scale);
        if (g.accumulate) {
          const float4 old = ld4(dst);
          o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
        }
        st4(dst, o);
      } else if (EK == EP_REPARAM_BWD) {
        // y = dL/dz_enc for latent feature n.  dmu = dz + kl_coef*mu ; dlogvar = dz*eps*0.5*exp(0.5 lv)
        // + kl_coef*0.5*(exp(lv)-1)   (SURVEY appendix A.7)
        const float4 mu = ld4(g.mu + off), lv = ld4(g.lv + off), e = ld4(g.eps + off);
        const float mm[4] = {mu.x, mu.y, mu.z, mu.w}, ll[4] = {lv.x, lv.y, lv.z, lv.w}, ee[4] = {e.x, e.y, e.z, e.w};
        float dmu[4], dlv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          dmu[i] = rowv[i] ? y[i] + g.kl_coef * mm[i] : 0.f;
          dlv[i] = rowv[i] ? y[i] * ee[i] * 0.5f * expf(0.5f * ll[i]) + g.kl_coef * 0.5f * (expf(ll[i]) - 1.0f) : 0.f;
        }
        st4(g.Y + off, make_float4(dmu[0], dmu[1], dmu[2], dmu[3]));
        st4(g.Y + (size_t)(g.N + n) * g.ld + m, make_float4(dlv[0], dlv[1], dlv[2], dlv[3]));
      }
    }
    if (g.ostats) {   // uniform branch; the 16 lanes of a half-warp share column n
      s1 = half_warp_sum_d(s1);
      s2 = half_warp_sum_d(s2);
      if ((tid & 15) == 0 && nvalid) {
        double* st = g.ostats + (long long)pass * g.sostats;
        atomicAdd(st + n, s1);
        atomicAdd(st + g.N + n, s2);
      }
    }
  }
  if (g.osum) {
    tot = warp_sum_d(tot);
    if ((tid & 31) == 0) atomicAdd(g.osum + pass, tot);
  }
  if (g.kl_acc) {
    klsum = warp_sum_d(klsum);
    if ((tid & 31) == 0) atomicAdd(g.kl_acc, klsum);
  }
  if (g.push)
    nvl_push_stats_tail(*g.nvl, g.ostats + (long long)(g.only_pass > 0 ? g.only_pass : 0) * g.sostats, g.sostats, (int)gridDim.z, g.N,
                        gridDim.x * gridDim.y * gridDim.z);
}

// ------------------------------------------------------------------------------------------------
// dW[n][k] += sum_m P[n][m] * Q[k][m]   (64 x 64 tile of dW per CTA, batch split over blockIdx.z)
// ------------------------------------------------------------------------------------------------
constexpr int DW_MC = 32;          // batch rows per staged chunk
constexpr int DW_LDS = DW_MC + 4;  // padded row (conflict-free 128-bit reads across rows)

// Deterministic split-batch reduction: each CTA adds its partial tile to `acc` ([tile][pass] slots of DW_PART int64) in
// fixed point (DET_FIX_SCALE), where addition is exact and so independent of the order the CTAs finish in; the last CTA of
// the tile (ticket on `tile_cnt`) converts the sums, adds them to the gradients and clears the slot and the counter.
constexpr int DW_PART = 64 * 64 + 64;   // dW tile + bias sums
constexpr double DET_FIX_SCALE = 1099511627776.0;   // 2^40: resolution 9.1e-13, range +-8.4e6
__device__ __forceinline__ unsigned long long det_fix(float v) {
  return (unsigned long long)__double2ll_rn((double)v * DET_FIX_SCALE);
}
__device__ __forceinline__ float det_unfix(unsigned long long v) { return (float)((double)(long long)v / DET_FIX_SCALE); }

template <int PK, int QK>
__global__ void __launch_bounds__(GEMM_THREADS, 2) gemm_dw_kernel(const DwArgs g, int nsplit, unsigned long long* acc64, unsigned* tile_cnt) {
  extern __shared__ __align__(16) float dyn_smem[];
  float* Ps = dyn_smem;                            // [2][64][DW_LDS]
  float* Qs = Ps + 2 * 64 * DW_LDS;                // [2][64][DW_LDS]
  float* cs_p = Qs + 2 * 64 * DW_LDS;
  float* cs_q = cs_p + operand_const_floats(g.p);

  const int tid = threadIdx.x;
  const int pass = blockIdx.z / nsplit, split = blockIdx.z % nsplit;
  const int k0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
  const int mbeg = split * g.rows_per_cta;
  const int mend = min(g.M, mbeg + g.rows_per_cta);

  const NvlDev* poll_p = ((PK == OP_BN_ACT || PK == OP_BN_BWD) && g.p.bn.poll) ? g.nvl : nullptr;
  const NvlDev* poll_q = ((QK == OP_BN_ACT || QK == OP_BN_BWD) && g.q.bn.poll) ? g.nvl : nullptr;
  if ((poll_p || poll_q) && blockIdx.x == 0 && blockIdx.y == 0 && split == 0) {   // this pass's write-back CTA
    if (poll_p) { bn_poll_writeback(g.p.bn, pass, 1, poll_p); if (g.p.bn.poll >> 20) bn_publish(g.p.bn, pass, 1); }
    if (poll_q) { bn_poll_writeback(g.q.bn, pass, 1, poll_q); if (g.q.bn.poll >> 20) bn_publish(g.q.bn, pass, 1); }
    __syncthreads();
    poll_p = poll_q = nullptr;
  } else {
    if (poll_p && (g.p.bn.poll >> 20)) { bn_wait_published(g.p.bn, pass); poll_p = nullptr; }
    if (poll_q && (g.q.bn.poll >> 20)) { bn_wait_published(g.q.bn, pass); poll_q = nullptr; }
  }
  operand_consts<PK>(g.p, pass, g.Bg, g.bn_eps, cs_p, poll_p);
  operand_consts<QK>(g.q, pass, g.Bg, g.bn_eps, cs_q, poll_q);
  // BatchNorm affine gradients are exactly the backward batch sums (appendix A.2): dbeta = sum dy,
  // dgamma = sum dy*xhat.  One CTA per pass adds them to the gradient buffer.
  // (added by the last CTA of tile (0, 0), pass by pass)
  __syncthreads();

  const int l_row = tid >> 3, l_m = (tid & 7) * 4;   // two rows per thread: l_row, l_row + 32
  const int tk = tid & 15, tn = tid >> 4;            // thread computes rows tn+16i (n) x tk+16j (k)
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float bsum[4] = {0.f, 0.f, 0.f, 0.f};
  const bool do_bias = (g.db != nullptr || g.label_col >= 0) && blockIdx.x == 0 && tk == 0;

  struct Regs { Raw p[2], q[2]; };
  auto gload = [&](int mb, Regs& r) {
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int row = l_row + 32 * t;
      // rows beyond this CTA's slice must not contribute: clamp through M = mend
      load_raw<PK>(g.p, pass, n0 + row, mb + l_m, mend, g.ld, r.p[t]);
      load_raw<QK>(g.q, pass, k0 + row, mb + l_m, mend, g.ld, r.q[t]);
    }
  };
  auto sstore = [&](int buf, int mb, const Regs& r) {
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int row = l_row + 32 * t;
      st4(Ps + ((size_t)buf * 64 + row) * DW_LDS + l_m,
          finish_operand<PK>(g.p, cs_p, pass, n0 + row, mb + l_m, mend, g.slope, r.p[t]));
      st4(Qs + ((size_t)buf * 64 + row) * DW_LDS + l_m,
          finish_operand<QK>(g.q, cs_q, pass, k0 + row, mb + l_m, mend, g.slope, r.q[t]));
    }
  };
  auto compute = [&](int cur) {
    const float* P = Ps + (size_t)cur * 64 * DW_LDS;
    const float* Q = Qs + (size_t)cur * 64 * DW_LDS;
#pragma unroll
    for (int mm = 0; mm < DW_MC; mm += 4) {
      float4 p[4], q[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) p[i] = ld4(P + (tn + 16 * i) * DW_LDS + mm);
#pragma unroll
      for (int j = 0; j < 4; ++j) q[j] = ld4(Q + (tk + 16 * j) * DW_LDS + mm);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[i][j] = fmaf(p[i].x, q[j].x, acc[i][j]);
          acc[i][j] = fmaf(p[i].y, q[j].y, acc[i][j]);
          acc[i][j] = fmaf(p[i].z, q[j].z, acc[i][j]);
          acc[i][j] = fmaf(p[i].w, q[j].w, acc[i][j]);
        }
      if (do_bias) {
#pragma unroll
        for (int i = 0; i < 4; ++i) bsum[i] += (p[i].x + p[i].y) + (p[i].z + p[i].w);
      }
    }
  };

  const int nchunks = mbeg < mend ? (mend - mbeg + DW_MC - 1) / DW_MC : 0;
  Regs rr;
  if (nchunks > 0) {
    gload(mbeg, rr);
    sstore(0, mbeg, rr);
  }
  __syncthreads();
  for (int c = 0; c < nchunks; ++c) {
    const int cur = c & 1;
    if (c + 1 < nchunks) gload(mbeg + (c + 1) * DW_MC, rr);
    compute(cur);
    if (c + 1 < nchunks) sstore(cur ^ 1, mbeg + (c + 1) * DW_MC, rr);
    __syncthreads();
  }

  const int tile = blockIdx.y * gridDim.x + blockIdx.x;
  unsigned long long* tacc = acc64 + (size_t)tile * g.npass * DW_PART;
  {
    unsigned long long* mine = tacc + (size_t)pass * DW_PART;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int n = n0 + tn + 16 * i;
      if (n >= g.N) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (k0 + tk + 16 * j < g.K) atomicAdd(mine + (tn + 16 * i) * 64 + tk + 16 * j, det_fix(acc[i][j]));
      if (do_bias) atomicAdd(mine + 64 * 64 + tn + 16 * i, det_fix(bsum[i]));
    }
  }
  __threadfence();
  __syncthreads();
  __shared__ unsigned s_last;
  if (tid == 0) s_last = atomicAdd(tile_cnt + tile, 1u) == gridDim.z - 1 ? 1u : 0u;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int ps = 0; ps < g.npass; ++ps) {
    if (g.add_affine && g.dgamma && tile == 0) {
      const double* bs = g.p.bn.bstats + (long long)ps * g.p.bn.sb;
      for (int c = tid; c < g.p.bn.C; c += GEMM_THREADS) {
        atomicAdd(g.dbeta + c, (float)__ldcg(bs + c));               // written by this pass's write-back CTA
        atomicAdd(g.dgamma + c, (float)__ldcg(bs + g.p.bn.C + c));
      }
    }
    unsigned long long* pa = tacc + (size_t)ps * DW_PART;
    float* dW = g.dW + (long long)ps * g.sdW;
    const bool bias = (g.db != nullptr || g.label_col >= 0) && blockIdx.x == 0;
    for (int el = tid; el < DW_PART; el += GEMM_THREADS) {
      const bool is_b = el >= 64 * 64;
      const int n = n0 + (is_b ? el - 64 * 64 : el >> 6), k = k0 + (el & 63);
      if (n >= g.N || (is_b ? !bias : k >= g.K)) continue;
      const float sum = det_unfix(__ldcg(pa + el));
      pa[el] = 0ull;
      if (!is_b) {
        atomicAdd(dW + (size_t)n * g.ldw + g.wcol0 + k, sum);
      } else {
        if (g.db) atomicAdd(g.db + n, sum);
        if (g.label_col >= 0) atomicAdd(dW + (size_t)n * g.ldw + g.label_col, sum);
      }
    }
  }
  if (tid == 0) tile_cnt[tile] = 0u;
}

inline size_t gemm_mn_smem(const GemmArgs& g) {
  size_t f = operand_const_floats(g.a);
  if (g.ekind == EP_DBN) f += 4 * (size_t)g.prev_bn.C;
  f = (f + 3) & ~(size_t)3;        // 16-byte aligned
  f += 4 * (size_t)TBN * RED_LD;   // split-K partial tiles
  return f * sizeof(float);
}
inline size_t gemm_dw_smem(const DwArgs& g) {
  size_t f = 4 * 64 * DW_LDS + operand_const_floats(g.p) + operand_const_floats(g.q);
  return f * sizeof(float);
}

// ------------------------------------------------------------------------------------------------
// host dispatch: one small straight-line kernel per (operand kind, epilogue kind) that the steps use
// ------------------------------------------------------------------------------------------------
template <bool WT, int AK, int EK>
inline cudaError_t launch_mn_inst(const GemmArgs& g, dim3 grid, size_t smem, cudaStream_t st) {
  gemm_mn_kernel<WT, AK, EK><<<grid, GEMM_THREADS, smem, st>>>(g);
  return cudaGetLastError();
}

inline cudaError_t dispatch_mn(bool wt, const GemmArgs& g, dim3 grid, size_t smem, cudaStream_t st) {
#define CVG_MN(W, A, E) \
  if (wt == W && g.a.kind == A && g.ekind == E) return launch_mn_inst<W, A, E>(g, grid, smem, st);
  CVG_MN(true, OP_PLAIN, EP_LINEAR)
  CVG_MN(true, OP_BN_ACT, EP_LINEAR)
  CVG_MN(true, OP_REPARAM, EP_LINEAR)
  CVG_MN(false, OP_PLAIN, EP_DACT)
  CVG_MN(false, OP_CONST, EP_DACT)
  CVG_MN(false, OP_PLAIN, EP_STORE)
  CVG_MN(false, OP_PLAIN, EP_DBN)
  CVG_MN(false, OP_BN_BWD, EP_DBN)
  CVG_MN(false, OP_BN_BWD, EP_REPARAM_BWD)
#undef CVG_MN
  return cudaErrorInvalidValue;
}

template <int PK, int QK>
inline cudaError_t launch_dw_inst(const DwArgs& g, int nsplit, unsigned long long* acc, unsigned* cnt, dim3 grid,
                                  size_t smem, cudaStream_t st) {
  gemm_dw_kernel<PK, QK><<<grid, GEMM_THREADS, smem, st>>>(g, nsplit, acc, cnt);
  return cudaGetLastError();
}

inline cudaError_t dispatch_dw(const DwArgs& g, int nsplit, unsigned long long* acc, unsigned* cnt, dim3 grid,
                               size_t smem, cudaStream_t st) {
#define CVG_DW(P, Q) \
  if (g.p.kind == P && g.q.kind == Q) return launch_dw_inst<P, Q>(g, nsplit, acc, cnt, grid, smem, st);
  CVG_DW(OP_PLAIN, OP_PLAIN)
  CVG_DW(OP_CONST, OP_PLAIN)
  CVG_DW(OP_PLAIN, OP_BN_ACT)
  CVG_DW(OP_BN_BWD, OP_BN_ACT)
  CVG_DW(OP_BN_BWD, OP_REPARAM)
  CVG_DW(OP_BN_BWD, OP_PLAIN)
#undef CVG_DW
  return cudaErrorInvalidValue;
}

}  // namespace cvg
