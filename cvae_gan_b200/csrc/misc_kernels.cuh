// cvaegan_b200 - row-wise and element-wise kernels (LayerNorm, cross-entropy, spectral norm, Adam,
// Philox noise, sampling, filter).  Activations are feature-major [features][ld] (see gemm.cuh).
#pragma once
#include "common.cuh"

namespace cvg {

// ------------------------------------------------------------------------------------------------
// device-resident control block: everything that changes from step to step lives HERE, not in kernel
// arguments, so that a whole label visit can be captured in a CUDA graph once and replayed
// ------------------------------------------------------------------------------------------------
struct StepCtl {
  unsigned long long seed;      // Philox key
  unsigned long long counter;   // Philox step counter (advanced by ctl_bump_kernel)
  long long adam_t[4];          // torch.optim.Adam state['step'] per network
  float lambda_class;           // current_lambda_class of this epoch (cvae_gan.py:198-204)
  float pad;
};

__global__ void ctl_set_kernel(StepCtl* c, unsigned long long seed, unsigned long long counter, int set_rng,
                               float lambda_class, int set_lambda) {
  if (threadIdx.x == 0) {
    if (set_rng) { c->seed = seed; c->counter = counter; }
    if (set_lambda) c->lambda_class = lambda_class;
  }
}
__global__ void ctl_bump_kernel(StepCtl* c, unsigned long long dcounter, int adam_mask) {
  if (threadIdx.x == 0) {
    c->counter += dcounter;
    for (int n = 0; n < 4; ++n)
      if (adam_mask & (1 << n)) c->adam_t[n] += 1;
  }
}

// ------------------------------------------------------------------------------------------------
// accumulator slots (doubles, zeroed at the start of every step)
// ------------------------------------------------------------------------------------------------
enum {
  L_DREAL = 0,  // sum of D(x_real) scores          (cvae_gan.py:118-119)
  L_DFAKE = 1,  // sum of D(x_fake) scores          (cvae_gan.py:122-123, 188-189)
  L_CE0 = 2,    // sum of -log softmax[label], pass 0
  L_CE1 = 3,    // pass 1
  L_RECON = 4,  // sum (x_rec - x)^2                (cvae_gan.py:184)
  L_KL = 5,     // sum -0.5(1 + lv - mu^2 - e^lv)   (cvae_gan.py:185)
  L_COUNT = 8
};

// ------------------------------------------------------------------------------------------------
// LayerNorm forward (classifier layer 2, cvae_gan_models.py:268-270): one thread per batch row.
//   n = (h - mean) * rstd * g + b ; a = dropout(relu(n))
// ------------------------------------------------------------------------------------------------
struct LnArgs {
  int M, ld, C, npass;
  const float* h; long long sh;        // [C][ld] pre-LN
  const float* g; const float* b;
  float eps;
  const uint8_t* mask; long long smask; float keep_inv;   // null in eval mode
  float* a; long long sa;              // [C][ld] output
  float* rs; long long srs;            // [2][ld] mean, rstd per row
};

// CTA = 256 threads = 32 batch rows (lane) x 8 feature groups (warp); each thread keeps C/8 features of its
// row in registers, row moments are combined through shared memory (two-pass variance like torch).
constexpr int LN_ROWS = 32;
constexpr int LN_MAXF = 32;        // features per thread (C <= 256: every width the reference's formulas give up to F = 512)
constexpr int LN_MAXF_WIDE = 64;   // second instantiation for the widened model (C <= 512, CvgConfig.hidden)

// The per-row body, shared with the fused classifier chain (chain.cuh): the thread of (lane, warp w) owns row `lane` of a
// 32-row tile and features [w * C/8, (w + 1) * C/8); all 256 threads of the CTA call it.  load_h(c) reads the row's pre-LN
// value of feature c, store_a(c, a) takes its output (valid rows only).
template <int MAXF, class LoadH, class StoreA>
__device__ __forceinline__ void ln_fwd_row(int C, bool valid, float eps, const float* gam, const float* bet, const uint8_t* mk,
                                           size_t ldm, float keep_inv, float (*red)[LN_ROWS], LoadH load_h, StoreA store_a,
                                           float& mean, float& rstd) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int fpt = (C + 7) / 8;            // features per thread
  const int c0 = w * fpt;
  float v[MAXF];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXF; ++i) {
    const int c = c0 + i;
    v[i] = (i < fpt && c < C && valid) ? load_h(c) : 0.f;
    s += v[i];
  }
  red[w][lane] = s;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) tot += red[k][lane];
  mean = tot / (float)C;
  __syncthreads();
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXF; ++i) {
    const int c = c0 + i;
    if (i < fpt && c < C) { const float d = v[i] - mean; q = fmaf(d, d, q); }
  }
  red[w][lane] = q;
  __syncthreads();
  tot = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) tot += red[k][lane];
  rstd = 1.0f / sqrtf(tot / (float)C + eps);
  if (!valid) return;
#pragma unroll
  for (int i = 0; i < MAXF; ++i) {
    const int c = c0 + i;
    if (i < fpt && c < C) {
      float n = (v[i] - mean) * rstd * gam[c] + bet[c];
      n = fmaxf(n, 0.f);
      if (mk) n = mk[(size_t)c * ldm] ? n * keep_inv : 0.f;
      store_a(c, n);
    }
  }
}

template <int MAXF>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const LnArgs g) {
  __shared__ float red[8][LN_ROWS];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int m = blockIdx.x * LN_ROWS + lane;
  const int pass = blockIdx.y;
  const bool valid = m < g.M;
  const float* h = g.h + (long long)pass * g.sh + (valid ? m : 0);
  float* a = g.a + (long long)pass * g.sa + m;
  const uint8_t* mk = g.mask ? g.mask + (long long)pass * g.smask + m : nullptr;
  float mean, rstd;
  ln_fwd_row<MAXF>(
      g.C, valid, g.eps, g.g, g.b, mk, g.ld, g.keep_inv, red, [&](int c) { return h[(size_t)c * g.ld]; },
      [&](int c, float n) { a[(size_t)c * g.ld] = n; }, mean, rstd);
  if (!valid) return;
  if (g.rs && w == 0) {
    float* rs = g.rs + (long long)pass * g.srs;
    rs[m] = mean;
    rs[g.ld + m] = rstd;
  }
}

// LayerNorm backward (appendix A.3): in place on dn -> dh.  dn already contains the ReLU/dropout
// derivative.  Optionally accumulates the affine gradients (classifier step only).
struct LnBwdArgs {
  int M, ld, C, npass;
  float* dn; long long sdn;            // in: dL/dn, out: dL/dh
  const float* h; long long sh;
  const float* rs; long long srs;
  const float* g;
  float* dg; float* db;                // null -> skipped
};

// The per-row body, shared with the fused classifier chain (chain.cuh); thread mapping as ln_fwd_row.  load_dn(c) / load_h(c)
// read the row's dL/dn and pre-LN value of feature c, store_dh(c, v) takes dL/dh (valid rows only).  acc != null: the 32-row
// sums of the affine gradients go into it in fixed point, [dgamma (C) | dbeta (C)].
template <int MAXF, class LoadDn, class LoadH, class StoreDh>
__device__ __forceinline__ void ln_bwd_row(int C, bool valid, float mean, float rstd, const float* gam, float (*red1)[LN_ROWS],
                                           float (*red2)[LN_ROWS], LoadDn load_dn, LoadH load_h, StoreDh store_dh,
                                           unsigned long long* acc) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int fpt = (C + 7) / 8;
  const int c0 = w * fpt;
  float xh[MAXF], d[MAXF];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < MAXF; ++i) {
    const int c = c0 + i;
    const bool on = i < fpt && c < C && valid;
    xh[i] = on ? (load_h(c) - mean) * rstd : 0.f;
    d[i] = on ? load_dn(c) : 0.f;
    const float dx = on ? d[i] * gam[c] : 0.f;
    s1 += dx;
    s2 = fmaf(dx, xh[i], s2);
  }
  red1[w][lane] = s1;
  red2[w][lane] = s2;
  __syncthreads();
  s1 = 0.f; s2 = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) { s1 += red1[k][lane]; s2 += red2[k][lane]; }
  s1 /= (float)C;
  s2 /= (float)C;
#pragma unroll
  for (int i = 0; i < MAXF; ++i) {
    const int c = c0 + i;
    const bool on = i < fpt && c < C;       // warp-uniform
    if (!on) continue;
    if (valid) store_dh(c, rstd * (d[i] * gam[c] - s1 - xh[i] * s2));
    if (acc) {
      const float a = warp_sum(d[i] * xh[i]), b = warp_sum(d[i]);
      if (lane == 0) {
        atomicAdd(acc + c, det_fix(a));
        atomicAdd(acc + C + c, det_fix(b));
      }
    }
  }
}

// The affine gradients are summed in fixed point in `acc` ([2C] int64, det_fix: exact, so independent of the block order);
// the last block (ticket on `cnt`) converts them, adds them to dg / db and clears `acc` and `cnt` (like gemm_dw_kernel).
template <int MAXF>
__global__ void __launch_bounds__(256) ln_bwd_kernel(const LnBwdArgs g, unsigned long long* acc, unsigned* cnt) {
  __shared__ float red1[8][LN_ROWS], red2[8][LN_ROWS];
  const int lane = threadIdx.x & 31;
  const int m = blockIdx.x * LN_ROWS + lane;
  const int pass = blockIdx.y;
  const bool valid = m < g.M;
  const int mm = valid ? m : 0;
  const float* h = g.h + (long long)pass * g.sh + mm;
  float* dn = g.dn + (long long)pass * g.sdn + mm;
  const float* rs = g.rs + (long long)pass * g.srs;
  ln_bwd_row<MAXF>(
      g.C, valid, rs[mm], rs[g.ld + mm], g.g, red1, red2, [&](int c) { return dn[(size_t)c * g.ld]; },
      [&](int c) { return h[(size_t)c * g.ld]; }, [&](int c, float v) { dn[(size_t)c * g.ld] = v; }, g.dg ? acc : nullptr);
  if (!g.dg) return;
  __threadfence();
  __syncthreads();
  __shared__ unsigned s_last;
  if (threadIdx.x == 0) s_last = atomicAdd(cnt, 1u) == gridDim.x * gridDim.y - 1 ? 1u : 0u;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int e = threadIdx.x; e < 2 * g.C; e += blockDim.x) {
    const float v = det_unfix(__ldcg(acc + e));
    acc[e] = 0ull;
    atomicAdd(e < g.C ? g.dg + e : g.db + (e - g.C), v);
  }
  if (threadIdx.x == 0) *cnt = 0u;
}

inline void launch_ln_fwd(const LnArgs& a, cudaStream_t st) {
  const dim3 grid((a.M + LN_ROWS - 1) / LN_ROWS, a.npass);
  if (a.C <= 8 * LN_MAXF) ln_fwd_kernel<LN_MAXF><<<grid, 256, 0, st>>>(a);
  else ln_fwd_kernel<LN_MAXF_WIDE><<<grid, 256, 0, st>>>(a);
}
inline void launch_ln_bwd(const LnBwdArgs& a, unsigned long long* acc, unsigned* cnt, cudaStream_t st) {
  const dim3 grid((a.M + LN_ROWS - 1) / LN_ROWS, a.npass);
  if (a.C <= 8 * LN_MAXF) ln_bwd_kernel<LN_MAXF><<<grid, 256, 0, st>>>(a, acc, cnt);
  else ln_bwd_kernel<LN_MAXF_WIDE><<<grid, 256, 0, st>>>(a, acc, cnt);
}

// ------------------------------------------------------------------------------------------------
// softmax cross-entropy with one shared target label (cvae_gan.py:147,151,194): one thread per row.
//   loss += -(l[y] - max - log sum exp(l - max)) ; dlogit = (softmax - onehot) * coef
// ------------------------------------------------------------------------------------------------
struct CeArgs {
  int M, ld, K, npass, label;
  const float* logits; long long sl;   // [K][ld]
  float* dlogits; long long sd;        // [K][ld]
  float coef;                          // 1/Bg; multiplied by ctl->lambda_class when `ctl` is set (generator step)
  const StepCtl* ctl;
  double* loss;                        // [npass] accumulators
  const long long* labels = nullptr;   // per-row targets (downstream Classifier.fit); null -> the shared `label`
};

// One row: K logits `ldl` apart in, K logit gradients `ldd` apart out; returns the row's negative log-likelihood.  Shared with
// the fused classifier chain (chain.cuh).
__device__ __forceinline__ double ce_row(const float* l, size_t ldl, float* d, size_t ldd, int K, int tgt, float coef) {
  float mx = -INFINITY;
  for (int k = 0; k < K; ++k) mx = fmaxf(mx, l[(size_t)k * ldl]);
  float s = 0.f;
  for (int k = 0; k < K; ++k) s += expf(l[(size_t)k * ldl] - mx);
  const float lse = logf(s);
  const double nll = -(double)(l[(size_t)tgt * ldl] - mx - lse);
  for (int k = 0; k < K; ++k) {
    const float p = expf(l[(size_t)k * ldl] - mx - lse);
    d[(size_t)k * ldd] = (p - (k == tgt ? 1.f : 0.f)) * coef;
  }
  return nll;
}

__global__ void ce_kernel(const CeArgs g) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  const int pass = blockIdx.y;
  double nll = 0.0;
  if (m < g.M) {
    const int tgt = g.labels ? (int)g.labels[m] : g.label;
    const float coef = g.ctl ? g.coef * g.ctl->lambda_class : g.coef;
    nll = ce_row(g.logits + (long long)pass * g.sl + m, g.ld, g.dlogits + (long long)pass * g.sd + m, g.ld, g.K, tgt, coef);
  }
  nll = warp_sum_d(nll);
  if ((threadIdx.x & 31) == 0 && nll != 0.0) atomicAdd(g.loss + pass, nll);
}

// ------------------------------------------------------------------------------------------------
// generator output seed gradient (cvae_gan.py:184 + sigmoid backward), element-wise over [F][ld]:
//   pass 0 (x_recon): dout = lambda_recon * 2 (o - x) / (Bg F)     and  recon += (o - x)^2
//   pass 1 (x_fake) : dout = dx (accumulated input gradient of critic + classifier)
//   dpre = dout * o * (1 - o)
// add_dx (sibling trainer CVAE, cvae.py:141-157): ONE pass, the classifier reads x_recon itself, so its input gradient
// joins the reconstruction term: dout = lambda_recon * 2 (o - x) / (Bg F) + dx
// ------------------------------------------------------------------------------------------------
struct SeedArgs {
  int M, ld, F;
  const float* out; long long sout;    // [2][F][ld] sigmoid outputs
  const float* x;                      // [F][ld] real batch
  const float* dx;                     // [F][ld]
  float* dpre; long long sdpre;        // [2][F][ld]
  float coef_recon;
  double* recon_acc;
  int prior_only = 0;                  // CGAN generator step: one pass, and it is the x_fake (dx) one
  int add_dx = 0;                      // CVAE generator step: pass 0 also receives dx (classification term on x_recon)
};

__global__ void g_seed_kernel(const SeedArgs g) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int pass = blockIdx.y;
  const int f = idx / g.ld, m = idx % g.ld;
  double sq = 0.0;
  if (f < g.F) {
    const size_t off = (size_t)f * g.ld + m;
    float d = 0.f;
    if (m < g.M) {
      const float o = g.out[(long long)pass * g.sout + off];
      float dout;
      if (pass == 0 && !g.prior_only) {
        const float diff = o - g.x[off];
        sq = (double)diff * (double)diff;
        dout = g.coef_recon * 2.0f * diff;
        if (g.add_dx) dout += g.dx[off];
      } else {
        dout = g.dx[off];
      }
      d = dout * (1.0f - o) * o;
    }
    g.dpre[(long long)pass * g.sdpre + off] = d;
  }
  if (pass == 0 && !g.prior_only) {
    sq = warp_sum_d(sq);
    if ((threadIdx.x & 31) == 0 && sq != 0.0) atomicAdd(g.recon_acc, sq);
  }
}

// ------------------------------------------------------------------------------------------------
// spectral norm (torch _SpectralNorm.forward, appendix A.4): one CTA per critic layer.  For each of
// `npass` consecutive train-mode forwards: u <- normalize(W v), v <- normalize(W^T u), sigma = u.(W v).
// Snapshots of (u, v, sigma) per pass are kept for the backward term.
// ------------------------------------------------------------------------------------------------
constexpr int SN_MAXDIM = 1024;
struct SnLayer {
  const float* W; int rows, cols;
  float* u; float* v;
  int snap_off;      // offset (floats) of this layer in the snapshot buffers
};
struct SnArgs {
  SnLayer L[4];
  int npass, do_power;
  float eps;
  float* sigma;      // [npass][4]
  float* inv_sigma;  // [4][npass]   (per layer contiguous over passes: GemmArgs.scale[pass])
  float* u_snap; float* v_snap; long long ssnap;   // [npass][ssnap]
  int w_smem_floats = 0;   // dynamic shared memory (floats) for a copy of W: the 3 mat-vecs per pass then read it from there
};

constexpr int SN_THREADS = 1024;

__global__ void __launch_bounds__(SN_THREADS) sn_power_kernel(const SnArgs g) {
  __shared__ float su[SN_MAXDIM], sv[SN_MAXDIM], st[SN_MAXDIM];
  __shared__ float part[SN_THREADS];
  __shared__ double red[32];
  extern __shared__ __align__(16) float sn_w[];
  SnLayer L = g.L[blockIdx.x];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  if (L.rows * L.cols <= g.w_smem_floats) {        // one pass over W in L2 instead of 3 * npass
    const int n_el = L.rows * L.cols;
    if ((n_el & 3) == 0 && ((size_t)L.W & 15) == 0) {
      for (int i = tid * 4; i < n_el; i += blockDim.x * 4) st4(sn_w + i, ld4(L.W + i));
    } else {
      for (int i = tid; i < n_el; i += blockDim.x) sn_w[i] = L.W[i];
    }
    L.W = sn_w;
  }
  for (int i = tid; i < L.rows; i += blockDim.x) su[i] = L.u[i];
  for (int i = tid; i < L.cols; i += blockDim.x) sv[i] = L.v[i];
  __syncthreads();
  // column-parallel W^T u: thread (k = tid % cp, group = tid / cp) sums rows group, group + ng, ...
  int cp = 1;
  while (cp < L.cols) cp <<= 1;
  if (cp > SN_THREADS) cp = SN_THREADS;
  const int ng = SN_THREADS / cp, kq = tid % cp, gq = tid / cp;
  for (int p = 0; p < g.npass; ++p) {
    if (g.do_power) {
      for (int n = w; n < L.rows; n += nw) {          // t = W v
        float s = 0.f;
        for (int k = lane; k < L.cols; k += 32) s = fmaf(L.W[(size_t)n * L.cols + k], sv[k], s);
        s = warp_sum(s);
        if (lane == 0) st[n] = s;
      }
      __syncthreads();
      double q = 0.0;
      for (int i = tid; i < L.rows; i += blockDim.x) q += (double)st[i] * st[i];
      q = block_sum_d(q, red);
      float nrm = fmaxf((float)sqrt(q), g.eps);
      for (int i = tid; i < L.rows; i += blockDim.x) su[i] = st[i] / nrm;
      __syncthreads();
      for (int k0 = 0; k0 < L.cols; k0 += cp) {       // s = W^T u
        const int k = k0 + kq;
        float s = 0.f;
        if (k < L.cols)
          for (int n = gq; n < L.rows; n += ng) s = fmaf(L.W[(size_t)n * L.cols + k], su[n], s);
        part[tid] = s;
        __syncthreads();
        if (gq == 0 && k < L.cols) {
          float t = 0.f;
          for (int j = 0; j < ng; ++j) t += part[j * cp + kq];
          st[k] = t;
        }
        __syncthreads();
      }
      q = 0.0;
      for (int i = tid; i < L.cols; i += blockDim.x) q += (double)st[i] * st[i];
      q = block_sum_d(q, red);
      nrm = fmaxf((float)sqrt(q), g.eps);
      for (int i = tid; i < L.cols; i += blockDim.x) sv[i] = st[i] / nrm;
      __syncthreads();
    }
    double sg = 0.0;                                  // sigma = u . (W v)
    for (int n = w; n < L.rows; n += nw) {
      float s = 0.f;
      for (int k = lane; k < L.cols; k += 32) s = fmaf(L.W[(size_t)n * L.cols + k], sv[k], s);
      s = warp_sum(s);
      if (lane == 0) sg += (double)s * su[n];
    }
    sg = block_sum_d(sg, red);
    if (tid == 0) {
      g.sigma[p * 4 + blockIdx.x] = (float)sg;
      g.inv_sigma[blockIdx.x * 2 + p] = 1.0f / (float)sg;
    }
    float* us = g.u_snap + (long long)p * g.ssnap + L.snap_off;
    float* vs = g.v_snap + (long long)p * g.ssnap + L.snap_off;
    for (int i = tid; i < L.rows; i += blockDim.x) us[i] = su[i];
    for (int i = tid; i < L.cols; i += blockDim.x) vs[i] = sv[i];
    __syncthreads();
  }
  if (g.do_power) {
    for (int i = tid; i < L.rows; i += blockDim.x) L.u[i] = su[i];
    for (int i = tid; i < L.cols; i += blockDim.x) L.v[i] = sv[i];
  }
}

// Gradient through W/sigma (appendix A.4): with G_p = dL/dWhat of pass p,
//   dL/dW += sum_p [ G_p / sigma_p - (<G_p, W> / sigma_p^2) u_p v_p^T ]
struct SnGradArgs {
  SnLayer L[4];
  int npass;
  const float* Gp; long long sG;    // per-pass raw gradients, same layout/offsets as the param buffer
  long long w_off[4];               // offset of each layer's weight in the param buffer
  const float* inv_sigma;           // [4][2]
  const float* u_snap; const float* v_snap; long long ssnap;
  float* grad;                      // param-layout gradient buffer (accumulated into)
  float* last_bias_grad;            // d(score bias): rows * sum_p seed_p, added analytically (exactly 0 in step D,
  float last_bias_value;            // where autograd's -1/B and +1/B sums cancel bit for bit)
};

// <G_p, W> per (layer, pass): grid (chunks, 4, npass); dots[layer * 2 + pass] accumulates in double
__global__ void __launch_bounds__(256) sn_dot_kernel(const SnGradArgs g, double* dots) {
  __shared__ double red[32];
  const int l = blockIdx.y, p = blockIdx.z;
  const SnLayer L = g.L[l];
  const int n_el = L.rows * L.cols;
  const float* G = g.Gp + (long long)p * g.sG + g.w_off[l];
  double d = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_el; i += gridDim.x * blockDim.x)
    d += (double)G[i] * (double)L.W[i];
  d = block_sum_d(d, red);
  if (threadIdx.x == 0 && d != 0.0) atomicAdd(dots + l * 2 + p, d);
}

__global__ void __launch_bounds__(256) sn_grad_kernel(const SnGradArgs g, const double* dots) {
  const int l = blockIdx.y;
  const SnLayer L = g.L[l];
  const int n_el = L.rows * L.cols;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_el; i += gridDim.x * blockDim.x) {
    const int n = i / L.cols, k = i % L.cols;
    float acc = 0.f;
    for (int p = 0; p < g.npass; ++p) {
      const float is = g.inv_sigma[l * 2 + p];
      const float* G = g.Gp + (long long)p * g.sG + g.w_off[l];
      const float u = g.u_snap[(long long)p * g.ssnap + L.snap_off + n];
      const float v = g.v_snap[(long long)p * g.ssnap + L.snap_off + k];
      acc += G[i] * is - (float)(dots[l * 2 + p] * (double)is * (double)is) * u * v;
    }
    g.grad[g.w_off[l] + i] += acc;
  }
  if (l == 3 && blockIdx.x == 0 && threadIdx.x == 0 && g.last_bias_grad) *g.last_bias_grad += g.last_bias_value;
}

// ------------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam, appendix A.8) over up to two flat parameter segments; also turns the loss
// accumulators into the user's loss_out.  The gradient is cleared after use.
// ------------------------------------------------------------------------------------------------
struct AdamSeg {
  float* p; float* g; float* m; float* v;
  long long n;
  float lr;
  const long long* t_prev;     // device: number of steps taken so far (this launch applies step t_prev + 1)
};
struct AdamArgs {
  AdamSeg seg[2];
  int nseg;
  float b1, b2, eps;
  int clear_grad;
  int t_add = 1;               // 0: the step counters were already advanced (loss_tail_kernel)
};

__global__ void adam_kernel(const AdamArgs a) {
  const AdamSeg s = a.seg[blockIdx.y];
  // bias corrections in double like torch's Python scalars: step_size = lr / (1 - beta1^t), sqrt(1 - beta2^t)
  __shared__ float sh[2];
  if (threadIdx.x == 0) {
    const double t = (double)(*s.t_prev + a.t_add);
    sh[0] = (float)((double)s.lr / (1.0 - pow((double)a.b1, t)));
    sh[1] = (float)sqrt(1.0 - pow((double)a.b2, t));
  }
  __syncthreads();
  const float step_size = sh[0], bc2_sqrt = sh[1];
  const float w = 1.0f - a.b1;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < s.n; i += (long long)gridDim.x * blockDim.x) {
    const float g = s.g[i];
    float m = s.m[i], v = s.v[i];
    // exp_avg.lerp_(grad, 1 - beta1)  (torch lerp: weight < 0.5 ? a + w (b - a) : b - (b - a)(1 - w))
    m = (w < 0.5f) ? m + w * (g - m) : g - (g - m) * (1.0f - w);
    v = v * a.b2 + (1.0f - a.b2) * g * g;
    const float denom = sqrtf(v) / bc2_sqrt + a.eps;
    s.p[i] = s.p[i] - step_size * (m / denom);
    s.m[i] = m;
    s.v[i] = v;
    if (a.clear_grad) s.g[i] = 0.f;
  }
}

// losses: accumulators (double, local sums) -> float partials in the gradient tail (so the data
// parallel all-reduce sums them with the gradients) -> loss_out after the reduction.
__global__ void pack_loss_kernel(const double* acc, float* tail) {
  if (threadIdx.x < L_COUNT) tail[threadIdx.x] = (float)acc[threadIdx.x];
}
// End of a step in one launch: pack; on one GPU (unpack != 0) also the unpack below; and the control block's bookkeeping -
// the Philox counter moves on by `dcounter`, Adam's state['step'] of the networks in `adam_mask` by one (the Adam launch
// that follows runs with t_add = 0).
__global__ void loss_tail_kernel(const double* acc, float* tail, float* out, int kind, float Bg, float F, int unpack,
                                 StepCtl* c, unsigned long long dcounter, int adam_mask) {
  __shared__ float t[L_COUNT];
  if (threadIdx.x < L_COUNT) t[threadIdx.x] = (float)acc[threadIdx.x];
  __syncthreads();
  if (threadIdx.x < L_COUNT && !unpack) tail[threadIdx.x] = t[threadIdx.x];
  if (threadIdx.x == 0) {
    if (unpack && out) {
      if (kind == 0) {
        const float r = t[L_DREAL] / Bg, f = t[L_DFAKE] / Bg;
        out[0] = -r + f; out[1] = r; out[2] = f; out[3] = 0.f;
      } else if (kind == 1) {
        const float r = t[L_CE0] / Bg, f = t[L_CE1] / Bg;
        out[0] = r + f; out[1] = r; out[2] = f; out[3] = 0.f;
      } else {
        out[0] = t[L_RECON] / (Bg * F);
        out[1] = t[L_KL] / Bg;
        out[2] = -t[L_DFAKE] / Bg;
        out[3] = t[L_CE0] / Bg;
      }
    }
    c->counter += dcounter;
    for (int n = 0; n < 4; ++n)
      if (adam_mask & (1 << n)) c->adam_t[n] += 1;
  }
}
// kind 0: step_d, 1: step_c, 2: step_g
__global__ void unpack_loss_kernel(const float* tail, float* out, int kind, float Bg, float F, int clear, float* tail_w) {
  if (threadIdx.x == 0) {
    if (kind == 0) {
      const float r = tail[L_DREAL] / Bg, f = tail[L_DFAKE] / Bg;
      out[0] = -r + f; out[1] = r; out[2] = f; out[3] = 0.f;
    } else if (kind == 1) {
      const float r = tail[L_CE0] / Bg, f = tail[L_CE1] / Bg;
      out[0] = r + f; out[1] = r; out[2] = f; out[3] = 0.f;
    } else {
      out[0] = tail[L_RECON] / (Bg * F);
      out[1] = tail[L_KL] / Bg;
      out[2] = -tail[L_DFAKE] / Bg;
      out[3] = tail[L_CE0] / Bg;
    }
  }
  __syncthreads();
  if (clear && threadIdx.x < CVG_GRAD_TAIL) tail_w[threadIdx.x] = 0.f;
}

// ------------------------------------------------------------------------------------------------
// noise: either transposes an injected row-major tensor into the feature-major workspace or draws it
// from Philox keyed by (seed, counter, stream, pass, global row, feature group).
// ------------------------------------------------------------------------------------------------
struct FillJob {
  void* out;             // float* (normal) or uint8_t* (mask), feature-major [npass][nfeat][ld]
  const void* injected;  // row-major [npass][M][nfeat] or null
  int kind;              // 0 normal float, 1 keep-mask uint8
  int nfeat, npass, stream;
  int cstep;             // != 0: pass i is the single pass of the step `i * cstep` counter values ahead (hoisted draws)
};
struct FillArgs {
  FillJob job[6];
  int njobs;
  int M, ld;
  uint64_t seed, counter, row_base;   // used when ctl == nullptr (generation path)
  const StepCtl* ctl = nullptr;       // training: seed = ctl->seed, counter = ctl->counter + counter_off
  uint64_t counter_off = 0;
  float keep_prob;
};

__global__ void fill_noise_kernel(const FillArgs a) {
  const FillJob j = a.job[blockIdx.y];
  const int ngroups = (j.nfeat + 3) >> 2;
  const long long total = (long long)j.npass * ngroups * a.M;
  const uint32_t keep_thr = (uint32_t)((double)a.keep_prob * 4294967296.0);
  const uint64_t seed = a.ctl ? a.ctl->seed : a.seed;
  const uint64_t counter = a.ctl ? a.ctl->counter + a.counter_off : a.counter;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(t % a.M);
    const int fg = (int)((t / a.M) % ngroups);
    const int pass = (int)(t / ((long long)a.M * ngroups));
    float vals[4];
    uint8_t bits[4];
    if (j.injected) {
      for (int i = 0; i < 4; ++i) {
        const int f = fg * 4 + i;
        if (f < j.nfeat) {
          const size_t src = ((size_t)pass * a.M + m) * j.nfeat + f;
          if (j.kind == 0) vals[i] = ((const float*)j.injected)[src];
          else bits[i] = ((const uint8_t*)j.injected)[src] ? 1 : 0;
        }
      }
    } else {
      const U4 r = j.cstep ? philox_at(seed, counter + (uint64_t)pass * j.cstep, (uint32_t)j.stream, 0u, a.row_base + (uint64_t)m, (uint32_t)fg)
                           : philox_at(seed, counter, (uint32_t)j.stream, (uint32_t)pass, a.row_base + (uint64_t)m, (uint32_t)fg);
      if (j.kind == 0) {
        box_muller(r.x, r.y, vals[0], vals[1]);
        box_muller(r.z, r.w, vals[2], vals[3]);
      } else {
        bits[0] = r.x < keep_thr; bits[1] = r.y < keep_thr; bits[2] = r.z < keep_thr; bits[3] = r.w < keep_thr;
      }
    }
    for (int i = 0; i < 4; ++i) {
      const int f = fg * 4 + i;
      if (f < j.nfeat) {
        const size_t dst = ((size_t)pass * j.nfeat + f) * a.ld + m;
        if (j.kind == 0) ((float*)j.out)[dst] = vals[i];
        else ((uint8_t*)j.out)[dst] = bits[i];
      }
    }
  }
}

// row-major [M][F] (optionally gathered through idx) -> feature-major [F][ld]
__global__ void to_feature_major_kernel(const float* src, const long long* idx, int M, int F, int ld, float* dst) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const long long r = idx ? idx[m] : m;
  for (int f = 0; f < F; ++f) dst[(size_t)f * ld + m] = src[(size_t)r * F + f];
}
// feature-major [F][ld] -> row-major [M][F]
__global__ void to_row_major_kernel(const float* src, int M, int F, int ld, float* dst) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  for (int f = 0; f < F; ++f) dst[(size_t)m * F + f] = src[(size_t)f * ld + m];
}

// ------------------------------------------------------------------------------------------------
// _get_target_samples on the device (cvae_gan.py:247-260)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
// keyed bijection of [0, 2^(2*half)) (balanced Feistel, 6 rounds)
__device__ __forceinline__ uint64_t feistel(uint64_t x, int half, const uint32_t* keys) {
  const uint32_t maskh = (half >= 32) ? 0xFFFFFFFFu : ((1u << half) - 1u);
  uint32_t L = (uint32_t)(x >> half) & maskh, R = (uint32_t)x & maskh;
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    const uint32_t f = mix32(R ^ keys[r]) & maskh;
    const uint32_t nl = R;
    R = L ^ f;
    L = nl;
  }
  return ((uint64_t)L << half) | R;
}

__global__ void sample_rows_kernel(const float* rows, long long n, long long B, long long draw_offset, int B_local,
                                   int F, uint64_t seed_arg, uint64_t counter_arg, const StepCtl* ctl,
                                   uint64_t counter_off, float* x_out, long long* idx_out) {
  const int il = blockIdx.x * blockDim.x + threadIdx.x;
  if (il >= B_local) return;
  const uint64_t seed = ctl ? ctl->seed : seed_arg;
  const uint64_t counter = ctl ? ctl->counter + counter_off : counter_arg;
  const long long i = draw_offset + il;      // index of this draw in the global batch
  long long r;
  if (n == B) {
    r = i;                                   // all rows, no draw (cvae_gan.py:254-256)
  } else if (n < B) {                        // with replacement (cvae_gan.py:250-253)
    const U4 u = philox_at(seed, counter, RS_SAMPLE, 0, (uint64_t)i, 0);
    const uint64_t w = ((uint64_t)u.x << 32) | u.y;
    r = (long long)(w % (uint64_t)n);
  } else {                                   // B distinct rows: first B images of a keyed permutation of [0, n)
    int bits = 1;
    while ((1ll << bits) < n) ++bits;
    const int half = (bits + 1) >> 1;
    uint32_t keys[6];
    const U4 k0 = philox_at(seed, counter, RS_SAMPLE, 1, 0, 0), k1 = philox_at(seed, counter, RS_SAMPLE, 1, 1, 0);
    keys[0] = k0.x; keys[1] = k0.y; keys[2] = k0.z; keys[3] = k0.w; keys[4] = k1.x; keys[5] = k1.y;
    uint64_t x = (uint64_t)i;
    do { x = feistel(x, half, keys); } while (x >= (uint64_t)n);   // cycle walking keeps it a bijection on [0, n)
    r = (long long)x;
  }
  if (idx_out) idx_out[il] = r;
  for (int f = 0; f < F; ++f) x_out[(size_t)il * F + f] = rows[(size_t)r * F + f];
}

// ------------------------------------------------------------------------------------------------
// filter decision (cvae_gan.py:366-370).  Softmax arithmetic follows torch's CUDA warp softmax for
// K <= 32 (softmax_warp_forward: exp(x - max) accumulated by a xor-butterfly over next_pow2(K)
// lanes, then a true division) so the decision equals torch.softmax -> torch.max on the same logits.
// ------------------------------------------------------------------------------------------------
constexpr int FILTER_MAXK = 32;

// P = next_pow2(K) known at compile time: everything stays in registers.  The decision is EXACTLY
//   p = e / sum (IEEE division);  (m, i) = max(p) with the first index on ties;  keep = m > thr && i == label
// but only p[label] is divided out unconditionally: IEEE division by a common positive divisor is monotonic, so
// p[k] can only tie with or beat p[label] when e[k] is within a few ulps of e[label] or above it, and only those
// (rare) candidates are divided and compared exactly.
template <int P, int KC = 0, typename LoadLogit>
__device__ __forceinline__ bool filter_decide_p(LoadLogit ld, int K_rt, int label, float thr) {
  const int K = KC > 0 ? KC : K_rt;     // KC > 0: class count known at compile time (no predicated-off work)
  float e[P];
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < P; ++k) {
    e[k] = (k < K) ? ld(k) : -INFINITY;
    if (k < K) mx = fmaxf(mx, e[k]);
  }
  bool nan = false;
  float el = ld(label);      // (re-read instead of indexing e[]: a dynamic index would push the array to local memory)
  // exact early-out: the largest exponential is expf(0) = 1; when the label's logit trails the maximum by more than
  // 2e-6 its exponential is below 1 / 1.000001, i.e. it is "clearly behind" in the sense used below
  if (mx - el > 2e-6f) return false;
#pragma unroll
  for (int k = 0; k < P; ++k) {
    if (k < K) { nan |= (e[k] != e[k]); e[k] = expf(e[k] - mx); } else e[k] = 0.f;
  }
  el = expf(el - mx);
  float s[P];
#pragma unroll
  for (int k = 0; k < P; ++k) s[k] = e[k];
#pragma unroll
  for (int o = P >> 1; o > 0; o >>= 1)
#pragma unroll
    for (int k = 0; k < o; ++k) s[k] = s[k] + s[k + o];
  const float sum = s[0];
  if (nan) return false;
  // cheap screen: some other class clearly ahead of the label -> the label cannot be the arg max
  const float lo = el * 0.999999f;    // "within ~8 ulps below e[label]"
  bool close = false, lost = false;
#pragma unroll
  for (int k = 0; k < P; ++k) {
    if (k < K && k != label) {
      if (e[k] > el * 1.000001f) lost = true;
      else if (e[k] >= lo) close = true;
    }
  }
  if (lost) return false;
  const float pl = el / sum;
  if (!(pl > thr)) return false;
  if (!close) return true;
  bool win = true;
#pragma unroll
  for (int k = 0; k < P; ++k) {
    if (k < K && k != label && e[k] >= lo) {
      const float pk = e[k] / sum;
      if (pk > pl || (pk == pl && k < label)) win = false;
    }
  }
  return win;
}

template <typename LoadLogit>
__device__ __forceinline__ bool filter_decide(LoadLogit ld, int K, int label, float thr) {
  if (K <= 2) return filter_decide_p<2>(ld, K, label, thr);
  if (K <= 4) return filter_decide_p<4>(ld, K, label, thr);
  if (K <= 8) return filter_decide_p<8>(ld, K, label, thr);
  if (K <= 16) return filter_decide_p<16>(ld, K, label, thr);
  return filter_decide_p<32>(ld, K, label, thr);
}

__global__ void filter_logits_kernel(const float* logits, long long n, int K, int label, float thr, uint8_t* keep) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* l = logits + i * K;
  keep[i] = filter_decide([&](int k) { return l[k]; }, K, label, thr) ? 1 : 0;
}

// Decision + order-preserving-within-block compaction.  FM = logits/x feature-major [.][ld] (fused
// generation path) or row-major (standalone filter over materialised tensors).
template <bool FM>
__global__ void __launch_bounds__(256) filter_compact_kernel(const float* x, const float* logits, long long n, int ld,
                                                             int F, int K, int label, float thr, uint64_t row_offset,
                                                             float* x_out, long long* idx_out, long long capacity,
                                                             unsigned long long* count, float* logits_out,
                                                             uint8_t* keep_out) {
  __shared__ int warp_cnt[8];
  __shared__ unsigned long long base;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool keep = false;
  if (i < n) {
    if (FM) keep = filter_decide([&](int k) { return logits[(size_t)k * ld + i]; }, K, label, thr);
    else keep = filter_decide([&](int k) { return logits[i * K + k]; }, K, label, thr);
    if (keep_out) keep_out[i] = keep ? 1 : 0;
    if (logits_out) {
      for (int k = 0; k < K; ++k) logits_out[i * K + k] = FM ? logits[(size_t)k * ld + i] : logits[i * K + k];
    }
  }
  const unsigned bal = __ballot_sync(0xffffffffu, keep);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) warp_cnt[w] = __popc(bal);
  __syncthreads();
  if (threadIdx.x == 0) {
    int tot = 0;
    for (int k = 0; k < 8; ++k) { const int c = warp_cnt[k]; warp_cnt[k] = tot; tot += c; }
    base = tot ? atomicAdd(count, (unsigned long long)tot) : 0ull;
  }
  __syncthreads();
  if (keep) {
    const long long pos = (long long)base + warp_cnt[w] + __popc(bal & ((1u << lane) - 1u));
    if (pos < capacity) {
      for (int f = 0; f < F; ++f) x_out[pos * F + f] = FM ? x[(size_t)f * ld + i] : x[i * F + f];
      if (idx_out) idx_out[pos] = (long long)(row_offset + (uint64_t)i);
    }
  }
}


// Standalone filter over MATERIALISED row-major tensors (the memory-bound kernel of SURVEY.md 8d).  One CTA takes
// `nsub` consecutive sub-blocks of 1024 rows.  Pass 1: each logits sub-block is fetched with coalesced 16-byte
// streaming loads into shared memory, every thread decides 4 rows from shared memory, and the warp ballots are kept
// in shared memory.  ONE atomic per CTA then orders its accepted rows (same-address atomics serialise in L2, so
// there must be few of them).  Pass 2 reads ONLY the accepted rows of x and copies them out - x of a rejected row
// is never touched: the traffic is 4K + a (4F read + 4F + 8 written) bytes per row, below SURVEY's 4F + 4K +
// a (4F + 8).
constexpr int FC_THREADS = 256;
constexpr int FC_MAXJ = 4;                          // rows per thread per sub-block
constexpr int FC_SUB_ROWS = FC_MAXJ * FC_THREADS;   // 1024
constexpr int FC_MAXSUB = 32;                        // sub-blocks per CTA (grid-strided)

__host__ __device__ constexpr int fc_pow2(int k) { return k <= 2 ? 2 : k <= 4 ? 4 : k <= 8 ? 8 : k <= 16 ? 16 : 32; }

// KC = number of classes (compile time)
template <int KC>
__global__ void __launch_bounds__(FC_THREADS, (KC <= 8) ? 6 : 2) filter_compact_stream_kernel(const float* __restrict__ x,
                                                                           const float* __restrict__ logits, long long n,
                                                                           int F, int K, int label, float thr,
                                                                           uint64_t row_offset, int nsub,
                                                                           float* __restrict__ x_out,
                                                                           long long* __restrict__ idx_out,
                                                                           long long capacity, unsigned long long* count) {
  extern __shared__ __align__(16) float fc_sl[];      // [1024][K] logits of the current sub-block
  __shared__ unsigned bals[FC_MAXSUB][FC_MAXJ][FC_THREADS / 32];
  __shared__ int pref[FC_MAXSUB * FC_MAXJ * (FC_THREADS / 32)];
  __shared__ int wsum[FC_THREADS / 32];
  __shared__ unsigned long long base;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const bool vec2 = (F & 1) == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(x_out)) & 7) == 0;
  // ---- pass 1: decisions ----
  // A cheap exact screen first (a row whose label logit trails the maximum by more than 2e-6 cannot win, see
  // filter_decide_p); the survivors are compacted into a shared list and only they pay for the softmax arithmetic -
  // without the compaction a warp runs the expensive path as soon as ONE of its 32 rows survives.
  __shared__ unsigned short surv[FC_SUB_ROWS];
  __shared__ unsigned int bitmap[FC_SUB_ROWS / 32];
  __shared__ int nsurv;
  for (int sb = 0; sb < nsub; ++sb) {
    const long long row0 = ((long long)sb * gridDim.x + blockIdx.x) * FC_SUB_ROWS;
    const int rows = (int)max(0ll, min((long long)FC_SUB_ROWS, n - row0));
    if (tid < FC_SUB_ROWS / 32) bitmap[tid] = 0u;
    if (tid == 0) nsurv = 0;
    if (rows > 0) {
      const float* src = logits + row0 * KC;
      const long long nfl = (long long)rows * KC;
      if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        const long long n4 = nfl >> 2;
        const float4* s4 = reinterpret_cast<const float4*>(src);
        float4* d4 = reinterpret_cast<float4*>(fc_sl);
        // batches of 4 independent 16-byte loads per thread (memory-level parallelism), then the stores
        for (long long i0 = 0; i0 < n4; i0 += 4 * FC_THREADS) {
          float4 t[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const long long i = i0 + q * FC_THREADS + tid;
            if (i < n4) t[q] = __ldcs(s4 + i);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const long long i = i0 + q * FC_THREADS + tid;
            if (i < n4) d4[i] = t[q];
          }
        }
        for (long long i = (n4 << 2) + tid; i < nfl; i += FC_THREADS) fc_sl[i] = __ldcs(src + i);
      } else {
        for (long long i = tid; i < nfl; i += FC_THREADS) fc_sl[i] = __ldcs(src + i);
      }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < FC_MAXJ; ++j) {
      const int r = j * FC_THREADS + tid;
      bool cand = false;
      if (r < rows) {
        float mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < KC; ++k) mx = fmaxf(mx, fc_sl[r * KC + k]);
        cand = !(mx - fc_sl[r * KC + label] > 2e-6f);      // NaNs stay candidates; the full decision rejects them
      }
      const unsigned cb = __ballot_sync(0xffffffffu, cand);
      int wbase = 0;
      if (lane == 0 && cb) wbase = atomicAdd(&nsurv, __popc(cb));
      wbase = __shfl_sync(0xffffffffu, wbase, 0);
      if (cand) surv[wbase + __popc(cb & ((1u << lane) - 1u))] = (unsigned short)r;
    }
    __syncthreads();
    for (int i = tid; i < nsurv; i += FC_THREADS) {
      const int r = surv[i];
      if (filter_decide_p<fc_pow2(KC), KC>([&](int k) { return fc_sl[r * KC + k]; }, KC, label, thr))
        atomicOr(&bitmap[r >> 5], 1u << (r & 31));
    }
    __syncthreads();
    // row j * 256 + tid sits in bit `lane` of bitmap word j * 8 + w: exactly the ballot layout
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < FC_MAXJ; ++j) {
        const unsigned bal = bitmap[j * (FC_THREADS / 32) + w];
        bals[sb][j][w] = bal;
        pref[(sb * FC_MAXJ + j) * (FC_THREADS / 32) + w] = __popc(bal);
      }
    }
    __syncthreads();
  }
  // ---- exclusive scan of the per-(sub-block, j, warp) counts; one atomic per CTA ----
  {
    const int nent = nsub * FC_MAXJ * (FC_THREADS / 32);           // <= 1024
    const int per = (nent + FC_THREADS - 1) / FC_THREADS;          // <= 4 consecutive entries per thread
    int loc[4] = {0, 0, 0, 0}, s = 0;
    for (int i = 0; i < per; ++i) {
      const int e = tid * per + i;
      loc[i] = e < nent ? pref[e] : 0;
      s += loc[i];
    }
    int incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    int woff = 0;
    for (int q = 0; q < w; ++q) woff += wsum[q];
    int run = woff + incl - s;
    for (int i = 0; i < per; ++i) {
      const int e = tid * per + i;
      if (e < nent) pref[e] = run;
      run += loc[i];
    }
    if (tid == FC_THREADS - 1) base = run ? atomicAdd(count, (unsigned long long)run) : 0ull;
    __syncthreads();
  }
  // ---- pass 2: copy the accepted rows ----
  for (int sb = 0; sb < nsub; ++sb) {
    const long long row0 = ((long long)sb * gridDim.x + blockIdx.x) * FC_SUB_ROWS;
#pragma unroll
    for (int j = 0; j < FC_MAXJ; ++j) {
      const unsigned bal = bals[sb][j][w];
      if ((bal >> lane) & 1u) {
        const long long r = row0 + j * FC_THREADS + tid;
        const long long pos = (long long)base + pref[(sb * FC_MAXJ + j) * (FC_THREADS / 32) + w] + __popc(bal & ((1u << lane) - 1u));
        if (pos < capacity) {
          const float* src = x + r * F;
          float* dst = x_out + pos * F;
          if (vec2) {
            const float2* s2 = reinterpret_cast<const float2*>(src);
            float2* d2 = reinterpret_cast<float2*>(dst);
            // all loads of a batch are in flight before the first store (a row costs one memory round trip, not F/2)
            for (int f0 = 0; f0 < (F >> 1); f0 += 8) {
              float2 t[8];
#pragma unroll
              for (int q = 0; q < 8; ++q)
                if (f0 + q < (F >> 1)) t[q] = __ldcs(s2 + f0 + q);
#pragma unroll
              for (int q = 0; q < 8; ++q)
                if (f0 + q < (F >> 1)) d2[f0 + q] = t[q];
            }
          } else {
            for (int f0 = 0; f0 < F; f0 += 8) {
              float t[8];
#pragma unroll
              for (int q = 0; q < 8; ++q)
                if (f0 + q < F) t[q] = __ldcs(src + f0 + q);
#pragma unroll
              for (int q = 0; q < 8; ++q)
                if (f0 + q < F) dst[f0 + q] = t[q];
            }
          }
          if (idx_out) idx_out[pos] = (long long)(row_offset + (uint64_t)r);
        }
      }
    }
  }
}

}  // namespace cvg
