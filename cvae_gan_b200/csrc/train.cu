// cvaegan_b200 - the three optimiser steps of a label visit (cvae_gan.py:104-216), as sequences of
// fused kernels on one stream.  Data parallel: batch rows are sharded; BatchNorm batch moments and
// the flat gradient buffers are all-reduced with NCCL between / after the kernels.
#include <dlfcn.h>
#include <math.h>

#include "chain.cuh"
#include "engine.cuh"
#include "mega.cuh"

namespace cvg {

// next op has no dependency on the ops of the current phase (step-program kernel only; a stream orders launches anyway)
#define CVG_PAR(e) do { (e).mk.par_next = true; } while (0)

// ------------------------------------------------------------------------------------------------
// NCCL, resolved at run time from the libnccl.so.2 that torch already loaded (no link dependency).
// ------------------------------------------------------------------------------------------------
struct Id128 {
  char b[128];   // ncclUniqueId is a 128-byte opaque struct passed by value
};
struct NcclApi {
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, Id128, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
};
static NcclApi g_nccl;

static int load_nccl() {
  if (g_nccl.ok) return 0;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) CVG_FAIL(std::string("cannot load libnccl: ") + dlerror());
  *(void**)&g_nccl.GetUniqueId = dlsym(h, "ncclGetUniqueId");
  *(void**)&g_nccl.CommInitRank = dlsym(h, "ncclCommInitRank");
  *(void**)&g_nccl.AllReduce = dlsym(h, "ncclAllReduce");
  *(void**)&g_nccl.CommDestroy = dlsym(h, "ncclCommDestroy");
  *(void**)&g_nccl.GetErrorString = dlsym(h, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce) CVG_FAIL("libnccl lacks required symbols");
  g_nccl.ok = true;
  return 0;
}

int comm_unique_id(void* out128) {
  CVG_TRY(load_nccl());
  int r = g_nccl.GetUniqueId(out128);
  if (r != 0) CVG_FAIL(std::string("ncclGetUniqueId: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"));
  return 0;
}

int comm_init(Engine& e, const void* id128, int rank, int world) {
  CVG_TRY(load_nccl());
  Id128 id;
  memcpy(id.b, id128, 128);
  int r = g_nccl.CommInitRank(&e.comm, world, id, rank);
  if (r != 0) CVG_FAIL(std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"));
  e.world = world;
  e.rank = rank;
  return 0;
}

void comm_destroy(Engine& e) {
  if (e.comm && g_nccl.CommDestroy) g_nccl.CommDestroy(e.comm);
  e.comm = nullptr;
}

// ------------------------------------------------------------------------------------------------
// NVLink peer-memory all-reduce (comm_nvl.cuh): staging buffer creation, CUDA IPC attach, launch
// ------------------------------------------------------------------------------------------------
int nvl_local_handle(Engine& e, void* out64) {
  if (e.world <= 1 || e.world > NVL_MAX_WORLD) CVG_FAIL("cvg_nvl_local_handle: world_size must be in [2, 8]");
  if (e.nvl.local) CVG_FAIL("cvg_nvl_local_handle: already created");
  size_t slot = (size_t)2 * 2 * STAT_C * sizeof(double);            // BatchNorm moments [2 passes][2][STAT_C]
  for (int net = 0; net < 4; ++net) {
    const size_t b = (size_t)(e.lay[net].n_param + CVG_GRAD_TAIL) * sizeof(float);
    if (b > slot) slot = b;
  }
  slot = 2 * ((slot + 255) & ~(size_t)255);      // LL packets: 8 bytes on the wire per 4-byte word
  const size_t total = (nvl_total_bytes(e.world, slot) + 255) & ~(size_t)255;      // one channel; two are allocated
  CVG_CUDA(cudaMalloc(&e.nvl.local, 3 * total));     // communication staging only (never tensor memory)
  CVG_CUDA(cudaMemset(e.nvl.local, 0, 3 * total));
  CVG_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  CVG_CUDA(cudaIpcGetMemHandle(&h, e.nvl.local));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  memcpy(out64, &h, 64);
  e.nvl.total_bytes = total;
  NvlDev& d = e.nvl.dev;
  d.world = e.world;
  d.rank = e.rank;
  d.slot_bytes = slot;
  d.peer[e.rank] = (unsigned char*)e.nvl.local;
  unsigned char* tail = (unsigned char*)e.nvl.local + 2 * (size_t)e.world * slot + 2 * (size_t)e.world * NVL_MAX_CTAS * sizeof(unsigned int);
  d.epoch = (unsigned long long*)tail;
  d.done = (unsigned int*)(tail + 64);
  NvlDev& d1 = e.nvl.dev1;
  d1 = d;
  d1.peer[e.rank] = d.peer[e.rank] + total;
  d1.epoch = (unsigned long long*)(tail + total);
  d1.done = (unsigned int*)(tail + total + 64);
  NvlDev& d2 = e.nvl.dev2;
  d2 = d;
  d2.peer[e.rank] = d.peer[e.rank] + 2 * total;
  d2.epoch = (unsigned long long*)(tail + 2 * total);
  d2.done = (unsigned int*)(tail + 2 * total + 64);
  return 0;
}

int nvl_attach(Engine& e, const void* handles) {
  if (!e.nvl.local) CVG_FAIL("cvg_nvl_attach: call cvg_nvl_local_handle first");
  for (int p = 0; p < e.world; ++p) {
    if (p == e.rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + (size_t)p * 64, 64);
    void* ptr = nullptr;
    CVG_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    e.nvl.dev.peer[p] = (unsigned char*)ptr;
    e.nvl.dev1.peer[p] = (unsigned char*)ptr + e.nvl.total_bytes;
    e.nvl.dev2.peer[p] = (unsigned char*)ptr + 2 * e.nvl.total_bytes;
    e.nvl.opened[p] = true;
  }
  CVG_CUDA(cudaMalloc(&e.nvl.dev_d[0], 2 * sizeof(NvlDev)));
  e.nvl.dev_d[1] = e.nvl.dev_d[0] + 1;
  CVG_CUDA(cudaMemcpy(e.nvl.dev_d[0], &e.nvl.dev, sizeof(NvlDev), cudaMemcpyHostToDevice));
  CVG_CUDA(cudaMemcpy(e.nvl.dev_d[1], &e.nvl.dev1, sizeof(NvlDev), cudaMemcpyHostToDevice));
  if (const char* f = getenv("CVG_FUSE_STATS")) e.nvl.fuse = atoi(f) != 0;
  // one-CTA polling (gemm.cuh bn_publish): measured slower than every CTA polling even at 8 ranks (4.51 vs 4.45 ms per
  // visit), so it stays an option
  e.nvl.via_lead = false;
  if (const char* f = getenv("CVG_POLL_LEAD")) e.nvl.via_lead = atoi(f) != 0;
  e.nvl.on = true;
  return 0;
}

void nvl_destroy(Engine& e) {
  for (int p = 0; p < NVL_MAX_WORLD; ++p)
    if (e.nvl.opened[p]) { cudaIpcCloseMemHandle(e.nvl.dev.peer[p]); e.nvl.opened[p] = false; }
  if (e.nvl.local) cudaFree(e.nvl.local);
  if (e.nvl.dev_d[0]) cudaFree(e.nvl.dev_d[0]);
  e.nvl.dev_d[0] = e.nvl.dev_d[1] = nullptr;
  e.nvl.local = nullptr;
  e.nvl.on = false;
}

// `nseg` segments of `seg_len` elements, `seg_stride` apart
template <typename T>
static int nvl_all_reduce(Engine& e, T* p, int64_t seg_len, int64_t seg_stride, int nseg, cudaStream_t st, int channel = 0) {
  const long long n = seg_len * nseg;
  if (e.mk.recording) {
    mk::NvlArgs a;
    a.data = p; a.seg_len = seg_len; a.seg_stride = seg_stride; a.nseg = nseg;
    a.exchange = e.mk.n_exchanges++;
    if ((unsigned long long)n * sizeof(T) * 2 > e.nvl.dev.slot_bytes) CVG_FAIL("step program: exchange larger than the NVLink staging slot");
    return mk_push(e, sizeof(T) == 8 ? mk::K_NVL_F64 : mk::K_NVL_F32, &a, sizeof(a), mk::NVL_VB);
  }
  if (e.nvl.n_pending && channel == 0) CVG_FAIL("internal: a folded BatchNorm exchange has no reader before the next exchange");
  int grid = (int)((n + NVL_THREADS - 1) / NVL_THREADS);     // one element per thread where possible
  if (grid < 1) grid = 1;
  if (grid > NVL_MAX_CTAS) grid = NVL_MAX_CTAS;
  nvl_allreduce_kernel<T><<<grid, NVL_THREADS, 0, st>>>(channel == 2 ? e.nvl.dev2 : (channel == 1 ? e.nvl.dev1 : e.nvl.dev), p, seg_len,
                                                        seg_stride, nseg);
  CVG_CUDA(cudaGetLastError());
  e.launches++;
  return 0;
}

// BatchNorm moments: per pass a slot of 2 * STAT_C doubles holding [sum (C)][sum of squares (C)] contiguously
int comm_all_reduce_stats(Engine& e, double* p, int npass, int C, cudaStream_t st) {
  if (e.world <= 1) return 0;
  if (e.nvl.on) return nvl_all_reduce<double>(e, p, 2 * C, 2 * STAT_C, npass, st);
  return comm_all_reduce_f64(e, p, (int64_t)npass * 2 * STAT_C, st);
}

int comm_all_reduce_f32(Engine& e, float* p, int64_t n, cudaStream_t st, int channel) {
  if (e.world <= 1) return 0;
  if (e.nvl.on && 2 * (size_t)n * sizeof(float) <= e.nvl.dev.slot_bytes) return nvl_all_reduce<float>(e, p, n, n, 1, st, channel);
  if (channel != 0) CVG_FAIL("internal: NCCL reduction requested on a side stream");
  if (!e.comm) CVG_FAIL("world_size > 1 but cvg_comm_init was not called");
  int r = g_nccl.AllReduce(p, p, (size_t)n, /*ncclFloat32*/ 7, /*ncclSum*/ 0, e.comm, st);
  if (r != 0) CVG_FAIL("ncclAllReduce(f32) failed");
  return 0;
}
int comm_all_reduce_f64(Engine& e, double* p, int64_t n, cudaStream_t st) {
  if (e.world <= 1) return 0;
  if (e.nvl.on && 2 * (size_t)n * sizeof(double) <= e.nvl.dev.slot_bytes) return nvl_all_reduce<double>(e, p, n, n, 1, st);
  if (!e.comm) CVG_FAIL("world_size > 1 but cvg_comm_init was not called");
  int r = g_nccl.AllReduce(p, p, (size_t)n, /*ncclFloat64*/ 8, /*ncclSum*/ 0, e.comm, st);
  if (r != 0) CVG_FAIL("ncclAllReduce(f64) failed");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------
#ifndef CVG_LAUNCH_CHECK
#define CVG_LAUNCH_CHECK()                 \
  do {                                     \
    CVG_CUDA(cudaGetLastError());          \
    e.launches++;                          \
  } while (0)
#endif

static void prof_begin(Engine& e, int cls, double flops, cudaStream_t st) {
  if (!e.prof) return;
  ProfRec r;
  cudaEventCreate(&r.a);
  cudaEventCreate(&r.b);
  r.cls = cls;
  r.flops = flops;
  cudaEventRecord(r.a, st);
  e.prof_recs.push_back(r);
}
static void prof_end(Engine& e, cudaStream_t st) {
  if (!e.prof) return;
  cudaEventRecord(e.prof_recs.back().b, st);
}

// first reader of batch sums a producer pushed over NVLink (launch_mn_stats below): it polls the packets
static const NvlDev* take_pending(Engine& e, Operand& o) {
  if (!e.nvl.n_pending || (o.kind != OP_BN_ACT && o.kind != OP_BN_BWD)) return nullptr;
  for (int i = 0; i < e.nvl.n_pending; ++i) {
    const NvlPending pd = e.nvl.pending[i];
    int which = 0;
    if (pd.stats == o.bn.fstats + (long long)pd.pass0 * o.bn.sf) which = 1;
    if (o.kind == OP_BN_BWD && pd.stats == o.bn.bstats + (long long)pd.pass0 * o.bn.sb) which = 2;
    if (!which) continue;
    o.bn.poll = which | (pd.npass << 4) | (pd.pass0 << 12) | (e.nvl.via_lead ? 1 << 20 : 0);
    e.nvl.pending[i] = e.nvl.pending[--e.nvl.n_pending];
    return e.nvl.dev_d[pd.channel];
  }
  return nullptr;
}

int launch_mn(Engine& e, bool wt, const GemmArgs& g_in, cudaStream_t st) {
  GemmArgs g = g_in;
  if (!e.mk.recording)
    if (const NvlDev* ch = take_pending(e, g.a)) g.nvl = ch;
  const int zp = g.only_pass >= 0 ? 1 : g.npass;
  if (e.mk.recording) {
    // 64-row tiles while they still fit one wave and a half of CTAs, 128-row tiles (full-rate MMAs) for larger batches
    const int nmt = (g.N + 127) / 128;
    int Nt = 64;
    if ((long long)((g.M + 63) / 64) * nmt * zp > 3 * e.num_sms / 2) Nt = 128;
    if (const char* f = getenv("CVG_MK_NT")) { if (atoi(f) == 128 && g.M > 64) Nt = 128; if (atoi(f) == 64) Nt = 64; }
    const int items = zp * nmt * ((g.M + Nt - 1) / Nt);
    const bool par = e.mk.par_next;
    const float* wp = nullptr;
    bool prepped_now = false;
    CVG_TRY(mk_weight_operand(e, g, wt, &wp, &prepped_now));   // may emit a prep op into the current phase ...
    e.mk.par_next = par && !prepped_now;                       // ... which this GEMM must then wait for
    return mk_push(e, mk::K_MN, &g, GEMM_ARGS_OP_BYTES, items, wt ? 1 : 0, Nt, 0, 0, &wp, sizeof(wp));
  }
  dim3 grid((g.M + TBM - 1) / TBM, (g.N + TBN - 1) / TBN, zp);
  const size_t smem = gemm_mn_smem(g);
  prof_begin(e, wt ? 0 : 1, 2.0 * g.M * (double)g.N * g.R * zp, st);
  const cudaError_t err = dispatch_mn(wt, g, grid, smem, st);
  prof_end(e, st);
  if (err != cudaSuccess)
    CVG_FAIL(std::string("gemm_mn launch (a.kind ") + std::to_string(g.a.kind) + ", ekind " + std::to_string(g.ekind) +
             "): " + cudaGetErrorString(err));
  e.launches++;
  return 0;
}

// the deterministic-reduction slot set of the stream a stand-alone kernel is launched on (Workspace::det_acc)
static int det_slot(const Engine& e, cudaStream_t st) {
  for (int i = 0; i < SIDE_STREAMS; ++i)
    if (st == e.ms.s[i]) return 1 + i;
  return 0;
}

int launch_dw(Engine& e, const DwArgs& g0, cudaStream_t st) {
  if (e.mk.recording) return mk_push_dw(e, g0);
  DwArgs g = g0;
  const int kt = (g.K + 63) / 64, nt = (g.N + 63) / 64;
  const int target = 2 * e.num_sms;
  int nsplit = (target + kt * nt * g.npass - 1) / (kt * nt * g.npass);
  const int max_split = (g.M + DW_MC - 1) / DW_MC;
  if (nsplit > max_split) nsplit = max_split;
  if (nsplit < 1) nsplit = 1;
  int rows = (g.M + nsplit - 1) / nsplit;
  rows = ((rows + DW_MC - 1) / DW_MC) * DW_MC;
  nsplit = (g.M + rows - 1) / rows;
  g.rows_per_cta = rows;
  if (const NvlDev* ch = take_pending(e, g.p)) g.nvl = ch;
  if (const NvlDev* ch = take_pending(e, g.q)) g.nvl = ch;
  dim3 grid(kt, nt, g.npass * nsplit);
  if ((long long)kt * nt * g.npass * DW_PART > e.ws.det_acc_n || kt * nt > e.ws.det_cnt_n)
    CVG_FAIL("internal: weight-gradient launch exceeds the deterministic-reduction slots");
  const int slot = det_slot(e, st);
  prof_begin(e, 2, 2.0 * g.M * (double)g.N * g.K * g.npass, st);
  const cudaError_t err = dispatch_dw(g, nsplit, e.ws.det_acc[slot], e.ws.det_cnt[slot], grid, gemm_dw_smem(g), st);
  prof_end(e, st);
  if (err != cudaSuccess)
    CVG_FAIL(std::string("gemm_dw launch (p.kind ") + std::to_string(g.p.kind) + ", q.kind " + std::to_string(g.q.kind) +
             "): " + cudaGetErrorString(err));
  e.launches++;
  return 0;
}

static const LinearP& lin(const Engine& e, int net, int l) { return e.lay[net].lin[l]; }

// One-hot concat of the first Linear of E / G / D == adding weight column (input width + label) to the bias (appendix A.1);
// unconditional networks (CvgConfig.unconditional, the VAE-GAN sibling) have no such columns.
static const float* label_column(const Engine& e, int net, const LinearP& p, int in_width, int label) {
  return e.Kc > 0 ? e.P(net, p.w) + in_width + label : nullptr;
}
static int label_col_index(const Engine& e, int in_width, int label) { return e.Kc > 0 ? in_width + label : -1; }

static double* fst_of(const Engine& e, int net, int l) {
  return net == CVG_NET_GENERATOR ? e.ws.g_fst + (size_t)l * 2 * 2 * STAT_C : e.ws.e_fst + (size_t)l * 2 * STAT_C;
}
static double* bst_of(const Engine& e, int net, int l) {
  return net == CVG_NET_GENERATOR ? e.ws.g_bst + (size_t)l * 2 * 2 * STAT_C : e.ws.e_bst + (size_t)l * 2 * STAT_C;
}

static BnRef bn_ref(const Engine& e, int net, int l, bool eval, bool update) {
  const LinearP& p = lin(e, net, l);
  BnRef b;
  b.fstats = fst_of(e, net, l);
  b.sf = 2 * STAT_C;
  b.bstats = bst_of(e, net, l);
  b.sb = 2 * STAT_C;
  b.gamma = e.P(net, p.gamma);
  b.beta = e.P(net, p.beta);
  b.rmean = e.S(net, p.rmean);
  b.rvar = e.S(net, p.rvar);
  b.C = p.out;
  b.eval = eval ? 1 : 0;
  b.update_running = (update && !eval) ? 1 : 0;
  return b;
}

static GemmArgs base_args(const Engine& e, int M, float Bg_bn, int npass) {
  GemmArgs g;
  g.M = M;
  g.ld = e.ws.ld;
  g.npass = npass;
  g.Bg = Bg_bn;
  g.bn_eps = e.cfg.bn_eps;
  g.momentum = e.cfg.bn_momentum;
  g.slope = e.cfg.lrelu_slope;
  return g;
}

static DwArgs base_dw(const Engine& e, int M, float Bg_bn, int npass) {
  DwArgs g;
  g.M = M;
  g.ld = e.ws.ld;
  g.npass = npass;
  g.Bg = Bg_bn;
  g.bn_eps = e.cfg.bn_eps;
  g.slope = e.cfg.lrelu_slope;
  return g;
}

static int sync_stats(Engine& e, double* p, int npass, int C, bool local_bn, cudaStream_t st) {
  if (e.world <= 1 || local_bn) return 0;
  return comm_all_reduce_stats(e, p, npass, C, st);
}

// Data parallel BatchNorm sums without a launch of their own (comm_nvl.cuh): the producing GEMM pushes them from its
// last CTA (g.push), the first GEMM that reads them polls (BnRef::poll, set by take_pending at its launch).
static bool fold_stats(const Engine& e, bool local_bn) {
  return e.world > 1 && !local_bn && e.nvl.on && e.nvl.fuse && e.nvl.dev_d[0] && !e.mk.recording;
}
// channel: 0 on the caller's stream, 1 on the side stream that runs a second GEMM chain beside it
static int launch_mn_stats(Engine& e, bool wt, GemmArgs& g, int npass_sync, bool local_bn, cudaStream_t st, int channel = 0) {
  const bool fold = fold_stats(e, local_bn);
  if (!fold && channel != 0 && e.world > 1 && !local_bn) CVG_FAIL("internal: an exchange launch on a side stream");
  if (fold) { g.push = 1; g.nvl = e.nvl.dev_d[channel]; }
  CVG_TRY(launch_mn(e, wt, g, st));
  if (!fold) return sync_stats(e, g.ostats, npass_sync, g.N, local_bn, st);
  if (e.nvl.n_pending >= 8) CVG_FAIL("internal: too many folded exchanges in flight");
  const int p0 = g.only_pass > 0 ? g.only_pass : 0;
  e.nvl.pending[e.nvl.n_pending++] = NvlPending{g.ostats + (long long)p0 * g.sostats, g.only_pass >= 0 ? 1 : g.npass, p0, channel};
  return 0;
}

// ------------------------------------------------------------------------------------------------
// noise + inputs
// ------------------------------------------------------------------------------------------------
// side stream `i`, ordered after everything enqueued on `st` so far (SideStreams, engine.cuh)
static cudaStream_t fork_to(Engine& e, int i, cudaStream_t st) {
  if (!e.ms.on || e.mk.recording) return st;
  cudaEvent_t ev = e.ms.ev[e.ms.next++ % SIDE_EVENTS];
  cudaEventRecord(ev, st);
  cudaStreamWaitEvent(e.ms.s[i], ev, 0);
  e.ms.dirty[i] = true;
  return e.ms.s[i];
}
// `waiter` continues after everything enqueued on `signaller` so far
static void wait_for(Engine& e, cudaStream_t waiter, cudaStream_t signaller) {
  if (waiter == signaller) return;
  cudaEvent_t ev = e.ms.ev[e.ms.next++ % SIDE_EVENTS];
  cudaEventRecord(ev, signaller);
  cudaStreamWaitEvent(waiter, ev, 0);
}
// `st` continues after everything enqueued on the side streams
static void join_sides(Engine& e, cudaStream_t st, int only = -1) {
  for (int i = 0; i < SIDE_STREAMS; ++i) {
    if (!e.ms.dirty[i] || (only >= 0 && only != i)) continue;
    cudaEvent_t ev = e.ms.ev[e.ms.next++ % SIDE_EVENTS];
    cudaEventRecord(ev, e.ms.s[i]);
    cudaStreamWaitEvent(st, ev, 0);
    e.ms.dirty[i] = false;
  }
}

static int launch_fill(Engine& e, FillArgs& a, cudaStream_t st) {
  if (a.njobs == 0) return 0;
  if (e.mk.recording) return mk_push(e, mk::K_FILL, &a, sizeof(a), a.njobs * mk::FILL_VB);
  long long mx = 0;
  for (int i = 0; i < a.njobs; ++i) {
    long long t = (long long)a.job[i].npass * ((a.job[i].nfeat + 3) / 4) * a.M;
    if (t > mx) mx = t;
  }
  int blocks = (int)((mx + 255) / 256);
  if (blocks > 4 * e.num_sms) blocks = 4 * e.num_sms;
  if (blocks < 1) blocks = 1;
  fill_noise_kernel<<<dim3(blocks, a.njobs), 256, 0, st>>>(a);
  CVG_LAUNCH_CHECK();
  return 0;
}

static void add_job(FillArgs& a, void* out, const void* inj, int kind, int nfeat, int npass, int stream) {
  FillJob& j = a.job[a.njobs++];
  j.out = out;
  j.injected = inj;
  j.kind = kind;
  j.nfeat = nfeat;
  j.npass = npass;
  j.stream = stream;
  j.cstep = 0;
}

static int emit_zero(Engine& e, void* p, size_t bytes, cudaStream_t st) {
  if (e.mk.recording) {
    mk::ZeroArgs a;
    a.p = p; a.bytes = (long long)bytes;
    const int items = (int)((bytes / 16 + mk::THREADS * 8 - 1) / (mk::THREADS * 8));
    return mk_push(e, mk::K_ZERO, &a, sizeof(a), items < 1 ? 1 : items);
  }
  CVG_CUDA(cudaMemsetAsync(p, 0, bytes, st));
  return 0;
}

static int stage_x(Engine& e, const float* x_real, int M, cudaStream_t st) {
  if (e.mk.recording) {
    // inside a visit program the batch is drawn from the class table right here (cvae_gan.py:247-260)
    const MkState& src = e.mk;
    mk::StageArgs a;
    memset(&a, 0, sizeof(a));
    a.src = src.src_rows ? src.src_rows : x_real;
    a.n_rows = src.src_rows ? src.src_n : 0;
    a.B_global = src.src_Bg; a.draw_offset = src.src_off;
    a.M = M; a.F = e.F; a.ld = e.ws.ld;
    a.ctl = e.ws.ctl; a.counter_off = e.mk.dcounter;
    a.xT = e.ws.xT;
    return mk_push(e, mk::K_STAGE, &a, sizeof(a), (M + mk::THREADS - 1) / mk::THREADS);
  }
  to_feature_major_kernel<<<(M + 127) / 128, 128, 0, st>>>(x_real, nullptr, M, e.F, e.ws.ld, e.ws.xT);
  CVG_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// forward passes
// ------------------------------------------------------------------------------------------------
int fwd_generator(Engine& e, int npass, bool train, bool reparam_pass0, int label, int M, float Bg, bool local_bn,
                  cudaStream_t st, const GenBufs* gb, const GenSplit* split) {
  const int net = CVG_NET_GENERATOR;
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  GenBufs b;
  if (gb) {
    b = *gb;
  } else {
    b.z = w.z; b.out = w.g_out;
    for (int l = 0; l < 3; ++l) { b.h[l] = w.g_h[l]; b.fst[l] = fst_of(e, net, l); }
  }
  for (int l = 0; l < 4; ++l) {
    const LinearP& p = lin(e, net, l);
    GemmArgs g = base_args(e, M, Bg, npass);
    g.R = (l == 0) ? e.Z : p.in;
    g.N = p.out;
    if (l == 0) {
      g.a.kind = (reparam_pass0 && !e.mk.recording) ? OP_REPARAM : OP_PLAIN;
      g.a.rows = e.Z;
      g.a.p = b.z;
      g.a.sp = (long long)e.Z * ld;
      g.a.mu = w.e_ml;
      g.a.lv = w.e_ml + (size_t)e.Z * ld;
      g.a.eps = w.z;
      g.a.reparam_pass = reparam_pass0 ? 0 : -1;
      g.wlabel = label_column(e, net, p, e.Z, label);   // one-hot concat == adding column Z+label (appendix A.1)
      g.ldwl = p.in;
    } else {
      g.a.kind = OP_BN_ACT;
      g.a.rows = p.in;
      g.a.p = b.h[l - 1];
      g.a.sp = (long long)p.in * ld;
      g.a.bn = bn_ref(e, net, l - 1, !train, true);
      g.a.bn.fstats = b.fst[l - 1];
    }
    g.W = e.P(net, p.w);
    g.ldw = p.in;
    g.bias = e.P(net, p.b);
    if (l < 3) {
      g.Y = b.h[l];
      g.sY = (long long)p.out * ld;
      if (train) {
        g.ostats = b.fst[l];
        g.sostats = 2 * STAT_C;
      }
    } else {
      g.act = ACT_SIGMOID;
      g.Y = b.out;
      g.sY = (long long)e.F * ld;
    }
    if (split) {
      // The z_enc pass applies the running-statistics update of BOTH passes, in the reference's order (z_enc, then
      // z_prior): it waits until the z_prior chain's reader of the same sums is done (their global values are in place).
      g.only_pass = split->only_pass;
      if (l > 0) g.a.bn.update_running = (split->only_pass == 0 && train) ? 1 : 0;
      if (l > 0 && split->wait) cudaStreamWaitEvent(st, split->wait[l], 0);
    }
    if (l < 3 && train) {
      CVG_TRY(launch_mn_stats(e, true, g, npass > 2 ? npass : 2, local_bn, st, split ? split->channel : 0));
    } else {
      CVG_TRY(launch_mn(e, true, g, st));
    }
    if (split && split->rec) cudaEventRecord(split->rec[l], st);
  }
  return 0;
}

int fwd_encoder(Engine& e, bool train, int label, int M, float Bg, bool local_bn, cudaStream_t st) {
  const int net = CVG_NET_ENCODER;
  const Workspace& w = e.ws;
  for (int l = 0; l < 4; ++l) {
    const LinearP& p = lin(e, net, l);
    GemmArgs g = base_args(e, M, Bg, 1);
    g.R = (l == 0) ? e.F : p.in;
    g.N = p.out;
    if (l == 0) {
      g.a.kind = OP_PLAIN;
      g.a.rows = e.F;
      g.a.p = w.xT;
      g.wlabel = label_column(e, net, p, e.F, label);
      g.ldwl = p.in;
    } else {
      g.a.kind = OP_BN_ACT;
      g.a.rows = p.in;
      g.a.p = w.e_h[l - 1];
      g.a.bn = bn_ref(e, net, l - 1, !train, true);
    }
    g.W = e.P(net, p.w);
    g.ldw = p.in;
    g.bias = e.P(net, p.b);
    if (l < 3) {
      g.Y = w.e_h[l];
      if (train) {
        g.ostats = fst_of(e, net, l);
        g.sostats = 2 * STAT_C;
      }
    } else {
      g.Y = w.e_ml;
      if (train) {
        g.kl_acc = w.loss + L_KL;
        g.kl_split = e.Z;
      }
    }
    if (l < 3 && train) {
      CVG_TRY(launch_mn_stats(e, true, g, 1, local_bn, st));
    } else {
      CVG_TRY(launch_mn(e, true, g, st));
    }
  }
  return 0;
}

constexpr int SN_W_SMEM_MAX = 160 * 1024;   // widest critic layer kept in shared memory by the power iteration (128 x 256 floats)
static int launch_sn(Engine& e, int npass, bool do_power, cudaStream_t st) {
  const int net = CVG_NET_DISCRIMINATOR;
  SnArgs a;
  int off = 0;
  for (int l = 0; l < 4; ++l) {
    const LinearP& p = lin(e, net, l);
    a.L[l].W = e.P(net, p.w);
    a.L[l].rows = p.out;
    a.L[l].cols = p.in;
    a.L[l].u = e.S(net, p.u);
    a.L[l].v = e.S(net, p.v);
    a.L[l].snap_off = off;
    off += ((p.out > p.in ? p.out : p.in) + 3) & ~3;
  }
  a.npass = npass;
  a.do_power = do_power ? 1 : 0;
  a.eps = e.cfg.sn_eps;
  a.sigma = e.ws.sn_sigma;
  a.inv_sigma = e.ws.sn_inv_sigma;
  a.u_snap = e.ws.sn_u;
  a.v_snap = e.ws.sn_v;
  a.ssnap = e.ws.sn_snap;
  if (e.mk.recording) return mk_push(e, mk::K_SN_POWER, &a, sizeof(a), 4);
  int wmax = 0;
  for (int l = 0; l < 4; ++l) wmax = a.L[l].rows * a.L[l].cols > wmax ? a.L[l].rows * a.L[l].cols : wmax;
  a.w_smem_floats = wmax * 4 <= SN_W_SMEM_MAX ? wmax : 0;
  sn_power_kernel<<<4, SN_THREADS, (size_t)a.w_smem_floats * sizeof(float), st>>>(a);
  CVG_LAUNCH_CHECK();
  return 0;
}

// critic forward (train mode).  xin: feature-major [F][ld] (+ pass * sxin).
static int fwd_critic(Engine& e, const float* xin, long long sxin, int npass, int label, int M, double* osum,
                      cudaStream_t st) {
  const int net = CVG_NET_DISCRIMINATOR;
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const float keep_inv = 1.0f / (1.0f - e.cfg.dropout_p);
  for (int l = 0; l < 4; ++l) {
    const LinearP& p = lin(e, net, l);
    GemmArgs g = base_args(e, M, (float)M, npass);
    g.R = (l == 0) ? e.F : p.in;
    g.N = p.out;
    g.a.kind = OP_PLAIN;
    g.a.rows = g.R;
    if (l == 0) {
      g.a.p = xin;
      g.a.sp = sxin;
      g.wlabel = label_column(e, net, p, e.F, label);
      g.ldwl = p.in;
    } else {
      g.a.p = w.d_a[l - 1];
      g.a.sp = (long long)p.in * ld;
    }
    g.W = e.P(net, p.w);
    g.ldw = p.in;
    g.bias = e.P(net, p.b);
    g.scale = w.sn_inv_sigma + l * 2;
    if (l < 3) {
      g.act = ACT_LRELU;
      g.Y = w.d_a[l];
      g.sY = (long long)p.out * ld;
      if (l == 0) { g.mask = w.d_m1; g.smask = (long long)p.out * ld; g.keep_inv = keep_inv; }
      if (l == 1) { g.mask = w.d_m2; g.smask = (long long)p.out * ld; g.keep_inv = keep_inv; }
    } else {
      g.Y = w.d_s;
      g.sY = (long long)ld;
      g.osum = osum;
    }
    CVG_TRY(launch_mn(e, true, g, st));
  }
  return 0;
}

int fwd_classifier(Engine& e, const float* xin, long long sxin, int npass, bool train, int M, cudaStream_t st) {
  const int net = CVG_NET_CLASSIFIER;
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const float keep_inv = 1.0f / (1.0f - e.cfg.dropout_p);
  for (int l = 0; l < 4; ++l) {
    const LinearP& p = lin(e, net, l);
    GemmArgs g = base_args(e, M, (float)M, npass);
    g.R = p.in;
    g.N = p.out;
    g.a.kind = OP_PLAIN;
    g.a.rows = p.in;
    g.W = e.P(net, p.w);
    g.ldw = p.in;
    g.bias = e.P(net, p.b);
    g.sY = (long long)p.out * ld;
    if (l == 0) {
      g.a.p = xin; g.a.sp = sxin;
      g.act = ACT_RELU;
      g.Y = w.c_a1;
      if (train) { g.mask = w.c_m1; g.smask = (long long)p.out * ld; g.keep_inv = keep_inv; }
    } else if (l == 1) {
      g.a.p = w.c_a1; g.a.sp = (long long)p.in * ld;
      g.Y = w.c_h2;
    } else if (l == 2) {
      g.a.p = w.c_a2; g.a.sp = (long long)p.in * ld;
      g.act = ACT_RELU;
      g.Y = w.c_a3;
    } else {
      g.a.p = w.c_a3; g.a.sp = (long long)p.in * ld;
      g.Y = w.c_logit;
    }
    CVG_TRY(launch_mn(e, true, g, st));
    if (l == 1) {
      LnArgs a;
      a.M = M; a.ld = w.ld; a.C = p.out; a.npass = npass;
      a.h = w.c_h2; a.sh = (long long)p.out * ld;
      a.g = e.P(net, p.gamma); a.b = e.P(net, p.beta);
      a.eps = e.cfg.ln_eps;
      a.mask = train ? w.c_m2 : nullptr; a.smask = (long long)p.out * ld; a.keep_inv = keep_inv;
      a.a = w.c_a2; a.sa = (long long)p.out * ld;
      a.rs = w.c_rs; a.srs = 2 * (long long)ld;
      if (e.mk.recording) {
        CVG_TRY(mk_push(e, mk::K_LN_FWD, &a, sizeof(a), npass * ((M + 31) / 32)));
      } else {
        launch_ln_fwd(a, st);
        CVG_LAUNCH_CHECK();
      }
    }
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// fused row-tile chains of the D and C steps (chain.cuh)
// ------------------------------------------------------------------------------------------------
// Used where the layer kernels would otherwise run stand-alone (the step-program kernel records layer ops) and at the widths
// the chains are built for; the widened model (CvgConfig.hidden) keeps the layer kernels.
static bool chain_usable(const Engine& e, int net) {
  if (!e.chain || e.mk.recording) return false;
  const int* h = net == CVG_NET_DISCRIMINATOR ? e.dh : e.ch;
  return h[0] == CH_H0 && h[1] == CH_H1 && h[2] == CH_H2 && e.F <= CH_MAX_IN && e.K <= CH_MAX_K;
}

// After a chain the weight gradients of the four layers are independent of each other: the largest (layer 1) runs on the
// caller's stream, the others beside it on the side streams (each stream has its own deterministic-reduction slot).
static cudaStream_t chain_dw_stream(Engine& e, int l, cudaStream_t st) { return l == 1 ? st : fork_to(e, l == 2 ? 1 : 0, st); }

// Critic forward (score sums into loss[L_DREAL + pass]) and input gradients from the per-pass seed, both passes, one launch.
static int launch_critic_chain(Engine& e, long long sx, int label, int M, const float* seed, cudaStream_t st) {
  const int net = CVG_NET_DISCRIMINATOR;
  const Workspace& w = e.ws;
  CriticChainArgs a;
  a.M = M; a.ld = w.ld; a.F = e.F;
  a.x = w.xT; a.sx = sx;
  double flops = 0.0;
  for (int l = 0; l < 4; ++l) {
    const LinearP& p = lin(e, net, l);
    a.W[l] = e.P(net, p.w); a.ldw[l] = p.in; a.b[l] = e.P(net, p.b);
    flops += 2.0 * ((l == 0) ? e.F : p.in) * p.out + (l > 0 ? 2.0 * p.in * p.out : 0.0);
  }
  a.wlabel = label_column(e, net, lin(e, net, 0), e.F, label);
  a.ldwl = lin(e, net, 0).in;
  a.inv_sigma = w.sn_inv_sigma;
  a.m1 = w.d_m1; a.m2 = w.d_m2;
  a.keep_inv = 1.0f / (1.0f - e.cfg.dropout_p);
  a.slope = e.cfg.lrelu_slope;
  for (int i = 0; i < 3; ++i) { a.a[i] = w.d_a[i]; a.g[i] = w.d_g[i]; }
  a.s = w.d_s;
  a.osum = w.loss + L_DREAL;
  a.seed[0] = seed[0]; a.seed[1] = seed[1];
  const dim3 grid(2 * ((M + TBM - 1) / TBM), 2);
  prof_begin(e, 3, flops * 2 * M, st);
  critic_chain_kernel<<<grid, CH_THREADS, critic_chain_smem(e.F), st>>>(a);
  prof_end(e, st);
  CVG_LAUNCH_CHECK();
  return 0;
}

// Classifier forward, cross-entropy with the step's label (loss[L_CE0 + pass]), input gradients with the LayerNorm backward
// and its affine gradients, both passes, one launch.
static int launch_classifier_chain(Engine& e, long long sx, int label, int M, float coef, cudaStream_t st) {
  const int net = CVG_NET_CLASSIFIER;
  const Workspace& w = e.ws;
  ClassifierChainArgs a;
  a.M = M; a.ld = w.ld; a.F = e.F; a.K = e.K; a.label = label;
  a.x = w.xT; a.sx = sx;
  double flops = 0.0;
  for (int l = 0; l < 4; ++l) {
    const LinearP& p = lin(e, net, l);
    a.W[l] = e.P(net, p.w); a.b[l] = e.P(net, p.b);
    flops += 2.0 * p.in * p.out * (l > 0 ? 2.0 : 1.0);
  }
  const LinearP& p1 = lin(e, net, 1);
  a.gamma = e.P(net, p1.gamma); a.beta = e.P(net, p1.beta);
  a.ln_eps = e.cfg.ln_eps;
  a.m1 = w.c_m1; a.m2 = w.c_m2;
  a.keep_inv = 1.0f / (1.0f - e.cfg.dropout_p);
  a.a1 = w.c_a1; a.h2 = w.c_h2; a.a2 = w.c_a2; a.rs = w.c_rs; a.a3 = w.c_a3; a.logit = w.c_logit; a.dlogit = w.c_dlogit;
  for (int i = 0; i < 3; ++i) a.g[i] = w.c_g[i];
  a.coef = coef;
  a.loss = w.loss + L_CE0;
  a.dgamma = e.G(net, p1.gamma); a.dbeta = e.G(net, p1.beta);
  const int slot = det_slot(e, st);
  if (2LL * CH_H1 > e.ws.det_acc_n) CVG_FAIL("internal: LayerNorm backward exceeds the deterministic-reduction slots");
  a.acc = e.ws.det_acc[slot]; a.cnt = e.ws.det_cnt[slot];
  const dim3 grid(2 * ((M + TBM - 1) / TBM), 2);
  prof_begin(e, 3, flops * 2 * M, st);
  classifier_chain_kernel<<<grid, CH_THREADS, classifier_chain_smem(e.F, e.K), st>>>(a);
  prof_end(e, st);
  CVG_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// backward passes
// ------------------------------------------------------------------------------------------------
// critic backward.  seed[pass] = dL/dscore (constant over rows).  want_dw: accumulate per-pass raw
// gradients into ws.sn_G (+ bias grads into the grad buffer).  want_dx: write dL/dx into ws.dx.
// dw_only: a fused chain (chain.cuh) has produced the input gradients; only the weight gradients are launched, spread over
// the streams (chain_dw_stream).
static int bwd_critic(Engine& e, const float* xin, long long sxin, int npass, int label, int M, const float* seed,
                      bool want_dw, bool want_dx, cudaStream_t st, bool dw_only = false) {
  const int net = CVG_NET_DISCRIMINATOR;
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const float keep_inv = 1.0f / (1.0f - e.cfg.dropout_p);
  const long long sG = e.lay[net].n_param;
  for (int l = 3; l >= 0; --l) {
    const LinearP& p = lin(e, net, l);
    // dY operand of this layer
    Operand dy;
    if (l == 3) {
      dy.kind = OP_CONST; dy.rows = 1; dy.cst = seed[0];
    } else {
      dy.kind = OP_PLAIN; dy.rows = p.out; dy.p = w.d_g[l]; dy.sp = (long long)p.out * ld;
    }
    if (want_dw) {
      // OP_CONST carries one value: run the two passes of layer 4 as separate launches
      const int reps = (l == 3 && npass > 1) ? npass : 1;
      // beside the input-gradient chain: both only read dY of layer l
      const cudaStream_t sw = dw_only ? chain_dw_stream(e, l, st) : fork_to(e, 0, st);
      for (int r = 0; r < reps; ++r) {
        if (r > 0) CVG_PAR(e);
        DwArgs d = base_dw(e, M, (float)M, reps > 1 ? 1 : npass);
        d.N = p.out;
        d.K = (l == 0) ? e.F : p.in;
        d.p = dy;
        if (l == 3) d.p.cst = seed[reps > 1 ? r : 0];
        d.q.kind = OP_PLAIN;
        d.q.rows = d.K;
        if (l == 0) { d.q.p = xin + (reps > 1 ? r * sxin : 0); d.q.sp = sxin; }
        else { d.q.p = w.d_a[l - 1] + (reps > 1 ? (long long)r * p.in * ld : 0); d.q.sp = (long long)p.in * ld; }
        d.dW = w.sn_G + p.w + (reps > 1 ? r * sG : 0);
        d.sdW = sG;
        d.ldw = p.in;
        d.db = (l == 3) ? nullptr : e.G(net, p.b);   // score-bias gradient is added analytically (sn_grad_kernel)
        d.label_col = (l == 0) ? label_col_index(e, e.F, label) : -1;
        CVG_TRY(launch_dw(e, d, sw));
      }
    }
    if (dw_only) continue;
    if (l == 0 && !want_dx) break;
    GemmArgs g = base_args(e, M, (float)M, npass);
    g.R = p.out;
    g.N = (l == 0) ? e.F : p.in;
    g.a = dy;
    g.W = e.P(net, p.w);
    g.ldw = p.in;
    g.scale = w.sn_inv_sigma + l * 2;
    if (want_dw) CVG_PAR(e);      // the input gradient and the weight gradient of a layer read the same dY
    if (l == 0) {
      g.ekind = EP_STORE;
      g.Y = w.dx;
      g.accumulate = 0;
      CVG_TRY(launch_mn(e, false, g, st));
    } else {
      g.ekind = EP_DACT;
      g.act = ACT_LRELU;
      g.prev = w.d_a[l - 1];
      g.sprev = (long long)p.in * ld;
      if (l - 1 == 0) { g.mask = w.d_m1; g.smask = (long long)p.in * ld; g.keep_inv = keep_inv; }
      if (l - 1 == 1) { g.mask = w.d_m2; g.smask = (long long)p.in * ld; g.keep_inv = keep_inv; }
      g.Y = w.d_g[l - 1];
      g.sY = (long long)p.in * ld;
      if (l == 3 && npass > 1) {
        for (int r = 0; r < npass; ++r) {   // per-pass constant seed
          if (r > 0) CVG_PAR(e);
          GemmArgs gr = g;
          gr.a.cst = seed[r];
          gr.only_pass = r;
          CVG_TRY(launch_mn(e, false, gr, st));
        }
      } else {
        CVG_TRY(launch_mn(e, false, g, st));
      }
    }
  }
  return 0;
}

// classifier backward from ws.c_dlogit.
// dx_after: a stream whose enqueued work writes ws.dx first (the critic's backward, when this one runs beside it).
// dw_only: as bwd_critic.
static int bwd_classifier(Engine& e, const float* xin, long long sxin, int npass, int M, bool want_dw, bool want_dx,
                          bool dx_accumulate, cudaStream_t st, cudaStream_t dx_after = nullptr, bool dw_only = false) {
  const int net = CVG_NET_CLASSIFIER;
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const float keep_inv = 1.0f / (1.0f - e.cfg.dropout_p);
  for (int l = 3; l >= 0; --l) {
    const LinearP& p = lin(e, net, l);
    Operand dy;
    dy.kind = OP_PLAIN;
    dy.rows = p.out;
    if (l == 3) { dy.p = w.c_dlogit; dy.sp = (long long)e.K * ld; }
    else { dy.p = w.c_g[l]; dy.sp = (long long)p.out * ld; }
    if (want_dw) {
      DwArgs d = base_dw(e, M, (float)M, npass);
      d.N = p.out;
      d.K = p.in;
      d.p = dy;
      d.q.kind = OP_PLAIN;
      d.q.rows = p.in;
      if (l == 0) { d.q.p = xin; d.q.sp = sxin; }
      else if (l == 1) { d.q.p = w.c_a1; d.q.sp = (long long)p.in * ld; }
      else if (l == 2) { d.q.p = w.c_a2; d.q.sp = (long long)p.in * ld; }
      else { d.q.p = w.c_a3; d.q.sp = (long long)p.in * ld; }
      d.dW = e.G(net, p.w);
      d.sdW = 0;
      d.ldw = p.in;
      d.db = e.G(net, p.b);
      CVG_TRY(launch_dw(e, d, dw_only ? chain_dw_stream(e, l, st) : fork_to(e, 0, st)));
    }
    if (dw_only) continue;
    if (l == 0 && !want_dx) break;
    if (l == 0 && dx_after) {
      wait_for(e, st, dx_after);
    }
    GemmArgs g = base_args(e, M, (float)M, npass);
    g.R = p.out;
    g.N = p.in;
    g.a = dy;
    g.W = e.P(net, p.w);
    g.ldw = p.in;
    if (l == 0) {
      g.ekind = EP_STORE;
      g.Y = w.dx;
      g.accumulate = dx_accumulate ? 1 : 0;
    } else {
      g.ekind = EP_DACT;
      g.act = ACT_RELU;
      g.sprev = (long long)p.in * ld;
      g.sY = (long long)p.in * ld;
      g.Y = w.c_g[l - 1];
      if (l == 3) g.prev = w.c_a3;
      if (l == 2) { g.prev = w.c_a2; g.mask = w.c_m2; g.smask = (long long)p.in * ld; g.keep_inv = keep_inv; }
      if (l == 1) { g.prev = w.c_a1; g.mask = w.c_m1; g.smask = (long long)p.in * ld; g.keep_inv = keep_inv; }
    }
    if (want_dw) CVG_PAR(e);
    CVG_TRY(launch_mn(e, false, g, st));
    if (l == 2) {   // c_g[1] holds dL/dn -> LayerNorm backward in place -> dL/dh2
      const LinearP& p1 = lin(e, net, 1);
      LnBwdArgs a;
      a.M = M; a.ld = w.ld; a.C = p1.out; a.npass = npass;
      a.dn = w.c_g[1]; a.sdn = (long long)p1.out * ld;
      a.h = w.c_h2; a.sh = (long long)p1.out * ld;
      a.rs = w.c_rs; a.srs = 2 * (long long)ld;
      a.g = e.P(net, p1.gamma);
      a.dg = want_dw ? e.G(net, p1.gamma) : nullptr;
      a.db = want_dw ? e.G(net, p1.beta) : nullptr;
      if (e.mk.recording) {
        CVG_TRY(mk_push(e, mk::K_LN_BWD, &a, sizeof(a), npass * ((M + 31) / 32)));
      } else {
        const int slot = det_slot(e, st);
        if (2LL * a.C > e.ws.det_acc_n) CVG_FAIL("internal: LayerNorm backward exceeds the deterministic-reduction slots");
        launch_ln_bwd(a, e.ws.det_acc[slot], e.ws.det_cnt[slot], st);
        CVG_LAUNCH_CHECK();
      }
    }
  }
  return 0;
}

// BatchNorm MLP backward shared by generator (npass 2) and encoder (npass 1).
//   top_dy      : dL/d(pre-activation of the last Linear) [Ntop][ld] per pass
//   h[], dy[]   : the net's pre-BN activations and gradient scratch
struct BnNetBwd {
  int net, npass;
  float* const* h;
  float* const* dy;
  const float* top_dy;
  long long s_top;
  Operand first_in;        // input operand of layer 0 (x, z or reparameterised z)
  int first_K;             // its width
  int label_col;
  bool want_first_dx;      // generator: dL/dz_enc of pass 0 -> encoder head gradient
};

// dY operand of layer l: the gradient w.r.t. the output of its Linear
static Operand bn_net_dy(const Engine& e, const BnNetBwd& b, int l) {
  const LinearP& p = lin(e, b.net, l);
  Operand dy;
  if (l == 3) {
    dy.kind = OP_PLAIN; dy.rows = p.out; dy.p = b.top_dy; dy.sp = b.s_top;
  } else {
    dy.kind = OP_BN_BWD; dy.rows = p.out;
    dy.p = b.dy[l]; dy.sp = (long long)p.out * e.ws.ld;
    dy.h = b.h[l]; dy.sh = (long long)p.out * e.ws.ld;
    dy.bn = bn_ref(e, b.net, l, false, false);
  }
  return dy;
}

// Input gradient of layer l: dY of layer l - 1 with its batch sums, or, at layer 0 with want_first_dx, the encoder head
// gradient (pass 0 only).  Nothing at layer 0 otherwise.  only_pass >= 0: that pass alone, in a grid of one pass slot.
static int bwd_bn_dx(Engine& e, const BnNetBwd& b, int l, int M, float Bg_bn, float kl_coef, bool local_bn, cudaStream_t st,
                     int only_pass = -1) {
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const int net = b.net;
  const LinearP& p = lin(e, net, l);
  if (l > 0) {
    const LinearP& pp = lin(e, net, l - 1);
    GemmArgs g = base_args(e, M, Bg_bn, b.npass);
    g.only_pass = only_pass;
    g.R = p.out;
    g.N = p.in;
    g.a = bn_net_dy(e, b, l);
    g.W = e.P(net, p.w);
    g.ldw = p.in;
    g.ekind = EP_DBN;
    g.prev = b.h[l - 1];
    g.sprev = (long long)pp.out * ld;
    g.prev_bn = bn_ref(e, net, l - 1, false, false);
    g.Y = b.dy[l - 1];
    g.sY = (long long)pp.out * ld;
    g.ostats = bst_of(e, net, l - 1);
    g.sostats = 2 * STAT_C;
    return launch_mn_stats(e, false, g, b.npass, local_bn, st);
  }
  if (!b.want_first_dx) return 0;
  GemmArgs g = base_args(e, M, Bg_bn, b.npass);
  g.only_pass = 0;
  g.R = p.out;
  g.N = e.Z;
  g.a = bn_net_dy(e, b, l);
  g.W = e.P(net, p.w);
  g.ldw = p.in;
  g.ekind = EP_REPARAM_BWD;
  g.mu = w.e_ml;
  g.lv = w.e_ml + (size_t)e.Z * ld;
  g.eps = e.mk.recording ? w.z_eps : w.z;
  g.kl_coef = kl_coef;
  g.Y = w.e_dml;
  return launch_mn(e, false, g, st);
}

// dW, db and the BatchNorm affine gradients of layer l, all passes in one launch
static int bwd_bn_dw(Engine& e, const BnNetBwd& b, int l, int M, float Bg_bn, bool local_bn, cudaStream_t st) {
  const int net = b.net;
  const LinearP& p = lin(e, net, l);
  DwArgs d = base_dw(e, M, Bg_bn, b.npass);
  d.N = p.out;
  d.p = bn_net_dy(e, b, l);
  if (l == 0) {
    d.K = b.first_K;
    d.q = b.first_in;
    d.label_col = b.label_col;
  } else {
    d.K = p.in;
    d.q.kind = OP_BN_ACT;
    d.q.rows = p.in;
    d.q.p = b.h[l - 1];
    d.q.sp = (long long)p.in * e.ws.ld;
    d.q.bn = bn_ref(e, net, l - 1, false, false);
  }
  d.dW = e.G(net, p.w);
  d.sdW = 0;
  d.ldw = p.in;
  d.db = e.G(net, p.b);
  if (l < 3) {
    d.dgamma = e.G(net, p.gamma);
    d.dbeta = e.G(net, p.beta);
    // with global BatchNorm the sums are already global: only rank 0 contributes them before the
    // gradient all-reduce (sum).  With local BatchNorm every rank adds its own.
    d.add_affine = (e.world <= 1 || local_bn || e.rank == 0) ? 1 : 0;
  }
  return launch_dw(e, d, st);
}

static int bwd_bn_net(Engine& e, const BnNetBwd& b, int M, float Bg_bn, float kl_coef, bool local_bn, cudaStream_t st) {
  for (int l = 3; l >= 0; --l) {
    // dX first: it produces the batch sums the next layer's kernels need
    CVG_TRY(bwd_bn_dx(e, b, l, M, Bg_bn, kl_coef, local_bn, st));
    if (l > 0 || b.want_first_dx) CVG_PAR(e);     // beside the input-gradient op just emitted: both read dY of layer l
    CVG_TRY(bwd_bn_dw(e, b, l, M, Bg_bn, local_bn, fork_to(e, 0, st)));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Adam + losses
// ------------------------------------------------------------------------------------------------
static float net_lr(const Engine& e, int net) {
  if (net == CVG_NET_DISCRIMINATOR) return e.cfg.d_lr;
  if (net == CVG_NET_CLASSIFIER) return e.cfg.c_lr;
  return e.cfg.g_lr;
}

int run_adam(Engine& e, int net_mask, cudaStream_t st, const AdamOverride* ov, bool steps_advanced) {
  AdamArgs a;
  a.nseg = 0;
  a.b1 = ov ? ov->beta1 : e.cfg.adam_beta1;
  a.b2 = ov ? ov->beta2 : e.cfg.adam_beta2;
  a.eps = ov ? ov->eps : e.cfg.adam_eps;
  a.clear_grad = 1;
  long long nmax = 0;
  for (int net = 0; net < 4; ++net) {
    if (!(net_mask & (1 << net))) continue;
    if (a.nseg == 2) CVG_FAIL("cvg_adam: at most two networks per call");
    AdamSeg& s = a.seg[a.nseg++];
    s.p = e.buf[net].params; s.g = e.buf[net].grads; s.m = e.buf[net].m; s.v = e.buf[net].v;
    s.n = e.lay[net].n_param;
    s.lr = ov ? ov->lr : net_lr(e, net);
    s.t_prev = &e.ws.ctl->adam_t[net];
    if (s.n > nmax) nmax = s.n;
  }
  if (a.nseg == 0) return 0;
  if (e.mk.recording) {
    mk::AdamOp op;
    op.a = a;
    op.t_off[0] = op.t_off[1] = 0;
    int si = 0;
    for (int net = 0; net < 4; ++net)
      if (net_mask & (1 << net)) { op.t_off[si++] = e.mk.adam_inc[net]; e.mk.adam_inc[net]++; }
    mk_weights_updated(e, net_mask);
    return mk_push(e, mk::K_ADAM, &op, sizeof(op), a.nseg * mk::ADAM_VB);
  }
  int blocks = (int)((nmax + 255) / 256);
  if (blocks > 2 * e.num_sms) blocks = 2 * e.num_sms;
  a.t_add = steps_advanced ? 0 : 1;
  adam_kernel<<<dim3(blocks, a.nseg), 256, 0, st>>>(a);
  CVG_LAUNCH_CHECK();
  if (!steps_advanced) {
    ctl_bump_kernel<<<1, 32, 0, st>>>(e.ws.ctl, 0ull, net_mask);   // state['step'] += 1
    CVG_LAUNCH_CHECK();
  }
  return 0;
}

// pack local loss sums into the first net's gradient tail, all-reduce gradients (+tail), Adam, unpack
static int finish_step(Engine& e, int net_mask, int kind, int M, int flags, float* loss_out, cudaStream_t st,
                       const AdamOverride* ov = nullptr) {
  int first = -1;
  for (int net = 0; net < 4; ++net)
    if (net_mask & (1 << net)) { first = net; break; }
  float* tail = e.buf[first].grads + e.lay[first].n_param;
  join_sides(e, st);
  if (e.mk.recording) {
    const bool had_red = !e.mk.pending_red.empty();
    CVG_TRY(mk_emit_dwred(e));                 // deterministic sums of the weight-gradient row slices
    mk::PackArgs pa;
    pa.acc = e.ws.loss; pa.tail = tail;
    if (had_red) CVG_PAR(e);                   // beside the reductions: the loss sums were complete phases ago
    CVG_TRY(mk_push(e, mk::K_PACK, &pa, sizeof(pa), 1));
    for (int net = 0; net < 4; ++net)
      if (net_mask & (1 << net))
        CVG_TRY(comm_all_reduce_f32(e, e.buf[net].grads, e.lay[net].n_param + (net == first ? CVG_GRAD_TAIL : 0), st));
    bool par = false;
    if (loss_out) {
      mk::UnpackArgs ua;
      ua.tail = tail; ua.out = loss_out; ua.kind = kind; ua.Bg = (float)M * (float)e.world; ua.F = (float)e.F; ua.tail_w = tail;
      CVG_TRY(mk_push(e, mk::K_UNPACK, &ua, sizeof(ua), 1));
      par = true;
    }
    if (!(flags & CVG_STEP_NO_UPDATE)) {
      if (par) CVG_PAR(e);
      CVG_TRY(run_adam(e, net_mask, st, ov));
    }
    return 0;
  }
  // one launch: loss sums -> gradient tail (or, on one GPU, straight to loss_out), Philox counter and Adam step counters
  const bool update = !(flags & CVG_STEP_NO_UPDATE);
  const bool one = e.world <= 1;
  loss_tail_kernel<<<1, 32, 0, st>>>(e.ws.loss, tail, loss_out, kind, (float)M * (float)e.world, (float)e.F, one ? 1 : 0,
                                     e.ws.ctl, e.step_dcounter, update ? net_mask : 0);
  CVG_LAUNCH_CHECK();
  e.step_dcounter = 0;
  // Inside a label visit the rest - gradient reduction (own exchange channel), loss read-out, Adam - runs on side stream 0
  // beside the next step's head (noise fill, batch draw and staging).  Whatever needs the updated network is ordered after
  // it: the power iteration is queued on the same stream, every step joins the side streams before its first GEMM on D or
  // C, the E/G step and the hoisted generator forward join before they start.
  bool beside = e.in_visit && e.ms.on && (one || e.nvl.on);
  for (int net = 0; net < 4 && beside && !one; ++net)
    if ((net_mask & (1 << net)) && 2 * (size_t)(e.lay[net].n_param + CVG_GRAD_TAIL) * sizeof(float) > e.nvl.dev.slot_bytes) beside = false;
  const cudaStream_t sx = beside ? fork_to(e, 0, st) : st;
  if (!one) {
    for (int net = 0; net < 4; ++net)
      if (net_mask & (1 << net))
        CVG_TRY(comm_all_reduce_f32(e, e.buf[net].grads, e.lay[net].n_param + (net == first ? CVG_GRAD_TAIL : 0), sx, beside ? 2 : 0));
    if (loss_out) {
      unpack_loss_kernel<<<1, 32, 0, sx>>>(tail, loss_out, kind, (float)M * (float)e.world, (float)e.F, 1, tail);
      CVG_LAUNCH_CHECK();
    }
  }
  if (update) CVG_TRY(run_adam(e, net_mask, sx, ov, true));
  return 0;
}

static int check_step(Engine& e, int B) {
  if (!e.ws_base) CVG_FAIL("workspace not bound");
  for (int n = 0; n < 4; ++n)
    if (!e.buf[n].params || !e.buf[n].grads || (!e.buf[n].state && e.lay[n].n_state > 0)) CVG_FAIL("network buffers not bound");
  if (B < 1 || B > e.ws.rows_cap) CVG_FAIL("batch size exceeds max_batch");
  if ((int64_t)B * e.world < 2) CVG_FAIL("BatchNorm in train mode needs more than 1 row");
  return 0;
}

static bool mk_usable(const Engine& e) { return e.mk.enabled && (e.world == 1 || e.nvl.on); }

// A step called on its own records (and at its end launches) its own program; inside a visit it appends to the visit's.
struct ProgramScope {
  Engine& e;
  bool own = false;
  explicit ProgramScope(Engine& en) : e(en) {
    if (mk_usable(e) && !e.mk.recording) { mk_begin(e); own = true; }
  }
  int finish(cudaStream_t st) {
    if (!own) return 0;
    own = false;
    return mk_flush(e, st);
  }
  ~ProgramScope() { if (own) e.mk.recording = false; }    // error path: drop the half-recorded program
};

static int begin_step(Engine& e, const StepRng& rng, bool with_lambda, cudaStream_t st) {
  e.nvl.n_pending = 0;
  e.mk.scratch_off = 0;      // the previous step's weight-gradient slices were reduced before its last barrier
  if (!rng.set) return 0;
  e.step_dcounter = 0;       // a step called on its own sets the Philox counter itself
  if (e.mk.recording) {
    // the ops of this program take the Philox key / counter from their own arguments (fill_args); the control block is
    // still brought up to date for ops that read lambda_class from it and for later calls
    mk::CtlSetArgs a;
    a.ctl = e.ws.ctl; a.seed = rng.seed; a.counter = rng.counter; a.set_rng = 1;
    a.lambda_class = rng.lambda_class; a.set_lambda = with_lambda ? 1 : 0;
    return mk_push(e, mk::K_CTL_SET, &a, sizeof(a), 1);
  }
  ctl_set_kernel<<<1, 32, 0, st>>>(e.ws.ctl, rng.seed, rng.counter, 1, rng.lambda_class, with_lambda ? 1 : 0);
  CVG_LAUNCH_CHECK();
  return 0;
}

// Philox addressing of a step's noise (see StepRng)
static void fill_args(Engine& e, FillArgs& f, const StepRng& rng, int B) {
  f.njobs = 0; f.M = B; f.ld = e.ws.ld; f.seed = 0; f.counter = 0; f.row_base = (uint64_t)e.rank * B;
  f.ctl = e.ws.ctl; f.counter_off = rng.off;
  f.keep_prob = 1.0f - e.cfg.dropout_p;
  if (e.mk.recording) {
    if (rng.set) { f.ctl = nullptr; f.seed = rng.seed; f.counter = rng.counter + rng.off; }
    else f.counter_off = rng.off + e.mk.dcounter;
  }
}

// Program kernel: pre-split (hi / lo, operand order) copies of the weight operands a step is going to use, emitted into the
// step's first phase so that no GEMM has to wait for its own prep op.  fwd: W[n][r]; dx: W[r][n]; first_dx: also the input
// gradient of the first Linear (without its one-hot label column).
static int prep_net(Engine& e, int net, bool fwd, bool dx, bool first_dx) {
  if (!e.mk.recording) return 0;
  const int first_k = (net == CVG_NET_GENERATOR) ? e.Z : e.F;
  for (int l = 0; l < e.lay[net].nlin; ++l) {
    const LinearP& p = e.lay[net].lin[l];
    GemmArgs g;
    g.W = e.P(net, p.w);
    g.ldw = p.in;
    g.wcol0 = 0;
    const float* wp = nullptr;
    if (fwd) {
      g.R = (l == 0) ? first_k : p.in;
      g.a.rows = g.R;
      g.N = p.out;
      e.mk.par_next = true;
      CVG_TRY(mk_weight_operand(e, g, true, &wp));
    }
    if (dx && (l > 0 || first_dx)) {
      g.R = p.out;
      g.a.rows = g.R;
      g.N = (l == 0) ? first_k : p.in;
      e.mk.par_next = true;
      CVG_TRY(mk_weight_operand(e, g, false, &wp));
    }
  }
  e.mk.par_next = false;
  return 0;
}

static int emit_ce(Engine& e, const CeArgs& c, int B, int npass, cudaStream_t st) {
  if (e.mk.recording) return mk_push(e, mk::K_CE, &c, sizeof(c), npass * ((B + mk::THREADS - 1) / mk::THREADS));
  ce_kernel<<<dim3((B + 127) / 128, npass), 128, 0, st>>>(c);
  CVG_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// step D (cvae_gan.py:104-128)
// ------------------------------------------------------------------------------------------------
int step_d(Engine& e, const float* x_real, int label, int B, const CvgNoise* nz, const StepRng& rng, int flags,
           float* loss_out, cudaStream_t st) {
  CVG_TRY(check_step(e, B));
  ProgramScope prog(e);
  CVG_TRY(begin_step(e, rng, false, st));
  const Workspace& w = e.ws;
  const bool local_bn = flags & CVG_STEP_LOCAL_BN;
  const float Bg = (float)B * (float)e.world;
  const float Bg_bn = local_bn ? (float)B : Bg;
  const int D = CVG_NET_DISCRIMINATOR;
  if (rng.set) CVG_PAR(e);
  CVG_TRY(emit_zero(e, w.acc, w.acc_bytes, st));
  CVG_PAR(e);
  CVG_TRY(emit_zero(e, w.sn_G, sizeof(float) * 2 * e.lay[D].n_param, st));
  CVG_TRY(prep_net(e, CVG_NET_GENERATOR, true, false, false));
  CVG_TRY(prep_net(e, D, true, true, false));
  FillArgs f;
  fill_args(e, f, rng, B);
  if (!e.hoist_x) add_job(f, w.z, nz ? nz->z : nullptr, 0, e.Z, 1, RS_Z);
  add_job(f, w.d_m1, nz ? nz->d_mask1 : nullptr, 1, e.dh[0], 2, RS_DMASK1);
  add_job(f, w.d_m2, nz ? nz->d_mask2 : nullptr, 1, e.dh[1], 2, RS_DMASK2);
  CVG_PAR(e);
  CVG_TRY(launch_fill(e, f, st));
  CVG_PAR(e);
  CVG_TRY(stage_x(e, x_real, B, fork_to(e, 1, st)));
  CVG_PAR(e);                           // the power iterations only touch the critic's weights and u / v: first phase
  CVG_TRY(launch_sn(e, 2, true, fork_to(e, 0, st)));   // D(real) then D(fake): two consecutive power iterations
  // G(z) under no_grad, still in train mode: batch stats, running stats updated (cvae_gan.py:113-115)
  if (!e.hoist_x) CVG_TRY(fwd_generator(e, 1, true, false, label, B, Bg_bn, local_bn, st));
  join_sides(e, st);
  const long long sx = (e.hoist_x ? e.hoist_x : w.g_out) - w.xT;  // pass 0 reads xT, pass 1 reads G(z)
  const float seedv[2] = {-1.0f / Bg, 1.0f / Bg};   // d_loss = -mean D(real) + mean D(fake)
  if (chain_usable(e, D)) {
    CVG_TRY(launch_critic_chain(e, sx, label, B, seedv, st));
    CVG_TRY(bwd_critic(e, w.xT, sx, 2, label, B, seedv, true, false, st, true));
  } else {
    CVG_TRY(fwd_critic(e, w.xT, sx, 2, label, B, w.loss + L_DREAL, st));
    CVG_TRY(bwd_critic(e, w.xT, sx, 2, label, B, seedv, true, false, st));
  }
  join_sides(e, st);
  {
    SnGradArgs a;
    int off = 0;
    for (int l = 0; l < 4; ++l) {
      const LinearP& p = lin(e, D, l);
      a.L[l].W = e.P(D, p.w); a.L[l].rows = p.out; a.L[l].cols = p.in;
      a.L[l].u = nullptr; a.L[l].v = nullptr; a.L[l].snap_off = off;
      off += ((p.out > p.in ? p.out : p.in) + 3) & ~3;
      a.w_off[l] = p.w;
    }
    a.npass = 2;
    a.Gp = w.sn_G; a.sG = e.lay[D].n_param;
    a.inv_sigma = w.sn_inv_sigma;
    a.u_snap = w.sn_u; a.v_snap = w.sn_v; a.ssnap = w.sn_snap;
    a.grad = e.buf[D].grads;
    a.last_bias_grad = e.G(D, lin(e, D, 3).b);
    a.last_bias_value = (float)B * (seedv[0] + seedv[1]);
    double* dots = w.loss + 8;   // 8 zeroed accumulator slots after the loss sums
    if (e.mk.recording) {
      CVG_TRY(mk_emit_dwred(e));   // per-pass raw critic gradients, summed over the row slices in a fixed order
      CVG_TRY(mk_push(e, mk::K_SN_DOT, &a, sizeof(a), mk::SN_DOT_VB * 4 * 2, 0, 0, 0, 0, &dots, sizeof(dots)));
      CVG_TRY(mk_push(e, mk::K_SN_GRAD, &a, sizeof(a), mk::SN_GRAD_VB * 4, 0, 0, 0, 0, &dots, sizeof(dots)));
      CVG_PAR(e);                  // the loss pack that follows is independent of the spectral-norm gradient
    } else {
      sn_dot_kernel<<<dim3(16, 4, 2), 256, 0, st>>>(a, dots);
      CVG_LAUNCH_CHECK();
      sn_grad_kernel<<<dim3(32, 4), 256, 0, st>>>(a, dots);
      CVG_LAUNCH_CHECK();
    }
  }
  CVG_TRY(finish_step(e, 1 << D, 0, B, flags, loss_out, st));
  return prog.finish(st);
}

// ------------------------------------------------------------------------------------------------
// step C (cvae_gan.py:131-157)
// ------------------------------------------------------------------------------------------------
int step_c(Engine& e, const float* x_real, int label, int B, const CvgNoise* nz, const StepRng& rng, int flags,
           float* loss_out, cudaStream_t st) {
  CVG_TRY(check_step(e, B));
  ProgramScope prog(e);
  CVG_TRY(begin_step(e, rng, false, st));
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const bool local_bn = flags & CVG_STEP_LOCAL_BN;
  const float Bg = (float)B * (float)e.world;
  const float Bg_bn = local_bn ? (float)B : Bg;
  const int C = CVG_NET_CLASSIFIER;
  if (rng.set) CVG_PAR(e);
  CVG_TRY(emit_zero(e, w.acc, w.acc_bytes, st));
  CVG_TRY(prep_net(e, CVG_NET_GENERATOR, true, false, false));
  CVG_TRY(prep_net(e, C, true, true, false));
  FillArgs f;
  fill_args(e, f, rng, B);
  if (!e.hoist_x) add_job(f, w.z, nz ? nz->z : nullptr, 0, e.Z, 1, RS_Z);
  add_job(f, w.c_m1, nz ? nz->c_mask1 : nullptr, 1, e.ch[0], 2, RS_CMASK1);
  add_job(f, w.c_m2, nz ? nz->c_mask2 : nullptr, 1, e.ch[1], 2, RS_CMASK2);
  CVG_PAR(e);
  CVG_TRY(launch_fill(e, f, st));
  CVG_PAR(e);
  CVG_TRY(stage_x(e, x_real, B, fork_to(e, 1, st)));
  if (!e.hoist_x) CVG_TRY(fwd_generator(e, 1, true, false, label, B, Bg_bn, local_bn, st));
  join_sides(e, st);
  const long long sx = (e.hoist_x ? e.hoist_x : w.g_out) - w.xT;
  if (chain_usable(e, C)) {
    CVG_TRY(launch_classifier_chain(e, sx, label, B, 1.0f / Bg, st));
    CVG_TRY(bwd_classifier(e, w.xT, sx, 2, B, true, false, false, st, nullptr, true));
  } else {
    CVG_TRY(fwd_classifier(e, w.xT, sx, 2, true, B, st));
    CeArgs c;
    c.M = B; c.ld = w.ld; c.K = e.K; c.npass = 2; c.label = label;
    c.logits = w.c_logit; c.sl = (long long)e.K * ld;
    c.dlogits = w.c_dlogit; c.sd = (long long)e.K * ld;
    c.coef = 1.0f / Bg;
    c.ctl = nullptr;
    c.loss = w.loss + L_CE0;
    CVG_TRY(emit_ce(e, c, B, 2, st));
    CVG_TRY(bwd_classifier(e, w.xT, sx, 2, B, true, false, false, st));
  }
  CVG_TRY(finish_step(e, 1 << C, 1, B, flags, loss_out, st));
  return prog.finish(st);
}

// ------------------------------------------------------------------------------------------------
// downstream fine-tuning step of the classifier network (classifier.py:24-45): logits = C(x) in train mode (dropout),
// loss = mean cross_entropy(logits, labels) with PER-ROW labels, Adam with the caller's hyper-parameters
// ------------------------------------------------------------------------------------------------
int step_classifier(Engine& e, const float* x, const long long* labels, int B, const CvgNoise* nz, const StepRng& rng,
                    const AdamOverride& ov, int flags, float* loss_out, cudaStream_t st) {
  if (!e.ws_base) CVG_FAIL("workspace not bound");
  if (B < 1 || B > e.ws.rows_cap) CVG_FAIL("batch size exceeds max_batch");
  ProgramScope prog(e);
  CVG_TRY(begin_step(e, rng, false, st));
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const int C = CVG_NET_CLASSIFIER;
  const float Bg = (float)B * (float)e.world;
  if (rng.set) CVG_PAR(e);
  CVG_TRY(emit_zero(e, w.acc, w.acc_bytes, st));
  CVG_TRY(prep_net(e, C, true, true, false));
  FillArgs f;
  fill_args(e, f, rng, B);
  add_job(f, w.c_m1, nz ? nz->c_mask1 : nullptr, 1, e.ch[0], 1, RS_CMASK1);
  add_job(f, w.c_m2, nz ? nz->c_mask2 : nullptr, 1, e.ch[1], 1, RS_CMASK2);
  CVG_PAR(e);
  CVG_TRY(launch_fill(e, f, st));
  CVG_PAR(e);
  CVG_TRY(stage_x(e, x, B, st));
  CVG_TRY(fwd_classifier(e, w.xT, 0, 1, true, B, st));
  CeArgs c;
  c.M = B; c.ld = w.ld; c.K = e.K; c.npass = 1; c.label = 0; c.labels = labels;
  c.logits = w.c_logit; c.sl = (long long)e.K * ld;
  c.dlogits = w.c_dlogit; c.sd = (long long)e.K * ld;
  c.coef = 1.0f / Bg;
  c.ctl = nullptr;
  c.loss = w.loss + L_CE0;
  CVG_TRY(emit_ce(e, c, B, 1, st));
  CVG_TRY(bwd_classifier(e, w.xT, 0, 1, B, true, false, false, st));
  CVG_TRY(finish_step(e, 1 << C, 1, B, flags, loss_out, st, &ov));
  return prog.finish(st);
}

// ------------------------------------------------------------------------------------------------
// step E+G (cvae_gan.py:160-216)
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// Sibling trainer CGAN (SURVEY 8 f4), generator step (/root/reference/src/cgan.py:138-178): x_fake = G(z_prior, onehot)
// only - no encoder, no reconstruction / KL terms, no real batch -, total = lambda_adv * (-mean D(x_fake)) +
// lambda_class_now * CE(C(x_fake), label), Adam on the generator alone.  The critic and classifier steps of CGAN are
// step_d / step_c (cgan.py:84-136 is cvae_gan.py:104-157 statement for statement).  Stand-alone kernels only.
// ------------------------------------------------------------------------------------------------
static int step_g_prior(Engine& e, int label, int B, const CvgNoise* nz, const StepRng& rng, int flags, float* loss_out,
                        cudaStream_t st) {
  CVG_TRY(check_step(e, B));
  if (e.mk.recording || mk_usable(e)) CVG_FAIL("the CGAN generator step runs on the stand-alone executor only (unset CVG_TRAIN_MODE)");
  CVG_TRY(begin_step(e, rng, true, st));
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const bool local_bn = flags & CVG_STEP_LOCAL_BN;
  const float Bg = (float)B * (float)e.world;
  const float Bg_bn = local_bn ? (float)B : Bg;
  const int G = CVG_NET_GENERATOR;
  CVG_TRY(emit_zero(e, w.acc, w.acc_bytes, st));
  FillArgs f;
  fill_args(e, f, rng, B);
  add_job(f, w.z, nz ? nz->z : nullptr, 0, e.Z, 1, RS_Z);
  add_job(f, w.d_m1, nz ? nz->d_mask1 : nullptr, 1, e.dh[0], 1, RS_DMASK1);
  add_job(f, w.d_m2, nz ? nz->d_mask2 : nullptr, 1, e.dh[1], 1, RS_DMASK2);
  add_job(f, w.c_m1, nz ? nz->c_mask1 : nullptr, 1, e.ch[0], 1, RS_CMASK1);
  add_job(f, w.c_m2, nz ? nz->c_mask2 : nullptr, 1, e.ch[1], 1, RS_CMASK2);
  CVG_TRY(launch_fill(e, f, st));
  join_sides(e, st);                                     // the previous step's Adam (visit: side stream 0)
  CVG_TRY(launch_sn(e, 1, true, fork_to(e, 0, st)));
  CVG_TRY(fwd_generator(e, 1, true, false, label, B, Bg_bn, local_bn, st));
  join_sides(e, st);
  const float* x_fake = w.g_out;
  const cudaStream_t sc = fork_to(e, 1, st);
  CVG_TRY(fwd_critic(e, x_fake, 0, 1, label, B, w.loss + L_DFAKE, st));
  {                                                      // the class loss is reported even while its weight is 0 (cgan.py:162,181)
    CVG_TRY(fwd_classifier(e, x_fake, 0, 1, true, B, sc));
    CeArgs c;
    c.M = B; c.ld = w.ld; c.K = e.K; c.npass = 1; c.label = label;
    c.logits = w.c_logit; c.sl = (long long)e.K * ld;
    c.dlogits = w.c_dlogit; c.sd = (long long)e.K * ld;
    c.coef = 1.0f / Bg;       // times ctl->lambda_class, read on the device
    c.ctl = w.ctl;
    c.loss = w.loss + L_CE0;
    CVG_TRY(emit_ce(e, c, B, 1, sc));
  }
  const float seedv[2] = {-e.cfg.lambda_adv / Bg, 0.f};
  CVG_TRY(bwd_critic(e, x_fake, 0, 1, label, B, seedv, false, true, st));
  if (rng.lambda_nonzero) CVG_TRY(bwd_classifier(e, x_fake, 0, 1, B, false, true, true, sc, st));
  join_sides(e, st);
  SeedArgs s;
  s.M = B; s.ld = w.ld; s.F = e.F;
  s.out = w.g_out; s.sout = (long long)e.F * ld;
  s.x = w.xT; s.dx = w.dx;
  s.dpre = w.g_dout; s.sdpre = (long long)e.F * ld;
  s.coef_recon = 0.f;
  s.recon_acc = w.loss + L_RECON;
  s.prior_only = 1;
  g_seed_kernel<<<dim3((unsigned)((e.F * ld + 255) / 256), 1), 256, 0, st>>>(s);
  CVG_LAUNCH_CHECK();
  BnNetBwd gb;
  gb.net = G; gb.npass = 1;
  gb.h = w.g_h; gb.dy = w.g_dy;
  gb.top_dy = w.g_dout; gb.s_top = (long long)e.F * ld;
  gb.first_in.kind = OP_PLAIN; gb.first_in.rows = e.Z;
  gb.first_in.p = w.z; gb.first_in.sp = (long long)e.Z * ld;
  gb.first_K = e.Z;
  gb.label_col = label_col_index(e, e.Z, label);
  gb.want_first_dx = false;
  CVG_TRY(bwd_bn_net(e, gb, B, Bg_bn, 0.f, local_bn, st));
  return finish_step(e, 1 << G, 2, B, flags, loss_out, st);
}

// ------------------------------------------------------------------------------------------------
// Sibling trainer CVAE (SURVEY 8 f4), encoder / generator step (/root/reference/src/cvae.py:117-166): mu, logvar = E(x);
// z_enc = mu + eps * std; x_recon = G(z_enc, onehot) - ONE generator pass, no critic, no z_prior -;
// total = lambda_recon * MSE(x_recon, x) + lambda_kl * KL + lambda_class_now * CE(C(x_recon), label): the classifier reads
// the RECONSTRUCTION, so its input gradient joins the reconstruction term at the generator's output (SeedArgs.add_dx).
// Adam on encoder and generator.  The classifier step of CVAE is step_c (cvae.py:89-115 is cvae_gan.py:131-157 statement for
// statement); there is no critic step.  Stand-alone kernels only, one stream.
// ------------------------------------------------------------------------------------------------
static int step_g_cvae(Engine& e, const float* x_real, int label, int B, const CvgNoise* nz, const StepRng& rng, int flags,
                       float* loss_out, cudaStream_t st) {
  CVG_TRY(check_step(e, B));
  if (e.mk.recording || mk_usable(e)) CVG_FAIL("the CVAE encoder/generator step runs on the stand-alone executor only (unset CVG_TRAIN_MODE)");
  CVG_TRY(begin_step(e, rng, true, st));
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const bool local_bn = flags & CVG_STEP_LOCAL_BN;
  const float Bg = (float)B * (float)e.world;
  const float Bg_bn = local_bn ? (float)B : Bg;
  const int E = CVG_NET_ENCODER, G = CVG_NET_GENERATOR;
  CVG_TRY(emit_zero(e, w.acc, w.acc_bytes, st));
  FillArgs f;
  fill_args(e, f, rng, B);
  add_job(f, w.z, nz ? nz->eps : nullptr, 0, e.Z, 1, RS_EPS);     // eps in slot 0: reparameterisation fused into G's first operand load
  add_job(f, w.c_m1, nz ? nz->c_mask1 : nullptr, 1, e.ch[0], 1, RS_CMASK1);
  add_job(f, w.c_m2, nz ? nz->c_mask2 : nullptr, 1, e.ch[1], 1, RS_CMASK2);
  CVG_TRY(launch_fill(e, f, st));
  join_sides(e, st);                                     // the previous step's Adam (visit: side stream 0)
  CVG_TRY(stage_x(e, x_real, B, st));
  CVG_TRY(fwd_encoder(e, true, label, B, Bg_bn, local_bn, st));
  CVG_TRY(fwd_generator(e, 1, true, true, label, B, Bg_bn, local_bn, st));
  const float* x_recon = w.g_out;
  {                                                      // the class loss is reported even while its weight is 0 (cvae.py:141-142,162)
    CVG_TRY(fwd_classifier(e, x_recon, 0, 1, true, B, st));
    CeArgs c;
    c.M = B; c.ld = w.ld; c.K = e.K; c.npass = 1; c.label = label;
    c.logits = w.c_logit; c.sl = (long long)e.K * ld;
    c.dlogits = w.c_dlogit; c.sd = (long long)e.K * ld;
    c.coef = 1.0f / Bg;       // times ctl->lambda_class, read on the device
    c.ctl = w.ctl;
    c.loss = w.loss + L_CE0;
    CVG_TRY(emit_ce(e, c, B, 1, st));
  }
  if (rng.lambda_nonzero) CVG_TRY(bwd_classifier(e, x_recon, 0, 1, B, false, true, false, st));   // -> ws.dx
  SeedArgs s;
  s.M = B; s.ld = w.ld; s.F = e.F;
  s.out = w.g_out; s.sout = (long long)e.F * ld;
  s.x = w.xT; s.dx = w.dx;
  s.dpre = w.g_dout; s.sdpre = (long long)e.F * ld;
  s.coef_recon = e.cfg.lambda_recon / (Bg * (float)e.F);
  s.recon_acc = w.loss + L_RECON;
  s.add_dx = rng.lambda_nonzero ? 1 : 0;
  g_seed_kernel<<<dim3((unsigned)((e.F * ld + 255) / 256), 1), 256, 0, st>>>(s);
  CVG_LAUNCH_CHECK();
  BnNetBwd gb;
  gb.net = G; gb.npass = 1;
  gb.h = w.g_h; gb.dy = w.g_dy;
  gb.top_dy = w.g_dout; gb.s_top = (long long)e.F * ld;
  gb.first_in.kind = OP_REPARAM; gb.first_in.rows = e.Z;
  gb.first_in.p = w.z; gb.first_in.sp = (long long)e.Z * ld;
  gb.first_in.mu = w.e_ml; gb.first_in.lv = w.e_ml + (size_t)e.Z * ld; gb.first_in.eps = w.z;
  gb.first_in.reparam_pass = 0;
  gb.first_K = e.Z;
  gb.label_col = label_col_index(e, e.Z, label);
  gb.want_first_dx = true;
  CVG_TRY(bwd_bn_net(e, gb, B, Bg_bn, e.cfg.lambda_kl / Bg, local_bn, st));
  BnNetBwd eb;
  eb.net = E; eb.npass = 1;
  eb.h = w.e_h; eb.dy = w.e_dy;
  eb.top_dy = w.e_dml; eb.s_top = 0;
  eb.first_in.kind = OP_PLAIN; eb.first_in.rows = e.F; eb.first_in.p = w.xT;
  eb.first_K = e.F;
  eb.label_col = label_col_index(e, e.F, label);
  eb.want_first_dx = false;
  CVG_TRY(bwd_bn_net(e, eb, B, Bg_bn, 0.f, local_bn, st));
  return finish_step(e, (1 << E) | (1 << G), 2, B, flags, loss_out, st);
}

int step_g(Engine& e, const float* x_real, int label, int B, const CvgNoise* nz, const StepRng& rng, int flags,
           float* loss_out, cudaStream_t st) {
  if (flags & CVG_STEP_PRIOR_ONLY) return step_g_prior(e, label, B, nz, rng, flags, loss_out, st);
  if (flags & CVG_STEP_CVAE) return step_g_cvae(e, x_real, label, B, nz, rng, flags, loss_out, st);
  CVG_TRY(check_step(e, B));
  ProgramScope prog(e);
  CVG_TRY(begin_step(e, rng, true, st));
  const Workspace& w = e.ws;
  const size_t ld = w.ld;
  const bool local_bn = flags & CVG_STEP_LOCAL_BN;
  const float Bg = (float)B * (float)e.world;
  const float Bg_bn = local_bn ? (float)B : Bg;
  const int E = CVG_NET_ENCODER, G = CVG_NET_GENERATOR;
  if (rng.set) CVG_PAR(e);
  CVG_TRY(emit_zero(e, w.acc, w.acc_bytes, st));
  CVG_TRY(prep_net(e, E, true, true, false));
  CVG_TRY(prep_net(e, G, true, true, true));
  CVG_TRY(prep_net(e, CVG_NET_DISCRIMINATOR, true, true, true));
  CVG_TRY(prep_net(e, CVG_NET_CLASSIFIER, true, rng.lambda_nonzero, true));
  FillArgs f;
  fill_args(e, f, rng, B);
  // eps: slot 0 of ws.z for the stand-alone kernels (reparameterisation fused into the operand load); the program
  // kernel keeps eps apart and materialises z_enc into slot 0 (mk::K_REPARAM below)
  add_job(f, e.mk.recording ? w.z_eps : w.z, nz ? nz->eps : nullptr, 0, e.Z, 1, RS_EPS);
  add_job(f, w.z + (size_t)e.Z * ld, nz ? nz->z : nullptr, 0, e.Z, 1, RS_Z);      // slot 1: z_prior
  add_job(f, w.d_m1, nz ? nz->d_mask1 : nullptr, 1, e.dh[0], 1, RS_DMASK1);
  add_job(f, w.d_m2, nz ? nz->d_mask2 : nullptr, 1, e.dh[1], 1, RS_DMASK2);
  add_job(f, w.c_m1, nz ? nz->c_mask1 : nullptr, 1, e.ch[0], 1, RS_CMASK1);
  add_job(f, w.c_m2, nz ? nz->c_mask2 : nullptr, 1, e.ch[1], 1, RS_CMASK2);
  CVG_PAR(e);
  CVG_TRY(launch_fill(e, f, st));
  const float* x_fake = w.g_out + (size_t)e.F * ld;
  CeArgs c;
  c.M = B; c.ld = w.ld; c.K = e.K; c.npass = 1; c.label = label;
  c.logits = w.c_logit; c.sl = (long long)e.K * ld;
  c.dlogits = w.c_dlogit; c.sd = (long long)e.K * ld;
  c.coef = 1.0f / Bg;       // times ctl->lambda_class, read on the device
  c.ctl = w.ctl;
  c.loss = w.loss + L_CE0;
  // backward to x_fake: adv = -mean D(x_fake) (cvae_gan.py:189), then the classification term
  const float seedv[2] = {-e.cfg.lambda_adv / Bg, 0.f};
  // Three chains side by side (stand-alone kernels, side streams on; data parallel: with the folded exchange, one channel
  // per chain): x_fake = G(z_prior) does not depend on the encoder, and the critic / classifier terms only on x_fake.
  //   caller's stream : E(x), G(z_enc)
  //   side 1          : batch staging, G(z_prior), then D(x_fake) forward and backward to x_fake
  //   side 0          : power iteration, then C(x_fake) forward, loss and backward to x_fake (after D's: both add to ws.dx)
  const bool three = !e.mk.recording && e.ms.on && (e.world <= 1 || local_bn || fold_stats(e, local_bn));
  // The backward continues as two chains, one per generator pass (their BatchNorm sums are per pass, and only pass 0
  // reaches the encoder):
  //   caller's stream : seed and generator input gradients of pass 0, the encoder head gradient, the encoder backward
  //   side 1          : after the critic's and classifier's dx, seed and generator input gradients of pass 1
  //   side 0          : the generator's weight gradients, each after both passes' dY of its layer (one launch for both
  //                     passes, so the fixed-point sums are converted once, as with one chain)
  //   side 2          : the encoder's weight gradients, which must not queue behind the generator's
  // Only where no BatchNorm sums are exchanged: a folded exchange of one pass cannot yet be told from the other pass's.
  const bool split = three && e.eg_split && (e.world <= 1 || local_bn);
  join_sides(e, st);      // the previous step's Adam (visit: side stream 0) beside the fill just launched
  if (three) {
    const cudaStream_t sA = fork_to(e, 0, st), sB = fork_to(e, 1, st);
    CVG_TRY(launch_sn(e, 1, true, sA));
    CVG_TRY(stage_x(e, x_real, B, sB));
    wait_for(e, st, sB);                                            // the encoder reads the staged batch
    GenSplit prior;
    prior.only_pass = 1; prior.channel = 1; prior.rec = e.ms.layer;
    CVG_TRY(fwd_generator(e, 2, true, false, label, B, Bg_bn, local_bn, sB, nullptr, &prior));
    wait_for(e, sB, sA);                                            // sigma of the critic's layers (all side 0 holds so far)
    if (rng.lambda_nonzero) {
      wait_for(e, sA, sB);                                          // x_fake
      CVG_TRY(fwd_classifier(e, x_fake, 0, 1, true, B, sA));
      CVG_TRY(emit_ce(e, c, B, 1, sA));
    }
    CVG_TRY(fwd_critic(e, x_fake, 0, 1, label, B, w.loss + L_DFAKE, sB));
    CVG_TRY(bwd_critic(e, x_fake, 0, 1, label, B, seedv, false, true, sB));
    if (rng.lambda_nonzero) CVG_TRY(bwd_classifier(e, x_fake, 0, 1, B, false, true, true, sA, sB));
    CVG_TRY(fwd_encoder(e, true, label, B, Bg_bn, local_bn, st));
    GenSplit enc;
    enc.only_pass = 0; enc.channel = 0; enc.wait = e.ms.layer;
    CVG_TRY(fwd_generator(e, 2, true, true, label, B, Bg_bn, local_bn, st, nullptr, &enc));
    if (!split) join_sides(e, st);
  } else {
  CVG_PAR(e);
  CVG_TRY(stage_x(e, x_real, B, fork_to(e, 1, st)));

  CVG_PAR(e);
  CVG_TRY(launch_sn(e, 1, true, fork_to(e, 0, st)));   // critic power iteration: independent of everything before D(x_fake)
  // forward: E -> (mu, logvar); G on z_enc (pass 0) and z_prior (pass 1); D and C on x_fake
  join_sides(e, st, 1);
  CVG_TRY(fwd_encoder(e, true, label, B, Bg_bn, local_bn, st));
  if (e.mk.recording) {
    mk::ReparamArgs ra;
    ra.mu = w.e_ml; ra.lv = w.e_ml + (size_t)e.Z * ld; ra.eps = w.z_eps; ra.out = w.z; ra.M = B; ra.ld = w.ld; ra.Z = e.Z;
    CVG_TRY(mk_push(e, mk::K_REPARAM, &ra, sizeof(ra), (int)(((long long)e.Z * ld + mk::THREADS - 1) / mk::THREADS)));
  }
  CVG_TRY(fwd_generator(e, 2, true, true, label, B, Bg_bn, local_bn, st));
  join_sides(e, st);
  // the classifier branch (forward, loss, backward to x_fake) runs beside the critic's; they meet at ws.dx
  const cudaStream_t sc = rng.lambda_nonzero ? fork_to(e, 1, st) : st;
  CVG_TRY(fwd_critic(e, x_fake, 0, 1, label, B, w.loss + L_DFAKE, st));
  CVG_TRY(fwd_classifier(e, x_fake, 0, 1, true, B, sc));
  CVG_TRY(emit_ce(e, c, B, 1, sc));
  CVG_TRY(bwd_critic(e, x_fake, 0, 1, label, B, seedv, false, true, st));
  if (rng.lambda_nonzero) CVG_TRY(bwd_classifier(e, x_fake, 0, 1, B, false, true, true, sc, st));
  join_sides(e, st);
  }

  // generator output gradients: recon MSE on pass 0, dx on pass 1, through the sigmoid
  SeedArgs s;
  s.M = B; s.ld = w.ld; s.F = e.F;
  s.out = w.g_out; s.sout = (long long)e.F * ld;
  s.x = w.xT; s.dx = w.dx;
  s.dpre = w.g_dout; s.sdpre = (long long)e.F * ld;
  s.coef_recon = e.cfg.lambda_recon / (Bg * (float)e.F);
  s.recon_acc = w.loss + L_RECON;
  const unsigned seed_blocks = (unsigned)((e.F * ld + 255) / 256);
  if (e.mk.recording) {
    CVG_TRY(mk_push(e, mk::K_SEED, &s, sizeof(s), 2 * (int)(((long long)e.F * ld + mk::THREADS - 1) / mk::THREADS)));
  } else if (split) {
    const cudaStream_t sB = e.ms.s[1];
    g_seed_kernel<<<dim3(seed_blocks, 1), 256, 0, st>>>(s);
    CVG_LAUNCH_CHECK();
    SeedArgs s1 = s;                                   // pass 1 alone: dx through the sigmoid
    s1.out += (size_t)e.F * ld;
    s1.dpre += (size_t)e.F * ld;
    s1.prior_only = 1;
    if (rng.lambda_nonzero) wait_for(e, sB, e.ms.s[0]);   // the classifier's share of dx
    g_seed_kernel<<<dim3(seed_blocks, 1), 256, 0, sB>>>(s1);
    CVG_LAUNCH_CHECK();
  } else {
    g_seed_kernel<<<dim3(seed_blocks, 2), 256, 0, st>>>(s);
    CVG_LAUNCH_CHECK();
  }

  BnNetBwd gb;
  gb.net = G; gb.npass = 2;
  gb.h = w.g_h; gb.dy = w.g_dy;
  gb.top_dy = w.g_dout; gb.s_top = (long long)e.F * ld;
  gb.first_in.kind = e.mk.recording ? OP_PLAIN : OP_REPARAM; gb.first_in.rows = e.Z;
  gb.first_in.p = w.z; gb.first_in.sp = (long long)e.Z * ld;
  gb.first_in.mu = w.e_ml; gb.first_in.lv = w.e_ml + (size_t)e.Z * ld; gb.first_in.eps = w.z;
  gb.first_in.reparam_pass = 0;
  gb.first_K = e.Z;
  gb.label_col = label_col_index(e, e.Z, label);
  gb.want_first_dx = true;
  const float kl_coef = e.cfg.lambda_kl / Bg;

  BnNetBwd eb;
  eb.net = E; eb.npass = 1;
  eb.h = w.e_h; eb.dy = w.e_dy;
  eb.top_dy = w.e_dml; eb.s_top = 0;
  eb.first_in.kind = OP_PLAIN; eb.first_in.rows = e.F; eb.first_in.p = w.xT;
  eb.first_K = e.F;
  eb.label_col = label_col_index(e, e.F, label);
  eb.want_first_dx = false;

  if (split) {
    const cudaStream_t sA = e.ms.s[0], sB = e.ms.s[1];
    for (int l = 3; l >= 0; --l) {
      wait_for(e, sA, st);                             // dY of layer l, pass 0 ...
      wait_for(e, sA, sB);                             // ... and pass 1
      CVG_TRY(bwd_bn_dx(e, gb, l, B, Bg_bn, kl_coef, local_bn, st, 0));
      if (l > 0) CVG_TRY(bwd_bn_dx(e, gb, l, B, Bg_bn, kl_coef, local_bn, sB, 1));
      CVG_TRY(bwd_bn_dw(e, gb, l, B, Bg_bn, local_bn, sA));
    }
    for (int l = 3; l >= 0; --l) {
      const cudaStream_t sw = fork_to(e, 2, st);       // dY of layer l
      CVG_TRY(bwd_bn_dx(e, eb, l, B, Bg_bn, 0.f, local_bn, st));
      CVG_TRY(bwd_bn_dw(e, eb, l, B, Bg_bn, local_bn, sw));
    }
  } else {
    CVG_TRY(bwd_bn_net(e, gb, B, Bg_bn, kl_coef, local_bn, st));
    CVG_TRY(bwd_bn_net(e, eb, B, Bg_bn, 0.f, local_bn, st));
  }

  CVG_TRY(finish_step(e, (1 << E) | (1 << G), 2, B, flags, loss_out, st));
  return prog.finish(st);
}

// ------------------------------------------------------------------------------------------------
// one label visit (cvae_gan.py:102-216): d_loop critic steps, c_loop classifier steps, g_loop encoder /
// generator steps, each on a freshly drawn batch.  Everything that varies between visits (Philox
// counter, Adam step counts, lambda_class) is read from the device control block, so the sequence can be
// captured into a CUDA graph once per (label, lambda_class != 0) and replayed.
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// The generator's parameters do not change during the critic and classifier steps of a visit (cvae_gan.py:104-157 only
// step D's and C's optimisers), so G(z) of all d_loop + c_loop of them is one forward with one pass per step, run before
// the first step: 4 launches and 3 BatchNorm exchanges instead of 4 and 3 per step.  Each pass has its own batch sums and
// its z comes from the step's own Philox counter (two values per step: draw, noise), so the values are the ones the
// steps would have computed; the running statistics take the passes' updates in step order (appendix A.2).
// ------------------------------------------------------------------------------------------------
static int hoist_generator(Engine& e, int nh, int label, int B, int flags, cudaStream_t st) {
  const Workspace& w = e.ws;
  const bool local_bn = flags & CVG_STEP_LOCAL_BN;
  const float Bg_bn = local_bn ? (float)B : (float)B * (float)e.world;
  StepRng rng;
  rng.set = false;
  rng.off = 1;
  if (e.mk.recording) e.mk.par_next = false;
  join_sides(e, st);
  CVG_TRY(emit_zero(e, w.hfst, sizeof(double) * 3 * HOIST_MAX * 2 * STAT_C, st));
  CVG_TRY(prep_net(e, CVG_NET_GENERATOR, true, false, false));
  FillArgs f;
  fill_args(e, f, rng, B);
  add_job(f, w.hz, nullptr, 0, e.Z, nh, RS_Z);
  f.job[0].cstep = 2;
  CVG_PAR(e);
  CVG_TRY(launch_fill(e, f, st));
  GenBufs b;
  b.z = w.hz; b.out = w.hout;
  for (int l = 0; l < 3; ++l) { b.h[l] = w.hh[l]; b.fst[l] = w.hfst + (size_t)l * HOIST_MAX * 2 * STAT_C; }
  return fwd_generator(e, nh, true, false, label, B, Bg_bn, local_bn, st, &b);
}

int visit(Engine& e, int label, int B, int64_t B_global, const float* class_rows, int64_t n_rows, const float* x_batches,
          int d_loop, int c_loop, int g_loop, int flags, float* loss_out, cudaStream_t st) {
  CVG_TRY(check_step(e, B));
  if (!x_batches && (!class_rows || n_rows < 1)) CVG_FAIL("cvg_visit: need class_rows or x_batches");
  if (B_global != (int64_t)B * e.world) CVG_FAIL("cvg_visit: B_global must be B_local * world_size");
  // step-program kernel: the whole visit is ONE program = one launch (batch draws included)
  ProgramScope prog(e);
  struct InVisit { Engine& e; explicit InVisit(Engine& en) : e(en) { e.in_visit = true; } ~InVisit() { e.in_visit = false; } } in_visit(e);
  const int nh = e.hoist ? (d_loop + c_loop < HOIST_MAX ? d_loop + c_loop : HOIST_MAX) : 0;
  if (nh > 0) CVG_TRY(hoist_generator(e, nh, label, B, flags, st));
  int i = 0;
  for (int kind = 0; kind < 3; ++kind) {
    const int reps = kind == 0 ? d_loop : (kind == 1 ? c_loop : g_loop);
    for (int r = 0; r < reps; ++r, ++i) {
      e.hoist_x = (kind < 2 && i < nh) ? e.ws.hout + (size_t)i * e.F * e.ws.ld : nullptr;
      const float* x = nullptr;
      const bool no_batch = kind == 2 && (flags & CVG_STEP_PRIOR_ONLY);     // the CGAN generator step draws no real rows
      if (no_batch) {
        x = nullptr;
      } else if (x_batches) {
        x = x_batches + (size_t)i * B * e.F;
      } else if (e.mk.recording) {
        e.mk.src_rows = class_rows; e.mk.src_n = n_rows; e.mk.src_Bg = B_global; e.mk.src_off = (long long)e.rank * B;
        x = class_rows;
      } else {
        sample_rows_kernel<<<(B + 127) / 128, 128, 0, fork_to(e, 1, st)>>>(class_rows, n_rows, B_global, (long long)e.rank * B,
                                                                            B, e.F, 0, 0, e.ws.ctl, 0, e.ws.x_stage, nullptr);
        CVG_LAUNCH_CHECK();
        x = e.ws.x_stage;
      }
      StepRng rng;
      rng.set = false;
      rng.off = 1;                                   // sampling used counter + 0
      rng.lambda_nonzero = !(flags & CVG_VISIT_LAMBDA_ZERO);
      float* lo = loss_out ? loss_out + 4 * i : nullptr;
      const int sf = flags & (CVG_STEP_LOCAL_BN | CVG_STEP_NO_UPDATE | CVG_STEP_PRIOR_ONLY | CVG_STEP_CVAE);
      if (!e.mk.recording) e.step_dcounter = 2;      // two counter values per step (draw + noise), advanced by the step's tail
      if (kind == 0) CVG_TRY(step_d(e, x, label, B, nullptr, rng, sf, lo, st));
      else if (kind == 1) CVG_TRY(step_c(e, x, label, B, nullptr, rng, sf, lo, st));
      else CVG_TRY(step_g(e, x, label, B, nullptr, rng, sf, lo, st));
      e.mk.src_rows = nullptr;
      e.hoist_x = nullptr;
      if (e.mk.recording) {
        e.mk.dcounter += 2;                                    // applied once by the program's finish op
      }
    }
  }
  join_sides(e, st);       // the caller's stream continues after everything the visit enqueued
  return prog.finish(st);
}

void set_all_kernel_attributes() {
  mk_set_kernel_attributes();
  cudaFuncSetAttribute(sn_power_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SN_W_SMEM_MAX);
  cudaFuncSetAttribute(critic_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)critic_chain_smem(CH_MAX_IN));
  cudaFuncSetAttribute(classifier_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)classifier_chain_smem(CH_MAX_IN, CH_MAX_K));
  // cudaFuncSetAttribute is done once, eagerly, so that nothing but launches happens during graph capture
#define CVG_MN_ATTR(W, A, E) cudaFuncSetAttribute(gemm_mn_kernel<W, A, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024);
  CVG_MN_ATTR(true, OP_PLAIN, EP_LINEAR) CVG_MN_ATTR(true, OP_BN_ACT, EP_LINEAR) CVG_MN_ATTR(true, OP_REPARAM, EP_LINEAR)
  CVG_MN_ATTR(false, OP_PLAIN, EP_DACT) CVG_MN_ATTR(false, OP_CONST, EP_DACT) CVG_MN_ATTR(false, OP_PLAIN, EP_STORE)
  CVG_MN_ATTR(false, OP_PLAIN, EP_DBN) CVG_MN_ATTR(false, OP_BN_BWD, EP_DBN) CVG_MN_ATTR(false, OP_BN_BWD, EP_REPARAM_BWD)
#undef CVG_MN_ATTR
#define CVG_DW_ATTR(P, Q) cudaFuncSetAttribute(gemm_dw_kernel<P, Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
  CVG_DW_ATTR(OP_PLAIN, OP_PLAIN) CVG_DW_ATTR(OP_CONST, OP_PLAIN) CVG_DW_ATTR(OP_PLAIN, OP_BN_ACT)
  CVG_DW_ATTR(OP_BN_BWD, OP_BN_ACT) CVG_DW_ATTR(OP_BN_BWD, OP_REPARAM) CVG_DW_ATTR(OP_BN_BWD, OP_PLAIN)
#undef CVG_DW_ATTR
}

}  // namespace cvg
