// cvaegan_b200 - extern "C" entry points (see include/cvaegan_b200.h for the contract).
#include "engine.cuh"

namespace cvg {
const char* last_error();
int comm_unique_id(void* out128);
int comm_init(Engine& e, const void* id128, int rank, int world);
void comm_destroy(Engine& e);
}  // namespace cvg

using namespace cvg;

struct CvgHandle {
  Engine e;
};

#define H_OR_FAIL(h)                      \
  if (!(h)) {                             \
    cvg::set_error("null handle");        \
    return 1;                             \
  }


// filter_compact_stream_kernel is instantiated for class counts 1..FC_MAX_KC; wider heads use the generic kernel
constexpr int FC_MAX_KC = 12;
template <int KC>
struct FcDispatch {
  static int attrs() {
    CVG_CUDA(cudaFuncSetAttribute(filter_compact_stream_kernel<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
    CVG_CUDA(cudaFuncSetAttribute(filter_compact_stream_kernel<KC>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    return FcDispatch<KC - 1>::attrs();
  }
  static int launch(int K, unsigned grid, size_t smem, cudaStream_t st, const float* x, const float* logits, long long n, int F,
                    int label, float thr, uint64_t row_offset, int nsub, float* x_out, long long* idx_out, long long capacity,
                    unsigned long long* count) {
    if (K == KC) {
      filter_compact_stream_kernel<KC><<<grid, FC_THREADS, smem, st>>>(x, logits, n, F, KC, label, thr, row_offset, nsub, x_out,
                                                                       idx_out, capacity, count);
      return 0;
    }
    return FcDispatch<KC - 1>::launch(K, grid, smem, st, x, logits, n, F, label, thr, row_offset, nsub, x_out, idx_out, capacity, count);
  }
};
template <>
struct FcDispatch<0> {
  static int attrs() { return 0; }
  static int launch(int, unsigned, size_t, cudaStream_t, const float*, const float*, long long, int, int, float, uint64_t, int, float*,
                    long long*, long long, unsigned long long*) {
    CVG_FAIL("cvg_filter_compact: unsupported class count");
  }
};
static int fc_set_attributes() { return FcDispatch<FC_MAX_KC>::attrs(); }
static int fc_launch(int K, unsigned grid, size_t smem, cudaStream_t st, const float* x, const float* logits, long long n, int F,
                     int label, float thr, uint64_t row_offset, int nsub, float* x_out, long long* idx_out, long long capacity,
                     unsigned long long* count) {
  return FcDispatch<FC_MAX_KC>::launch(K, grid, smem, st, x, logits, n, F, label, thr, row_offset, nsub, x_out, idx_out, capacity, count);
}

extern "C" {

const char* cvg_last_error(void) { return cvg::last_error(); }
int cvg_abi_version(void) { return CVG_ABI_VERSION; }
int cvg_config_bytes(void) { return (int)sizeof(CvgConfig); }

int cvg_create(const CvgConfig* cfg, CvgHandle** out) {
  if (!cfg || !out) CVG_FAIL("cvg_create: null argument");
  *out = nullptr;
  int dev = 0;
  CVG_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CVG_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10)
    CVG_FAIL(std::string("cvaegan_b200 runs on sm_100 (B200) only; device is sm_") + std::to_string(prop.major) +
             std::to_string(prop.minor) + " - there is no fallback path");
  if (cfg->feature_num < 1 || cfg->label_num < 1 || cfg->z_size < 4 || cfg->max_batch < 1)
    CVG_FAIL("cvg_create: bad dimensions");
  if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size) CVG_FAIL("cvg_create: bad rank/world_size");
  CvgHandle* h = new CvgHandle();
  Engine& e = h->e;
  e.cfg = *cfg;
  e.F = cfg->feature_num;
  e.K = cfg->label_num;
  e.Kc = cfg->unconditional ? 0 : cfg->label_num;
  e.Z = cfg->z_size;
  e.world = cfg->world_size;
  e.rank = cfg->rank;
  e.num_sms = prop.multiProcessorCount;
  if (build_layouts(e) != 0) {
    delete h;
    return 1;
  }
  set_all_kernel_attributes();
  tc_set_kernel_attributes();
  {
    const char* off = getenv("CVG_DISABLE_TC");
    e.use_tc = tc_supported(e) && !(off && off[0] == '1');
    // training executors: the stand-alone FP32-FMA layer kernels (default: faster at the benchmarked batch of 4096), or -
    // CVG_TRAIN_MODE=mk / cvg_debug_set("train_mode", 1) - ONE persistent tcgen05 kernel per step / label visit (mega.cuh)
    const char* tm = getenv("CVG_TRAIN_MODE");
    e.mk.enabled = mk_supported(e) && tm && !strcmp(tm, "mk");
    if (const char* hv = getenv("CVG_HOIST")) e.hoist = atoi(hv) != 0;   // 0: every step of a visit runs its own G(z)
    const char* coop = getenv("CVG_MK_COOP");
    e.mk.coop = !(coop && coop[0] == '0');
    const char* ab = getenv("CVG_MK_ALLBAR");
    e.mk.allbar = ab && ab[0] == '1';
  }
  if (cudaGetLastError() != cudaSuccess) {
    cvg::set_error("cudaFuncSetAttribute failed");
    delete h;
    return 1;
  }
  {
    SideStreams& ms = h->e.ms;
    const char* off = getenv("CVG_STREAMS");
    ms.on = !(off && off[0] == '0');
    bool ok = true;
    for (int i = 0; i < SIDE_STREAMS && ok; ++i) ok = cudaStreamCreateWithFlags(&ms.s[i], cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < SIDE_EVENTS && ok; ++i) ok = cudaEventCreateWithFlags(&ms.ev[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 4 && ok; ++i) ok = cudaEventCreateWithFlags(&ms.layer[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
      cvg::set_error("creating the side streams failed");
      cvg_destroy(h);
      return 1;
    }
  }
  *out = h;
  return 0;
}

void cvg_destroy(CvgHandle* h) {
  if (!h) return;
  for (int i = 0; i < SIDE_STREAMS; ++i)
    if (h->e.ms.s[i]) cudaStreamDestroy(h->e.ms.s[i]);
  for (int i = 0; i < SIDE_EVENTS; ++i)
    if (h->e.ms.ev[i]) cudaEventDestroy(h->e.ms.ev[i]);
  for (int i = 0; i < 4; ++i)
    if (h->e.ms.layer[i]) cudaEventDestroy(h->e.ms.layer[i]);
  nvl_destroy(h->e);
  comm_destroy(h->e);
  mk_destroy(h->e);
  delete h;
}

int cvg_net_sizes(const CvgHandle* h, int net, int64_t* n_param_floats, int64_t* n_state_floats) {
  H_OR_FAIL(h);
  if (net < 0 || net >= CVG_NUM_NETS) CVG_FAIL("bad net id");
  if (n_param_floats) *n_param_floats = h->e.lay[net].n_param;
  if (n_state_floats) *n_state_floats = h->e.lay[net].n_state;
  return 0;
}

int cvg_tensor_table(const CvgHandle* h, int net, CvgTensorDesc* out, int32_t capacity, int32_t* count) {
  H_OR_FAIL(h);
  if (net < 0 || net >= CVG_NUM_NETS) CVG_FAIL("bad net id");
  const auto& t = h->e.lay[net].table;
  if (count) *count = (int32_t)t.size();
  if (out) {
    if (capacity < (int32_t)t.size()) CVG_FAIL("tensor table capacity too small");
    for (size_t i = 0; i < t.size(); ++i) out[i] = t[i];
  }
  return 0;
}

int64_t cvg_workspace_bytes(const CvgHandle* h) { return h ? workspace_bytes(h->e) : -1; }

int cvg_bind_net(CvgHandle* h, int net, float* params, float* grads, float* adam_m, float* adam_v, float* state) {
  H_OR_FAIL(h);
  if (net < 0 || net >= CVG_NUM_NETS) CVG_FAIL("bad net id");
  if (!params || !grads || !adam_m || !adam_v) CVG_FAIL("cvg_bind_net: null buffer");
  if (h->e.lay[net].n_state > 0 && !state) CVG_FAIL("cvg_bind_net: this network needs a state buffer");
  if ((((uintptr_t)params | (uintptr_t)grads | (uintptr_t)adam_m | (uintptr_t)adam_v | (uintptr_t)state) & 15) != 0)
    CVG_FAIL("cvg_bind_net: buffers must be 16-byte aligned");
  NetBuffers& b = h->e.buf[net];
  b.params = params; b.grads = grads; b.m = adam_m; b.v = adam_v; b.state = state;
  return 0;
}

int cvg_bind_workspace(CvgHandle* h, void* workspace, int64_t bytes, void* stream) {
  H_OR_FAIL(h);
  if (!workspace) CVG_FAIL("null workspace");
  CVG_TRY(carve_workspace(h->e, workspace, bytes));
  if (mk_supported(h->e)) CVG_TRY(mk_alloc_slots(h->e));   // program buffers of the step-program executor
  // rows beyond the batch are never read un-masked, but start from a defined state
  CVG_CUDA(cudaMemsetAsync(workspace, 0, (size_t)bytes, (cudaStream_t)stream));
  return 0;
}

int cvg_set_adam_step(CvgHandle* h, int net, int64_t t) {
  H_OR_FAIL(h);
  if (net < 0 || net >= CVG_NUM_NETS) CVG_FAIL("bad net id");
  if (!h->e.ws_base) CVG_FAIL("workspace not bound");
  long long v = (long long)t;
  CVG_CUDA(cudaMemcpy(&h->e.ws.ctl->adam_t[net], &v, sizeof(v), cudaMemcpyHostToDevice));
  return 0;
}
int64_t cvg_get_adam_step(const CvgHandle* h, int net) {
  if (!h || net < 0 || net >= CVG_NUM_NETS) return -1;
  if (!h->e.ws_base) return -1;
  long long v = -1;
  if (cudaMemcpy(&v, &h->e.ws.ctl->adam_t[net], sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return (int64_t)v;
}

int cvg_comm_unique_id(void* out128) {
  if (!out128) CVG_FAIL("null argument");
  return comm_unique_id(out128);
}
int cvg_comm_init(CvgHandle* h, const void* id128, int rank, int world_size) {
  H_OR_FAIL(h);
  if (world_size != h->e.cfg.world_size || rank != h->e.cfg.rank) CVG_FAIL("rank/world_size differ from cvg_create");
  return comm_init(h->e, id128, rank, world_size);
}

int cvg_nvl_local_handle(CvgHandle* h, void* out64) {
  H_OR_FAIL(h);
  if (!out64) CVG_FAIL("null argument");
  return nvl_local_handle(h->e, out64);
}
int cvg_nvl_attach(CvgHandle* h, const void* handles) {
  H_OR_FAIL(h);
  if (!handles) CVG_FAIL("null argument");
  return nvl_attach(h->e, handles);
}

int cvg_nvl_disable(CvgHandle* h) {
  H_OR_FAIL(h);
  nvl_destroy(h->e);
  return 0;
}

int cvg_step_d(CvgHandle* h, const float* x_real, int label, int B, const CvgNoise* noise, uint64_t seed,
               uint64_t counter, int flags, float* loss_out, void* stream) {
  H_OR_FAIL(h);
  if (!x_real) CVG_FAIL("null x_real");
  if (label < 0 || label >= h->e.K) CVG_FAIL("label out of range");
  StepRng rng;
  rng.seed = seed; rng.counter = counter;
  return step_d(h->e, x_real, label, B, noise, rng, flags, loss_out, (cudaStream_t)stream);
}
int cvg_step_c(CvgHandle* h, const float* x_real, int label, int B, const CvgNoise* noise, uint64_t seed,
               uint64_t counter, int flags, float* loss_out, void* stream) {
  H_OR_FAIL(h);
  if (!x_real) CVG_FAIL("null x_real");
  if (label < 0 || label >= h->e.K) CVG_FAIL("label out of range");
  StepRng rng;
  rng.seed = seed; rng.counter = counter;
  return step_c(h->e, x_real, label, B, noise, rng, flags, loss_out, (cudaStream_t)stream);
}
int cvg_step_g(CvgHandle* h, const float* x_real, int label, int B, const CvgNoise* noise, uint64_t seed,
               uint64_t counter, float lambda_class_now, int flags, float* loss_out, void* stream) {
  H_OR_FAIL(h);
  if (!x_real && !(flags & CVG_STEP_PRIOR_ONLY)) CVG_FAIL("null x_real");
  if ((flags & CVG_STEP_PRIOR_ONLY) && (flags & CVG_STEP_CVAE)) CVG_FAIL("CVG_STEP_PRIOR_ONLY and CVG_STEP_CVAE are mutually exclusive");
  if (label < 0 || label >= h->e.K) CVG_FAIL("label out of range");
  StepRng rng;
  rng.seed = seed; rng.counter = counter;
  rng.lambda_class = lambda_class_now; rng.lambda_nonzero = lambda_class_now != 0.f;
  return step_g(h->e, x_real, label, B, noise, rng, flags, loss_out, (cudaStream_t)stream);
}

int cvg_step_classifier(CvgHandle* h, const float* x, const int64_t* labels, int B, const CvgNoise* noise, uint64_t seed,
                        uint64_t counter, float lr, float beta1, float beta2, float eps, int flags, float* loss_out,
                        void* stream) {
  H_OR_FAIL(h);
  if (!x || !labels) CVG_FAIL("cvg_step_classifier: null argument");
  StepRng rng;
  rng.seed = seed; rng.counter = counter;
  AdamOverride ov{lr, beta1, beta2, eps};
  return step_classifier(h->e, x, (const long long*)labels, B, noise, rng, ov, flags, loss_out, (cudaStream_t)stream);
}

int cvg_visit(CvgHandle* h, int label, int B_local, int64_t B_global, const float* class_rows, int64_t n_rows,
              const float* x_batches, int d_loop, int c_loop, int g_loop, int flags, float* loss_out, void* stream) {
  H_OR_FAIL(h);
  if (label < 0 || label >= h->e.K) CVG_FAIL("label out of range");
  if (d_loop < 0 || c_loop < 0 || g_loop < 0) CVG_FAIL("cvg_visit: negative loop count");
  if ((flags & CVG_STEP_PRIOR_ONLY) && (flags & CVG_STEP_CVAE)) CVG_FAIL("CVG_STEP_PRIOR_ONLY and CVG_STEP_CVAE are mutually exclusive");
  if ((flags & CVG_STEP_CVAE) && d_loop != 0) CVG_FAIL("cvg_visit: a CVAE visit has no critic steps (d_loop must be 0, cvae.py:86-166)");
  return visit(h->e, label, B_local, B_global, class_rows, n_rows, x_batches, d_loop, c_loop, g_loop, flags, loss_out,
               (cudaStream_t)stream);
}

int cvg_ctl_set(CvgHandle* h, uint64_t seed, uint64_t counter, int set_rng, float lambda_class, int set_lambda, void* stream) {
  H_OR_FAIL(h);
  if (!h->e.ws_base) CVG_FAIL("workspace not bound");
  ctl_set_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->e.ws.ctl, seed, counter, set_rng, lambda_class, set_lambda);
  CVG_CUDA(cudaGetLastError());
  h->e.launches++;
  return 0;
}

int cvg_adam(CvgHandle* h, int net_mask, void* stream) {
  H_OR_FAIL(h);
  return run_adam(h->e, net_mask, (cudaStream_t)stream);
}

int cvg_sample_rows(CvgHandle* h, const float* class_rows, int64_t n, int64_t B_global, int64_t draw_offset,
                    int B_local, uint64_t seed, uint64_t counter, float* x_out, int64_t* idx_out, void* stream) {
  H_OR_FAIL(h);
  if (!class_rows || !x_out || n < 1 || B_local < 1 || draw_offset < 0 || draw_offset + B_local > B_global)
    CVG_FAIL("cvg_sample_rows: bad argument");
  sample_rows_kernel<<<(B_local + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      class_rows, n, B_global, draw_offset, B_local, h->e.F, seed, counter, nullptr, 0, x_out, (long long*)idx_out);
  CVG_CUDA(cudaGetLastError());
  h->e.launches++;
  return 0;
}

int cvg_generate(CvgHandle* h, int label, int64_t n, const float* z, uint64_t seed, uint64_t row_offset, int train_mode,
                 float* x_out, void* stream) {
  H_OR_FAIL(h);
  if (n < 0 || (n > 0 && !x_out)) CVG_FAIL("cvg_generate: bad argument");
  return generate(h->e, label, n, z, seed, row_offset, train_mode, x_out, (cudaStream_t)stream);
}

int cvg_generate_filter(CvgHandle* h, int label, int64_t n, float thr, const float* z, uint64_t seed,
                        uint64_t row_offset, float* x_out, int64_t* idx_out, int64_t capacity,
                        unsigned long long* count_out, float* logits_out, uint8_t* keep_out, void* stream) {
  H_OR_FAIL(h);
  if (n < 0 || !count_out || (capacity > 0 && !x_out)) CVG_FAIL("cvg_generate_filter: bad argument");
  return generate_filter(h->e, label, n, thr, z, seed, row_offset, x_out, idx_out, capacity, count_out, logits_out,
                         keep_out, (cudaStream_t)stream);
}

int cvg_filter_logits(const float* logits, int64_t n, int K, int label, float thr, uint8_t* keep_out, void* stream) {
  if (!logits || !keep_out || n < 0) CVG_FAIL("cvg_filter_logits: bad argument");
  if (K < 1 || K > FILTER_MAXK) CVG_FAIL("cvg_filter_logits: K must be in [1, 32]");
  if (n == 0) return 0;
  filter_logits_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(logits, n, K, label, thr, keep_out);
  CVG_CUDA(cudaGetLastError());
  return 0;
}

int cvg_filter_compact(const float* x, const float* logits, int64_t n, int F, int K, int label, float thr,
                       uint64_t row_offset, float* x_out, int64_t* idx_out, int64_t capacity,
                       unsigned long long* count_out, void* stream) {
  if (!x || !logits || !count_out || n < 0) CVG_FAIL("cvg_filter_compact: bad argument");
  if (K < 1 || K > FILTER_MAXK) CVG_FAIL("cvg_filter_compact: K must be in [1, 32]");
  if (n == 0) return 0;
  if (K > FC_MAX_KC) {
    filter_compact_kernel<false><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        x, logits, n, 0, F, K, label, thr, row_offset, x_out, (long long*)idx_out, capacity, count_out, nullptr, nullptr);
  } else {
    const size_t smem = (size_t)FC_SUB_ROWS * K * sizeof(float);      // K <= 32 -> at most 128 KB
    static int sms = 0;
    if (!sms) {
      int dev = 0;
      CVG_CUDA(cudaGetDevice(&dev));
      CVG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
      CVG_TRY(fc_set_attributes());
    }
    // few CTAs (one same-address atomic each), one full wave of 6 per SM (__launch_bounds__); sub-blocks are grid-strided over the CTAs.
    // A launch covers at most grid * FC_MAXSUB sub-blocks; longer streams take several launches.
    const long long slots = (long long)sms * 6;
    long long done = 0;
    while (done < n) {
      const long long left = n - done;
      const long long nblk1k = (left + FC_SUB_ROWS - 1) / FC_SUB_ROWS;
      const long long grid = nblk1k < slots ? nblk1k : slots;
      long long nsub = (nblk1k + grid - 1) / grid;
      long long rows_now = left;
      if (nsub > FC_MAXSUB) {
        nsub = FC_MAXSUB;
        rows_now = grid * nsub * FC_SUB_ROWS;
      }
      CVG_TRY(fc_launch(K, (unsigned)grid, smem, (cudaStream_t)stream, x + done * F, logits + done * K, rows_now, F, label, thr,
                        row_offset + (uint64_t)done, (int)nsub, x_out, (long long*)idx_out, capacity, count_out));
      CVG_CUDA(cudaGetLastError());
      done += rows_now;
    }
  }
  CVG_CUDA(cudaGetLastError());
  return 0;
}

int cvg_classifier_forward(CvgHandle* h, const float* x, int64_t n, float* logits_out, void* stream) {
  H_OR_FAIL(h);
  if (!x || !logits_out || n < 0) CVG_FAIL("cvg_classifier_forward: bad argument");
  return classifier_forward(h->e, x, n, logits_out, (cudaStream_t)stream);
}
int cvg_encoder_forward(CvgHandle* h, const float* x, int label, int64_t n, float* mu_out, float* logvar_out,
                        void* stream) {
  H_OR_FAIL(h);
  if (!x || !mu_out || !logvar_out || n < 0) CVG_FAIL("cvg_encoder_forward: bad argument");
  return encoder_forward(h->e, x, label, n, mu_out, logvar_out, (cudaStream_t)stream);
}

int cvg_patience_scan(const uint8_t* keep, int64_t n, int64_t num, int chunk, int patience, int64_t* rows_consumed,
                      int64_t* rows_accepted) {
  if (!keep || !rows_consumed || !rows_accepted || chunk < 1) CVG_FAIL("cvg_patience_scan: bad argument");
  int64_t pos = 0, got = 0;
  while (got < num && patience > 0) {
    const int64_t c = (num - got) < chunk ? (num - got) : chunk;
    if (pos + c > n) CVG_FAIL("cvg_patience_scan: row stream too short");
    int64_t k = 0;
    for (int64_t i = 0; i < c; ++i) k += keep[pos + i] ? 1 : 0;
    pos += c;
    got += k;
    if (k == 0) --patience;
  }
  *rows_consumed = pos;
  *rows_accepted = got;
  return 0;
}

int cvg_debug_read(CvgHandle* h, const char* name, int pass, int rows, float* dst, int* features_out, void* stream) {
  H_OR_FAIL(h);
  if (!name) CVG_FAIL("null name");
  Engine& e = h->e;
  const Workspace& w = e.ws;
  if (!e.ws_base) CVG_FAIL("workspace not bound");
  const std::string n(name);
  const float* p = nullptr;
  int C = 0;
  auto idx = [&](const char* prefix) -> int {
    const size_t L = strlen(prefix);
    if (n.size() == L + 1 && n.compare(0, L, prefix) == 0 && n[L] >= '0' && n[L] <= '2') return n[L] - '0';
    return -1;
  };
  int i;
  if (n == "xT") { p = w.xT; C = e.F; }
  else if (n == "z") { p = w.z; C = e.Z; }
  else if ((i = idx("g_h")) >= 0) { p = w.g_h[i]; C = e.gh[i]; }
  else if ((i = idx("g_dy")) >= 0) { p = w.g_dy[i]; C = e.gh[i]; }
  else if (n == "g_out") { p = w.g_out; C = e.F; }
  else if (n == "g_dout") { p = w.g_dout; C = e.F; }
  else if ((i = idx("e_h")) >= 0) { p = w.e_h[i]; C = e.eh[i]; }
  else if ((i = idx("e_dy")) >= 0) { p = w.e_dy[i]; C = e.eh[i]; }
  else if (n == "e_ml") { p = w.e_ml; C = 2 * e.Z; }
  else if (n == "e_dml") { p = w.e_dml; C = 2 * e.Z; }
  else if ((i = idx("d_a")) >= 0) { p = w.d_a[i]; C = e.dh[i]; }
  else if ((i = idx("d_g")) >= 0) { p = w.d_g[i]; C = e.dh[i]; }
  else if (n == "d_s") { p = w.d_s; C = 1; }
  else if (n == "c_a1") { p = w.c_a1; C = e.ch[0]; }
  else if (n == "c_h2") { p = w.c_h2; C = e.ch[1]; }
  else if (n == "c_a2") { p = w.c_a2; C = e.ch[1]; }
  else if (n == "c_a3") { p = w.c_a3; C = e.ch[2]; }
  else if (n == "c_logit") { p = w.c_logit; C = e.K; }
  else if (n == "c_dlogit") { p = w.c_dlogit; C = e.K; }
  else if ((i = idx("c_g")) >= 0) { p = w.c_g[i]; C = e.ch[i]; }
  else if (n == "dx") { p = w.dx; C = e.F; }
  else CVG_FAIL("cvg_debug_read: unknown buffer name");
  if (features_out) *features_out = C;
  if (!dst) return 0;
  if (rows < 1 || rows > w.ld || pass < 0 || pass > 1) CVG_FAIL("cvg_debug_read: bad rows/pass");
  to_row_major_kernel<<<(rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p + (size_t)pass * C * w.ld, rows, C, w.ld, dst);
  CVG_CUDA(cudaGetLastError());
  return 0;
}

int cvg_debug_tc_counters(CvgHandle* h, long long* dev_counters) {
  H_OR_FAIL(h);
  h->e.tc_dbg = dev_counters;
  return 0;
}

int cvg_profile_enable(CvgHandle* h, int enable) {
  H_OR_FAIL(h);
  Engine& e = h->e;
  for (auto& r : e.prof_recs) {
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  e.prof_recs.clear();
  e.prof = enable != 0;
  return 0;
}

int cvg_profile_read(CvgHandle* h, int kernel_class, int64_t* launches, double* flops, double* ms) {
  H_OR_FAIL(h);
  if (!launches || !flops || !ms) CVG_FAIL("cvg_profile_read: null argument");
  Engine& e = h->e;
  *launches = 0;
  *flops = 0.0;
  *ms = 0.0;
  for (auto& r : e.prof_recs) {
    if (r.cls != kernel_class) continue;
    CVG_CUDA(cudaEventSynchronize(r.b));
    float t = 0.f;
    CVG_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
    *launches += 1;
    *flops += r.flops;
    *ms += (double)t;
  }
  return 0;
}

int64_t cvg_launch_count(const CvgHandle* h) { return h ? h->e.launches : -1; }

int cvg_debug_set(CvgHandle* h, const char* key, int value) {
  H_OR_FAIL(h);
  if (!key) CVG_FAIL("null key");
  Engine& e = h->e;
  const std::string k(key);
  if (k == "train_mode") {            // 0: stand-alone FFMA kernels, 1: step-program kernel (tcgen05)
    if (value && !mk_supported(e)) CVG_FAIL("cvg_debug_set: the step-program kernel does not cover these layer widths");
    e.mk.enabled = value != 0;
  } else if (k == "mk_max_ops") e.mk.max_ops = value;
  else if (k == "mk_allbar") e.mk.allbar = value != 0;
  else if (k == "mk_coop") e.mk.coop = value != 0;
  else if (k == "hoist") e.hoist = value != 0;
  else if (k == "streams") e.ms.on = value != 0;
  else if (k == "chain") e.chain = value != 0;      // 0: the D / C steps run the layer kernels (the chains' reference)
  else if (k == "eg_split") e.eg_split = value != 0;   // 0: the E/G step's generator backward runs both passes per launch
  else if (k == "fuse_stats") e.nvl.fuse = value != 0;
  else CVG_FAIL("cvg_debug_set: unknown key");
  return 0;
}

int cvg_debug_get(const CvgHandle* h, const char* key, int* value) {
  H_OR_FAIL(h);
  if (!key || !value) CVG_FAIL("null argument");
  const Engine& e = h->e;
  const std::string k(key);
  if (k == "train_mode") *value = e.mk.enabled ? 1 : 0;
  else if (k == "mk_last_nops") *value = e.mk.last_nops;
  else if (k == "mk_supported") *value = mk_supported(e) ? 1 : 0;
  else CVG_FAIL("cvg_debug_get: unknown key");
  return 0;
}

int cvg_debug_mk_cycles(CvgHandle* h, long long* out, int capacity, int* count) {
  H_OR_FAIL(h);
  Engine& e = h->e;
  if (!e.ws_base) CVG_FAIL("workspace not bound");
  // capacity >= 2048 + 64: also returns the GEMM section counters at out[2048 ...]
  const int n = e.mk.last_nops < capacity ? e.mk.last_nops : capacity;
  if (count) *count = n;
  if (out && n > 0) CVG_CUDA(cudaMemcpy(out, e.ws.mk_dbg, sizeof(long long) * n, cudaMemcpyDeviceToHost));
  if (out && capacity >= 2048 + 64 && n <= 1024) {
    // out[1024 + i]: start clock of op i (CTA 0);  out[3072 + i] (capacity >= 4096): kind | bar_before << 8 | items << 16
    CVG_CUDA(cudaMemcpy(out + 1024, e.ws.mk_dbg + 1024, sizeof(long long) * n, cudaMemcpyDeviceToHost));
    if (capacity >= 4096)
      for (int i = 0; i < n && i < (int)e.mk.last_kinds.size(); ++i) out[3072 + i] = e.mk.last_kinds[i];
  }
  if (out && capacity >= 2048 + 64) CVG_CUDA(cudaMemcpy(out + 2048, e.ws.mk_dbg + 2048, sizeof(long long) * 64, cudaMemcpyDeviceToHost));
  return 0;
}

}  // extern "C"
