// cvaegan_b200 - engine state: network layouts, borrowed buffers, workspace carving.
#pragma once
#include "common.cuh"
#include "gemm.cuh"
#include "misc_kernels.cuh"
#include "comm_nvl.cuh"

typedef struct ncclComm* ncclComm_t;

namespace cvg {

constexpr int HOIST_MAX = 16;  // generator passes one hoisted forward can hold (d_loop + c_loop of a visit)
constexpr int STAT_C = 1024;   // max features of a BatchNorm layer (stats slots are [2][STAT_C])

constexpr int DET_MAX_PASS = 4;   // passes per launch the deterministic-reduction slots are sized for
constexpr int SIDE_STREAMS = 3;   // streams beside the caller's (SideStreams)

// feature-major workspace (all float matrices are [features][ld], two pass slots where noted)
struct Workspace {
  int ld = 0;          // rows rounded up to 64
  int rows_cap = 0;
  // inputs / noise
  float* xT = nullptr;      // [F][ld]
  float* z = nullptr;       // [2][Z][ld]      slot 0: z (D/C steps) or eps (G step); slot 1: z_prior (G step)
  uint8_t* d_m1 = nullptr;  // [2][H1][ld]
  uint8_t* d_m2 = nullptr;  // [2][H2][ld]
  uint8_t* c_m1 = nullptr;
  uint8_t* c_m2 = nullptr;
  // generator
  float *g_h[3] = {nullptr, nullptr, nullptr};   // [2][Hi][ld] pre-BN
  float* g_out = nullptr;                        // [2][F][ld]
  // generator forward of every critic / classifier step of a visit, run once up front (train.cu hoist_generator)
  float* hz = nullptr;                           // [HOIST_MAX][Z][ld]
  float* hh[3] = {nullptr, nullptr, nullptr};    // [HOIST_MAX][Hi][ld] pre-BN
  float* hout = nullptr;                         // [HOIST_MAX][F][ld]
  double* hfst = nullptr;                        // [3 layers][HOIST_MAX][2 * STAT_C]
  float *g_dy[3] = {nullptr, nullptr, nullptr};
  float* g_dout = nullptr;                       // [2][F][ld]
  // encoder
  float *e_h[3] = {nullptr, nullptr, nullptr};   // [Hi][ld]
  float* e_ml = nullptr;                         // [2Z][ld]  mu | logvar
  float *e_dy[3] = {nullptr, nullptr, nullptr};
  float* e_dml = nullptr;
  // critic
  float *d_a[3] = {nullptr, nullptr, nullptr};   // [2][Hi][ld] post activation/dropout
  float* d_s = nullptr;                          // [2][1][ld]
  float *d_g[3] = {nullptr, nullptr, nullptr};   // [2][Hi][ld] grads w.r.t. pre-activations
  // classifier
  float* c_a1 = nullptr;    // [2][H1][ld]
  float* c_h2 = nullptr;    // [2][H2][ld]
  float* c_a2 = nullptr;
  float* c_rs = nullptr;    // [2][2][ld]
  float* c_a3 = nullptr;    // [2][H3][ld]
  float* c_logit = nullptr; // [2][K][ld]
  float* c_dlogit = nullptr;
  float *c_g[3] = {nullptr, nullptr, nullptr};
  float* dx = nullptr;      // [F][ld]
  // spectral norm scratch
  float* sn_sigma = nullptr;      // [2][4]
  float* sn_inv_sigma = nullptr;  // [4][2]
  float* sn_u = nullptr;          // [2][sn_snap]
  float* sn_v = nullptr;
  long long sn_snap = 0;
  float* sn_G = nullptr;          // [2][n_param(D)] per-pass raw critic gradients
  // accumulators (doubles), zeroed every step
  double* acc = nullptr;
  size_t acc_bytes = 0;
  double* loss = nullptr;         // [L_COUNT]
  double* g_fst = nullptr;        // [3 layers][2 pass][2][STAT_C]
  double* g_bst = nullptr;
  double* e_fst = nullptr;        // [3][1][2][STAT_C]
  double* e_bst = nullptr;
  // generation scratch
  unsigned long long* gen_count = nullptr;
  // device-resident step control block + staging for device-side sampling
  StepCtl* ctl = nullptr;
  float* x_stage = nullptr;        // [rows][F] row-major batch drawn by sample_rows_kernel
  // tensor-core path: pre-split weights in shared-memory operand order + per-feature epilogue constants
  float* tc_w = nullptr;
  float* tc_c = nullptr;
  // step-program kernel (mega.cuh): weight-gradient partial slots, grid-barrier counter, materialised z_enc slot
  float* dw_scratch = nullptr;
  long long dw_scratch_floats = 0;
  // stand-alone kernels' deterministic reductions (gemm_dw_kernel, ln_bwd_kernel): fixed-point accumulators and ticket
  // counters, one set per stream the engine launches on (0: the caller's, 1 + i: side stream i), since launches on one
  // stream never overlap
  unsigned long long* det_acc[SIDE_STREAMS + 1] = {};
  unsigned* det_cnt[SIDE_STREAMS + 1] = {};
  long long det_acc_n = 0;
  int det_cnt_n = 0;
  unsigned int* mk_bar = nullptr;
  float* z_eps = nullptr;          // [Z][ld] reparameterisation noise of the E+G step when the program kernel runs it
  float* mk_wprep = nullptr;       // hi / lo pre-split weight chunks of every layer, both GEMM orientations
  long long mk_wprep_floats = 0;
  long long* mk_dbg = nullptr;     // per-op cycle counters of the last program (development)
};

// ---- step-program recorder (mega.cu) ---------------------------------------------------------------------------------
struct MkSlot {
  void* dev = nullptr;
  void* host = nullptr;            // pinned mirror (a captured graph re-reads it at every replay)
  size_t bytes = 0;
  unsigned long long hash = 0;
  cudaEvent_t ev = nullptr;        // completion of the last upload from `host`
  bool in_graph = false;           // uploaded during stream capture: never recycled
  unsigned long long last_use = 0;
};
struct MkPrepSlot {
  const float* W = nullptr;
  int ldw = 0, wcol0 = 0, wt = 0, R = 0, N = 0, net = -1;
  long long off = 0;               // floats into ws.mk_wprep
  bool fresh = false;              // prepped in this program and the net has not been updated since
};
struct MkPendingRed {
  unsigned char bytes[160];
  int items;
};
struct MkState {
  bool enabled = true;             // CVG_TRAIN_MODE=ffma (or an unsupported shape) keeps the stand-alone FFMA kernels
  bool coop = true;                // cooperative launch (CVG_MK_COOP=0: plain launch of one CTA per SM)
  bool allbar = false;             // CVG_MK_ALLBAR=1: a grid barrier before every op (debugging)
  int max_ops = -1;                // development: truncate every program after this many ops
  bool recording = false;
  bool par_next = false;
  std::vector<unsigned char> ops;  // mk::OpRec records
  int nops = 0;
  int phase_items = 0;
  long long scratch_off = 0;
  int n_exchanges = 0;
  int adam_inc[4] = {0, 0, 0, 0};
  unsigned long long dcounter = 0;
  std::vector<MkPendingRed> pending_red;
  std::vector<MkPrepSlot> prep;    // per program: which weight operands have been pre-split, and where
  long long prep_off = 0;
  bool prep_open = false;          // the newest op is a prep op that can still take entries
  const float* src_rows = nullptr;   // inside a visit program: class table the next step draws its batch from
  long long src_n = 0, src_Bg = 0, src_off = 0;
  std::vector<MkSlot> slots;
  unsigned long long clock = 0;
  int last_nops = 0;
  std::vector<int> last_kinds;     // per op of the last program: kind | bar_before << 8 | items << 16
};

struct ProfRec {
  cudaEvent_t a, b;
  int cls;
  double flops;
};

// Extra streams beside the caller's: the stand-alone layer kernels are latency bound at the benchmarked sizes, so
// independent ones (weight gradients beside the input-gradient chain, the critic's power iteration and the batch staging
// beside the noise fill, C beside D in the E/G step) run concurrently.  Fork / join with events, so the work stays
// capturable in the caller's CUDA graph and ordered with the caller's stream.  The third side stream only carries the
// encoder's weight gradients of the E/G step, whose generator backward runs as two per-pass chains on the caller's stream
// and side stream 1, with the generator's weight gradients on side stream 0.
constexpr int SIDE_EVENTS = 32;   // fork / join events, used round-robin (far more than are ever pending at once)
struct SideStreams {
  bool on = false;
  cudaStream_t s[SIDE_STREAMS] = {};
  cudaEvent_t ev[SIDE_EVENTS] = {};
  cudaEvent_t layer[4] = {};        // E/G step: layer l of the generator's z_prior pass is done (the z_enc pass waits for it)
  unsigned next = 0;
  bool dirty[SIDE_STREAMS] = {};
};

struct Engine {
  bool prof = false;
  std::vector<ProfRec> prof_recs;
  CvgConfig cfg{};
  int F = 0, K = 0, Z = 0;
  int Kc = 0;                      // one-hot label columns beside the input of E, G and D: K, or 0 (CvgConfig.unconditional)
  int eh[3]{}, gh[3]{}, dh[3]{}, ch[3]{};
  NetLayout lay[4];
  NetBuffers buf[4];
  Workspace ws;
  void* ws_base = nullptr;
  int64_t ws_bytes = 0;
  int64_t launches = 0;
  const float* hoist_x = nullptr;   // visit(): G(z) of the step being emitted, computed up front (null: the step runs G)
  SideStreams ms;
  bool in_visit = false;            // steps emitted by visit(): their gradient reduction + Adam may run beside the next step
  unsigned long long step_dcounter = 0;   // visit(): Philox counter values the step being emitted uses (advanced at its end)
  int hoist = 1;                    // CVG_HOIST=0: every step runs its own generator forward
  bool chain = true;                // D / C steps run the critic / classifier as fused row-tile chains (chain.cuh) where they fit
  bool eg_split = true;             // the E/G step runs the generator backward of its two passes as two chains (train.cu step_g)
  ncclComm_t comm = nullptr;
  int world = 1, rank = 0;
  NvlState nvl;            // NVLink peer-memory all-reduce for the latency-bound exchanges (comm_nvl.cuh)
  int num_sms = 148;
  long long* tc_dbg = nullptr;   // development: device cycle counters of tc_eval_kernel (cvg_debug_tc_counters)
  bool use_tc = true;      // tensor-core chains (CVG_DISABLE_TC=1 forces the FFMA layer kernels)
  MkState mk;              // training steps as ONE persistent tcgen05 kernel per step / label visit (mega.cuh)

  float* P(int net, int64_t off) const { return buf[net].params + off; }
  float* G(int net, int64_t off) const { return buf[net].grads + off; }
  float* S(int net, int64_t off) const { return buf[net].state + off; }
};

struct CvgHandleImpl {
  Engine e;
};

// layout.cu
int build_layouts(Engine& e);
int64_t workspace_bytes(const Engine& e);
int carve_workspace(Engine& e, void* base, int64_t bytes);

// train.cu
// How a step obtains its Philox key/counter and lambda_class: the C-ABI step calls write them into the control
// block first (set = true); a label visit leaves the block alone and addresses counter + off.
struct StepRng {
  bool set = true;
  uint64_t seed = 0, counter = 0, off = 0;
  float lambda_class = 0.f;
  bool lambda_nonzero = true;
};
int step_d(Engine& e, const float* x_real, int label, int B, const CvgNoise* noise, const StepRng& rng, int flags,
           float* loss_out, cudaStream_t st);
int step_c(Engine& e, const float* x_real, int label, int B, const CvgNoise* noise, const StepRng& rng, int flags,
           float* loss_out, cudaStream_t st);
int step_g(Engine& e, const float* x_real, int label, int B, const CvgNoise* noise, const StepRng& rng, int flags,
           float* loss_out, cudaStream_t st);
int visit(Engine& e, int label, int B, int64_t B_global, const float* class_rows, int64_t n_rows, const float* x_batches,
          int d_loop, int c_loop, int g_loop, int flags, float* loss_out, cudaStream_t st);
void set_all_kernel_attributes();
struct AdamOverride {
  float lr, beta1, beta2, eps;
};
int run_adam(Engine& e, int net_mask, cudaStream_t st, const AdamOverride* ov = nullptr, bool steps_advanced = false);
int step_classifier(Engine& e, const float* x, const long long* labels, int B, const CvgNoise* noise, const StepRng& rng,
                    const AdamOverride& ov, int flags, float* loss_out, cudaStream_t st);
int nvl_local_handle(Engine& e, void* out64);
int nvl_attach(Engine& e, const void* handles);
void nvl_destroy(Engine& e);
int comm_all_reduce_f32(Engine& e, float* p, int64_t n, cudaStream_t st, int channel = 0);
int comm_all_reduce_f64(Engine& e, double* p, int64_t n, cudaStream_t st);
int comm_all_reduce_stats(Engine& e, double* p, int npass, int C, cudaStream_t st);

// mega.cu: step programs
bool mk_supported(const Engine& e);
void mk_set_kernel_attributes();
void mk_destroy(Engine& e);
int mk_alloc_slots(Engine& e);
int mk_begin(Engine& e);                                   // start recording (no-op when the program kernel is off)
int mk_flush(Engine& e, cudaStream_t st);                  // finish + upload + launch the recorded program
int mk_push(Engine& e, int kind, const void* payload, size_t bytes, int items, int a0 = 0, int a1 = 0, int a2 = 0, int a3 = 0,
            const void* extra = nullptr, size_t extra_bytes = 0);
int mk_weight_operand(Engine& e, const GemmArgs& g, bool wt, const float** out, bool* emitted = nullptr);   // pre-split weights (+ prep op when stale)
void mk_weights_updated(Engine& e, int net_mask);          // Adam recorded for these networks: their pre-split copies are stale
int mk_push_dw(Engine& e, const DwArgs& g);                // weight-gradient op + its deferred deterministic reduction
int mk_emit_dwred(Engine& e);                              // emits the pending reductions (one phase)

// generate.cu
int generate(Engine& e, int label, int64_t n, const float* z, uint64_t seed, uint64_t row_offset, int train_mode,
             float* x_out, cudaStream_t st);
int generate_filter(Engine& e, int label, int64_t n, float thr, const float* z, uint64_t seed, uint64_t row_offset,
                    float* x_out, int64_t* idx_out, int64_t capacity, unsigned long long* count_out, float* logits_out,
                    uint8_t* keep_out, cudaStream_t st);
int classifier_forward(Engine& e, const float* x, int64_t n, float* logits_out, cudaStream_t st);
int encoder_forward(Engine& e, const float* x, int label, int64_t n, float* mu_out, float* lv_out, cudaStream_t st);

// eval_tc.cu: fused eval-mode chains on tcgen05 (no CPU or library fallback; unsupported widths use the FFMA kernels)
bool tc_supported(const Engine& e);
int64_t tc_prep_floats(const Engine& e);
int64_t tc_const_floats();
void tc_set_kernel_attributes();
int tc_generate(Engine& e, int label, int64_t n, const float* z, uint64_t seed, uint64_t row_offset, float* x_out, cudaStream_t st);
int tc_generate_filter(Engine& e, int label, int64_t n, float thr, const float* z, uint64_t seed, uint64_t row_offset, float* x_out,
                       int64_t* idx_out, int64_t capacity, unsigned long long* count_out, float* logits_out, uint8_t* keep_out,
                       cudaStream_t st);
int tc_classifier_forward(Engine& e, const float* x, int64_t n, float* logits_out, cudaStream_t st);
int tc_encoder_forward(Engine& e, const float* x, int label, int64_t n, float* mu_out, float* lv_out, cudaStream_t st);

// shared launch helpers (train.cu)
int launch_mn(Engine& e, bool wt, const GemmArgs& g, cudaStream_t st);
int launch_dw(Engine& e, const DwArgs& g, cudaStream_t st);
// where a generator forward reads z and keeps its activations / batch sums (default: the two-pass step buffers)
struct GenBufs {
  const float* z;
  float* h[3];
  float* out;
  double* fst[3];
  uint64_t pad = 0;
};
// one pass of a two-pass generator forward run as a chain of its own (E/G step): which pass, the exchange channel of its
// stream, and the per-layer events it records (rec) or waits for before each layer after the first (wait)
struct GenSplit {
  int only_pass = -1;
  int channel = 0;
  cudaEvent_t* rec = nullptr;
  cudaEvent_t* wait = nullptr;
};
int fwd_generator(Engine& e, int npass, bool train, bool reparam_pass0, int label, int M, float Bg, bool local_bn,
                  cudaStream_t st, const GenBufs* gb = nullptr, const GenSplit* split = nullptr);
int fwd_classifier(Engine& e, const float* xin, long long sxin, int npass, bool train, int M, cudaStream_t st);
int fwd_encoder(Engine& e, bool train, int label, int M, float Bg, bool local_bn, cudaStream_t st);

}  // namespace cvg
