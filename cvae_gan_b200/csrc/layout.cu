// cvaegan_b200 - network layouts (reference state_dict keys -> offsets) and workspace carving.
#include "engine.cuh"

namespace cvg {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error() { return g_err.c_str(); }

static int64_t pad4(int64_t n) { return (n + 3) & ~(int64_t)3; }

struct Builder {
  NetLayout& L;
  int64_t po = 0, so = 0;
  explicit Builder(NetLayout& l) : L(l) {}
  int64_t add(const std::string& key, int kind, int64_t d0, int64_t d1) {
    CvgTensorDesc t;
    memset(&t, 0, sizeof(t));
    snprintf(t.key, sizeof(t.key), "%s", key.c_str());
    t.kind = kind;
    t.ndim = d1 > 0 ? 2 : 1;
    t.shape[0] = d0;
    t.shape[1] = d1 > 0 ? d1 : 0;
    const int64_t n = d0 * (d1 > 0 ? d1 : 1);
    int64_t& o = kind == 0 ? po : so;
    t.offset = o;
    o += pad4(n);
    L.table.push_back(t);
    return t.offset;
  }
};

static void hidden(const CvgConfig& cfg, int tin, bool fixed3, int* h) {
  if (cfg.hidden[0] > 0) {            // widened model (BASELINE.json configs[4]): the same three widths for every network
    for (int i = 0; i < 3; ++i) h[i] = cfg.hidden[i];
    return;
  }
  // cvae_gan_models.py:16-18, 85-87, 173-175, 257-259
  h[0] = tin > 256 ? tin : 256;
  h[1] = tin / 2 > 128 ? tin / 2 : 128;
  h[2] = fixed3 ? 64 : (tin / 4 > 64 ? tin / 4 : 64);
}

int build_layouts(Engine& e) {
  const int F = e.F, Z = e.Z;
  const int K = e.Kc;                  // label columns of E / G / D (0: unconditional networks); the classifier has e.K outputs
  const int* hv = e.cfg.hidden;
  if (hv[0] != 0 || hv[1] != 0 || hv[2] != 0)
    for (int i = 0; i < 3; ++i)
      if (hv[i] < 64 || hv[i] % 64 != 0) CVG_FAIL("CvgConfig.hidden: all zero, or three multiples of 64");
  hidden(e.cfg, F + K, false, e.eh);
  hidden(e.cfg, Z + K, false, e.gh);
  hidden(e.cfg, F + K, true, e.dh);
  hidden(e.cfg, F, true, e.ch);
  for (int i = 0; i < 3; ++i)
    if (e.eh[i] > STAT_C || e.gh[i] > STAT_C || e.dh[i] > SN_MAXDIM || e.ch[i] > STAT_C)
      CVG_FAIL("layer wider than supported (1024)");
  if (Z % 4 != 0) CVG_FAIL("z_size must be a multiple of 4");
  if (e.K > FILTER_MAXK) CVG_FAIL("label_num > 32 is not supported");
  if (e.ch[1] > 8 * LN_MAXF_WIDE) CVG_FAIL("classifier LayerNorm wider than 512 is not supported");

  {  // encoder (cvae_gan_models.py:20-35)
    NetLayout& L = e.lay[CVG_NET_ENCODER];
    Builder b(L);
    int dims[4] = {F + K, e.eh[0], e.eh[1], e.eh[2]};
    const int li[3] = {0, 3, 6};
    for (int i = 0; i < 3; ++i) {
      LinearP& p = L.lin[i];
      p.out = dims[i + 1];
      p.in = dims[i];
      std::string s = "encoder." + std::to_string(li[i]), n = "encoder." + std::to_string(li[i] + 1);
      p.w = b.add(s + ".weight", 0, p.out, p.in);
      p.b = b.add(s + ".bias", 0, p.out, 0);
      p.gamma = b.add(n + ".weight", 0, p.out, 0);
      p.beta = b.add(n + ".bias", 0, p.out, 0);
      p.rmean = b.add(n + ".running_mean", 1, p.out, 0);
      p.rvar = b.add(n + ".running_var", 1, p.out, 0);
    }
    LinearP& h = L.lin[3];  // fc_mu and fc_logvar stored back to back -> one [2Z][h3] matrix
    h.out = 2 * Z;
    h.in = e.eh[2];
    h.w = b.add("fc_mu.weight", 0, Z, h.in);
    b.add("fc_logvar.weight", 0, Z, h.in);
    h.b = b.add("fc_mu.bias", 0, Z, 0);
    b.add("fc_logvar.bias", 0, Z, 0);
    if (((int64_t)Z * h.in) % 4 != 0) CVG_FAIL("encoder head size not 16-byte aligned");
    L.nlin = 4;
    L.n_param = b.po;
    L.n_state = b.so;
  }
  {  // generator (cvae_gan_models.py:89-108)
    NetLayout& L = e.lay[CVG_NET_GENERATOR];
    Builder b(L);
    int dims[4] = {Z + K, e.gh[0], e.gh[1], e.gh[2]};
    const int li[3] = {0, 3, 6};
    for (int i = 0; i < 3; ++i) {
      LinearP& p = L.lin[i];
      p.out = dims[i + 1];
      p.in = dims[i];
      std::string s = "main_model." + std::to_string(li[i]), n = "main_model." + std::to_string(li[i] + 1);
      p.w = b.add(s + ".weight", 0, p.out, p.in);
      p.b = b.add(s + ".bias", 0, p.out, 0);
      p.gamma = b.add(n + ".weight", 0, p.out, 0);
      p.beta = b.add(n + ".bias", 0, p.out, 0);
      p.rmean = b.add(n + ".running_mean", 1, p.out, 0);
      p.rvar = b.add(n + ".running_var", 1, p.out, 0);
    }
    LinearP& o = L.lin[3];
    o.out = F;
    o.in = e.gh[2];
    o.w = b.add("last_layer.0.weight", 0, o.out, o.in);
    o.b = b.add("last_layer.0.bias", 0, o.out, 0);
    L.nlin = 4;
    L.n_param = b.po;
    L.n_state = b.so;
  }
  {  // critic (cvae_gan_models.py:177-190); parameters() order of a parametrised Linear: bias, original
    NetLayout& L = e.lay[CVG_NET_DISCRIMINATOR];
    Builder b(L);
    int dims[5] = {F + K, e.dh[0], e.dh[1], e.dh[2], 1};
    const int li[4] = {0, 3, 6, 8};
    for (int i = 0; i < 4; ++i) {
      LinearP& p = L.lin[i];
      p.out = dims[i + 1];
      p.in = dims[i];
      std::string s = "discriminator_network." + std::to_string(li[i]);
      p.b = b.add(s + ".bias", 0, p.out, 0);
      p.w = b.add(s + ".parametrizations.weight.original", 0, p.out, p.in);
      p.u = b.add(s + ".parametrizations.weight.0._u", 1, p.out, 0);
      p.v = b.add(s + ".parametrizations.weight.0._v", 1, p.in, 0);
    }
    L.nlin = 4;
    L.n_param = b.po;
    L.n_state = b.so;
  }
  {  // classifier (cvae_gan_models.py:261-276)
    NetLayout& L = e.lay[CVG_NET_CLASSIFIER];
    Builder b(L);
    int dims[5] = {F, e.ch[0], e.ch[1], e.ch[2], e.K};
    const int li[4] = {0, 3, 7, 9};
    for (int i = 0; i < 4; ++i) {
      LinearP& p = L.lin[i];
      p.out = dims[i + 1];
      p.in = dims[i];
      std::string s = "classifier_network." + std::to_string(li[i]);
      p.w = b.add(s + ".weight", 0, p.out, p.in);
      p.b = b.add(s + ".bias", 0, p.out, 0);
      if (i == 1) {
        p.gamma = b.add("classifier_network.4.weight", 0, p.out, 0);
        p.beta = b.add("classifier_network.4.bias", 0, p.out, 0);
      }
    }
    L.nlin = 4;
    L.n_param = b.po;
    L.n_state = b.so;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// workspace
// ------------------------------------------------------------------------------------------------
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base((char*)b) {}
  template <typename T>
  T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? (T*)(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

static size_t carve(const Engine& e, Workspace& w, void* base) {
  Carver c(base);
  const int rows = e.cfg.max_batch;
  const size_t ld = (size_t)((rows + 63) / 64) * 64;
  w.ld = (int)ld;
  w.rows_cap = rows;
  const int F = e.F, K = e.K, Z = e.Z;
  w.xT = c.take<float>(F * ld);
  w.z = c.take<float>(2 * Z * ld);
  w.d_m1 = c.take<uint8_t>(2 * e.dh[0] * ld);
  w.d_m2 = c.take<uint8_t>(2 * e.dh[1] * ld);
  w.c_m1 = c.take<uint8_t>(2 * e.ch[0] * ld);
  w.c_m2 = c.take<uint8_t>(2 * e.ch[1] * ld);
  for (int i = 0; i < 3; ++i) {
    w.g_h[i] = c.take<float>(2 * e.gh[i] * ld);
    w.g_dy[i] = c.take<float>(2 * e.gh[i] * ld);
    w.e_h[i] = c.take<float>(e.eh[i] * ld);
    w.e_dy[i] = c.take<float>(e.eh[i] * ld);
    w.d_a[i] = c.take<float>(2 * e.dh[i] * ld);
    w.d_g[i] = c.take<float>(2 * e.dh[i] * ld);
    w.c_g[i] = c.take<float>(2 * e.ch[i] * ld);
  }
  w.g_out = c.take<float>(2 * F * ld);
  w.g_dout = c.take<float>(2 * F * ld);
  w.e_ml = c.take<float>(2 * Z * ld);
  w.e_dml = c.take<float>(2 * Z * ld);
  w.d_s = c.take<float>(2 * ld);
  w.c_a1 = c.take<float>(2 * e.ch[0] * ld);
  w.c_h2 = c.take<float>(2 * e.ch[1] * ld);
  w.c_a2 = c.take<float>(2 * e.ch[1] * ld);
  w.c_rs = c.take<float>(2 * 2 * ld);
  w.c_a3 = c.take<float>(2 * e.ch[2] * ld);
  w.c_logit = c.take<float>(2 * K * ld);
  w.c_dlogit = c.take<float>(2 * K * ld);
  w.dx = c.take<float>(F * ld);
  w.sn_sigma = c.take<float>(8);
  w.sn_inv_sigma = c.take<float>(8);
  long long snap = 0;
  for (int i = 0; i < 4; ++i) {
    const LinearP& p = e.lay[CVG_NET_DISCRIMINATOR].lin[i];
    snap += pad4(p.out > p.in ? p.out : p.in);
  }
  w.sn_snap = snap;
  w.sn_u = c.take<float>(2 * snap);
  w.sn_v = c.take<float>(2 * snap);
  w.sn_G = c.take<float>(2 * e.lay[CVG_NET_DISCRIMINATOR].n_param);
  // accumulators: one contiguous block so a single memset clears them
  const size_t n_acc = 16 + (size_t)(3 * 2 + 3 * 2 + 3 + 3) * 2 * STAT_C;
  w.acc = c.take<double>(n_acc);
  w.acc_bytes = n_acc * sizeof(double);
  if (w.acc) {
    w.loss = w.acc;
    w.g_fst = w.acc + 16;
    w.g_bst = w.g_fst + (size_t)3 * 2 * 2 * STAT_C;
    w.e_fst = w.g_bst + (size_t)3 * 2 * 2 * STAT_C;
    w.e_bst = w.e_fst + (size_t)3 * 2 * STAT_C;
  }
  w.gen_count = c.take<unsigned long long>(4);
  w.ctl = c.take<StepCtl>(1);
  w.x_stage = c.take<float>((size_t)rows * F);
  w.tc_w = c.take<float>((size_t)tc_prep_floats(e));
  w.tc_c = c.take<float>((size_t)tc_const_floats());
  // step-program kernel: 32 row slices of every weight gradient of the E+G step (the largest) fit
  {
    long long per = 0;
    for (int net = 0; net < 4; ++net) {
      long long t = 0;
      for (int i = 0; i < e.lay[net].nlin; ++i) {
        const LinearP& p = e.lay[net].lin[i];
        t += (long long)p.out * (((p.in + 15) & ~15) + 1);
      }
      per += t * (net == CVG_NET_GENERATOR || net == CVG_NET_DISCRIMINATOR ? 2 : 1);
    }
    w.dw_scratch_floats = 32 * per;
  }
  w.dw_scratch = c.take<float>((size_t)w.dw_scratch_floats);
  {
    int tiles = 1, cmax = 1;
    for (int net = 0; net < 4; ++net)
      for (int i = 0; i < e.lay[net].nlin; ++i) {
        const LinearP& p = e.lay[net].lin[i];
        tiles = std::max(tiles, ((p.in + 63) / 64) * ((p.out + 63) / 64));
        cmax = std::max(cmax, std::max(p.in, p.out));
      }
    w.det_acc_n = std::max((long long)tiles * DET_MAX_PASS * DW_PART, 2LL * cmax);
    w.det_cnt_n = tiles;
    for (int i = 0; i < SIDE_STREAMS + 1; ++i) {
      w.det_acc[i] = c.take<unsigned long long>((size_t)w.det_acc_n);
      w.det_cnt[i] = c.take<unsigned>((size_t)w.det_cnt_n);
    }
  }
  {
    // pre-split weight chunks (128 rows x 32 k, hi + lo = 8192 floats): both orientations of every Linear; the heads and
    // first layers are prepped with a narrower contraction, never a wider one
    long long chunks = 0;
    for (int net = 0; net < 4; ++net)
      for (int i = 0; i < e.lay[net].nlin; ++i) {
        const LinearP& p = e.lay[net].lin[i];
        chunks += (long long)((p.out + 127) / 128) * ((p.in + 31) / 32) + (long long)((p.in + 127) / 128) * ((p.out + 31) / 32);
      }
    w.mk_wprep_floats = chunks * 8192;
  }
  w.mk_wprep = c.take<float>((size_t)w.mk_wprep_floats);
  w.mk_bar = c.take<unsigned int>(64);
  w.z_eps = c.take<float>((size_t)Z * ld);
  w.mk_dbg = c.take<long long>(2048 + 64);
  w.hz = c.take<float>((size_t)HOIST_MAX * Z * ld);
  for (int i = 0; i < 3; ++i) w.hh[i] = c.take<float>((size_t)HOIST_MAX * e.gh[i] * ld);
  w.hout = c.take<float>((size_t)HOIST_MAX * F * ld);
  w.hfst = c.take<double>((size_t)3 * HOIST_MAX * 2 * STAT_C);
  return c.off + 256;
}

int64_t workspace_bytes(const Engine& e) {
  Workspace tmp;
  return (int64_t)carve(e, tmp, nullptr);
}

int carve_workspace(Engine& e, void* base, int64_t bytes) {
  if ((int64_t)workspace_bytes(e) > bytes) CVG_FAIL("workspace too small");
  if (((uintptr_t)base & 255) != 0) CVG_FAIL("workspace must be 256-byte aligned");
  carve(e, e.ws, base);
  e.ws_base = base;
  e.ws_bytes = bytes;
  return 0;
}

}  // namespace cvg
