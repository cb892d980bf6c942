// C-ABI layer of npbnn_b200 (include/npbnn_b200.h): context, workspace management, launch sequencing.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "bnn_kernels.h"

static thread_local std::string g_last_error;

static int fail(const std::string& msg) {
  g_last_error = msg;
  return 1;
}
#define CUDA_TRY(expr)                                                                         \
  do {                                                                                         \
    cudaError_t e__ = (expr);                                                                  \
    if (e__ != cudaSuccess)                                                                    \
      return fail(std::string(#expr) + ": " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" + \
                  std::to_string(__LINE__) + ")");                                             \
  } while (0)
#define REQUIRE(cond, msg) \
  do {                     \
    if (!(cond)) return fail(msg); \
  } while (0)

// device buffer that frees itself; one owner, so not copyable
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  // grow-only; newly allocated memory is zero-filled when `zero`
  cudaError_t ensure(size_t n, bool zero, cudaStream_t st, bool* grew = nullptr) {
    if (grew) *grew = false;
    if (n <= bytes) return cudaSuccess;
    if (p) {
      cudaError_t e = cudaFree(p);
      p = nullptr; bytes = 0;
      if (e != cudaSuccess) return e;
    }
    cudaError_t e = cudaMalloc(&p, n);
    if (e != cudaSuccess) return e;
    bytes = n;
    if (grew) *grew = true;
    if (zero) return cudaMemsetAsync(p, 0, n, st);
    return cudaSuccess;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr; bytes = 0;
  }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct bnn_ctx {
  int device = 0, n_sms = 0;
  bool have_net = false, have_data = false, have_chains = false;
  int force_generic = 0;
  long long launches = 0;
  NetGeom g{};                      // geometry in use: g_base, or padded up to a k_fwd3 width family by bnn_set_data
  NetGeom g_base{};                 // minimal padding (bnn_set_net)
  NetGeom wp_geom{};                // layout the zero padding of wp_scratch was prepared for
  // staged data
  DevBuf xs, labels, targets, lgk1, inst_w, class_w;     // lgk1: lgamma(k + 1) of the targets (count likelihoods)
  bool has_iw = false, has_cw = false;
  long long n_train = 0, n_test = 0, n_total = 0, n_pad = 0, n_tiles16 = 0;
  // workspaces
  DevBuf exp_tab, exp_tab_small, wp_scratch, part, counts_scratch, xs_pred, ov_cols, ov_vals;
  DevBuf h_w, h_alpha, h_sigma, h_loglik, h_sums, h_counts;    // device staging of the *_host entry points
  DevBuf flag;                      // one int: bnn_set_data's label check
  // chains
  int C = 0;
  bnn_sampler_config cfg{};
  PriorScales ps{};
  DevBuf w_cur, w_prop, wp_prop, mask, owner, sf, si, counts_prop, alpha_chain;
  DevBuf ps_entry, pls_entry, ps_tmp, pls_tmp;   // per-entry prior scales of the chains (hyper-priors) / of a scoring call
  DevBuf ind_cur, ind_prop, fi_cur, fi_prop, feat_mean, inj_ind_move, inj_ind_flip, inj_fi_move, inj_fi_flip;   // indicators
  bool have_feat_mean = false;
  bool have_ps_entry = false;
  // additional_prob of free-running chains (bnn_chains_set_additional_prob): [C], read by the proposal step when no
  // injection carries one.  Allocated by the first set after bnn_chains_init and kept at that address, so that captured
  // graphs see a new value through the copy into it.
  DevBuf add_prob;
  bool have_add_prob = false;
  // row sharding: the chains' accept step reads the all-reduced sums from part_red (one pseudo tile)
  bool rowshard = false;
  long long n_train_global = 0;
  DevBuf part_red;
  DevBuf part_sl;                   // [C, NF, n_slices]: slice sums of the tile partials (k_reduce_part), read by k_mh_update
  DevBuf inj_alpha_ix, inj_alpha_dz, inj_add_prob;
  // the six arrays every injection carries travel in ONE host-to-device transfer: packed into a pinned staging buffer
  // (so the caller's arrays are free on return whatever memory they live in), copied into one device arena
  DevBuf inj_arena;
  void* inj_host = nullptr;
  size_t inj_host_bytes = 0;
  cudaEvent_t inj_copied = nullptr;   // the last transfer out of inj_host
  const char* last_kernel = "";
  // block-masked networks: dataflow program of the chains' mask (bnn_sparse.cu); sp.prog null: the dense kernels run
  struct { DevBuf prog, widx; SparseParams sp{}; } sparse;
  int opt_sparse = 1;               // option "sparse": 0 forces the dense kernels for masked chains
  // optional per-launch timing of the forward kernel (bench.py roofline): event pairs on the launch stream
  int time_forward = 0;
  std::vector<cudaEvent_t> ev;      // start/stop pairs, recorded but not yet read
  size_t ev_used = 0;
  double fwd_ms_sum = 0.0;
  long long fwd_count = 0;
  // asynchronous state snapshots (logger ring): device staging + pinned host copy per slot, own copy stream
  struct Snap {
    DevBuf dev;
    void* host = nullptr;
    size_t bytes = 0;
    cudaEvent_t staged = nullptr, done = nullptr;
    bool pending = false;
    ~Snap() {
      if (host) cudaFreeHost(host);
      if (staged) cudaEventDestroy(staged);
      if (done) cudaEventDestroy(done);
    }
  };
  static constexpr int kSnapSlots = 64;
  Snap snaps[kSnapSlots];
  cudaStream_t copy_stream = nullptr;
  // CUDA graphs of the free-running MH loop (bnn_mh_steps without injection): launch-bound at small N
  struct StepGraph { int n_steps; cudaGraphExec_t exec; long long launches; };
  std::vector<StepGraph> graphs;
  cudaStream_t capture_stream = nullptr;
  int opt_graphs = 1;               // option "graphs"
  int opt_chain_loop = 1;           // option "chain_loop": 1 = small data sets step inside one persistent launch (k_chain_loop)
                                    // where that beats the launch sequence, 2 = wherever it fits (tests), 0 = never
  int opt_chain_cluster = 16;       // option "chain_loop_cluster": largest thread-block cluster per chain
  int opt_pred_tf32 = 0;            // option "predict_tf32": opt-in 3xTF32 prediction summaries (bnn_pred_lp.cu), never the MH path
  bool mh_warm = false;             // one eager bnn_mh_steps has run since the last (re)configuration

  // the owner of the device resources above (the DevBufs and Snaps free themselves); the caller has made this context's
  // device current and synchronised it
  ~bnn_ctx() {
    for (auto& gph : graphs) cudaGraphExecDestroy(gph.exec);
    if (capture_stream) cudaStreamDestroy(capture_stream);
    if (copy_stream) cudaStreamDestroy(copy_stream);
    if (inj_host) cudaFreeHost(inj_host);
    if (inj_copied) cudaEventDestroy(inj_copied);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
};

// every call that changes what a captured launch sequence would contain (pointers, kernel choice, chain count)
static void invalidate_graphs(bnn_ctx* c) {
  for (auto& gph : c->graphs) cudaGraphExecDestroy(gph.exec);
  c->graphs.clear();
  c->mh_warm = false;
}

static cudaError_t timed_forward(bnn_ctx* c, const FwdParams& p, bool predict, cudaStream_t st) {
  if (!c->time_forward) return bnn_launch_forward(p, predict, c->n_sms, c->force_generic, st, &c->last_kernel);
  if (c->ev_used + 2 > c->ev.size()) {
    for (int i = 0; i < 2; ++i) {
      cudaEvent_t e;
      cudaError_t r = cudaEventCreate(&e);
      if (r != cudaSuccess) return r;
      c->ev.push_back(e);
    }
  }
  cudaError_t r = cudaEventRecord(c->ev[c->ev_used], st);
  if (r != cudaSuccess) return r;
  r = bnn_launch_forward(p, predict, c->n_sms, c->force_generic, st, &c->last_kernel);
  if (r != cudaSuccess) return r;
  r = cudaEventRecord(c->ev[c->ev_used + 1], st);
  c->ev_used += 2;
  return r;
}

static int sets_per_pass(const NetGeom& g) {
  int nc = bnn_n_counts(g.K);
  int byc = 16384 / (nc * 4);
  int v = byc < BNN_MAX_SETS_PER_PASS ? byc : BNN_MAX_SETS_PER_PASS;
  return v < 1 ? 1 : v;
}
// the forward parameters every launch over the packed rows x (n_total rows, the first n_train of them training rows) shares
static FwdParams fwd_params(const bnn_ctx* c, const NetGeom& g, const double* x, long long n_train, long long n_total) {
  FwdParams p{};
  p.g = g;
  p.x = x;
  p.n_train = n_train;
  p.n_total = n_total;
  p.n_tiles16 = (n_total + 15) / 16;
  p.exp_tab = c->exp_tab.as<double>();
  p.exp_tab_small = c->exp_tab_small.as<double>();
  p.NF = bnn_n_slots(g);
  p.inv_sets = 1.0;
  return p;
}

// ... over the staged data set
static FwdParams base_params(const bnn_ctx* c) {
  FwdParams p = fwd_params(c, c->g, c->xs.as<double>(), c->n_train, c->n_total);
  p.labels = c->labels.as<int>();
  p.targets = c->targets.as<double>();
  p.lgk1 = c->lgk1.as<double>();
  p.inst_w = c->has_iw ? c->inst_w.as<double>() : nullptr;
  p.class_w = c->has_cw ? c->class_w.as<double>() : nullptr;
  return p;
}

template <typename T>
static int upload(DevBuf& b, const T* src, size_t n, cudaStream_t st) {
  CUDA_TRY(b.ensure(sizeof(T) * n, false, st));
  CUDA_TRY(cudaMemcpyAsync(b.p, src, sizeof(T) * n, cudaMemcpyHostToDevice, st));
  return 0;
}

// (Re)compute the packed layout of a network for the given padded widths: F_pad for the features, out_pad[l] per layer
// (each layer's padded input width is the previous layer's padded output width).
static void geom_layout(NetGeom& g, int f_pad, const int* out_pad) {
  int off = 0, in_pad = f_pad;
  g.max_w = 8;
  for (int l = 0; l < g.L; ++l) {
    LayerGeom& lg = g.l[l];
    lg.in_pad = in_pad;
    lg.out_pad = out_pad[l];
    lg.stride = lg.in_pad;
    lg.swz = bnn_swz_for(lg.stride);
    lg.w_off = off;
    off += lg.out_pad * lg.stride;
    lg.b_off = off;
    off += lg.out_pad;
    if (l >= 1 && lg.in_pad > g.max_w) g.max_w = lg.in_pad;
    in_pad = lg.out_pad;
  }
  g.F_pad = g.l[0].in_pad;
  g.x_swz = g.l[0].swz;
  g.PB = off;
}

// Three-layer networks that fit one of the two k_fwd3 width families (64 -> 64 -> 32 or 32 -> 32 -> 16, last layer 16
// columns for classes / 8 for Gaussian outputs) are padded UP to that family when the data set is large enough for the
// specialised kernel to pay (at least one full round of 148 x 12 warp tiles); padded weights are zero, so the padded
// hidden units are act(0) = 0 for every supported activation and contribute nothing.  Small data sets keep the
// minimal padding (rounded up to 8) and the generic kernel.
static const long long kFwd3PromoteRows = 16LL * 148 * 12;
static NetGeom geom_for_rows(const NetGeom& base, long long n_rows) {
  if (base.L != 3 || n_rows < kFwd3PromoteRows || bnn_fwd3_family(base)) return base;
  const int n3 = (base.lik == BNN_LIK_CATEGORICAL) ? 16 : 8;
  if (base.l[2].out > n3) return base;
  NetGeom g = base;
  if (base.F <= 32 && base.l[0].out <= 32 && base.l[1].out <= 16) {
    const int pads[3] = {32, 16, n3};
    geom_layout(g, 32, pads);
    return g;
  }
  if (base.F <= 64 && base.l[0].out <= 64 && base.l[1].out <= 32) {
    const int pads[3] = {64, 32, n3};
    geom_layout(g, 64, pads);
    return g;
  }
  return base;
}
static bool same_layout(const NetGeom& a, const NetGeom& b) {
  if (a.L != b.L || a.F_pad != b.F_pad || a.PB != b.PB) return false;
  for (int l = 0; l < a.L; ++l)
    if (a.l[l].out_pad != b.l[l].out_pad) return false;
  return true;
}

// wp_scratch holds packed weight sets; its padding entries are zeroed when it is (re)allocated and never written, so a
// change of layout (prediction on a different number of rows may pick another padding) needs a fresh buffer
static int ensure_wp_scratch(bnn_ctx* c, const NetGeom& g, size_t n_sets, cudaStream_t st) {
  if (!same_layout(c->wp_geom, g)) {
    c->wp_scratch.release();
    c->wp_geom = g;
  }
  CUDA_TRY(c->wp_scratch.ensure(sizeof(double) * n_sets * g.PB, true, st));
  return 0;
}

extern "C" {

const char* bnn_last_error(void) { return g_last_error.c_str(); }
int bnn_abi_version(void) { return BNN_ABI_VERSION; }

int bnn_ctx_create(bnn_ctx** out, int device) {
  REQUIRE(out != nullptr, "bnn_ctx_create: null output pointer");
  int n = 0;
  CUDA_TRY(cudaGetDeviceCount(&n));
  REQUIRE(device >= 0 && device < n, "bnn_ctx_create: no such CUDA device");
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  REQUIRE(prop.major == 10, "npbnn_b200 kernels are built for sm_100a (Blackwell B200) only; found sm_" +
                                std::to_string(prop.major) + std::to_string(prop.minor));
  bnn_ctx* c = new bnn_ctx();
  c->device = device;
  c->n_sms = prop.multiProcessorCount;
  const char* pt = getenv("NPBNN_PREDICT_TF32");           // opt-in reduced-precision prediction summaries (bnn_pred_lp.cu)
  if (pt) c->opt_pred_tf32 = atoi(pt);
  std::vector<double> tab(BNN_EXP_TAB_SIZE);
  for (int j = 0; j < BNN_EXP_TAB_SIZE; ++j) tab[j] = exp2((double)j / BNN_EXP_TAB_SIZE);
  cudaError_t e = c->exp_tab.ensure(sizeof(double) * BNN_EXP_TAB_SIZE, false, 0);
  if (e == cudaSuccess) e = cudaMemcpy(c->exp_tab.p, tab.data(), sizeof(double) * BNN_EXP_TAB_SIZE, cudaMemcpyHostToDevice);
  for (int j = 0; j < 256; ++j) tab[j] = exp2((double)j / 256.0);
  if (e == cudaSuccess) e = c->exp_tab_small.ensure(sizeof(double) * 256, false, 0);
  if (e == cudaSuccess) e = cudaMemcpy(c->exp_tab_small.p, tab.data(), sizeof(double) * 256, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    delete c;
    return fail(std::string("bnn_ctx_create: ") + cudaGetErrorString(e));
  }
  *out = c;
  return 0;
}

int bnn_ctx_destroy(bnn_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  delete c;
  return 0;
}

int bnn_set_option(bnn_ctx* c, const char* name, int value) {
  REQUIRE(c && name, "bnn_set_option: null argument");
  invalidate_graphs(c);
  if (strcmp(name, "force_generic") == 0) { c->force_generic = value; return 0; }
  if (strcmp(name, "time_forward") == 0) { c->time_forward = value; return 0; }
  if (strcmp(name, "sparse") == 0) { c->opt_sparse = value; return 0; }
  if (strcmp(name, "graphs") == 0) { c->opt_graphs = value; return 0; }
  if (strcmp(name, "chain_loop") == 0) { c->opt_chain_loop = value; return 0; }
  if (strcmp(name, "predict_tf32") == 0) { c->opt_pred_tf32 = value; return 0; }
  if (strcmp(name, "chain_loop_cluster") == 0) {
    REQUIRE(value == 1 || value == 2 || value == 4 || value == 8 || value == 16, "bnn_set_option: chain_loop_cluster must be 1, 2, 4, 8 or 16");
    c->opt_chain_cluster = value;
    return 0;
  }
  return fail(std::string("bnn_set_option: unknown option ") + name);
}

// debugging aid: per-warp-tile partial sums of the last forward pass, [n_sets_in_pass][NF][n_tiles16]
int bnn_debug_read_part(bnn_ctx* c, double* out_host, int64_t n_doubles) {
  REQUIRE(c && out_host, "bnn_debug_read_part: null argument");
  CUDA_TRY(cudaSetDevice(c->device));
  CUDA_TRY(cudaDeviceSynchronize());
  REQUIRE((size_t)n_doubles * sizeof(double) <= c->part.bytes, "bnn_debug_read_part: more than the workspace holds");
  CUDA_TRY(cudaMemcpy(out_host, c->part.p, sizeof(double) * (size_t)n_doubles, cudaMemcpyDeviceToHost));
  return 0;
}

const char* bnn_last_kernel(const bnn_ctx* c) { return c ? c->last_kernel : ""; }

int bnn_set_net(bnn_ctx* c, const bnn_net_spec* s) {
  REQUIRE(c && s, "bnn_set_net: null argument");
  REQUIRE(s->n_layers >= 1 && s->n_layers <= BNN_MAX_LAYERS, "bnn_set_net: n_layers must be in [1, 8]");
  REQUIRE(s->n_features >= 1, "bnn_set_net: n_features must be positive");
  REQUIRE(s->act >= BNN_ACT_RELU && s->act <= BNN_ACT_TANH, "bnn_set_net: unknown activation");
  REQUIRE(s->lik >= BNN_LIK_CATEGORICAL && s->lik <= BNN_LIK_NEGBIN10, "bnn_set_net: unknown likelihood");
  NetGeom g{};
  g.L = s->n_layers;
  g.F = s->n_features;
  g.act = s->act;
  g.lik = s->lik;
  int in = s->n_features, coff = 0;
  int out_pad[BNN_MAX_LAYERS];
  for (int l = 0; l < g.L; ++l) {
    LayerGeom& lg = g.l[l];
    REQUIRE(s->out_dim[l] >= 1, "bnn_set_net: layer width must be positive");
    lg.in = in;
    lg.out = s->out_dim[l];
    lg.bias = s->has_bias[l] ? 1 : 0;
    lg.c_off = coff;
    coff += lg.out * (lg.in + lg.bias);
    out_pad[l] = bnn_round_up(lg.out, 8);
    in = lg.out;
  }
  geom_layout(g, bnn_round_up(g.F, 8), out_pad);
  g.P = coff;
  g.O = g.l[g.L - 1].out;
  REQUIRE(g.O <= BNN_MAX_OUT, "bnn_set_net: output layer wider than BNN_MAX_OUT (32)");
  if (g.lik == BNN_LIK_GAUSSIAN_HEAD) {
    REQUIRE(g.O % 2 == 0, "bnn_set_net: the sigma-head likelihood needs an even output width");
    g.K = g.O / 2;
  } else if (g.lik == BNN_LIK_POISSON) {
    g.K = 1;                                     // poi_likelihood reads output column 0 only (BNN_lik.py:5-14)
  } else if (g.lik == BNN_LIK_NEGBIN || g.lik == BNN_LIK_NEGBIN10) {
    REQUIRE(g.O % 2 == 0, "bnn_set_net: the negative-binomial likelihood needs an even output width (mean | dispersion)");
    g.K = g.O / 2;
  } else {
    g.K = g.O;
  }
  c->g = g;
  c->g_base = g;
  c->wp_scratch.release();   // packed layout changed: padding entries must be re-zeroed
  c->wp_geom = g;
  c->have_net = true;
  c->have_data = false;
  c->have_chains = false;
  return 0;
}

int64_t bnn_n_params(const bnn_ctx* c) { return (c && c->have_net) ? c->g.P : -1; }
int64_t bnn_launch_count(const bnn_ctx* c) { return c ? c->launches : -1; }

int bnn_set_data(bnn_ctx* c, const double* x_dev, int64_t n_train, int64_t n_test, const int32_t* labels_dev,
                 const double* targets_dev, const double* inst_w_dev, const double* class_w_dev, void* stream) {
  REQUIRE(c && c->have_net, "bnn_set_data: call bnn_set_net first");
  invalidate_graphs(c);
  REQUIRE(x_dev != nullptr && n_train >= 1 && n_test >= 0, "bnn_set_data: bad arguments");
  c->have_data = false;        // a failed call leaves no half-staged data set behind
  c->have_chains = false;
  c->g = geom_for_rows(c->g_base, n_train + n_test);
  const NetGeom& g = c->g;
  if (g.lik == BNN_LIK_CATEGORICAL) REQUIRE(labels_dev != nullptr, "bnn_set_data: labels_dev required for the categorical likelihood");
  else REQUIRE(targets_dev != nullptr, "bnn_set_data: targets_dev required for the Gaussian likelihoods");
  if (g.lik != BNN_LIK_CATEGORICAL) REQUIRE(inst_w_dev == nullptr, "instance_weight not implemented for regression (BNN_lib.py:129-130)");
  if (bnn_lik_is_count(g.lik)) REQUIRE(class_w_dev == nullptr, "class_weight is not used by the count likelihoods (BNN_lik.py)");
  REQUIRE(!(inst_w_dev && class_w_dev), "class_weight together with instance_weight is an AxisError in the reference (BNN_lib.py:105)");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  c->n_train = n_train; c->n_test = n_test; c->n_total = n_train + n_test;
  c->n_pad = (c->n_total + 15) / 16 * 16;
  c->n_tiles16 = c->n_pad / 16;
  CUDA_TRY(c->xs.ensure(sizeof(double) * c->n_pad * g.F_pad, false, st));
  CUDA_TRY(bnn_launch_pack_x(x_dev, c->xs.as<double>(), c->n_total, c->n_pad, g.F, g.F_pad, g.x_swz, nullptr, nullptr, 0, st));
  c->launches++;
  if (g.lik == BNN_LIK_CATEGORICAL) {
    CUDA_TRY(c->labels.ensure(sizeof(int) * c->n_total, false, st));
    CUDA_TRY(cudaMemcpyAsync(c->labels.p, labels_dev, sizeof(int) * c->n_total, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(c->flag.ensure(sizeof(int), false, st));
    CUDA_TRY(cudaMemsetAsync(c->flag.p, 0, sizeof(int), st));
    CUDA_TRY(bnn_launch_check_labels(c->labels.as<int>(), n_train, c->n_total, g.K, c->flag.as<int>(), st));
    c->launches++;
    int bad_label = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad_label, c->flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    REQUIRE(bad_label == 0, "bnn_set_data: class labels must lie in [0, K) with K = the output width of the network "
                            "(the reference raises IndexError at BNN_lib.py:104)");
  } else {
    CUDA_TRY(c->targets.ensure(sizeof(double) * c->n_total * g.K, false, st));
    CUDA_TRY(cudaMemcpyAsync(c->targets.p, targets_dev, sizeof(double) * c->n_total * g.K, cudaMemcpyDeviceToDevice, st));
    if (bnn_lik_is_count(g.lik)) {
      CUDA_TRY(c->lgk1.ensure(sizeof(double) * c->n_total * g.K, false, st));
      CUDA_TRY(bnn_launch_lgamma1(c->targets.as<double>(), c->lgk1.as<double>(), c->n_total * g.K, st));
      c->launches++;
    }
  }
  c->has_iw = inst_w_dev != nullptr;
  if (c->has_iw) {
    CUDA_TRY(c->inst_w.ensure(sizeof(double) * n_train, false, st));
    CUDA_TRY(cudaMemcpyAsync(c->inst_w.p, inst_w_dev, sizeof(double) * n_train, cudaMemcpyDeviceToDevice, st));
  }
  c->has_cw = class_w_dev != nullptr;
  if (c->has_cw) {
    CUDA_TRY(c->class_w.ensure(sizeof(double) * g.K, false, st));
    CUDA_TRY(cudaMemcpyAsync(c->class_w.p, class_w_dev, sizeof(double) * g.K, cudaMemcpyDeviceToDevice, st));
  }
  c->have_data = true;
  c->have_chains = false;
  return 0;
}

int bnn_forward_lik(bnn_ctx* c, const double* w_dev, int32_t n_sets, const double* alpha_dev, const double* sigma_dev,
                    int32_t sigma_mode, double lik_temp, double* loglik_dev, double* sums_dev, int32_t* counts_dev,
                    void* stream) {
  REQUIRE(c && c->have_data, "bnn_forward_lik: call bnn_set_net and bnn_set_data first");
  REQUIRE(w_dev && loglik_dev && n_sets >= 1, "bnn_forward_lik: bad arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const NetGeom& g = c->g;
  const int NC = bnn_n_counts(g.K);
  if (int rc = ensure_wp_scratch(c, g, (size_t)n_sets, st)) return rc;
  CUDA_TRY(bnn_launch_pack_w(g, w_dev, c->wp_scratch.as<double>(), n_sets, st));
  c->launches++;
  int* counts = counts_dev;
  if (g.lik == BNN_LIK_CATEGORICAL) {
    if (!counts) {
      CUDA_TRY(c->counts_scratch.ensure(sizeof(int) * (size_t)n_sets * NC, false, st));
      counts = c->counts_scratch.as<int>();
    }
    CUDA_TRY(cudaMemsetAsync(counts, 0, sizeof(int) * (size_t)n_sets * NC, st));
  }
  const int per = sets_per_pass(g);
  FwdParams p = base_params(c);
  CUDA_TRY(c->part.ensure(sizeof(double) * (size_t)p.NF * per * c->n_tiles16, false, st));
  p.part = c->part.as<double>();
  for (int s0 = 0; s0 < n_sets; s0 += per) {
    const int n = (n_sets - s0 < per) ? n_sets - s0 : per;
    p.wp = c->wp_scratch.as<double>() + (size_t)s0 * g.PB;
    p.alpha = alpha_dev ? alpha_dev + (size_t)s0 * g.L : nullptr;
    p.C = n;
    p.counts = counts ? counts + (size_t)s0 * NC : nullptr;
    CUDA_TRY(timed_forward(c, p, false, st));
    CUDA_TRY(bnn_launch_finalize_lik(g, p.part, p.NF, c->n_tiles16, c->n_train, lik_temp, sigma_mode, sigma_dev,
                                     loglik_dev, sums_dev, s0, n, st));
    c->launches += 2;
  }
  return 0;
}

int bnn_forward_lik_host(bnn_ctx* c, const double* w_host, int32_t n_sets, const double* alpha_host,
                         const double* sigma_host, int32_t sigma_mode, double lik_temp, double* loglik_host,
                         double* sums_host, int32_t* counts_host, void* stream) {
  REQUIRE(c && c->have_data, "bnn_forward_lik_host: call bnn_set_net and bnn_set_data first");
  REQUIRE(w_host && loglik_host && n_sets >= 1, "bnn_forward_lik_host: bad arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const NetGeom& g = c->g;
  const int NC = bnn_n_counts(g.K);
  CUDA_TRY(c->h_w.ensure(sizeof(double) * (size_t)n_sets * g.P, false, st));
  CUDA_TRY(cudaMemcpyAsync(c->h_w.p, w_host, sizeof(double) * (size_t)n_sets * g.P, cudaMemcpyHostToDevice, st));
  if (alpha_host) {
    CUDA_TRY(c->h_alpha.ensure(sizeof(double) * (size_t)n_sets * g.L, false, st));
    CUDA_TRY(cudaMemcpyAsync(c->h_alpha.p, alpha_host, sizeof(double) * (size_t)n_sets * g.L, cudaMemcpyHostToDevice, st));
  }
  if (sigma_host) {
    CUDA_TRY(c->h_sigma.ensure(sizeof(double) * (size_t)n_sets * g.K, false, st));
    CUDA_TRY(cudaMemcpyAsync(c->h_sigma.p, sigma_host, sizeof(double) * (size_t)n_sets * g.K, cudaMemcpyHostToDevice, st));
  }
  CUDA_TRY(c->h_loglik.ensure(sizeof(double) * n_sets, false, st));
  CUDA_TRY(c->h_sums.ensure(sizeof(double) * (size_t)n_sets * 3 * g.K, false, st));
  CUDA_TRY(c->h_counts.ensure(sizeof(int) * (size_t)n_sets * NC, false, st));
  int rc = bnn_forward_lik(c, c->h_w.as<double>(), n_sets, alpha_host ? c->h_alpha.as<double>() : nullptr,
                           sigma_host ? c->h_sigma.as<double>() : nullptr, sigma_mode, lik_temp,
                           c->h_loglik.as<double>(), c->h_sums.as<double>(), c->h_counts.as<int>(), stream);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(loglik_host, c->h_loglik.p, sizeof(double) * n_sets, cudaMemcpyDeviceToHost, st));
  if (sums_host && g.lik != BNN_LIK_CATEGORICAL)
    CUDA_TRY(cudaMemcpyAsync(sums_host, c->h_sums.p, sizeof(double) * (size_t)n_sets * 3 * g.K, cudaMemcpyDeviceToHost, st));
  if (counts_host && g.lik == BNN_LIK_CATEGORICAL)
    CUDA_TRY(cudaMemcpyAsync(counts_host, c->h_counts.p, sizeof(int) * (size_t)n_sets * NC, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

static void fill_prior_scales(PriorScales& ps, const double* s, int L) {
  for (int l = 0; l < BNN_MAX_LAYERS; ++l) {
    ps.s[l] = (l < L) ? s[l] : 1.0;
    ps.ls[l] = log(ps.s[l]);
  }
}

int bnn_log_prior(bnn_ctx* c, const double* w_dev, int32_t n_sets, int32_t prior, const double* prior_scale,
                  double* logprior_dev, void* stream) {
  REQUIRE(c && c->have_net, "bnn_log_prior: call bnn_set_net first");
  REQUIRE(w_dev && logprior_dev && prior_scale && n_sets >= 1, "bnn_log_prior: bad arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  PriorScales ps;
  fill_prior_scales(ps, prior_scale, c->g.L);
  CUDA_TRY(bnn_launch_log_prior(c->g, w_dev, n_sets, prior, ps, nullptr, nullptr, 0, logprior_dev, (cudaStream_t)stream));
  c->launches++;
  return 0;
}

// scales > 0 and finite, logs taken on the host (libm log, as scipy's logpdf does)
static int upload_entry_scales(DevBuf& sc, DevBuf& lg, const double* scale_host, size_t n, cudaStream_t st, const char* who) {
  std::vector<double> ls(n);
  for (size_t i = 0; i < n; ++i) {
    if (!(scale_host[i] > 0.0) || !std::isfinite(scale_host[i])) {
      g_last_error = std::string(who) + ": prior scales must be positive and finite";
      return 1;
    }
    ls[i] = std::log(scale_host[i]);
  }
  if (upload(sc, scale_host, n, st) || upload(lg, ls.data(), n, st)) return 1;
  CUDA_TRY(cudaStreamSynchronize(st));     // `ls` leaves scope
  return 0;
}

int bnn_log_prior_entries(bnn_ctx* c, const double* w_dev, int32_t n_sets, int32_t prior, const double* entry_scale_host,
                          double* logprior_dev, void* stream) {
  REQUIRE(c && c->have_net, "bnn_log_prior_entries: call bnn_set_net first");
  REQUIRE(w_dev && logprior_dev && entry_scale_host && n_sets >= 1, "bnn_log_prior_entries: bad arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = upload_entry_scales(c->ps_tmp, c->pls_tmp, entry_scale_host, (size_t)c->g.P, st, "bnn_log_prior_entries")) return rc;
  PriorScales ps{};
  CUDA_TRY(bnn_launch_log_prior(c->g, w_dev, n_sets, prior, ps, c->ps_tmp.as<double>(), c->pls_tmp.as<double>(), 0,
                                logprior_dev, st));
  c->launches++;
  return 0;
}

static ChainDev chain_dev(bnn_ctx* c) {
  ChainDev d{};
  d.g = c->g;
  d.cfg = c->cfg;
  d.ps = c->ps;
  d.C = c->C;
  d.n_train = c->n_train;
  d.n_tiles16 = c->n_tiles16;
  d.w_cur = c->w_cur.as<double>();
  d.w_prop = c->w_prop.as<double>();
  d.wp_prop = c->wp_prop.as<double>();
  d.mask = c->cfg.use_mask ? c->mask.as<double>() : nullptr;
  d.ps_entry = c->have_ps_entry ? c->ps_entry.as<double>() : nullptr;
  d.pls_entry = c->have_ps_entry ? c->pls_entry.as<double>() : nullptr;
  if (c->cfg.use_indicators) { d.ind_cur = c->ind_cur.as<double>(); d.ind_prop = c->ind_prop.as<double>(); }
  if (c->cfg.use_feature_indicators) {
    d.fi_cur = c->fi_cur.as<double>(); d.fi_prop = c->fi_prop.as<double>(); d.feat_mean = c->feat_mean.as<double>();
  }
  d.owner = c->owner.as<int>();
  d.sf = c->sf.as<double>();
  d.si = c->si.as<int>();
  d.part = c->part.as<double>();
  d.NF = bnn_n_slots(c->g);
  d.counts_prop = c->counts_prop.as<int>();
  d.alpha_fwd = c->alpha_chain.as<double>();
  d.add_prob = c->have_add_prob ? c->add_prob.as<double>() : nullptr;
  if (const int ns = bnn_part_slices(c->n_tiles16)) {     // chains_forward folds the tile partials into ns slices per chain
    d.part = c->part_sl.as<double>();
    d.n_tiles16 = ns;
  }
  if (c->rowshard) {                 // accept step on the sums over all ranks (k_rowshard_commit)
    d.part = c->part_red.as<double>();
    d.n_tiles16 = 1;
    d.n_train = c->n_train_global;
  }
  return d;
}

// forward pass of every chain's packed proposal -> partials + proposal counters
static int chains_forward(bnn_ctx* c, cudaStream_t st) {
  const NetGeom& g = c->g;
  const int NC = bnn_n_counts(g.K);
  const int per = sets_per_pass(g);
  FwdParams p = base_params(c);
  if (c->opt_sparse) p.sp = c->sparse.sp;
  for (int s0 = 0; s0 < c->C; s0 += per) {
    const int n = (c->C - s0 < per) ? c->C - s0 : per;
    p.wp = c->wp_prop.as<double>() + (size_t)s0 * g.PB;
    p.alpha = c->alpha_chain.as<double>() + (size_t)s0 * g.L;
    p.C = n;
    p.part = c->part.as<double>() + (size_t)s0 * p.NF * c->n_tiles16;
    p.counts = c->counts_prop.as<int>() + (size_t)s0 * NC;
    CUDA_TRY(timed_forward(c, p, false, st));
    c->launches++;
  }
  if (const int ns = bnn_part_slices(c->n_tiles16)) {
    if (!c->rowshard) {              // (row-sharded chains fold the full partials in k_rowshard_local)
      CUDA_TRY(bnn_launch_reduce_part(c->part.as<double>(), c->n_tiles16, ns, c->C * p.NF, c->part_sl.as<double>(), st));
      c->launches++;
    }
  }
  return 0;
}

int bnn_chains_init(bnn_ctx* c, int32_t n_chains, const bnn_sampler_config* cfg, const double* w0_host,
                    const double* mask_host, const double* temperature, const double* update_f,
                    const double* update_ws, const double* alpha, const double* sigma0, void* stream) {
  REQUIRE(c && c->have_data, "bnn_chains_init: call bnn_set_net and bnn_set_data first");
  invalidate_graphs(c);
  REQUIRE(cfg && w0_host && temperature && update_f && update_ws && n_chains >= 1, "bnn_chains_init: bad arguments");
  REQUIRE(cfg->adapt_freq >= 1, "bnn_chains_init: adapt_freq must be >= 1");
  REQUIRE(cfg->n_act_prm >= 0 && cfg->n_act_prm <= c->g.L, "bnn_chains_init: n_act_prm must be in [0, n_layers]");
  REQUIRE(!cfg->use_mask || mask_host, "bnn_chains_init: use_mask set but mask_host is null");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const NetGeom& g = c->g;
  const int C = n_chains, NC = bnn_n_counts(g.K);
  c->C = C;
  c->have_ps_entry = false;          // per-entry prior scales belong to the previous set of chains
  c->have_add_prob = false;          // and so does their additional_prob
  for (auto& sn : c->snaps) sn.pending = false;
  c->cfg = *cfg;
  fill_prior_scales(c->ps, cfg->prior_scale, g.L);
  CUDA_TRY(c->w_cur.ensure(sizeof(double) * (size_t)C * g.P, false, st));
  CUDA_TRY(c->w_prop.ensure(sizeof(double) * (size_t)C * g.P, false, st));
  CUDA_TRY(c->wp_prop.ensure(sizeof(double) * (size_t)C * g.PB, false, st));
  CUDA_TRY(cudaMemsetAsync(c->wp_prop.p, 0, sizeof(double) * (size_t)C * g.PB, st));
  CUDA_TRY(c->owner.ensure(sizeof(int) * (size_t)C * g.P, false, st));
  CUDA_TRY(cudaMemsetAsync(c->owner.p, 0xff, sizeof(int) * (size_t)C * g.P, st));
  CUDA_TRY(c->sf.ensure(sizeof(double) * (size_t)C * BNN_F_STRIDE, false, st));
  CUDA_TRY(c->si.ensure(sizeof(int) * (size_t)C * BNN_I_STRIDE, false, st));
  CUDA_TRY(c->counts_prop.ensure(sizeof(int) * (size_t)C * NC, false, st));
  CUDA_TRY(c->alpha_chain.ensure(sizeof(double) * (size_t)C * g.L, false, st));
  CUDA_TRY(c->part.ensure(sizeof(double) * (size_t)bnn_n_slots(g) * C * c->n_tiles16, false, st));
  if (c->rowshard) CUDA_TRY(c->part_red.ensure(sizeof(double) * (size_t)C * bnn_n_slots(g), true, st));
  CUDA_TRY(c->part_sl.ensure(sizeof(double) * (size_t)C * bnn_n_slots(g) * 64, false, st));
  c->sparse.sp = SparseParams{};
  if (cfg->use_mask) {
    CUDA_TRY(c->mask.ensure(sizeof(double) * g.P, false, st));
    CUDA_TRY(cudaMemcpyAsync(c->mask.p, mask_host, sizeof(double) * g.P, cudaMemcpyHostToDevice, st));
    // block-sparse forward: only when the cover is thin and the initial weights respect the mask (the
    // reference applies the mask at construction, BNN_env.py:259-267; proposals are masked in k_mh_update)
    SparseProgram sp;
    bool ok = bnn_sparse_build(g, mask_host, &sp);
    for (size_t i = 0; ok && i < (size_t)C * g.P; ++i)
      if (mask_host[i % g.P] == 0.0 && w0_host[i] != 0.0) ok = false;
    if (ok) {
      if (upload(c->sparse.prog, sp.prog.data(), sp.prog.size(), st)) return 1;
      if (upload(c->sparse.widx, sp.widx.data(), sp.widx.size(), st)) return 1;
      c->sparse.sp = sp.sp;
      c->sparse.sp.prog = c->sparse.prog.as<int>();
      c->sparse.sp.widx = c->sparse.widx.as<int>();
    }
  }
  CUDA_TRY(cudaMemcpyAsync(c->w_cur.p, w0_host, sizeof(double) * (size_t)C * g.P, cudaMemcpyHostToDevice, st));

  std::vector<double> sf((size_t)C * BNN_F_STRIDE, 0.0), al((size_t)C * g.L, 0.0);
  std::vector<int> si((size_t)C * BNN_I_STRIDE, 0);
  for (int ch = 0; ch < C; ++ch) {
    double* f = sf.data() + (size_t)ch * BNN_F_STRIDE;
    int* i = si.data() + (size_t)ch * BNN_I_STRIDE;
    f[BNN_F_TEMPERATURE] = temperature[ch];
    for (int l = 0; l < g.L; ++l) {
      const int size = g.l[l].out * (g.l[l].in + g.l[l].bias);
      f[BNN_F_UPDATE_F + l] = update_f[ch * g.L + l];
      f[BNN_F_UPDATE_WS + l] = update_ws[ch * g.L + l];
      f[BNN_F_FREQ_LAYER + l] = 1.0;
      f[BNN_F_ALPHA + l] = alpha ? alpha[ch * g.L + l] : 0.0;
      al[(size_t)ch * g.L + l] = f[BNN_F_ALPHA + l];
      // update_n = max(1, round(size * update_f)) with numpy's half-to-even rounding (BNN_env.py:292-293)
      int n = (int)nearbyint((double)size * update_f[ch * g.L + l]);
      i[BNN_I_UPDATE_N + l] = n < 1 ? 1 : n;
      i[BNN_I_MAX_N + l] = size;
    }
    for (int j = 0; j < g.K; ++j) f[BNN_F_SIGMA + j] = sigma0 ? sigma0[ch * g.K + j] : 1.0;
    // _last_accepted = 1, _last_accepted_mem = [1], _acceptance_rate = 0 (BNN_env.py:356-358)
    i[BNN_I_LAST_ACCEPTED] = 1;
    i[BNN_I_RING_LEN] = 1; i[BNN_I_RING_SUM] = 1; i[BNN_I_RING + 0] = 1;
  }
  CUDA_TRY(cudaMemcpyAsync(c->sf.p, sf.data(), sizeof(double) * sf.size(), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(c->si.p, si.data(), sizeof(int) * si.size(), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(c->alpha_chain.p, al.data(), sizeof(double) * al.size(), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaStreamSynchronize(st));   // host staging vectors go out of scope
  if (cfg->use_indicators || cfg->use_feature_indicators) {
    // both kinds of indicators start as all ones (BNN_env.py:124,170-171)
    REQUIRE(!cfg->use_indicators || (cfg->prior_ind1 > 0.0 && cfg->prior_ind1 < 1.0), "bnn_chains_init: prior_ind1 must be in (0, 1)");
    REQUIRE(!cfg->use_feature_indicators || c->have_feat_mean, "bnn_chains_init: call bnn_set_feature_means first");
    const size_t P0 = (size_t)g.l[0].out * (g.l[0].in + g.l[0].bias);
    std::vector<double> ones((size_t)C * (P0 > (size_t)g.F ? P0 : (size_t)g.F), 1.0);
    if (cfg->use_indicators)
      if (upload(c->ind_cur, ones.data(), (size_t)C * P0, st) || upload(c->ind_prop, ones.data(), (size_t)C * P0, st)) return 1;
    if (cfg->use_feature_indicators)
      if (upload(c->fi_cur, ones.data(), (size_t)C * g.F, st) || upload(c->fi_prop, ones.data(), (size_t)C * g.F, st)) return 1;
    CUDA_TRY(cudaStreamSynchronize(st));
  }

  // initial state: forward + likelihood + prior + counters of w0 (MCMC.__init__, BNN_env.py:299-353)
  ChainDev d = chain_dev(c);
  CUDA_TRY(bnn_launch_mh_update(d, 0, 2, 0, st));
  c->launches++;
  int rc = chains_forward(c, st);
  if (rc) return rc;
  c->have_chains = true;
  if (c->rowshard) return 0;          // the caller reduces over the ranks first, then bnn_rowshard_update(accept = 2)
  CUDA_TRY(bnn_launch_mh_update(d, 2, 0, 0, st));
  c->launches++;
  return 0;
}

// validate and upload the injected draws of n_steps iterations; fills the injection pointers of d
static int stage_injection(bnn_ctx* c, int32_t n_steps, const bnn_injection* inj, ChainDev& d, cudaStream_t st) {
  const NetGeom& g = c->g;
  if (inj) {
    REQUIRE(inj->n_steps >= n_steps && inj->cap >= 1, "bnn_mh_steps: injection shorter than n_steps");
    REQUIRE(inj->proposed && inj->count && inj->ix && inj->iy && inj->dz && inj->log_u, "bnn_mh_steps: null injection array");
    const size_t nl = (size_t)n_steps * c->C * g.L, nc = (size_t)n_steps * c->C * inj->cap;
    // bounds check on the host: indices address the canonical matrices directly
    for (size_t s = 0; s < (size_t)n_steps * c->C; ++s) {
      size_t off = 0;
      for (int l = 0; l < g.L; ++l) {
        if (!inj->proposed[s * g.L + l]) continue;
        const int cnt = inj->count[s * g.L + l];
        REQUIRE(cnt >= 0 && off + cnt <= (size_t)inj->cap, "bnn_mh_steps: injection count exceeds cap");
        for (int k = 0; k < cnt; ++k) {
          const int ix = inj->ix[s * inj->cap + off + k], iy = inj->iy[s * inj->cap + off + k];
          REQUIRE(ix >= 0 && ix < g.l[l].out && iy >= 0 && iy < g.l[l].in + g.l[l].bias, "bnn_mh_steps: injected index out of range");
        }
        off += cnt;
      }
    }
    const size_t ns = (size_t)n_steps * c->C;
    {
      // one transfer instead of six (a single-step injection is latency, not bandwidth: 6 x ~8 us of copy-engine
      // round trips in front of the step's first kernel)
      auto al = [](size_t b) { return (b + 15) & ~(size_t)15; };
      const size_t o_dz = 0, o_lu = o_dz + al(8 * nc), o_pr = o_lu + al(8 * ns), o_ct = o_pr + al(4 * nl),
                   o_ix = o_ct + al(4 * nl), o_iy = o_ix + al(4 * nc), total = o_iy + al(4 * nc);
      if (c->inj_copied) CUDA_TRY(cudaEventSynchronize(c->inj_copied));      // the staging buffer is free again
      else CUDA_TRY(cudaEventCreateWithFlags(&c->inj_copied, cudaEventDisableTiming));
      if (total > c->inj_host_bytes) {
        if (c->inj_host) CUDA_TRY(cudaFreeHost(c->inj_host));
        c->inj_host = nullptr; c->inj_host_bytes = 0;
        CUDA_TRY(cudaMallocHost(&c->inj_host, 2 * total));
        c->inj_host_bytes = 2 * total;
      }
      CUDA_TRY(c->inj_arena.ensure(total, false, st));
      char* h = static_cast<char*>(c->inj_host);
      memcpy(h + o_dz, inj->dz, 8 * nc);
      memcpy(h + o_lu, inj->log_u, 8 * ns);
      memcpy(h + o_pr, inj->proposed, 4 * nl);
      memcpy(h + o_ct, inj->count, 4 * nl);
      memcpy(h + o_ix, inj->ix, 4 * nc);
      memcpy(h + o_iy, inj->iy, 4 * nc);
      CUDA_TRY(cudaMemcpyAsync(c->inj_arena.p, h, total, cudaMemcpyHostToDevice, st));
      CUDA_TRY(cudaEventRecord(c->inj_copied, st));
      char* dv = static_cast<char*>(c->inj_arena.p);
      d.inj_dz = reinterpret_cast<double*>(dv + o_dz);
      d.inj_logu = reinterpret_cast<double*>(dv + o_lu);
      d.inj_proposed = reinterpret_cast<int*>(dv + o_pr);
      d.inj_count = reinterpret_cast<int*>(dv + o_ct);
      d.inj_ix = reinterpret_cast<int*>(dv + o_ix);
      d.inj_iy = reinterpret_cast<int*>(dv + o_iy);
    }
    d.inj_cap = inj->cap;
    if (c->cfg.n_act_prm > 0) {
      REQUIRE(inj->alpha_ix && inj->alpha_dz, "bnn_mh_steps: trainable activation parameters need alpha_ix / alpha_dz");
      for (size_t s = 0; s < ns; ++s)
        REQUIRE(inj->alpha_ix[s] >= 0 && inj->alpha_ix[s] < c->cfg.n_act_prm, "bnn_mh_steps: alpha_ix out of range");
      if (upload(c->inj_alpha_ix, inj->alpha_ix, ns, st) || upload(c->inj_alpha_dz, inj->alpha_dz, ns, st)) return 1;
      d.inj_alpha_ix = c->inj_alpha_ix.as<int>();
      d.inj_alpha_dz = c->inj_alpha_dz.as<double>();
    }
    if (inj->add_prob) {
      if (upload(c->inj_add_prob, inj->add_prob, ns, st)) return 1;
      d.inj_add_prob = c->inj_add_prob.as<double>();
    }
    if (inj->ind_move) {
      REQUIRE(c->cfg.use_indicators && inj->ind_flip, "bnn_mh_steps: ind_move needs cfg.use_indicators and ind_flip");
      const size_t P0 = (size_t)g.l[0].out * (g.l[0].in + g.l[0].bias);
      if (upload(c->inj_ind_move, inj->ind_move, ns, st) || upload(c->inj_ind_flip, inj->ind_flip, ns * P0, st)) return 1;
      d.inj_ind_move = c->inj_ind_move.as<int>();
      d.inj_ind_flip = c->inj_ind_flip.as<uint8_t>();
    }
    if (inj->fi_move) {
      REQUIRE(c->cfg.use_feature_indicators && inj->fi_flip, "bnn_mh_steps: fi_move needs cfg.use_feature_indicators and fi_flip");
      if (upload(c->inj_fi_move, inj->fi_move, ns, st) || upload(c->inj_fi_flip, inj->fi_flip, ns * (size_t)g.F, st)) return 1;
      d.inj_fi_move = c->inj_fi_move.as<int>();
      d.inj_fi_flip = c->inj_fi_flip.as<uint8_t>();
    }
  } else {
    // free-running chains: every branch of the proposal is drawn on the device (Philox); the weight-indicator move
    // reads update_f[3] like the reference (BNN_env.py:460), i.e. it exists from four layers on
    REQUIRE(!(c->cfg.use_indicators && c->cfg.freq_indicator > 0.0 && g.L < 4),
            "bnn_mh_steps: weight-indicator moves need a network of at least four layers (update_f[3])");
  }
  return 0;
}

// the launch sequence of n_steps MH iterations: [accept s-1 + propose s] [forward] ... [accept n-1]
static int launch_mh_sequence(bnn_ctx* c, const ChainDev& d, int32_t n_steps, cudaStream_t st) {
  for (int s = 0; s < n_steps; ++s) {
    CUDA_TRY(bnn_launch_mh_update(d, s > 0 ? 1 : 0, 1, s, st));
    c->launches++;
    int rc = chains_forward(c, st);
    if (rc) return rc;
  }
  CUDA_TRY(bnn_launch_mh_update(d, 1, 0, n_steps, st));
  c->launches++;
  return 0;
}

int bnn_mh_steps(bnn_ctx* c, int32_t n_steps, const bnn_injection* inj, void* stream) {
  REQUIRE(c && c->have_chains, "bnn_mh_steps: call bnn_chains_init first");
  REQUIRE(n_steps >= 1, "bnn_mh_steps: n_steps must be >= 1");
  REQUIRE(!c->rowshard, "bnn_mh_steps: row-sharded chains are stepped with bnn_rowshard_update / _local / _commit");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  ChainDev d = chain_dev(c);
  if (int rc = stage_injection(c, n_steps, inj, d, st)) return rc;
  // Small data sets (a few thousand rows, <= 2048 weights, dense generic forward path): all n_steps iterations run
  // inside ONE persistent launch, a thread-block cluster per chain (bnn_chainloop.cu) -- injected or device-generated
  // proposals alike.  Same update / forward bodies and reduction order as the launch sequence below: identical chains.
  if (c->opt_chain_loop && !c->time_forward && !(c->sparse.sp.prog && c->opt_sparse) &&
      (c->force_generic || !bnn_fwd3_family(c->g)) && !bnn_part_slices(c->n_tiles16) &&
      bnn_chain_loop_fits(c->g, d.NF, d.n_tiles16, c->C, c->n_sms, c->opt_chain_cluster, c->opt_chain_loop)) {
    FwdParams p = base_params(c);
    p.C = 1;
    int cl = 0;
    cudaError_t e = bnn_launch_chain_loop(d, p, n_steps, c->n_sms, c->opt_chain_cluster, c->opt_chain_loop, st, &cl);
    if (e == cudaSuccess) {
      c->launches++;
      c->last_kernel = "k_chain_loop";
      if (inj) CUDA_TRY(cudaStreamSynchronize(st));
      return 0;
    }
    cudaGetLastError();
    if (e != cudaErrorNotSupported) {
      // a cluster shape this GPU cannot schedule (MIG slices, non-portable size): halve it once, then give the path up
      if (c->opt_chain_cluster > 8) c->opt_chain_cluster = 8; else c->opt_chain_loop = 0;
      return bnn_mh_steps(c, n_steps, inj, stream);
    }
  }
  // Free-running chains: the sequence depends on nothing but n_steps (Philox counters come from the chain state), so
  // it is captured once per n_steps into a CUDA graph and replayed -- at small N the loop is bound by launch latency,
  // not by the kernels.  The first call after any (re)configuration runs eagerly (function attributes, lazily
  // allocated workspaces); capture uses a private stream because the caller's may be the legacy default stream.
  const bool graphable = !inj && c->opt_graphs && c->mh_warm && !c->time_forward && n_steps >= 2 && n_steps <= 512;
  if (graphable) {
    cudaGraphExec_t exec = nullptr;
    long long per_launch = 0;
    for (auto& gph : c->graphs)
      if (gph.n_steps == n_steps) { exec = gph.exec; per_launch = gph.launches; }
    if (!exec) {
      // capture; any failure (a launch path that is not capturable on this driver) turns graphs off for this context
      // and falls through to the eager sequence below -- never an error for the caller
      const long long l0 = c->launches;
      bool ok = true;
      if (!c->capture_stream) ok = cudaStreamCreateWithFlags(&c->capture_stream, cudaStreamNonBlocking) == cudaSuccess;
      ok = ok && cudaStreamBeginCapture(c->capture_stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
      if (ok) {
        const int rc = launch_mh_sequence(c, d, n_steps, c->capture_stream);
        cudaGraph_t graph = nullptr;
        ok = cudaStreamEndCapture(c->capture_stream, &graph) == cudaSuccess && rc == 0 && graph != nullptr;
        ok = ok && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
        if (graph) cudaGraphDestroy(graph);
      }
      per_launch = c->launches - l0;          // kernels in the sequence (counted while capturing, launched on replay)
      c->launches = l0;
      if (!ok) {
        cudaGetLastError();
        c->opt_graphs = 0;
        exec = nullptr;
      } else {
        if (c->graphs.size() >= 8) { cudaGraphExecDestroy(c->graphs.front().exec); c->graphs.erase(c->graphs.begin()); }
        c->graphs.push_back({n_steps, exec, per_launch});
      }
    }
    if (exec) {
      CUDA_TRY(cudaGraphLaunch(exec, st));
      c->launches += per_launch;
      return 0;
    }
  }
  if (int rc = launch_mh_sequence(c, d, n_steps, st)) return rc;
  if (!inj) c->mh_warm = true;
  if (inj) CUDA_TRY(cudaStreamSynchronize(st));   // the caller may free the host arrays after return
  return 0;
}

// ---- row sharding (include/npbnn_b200.h) -------------------------------------------------------------------
int bnn_rowshard_config(bnn_ctx* c, int64_t n_train_global) {
  REQUIRE(c && c->have_data, "bnn_rowshard_config: call bnn_set_data (this rank's rows) first");
  invalidate_graphs(c);
  REQUIRE(n_train_global >= c->n_train, "bnn_rowshard_config: n_train_global is smaller than the local shard");
  c->rowshard = true;
  c->n_train_global = n_train_global;
  c->have_chains = false;
  return 0;
}

int bnn_rowshard_n_values(const bnn_ctx* c) { return c ? bnn_n_slots(c->g) + bnn_n_counts(c->g.K) : 0; }

int bnn_rowshard_local(bnn_ctx* c, double* red_dev, void* stream) {
  REQUIRE(c && c->have_chains && c->rowshard && red_dev, "bnn_rowshard_local: bad arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  const NetGeom& g = c->g;
  const int* counts = (g.lik == BNN_LIK_CATEGORICAL) ? c->counts_prop.as<int>() : nullptr;
  CUDA_TRY(bnn_launch_rowshard_local(g, c->part.as<double>(), bnn_n_slots(g), c->n_tiles16, counts, bnn_n_counts(g.K), red_dev, c->C,
                                     (cudaStream_t)stream));
  c->launches++;
  return 0;
}

int bnn_rowshard_commit(bnn_ctx* c, const double* red_global_dev, void* stream) {
  REQUIRE(c && c->have_chains && c->rowshard && red_global_dev, "bnn_rowshard_commit: bad arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  const NetGeom& g = c->g;
  int* counts = (g.lik == BNN_LIK_CATEGORICAL) ? c->counts_prop.as<int>() : nullptr;
  CUDA_TRY(bnn_launch_rowshard_commit(red_global_dev, bnn_n_slots(g), bnn_n_counts(g.K), c->part_red.as<double>(), counts, c->C,
                                      (cudaStream_t)stream));
  c->launches++;
  return 0;
}

int bnn_rowshard_update(bnn_ctx* c, int32_t accept_mode, int32_t propose, const bnn_injection* inj, void* stream) {
  REQUIRE(c && c->have_chains && c->rowshard, "bnn_rowshard_update: call bnn_rowshard_config and bnn_chains_init first");
  REQUIRE(accept_mode >= 0 && accept_mode <= 2, "bnn_rowshard_update: accept_mode must be 0, 1 or 2");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  ChainDev d = chain_dev(c);
  if (propose)
    if (int rc = stage_injection(c, 1, inj, d, st)) return rc;
  CUDA_TRY(bnn_launch_mh_update(d, accept_mode, propose ? 1 : 0, 0, st));
  c->launches++;
  if (propose) {
    if (int rc = chains_forward(c, st)) return rc;
    if (inj) CUDA_TRY(cudaStreamSynchronize(st));
  }
  return 0;
}

int bnn_chains_read(bnn_ctx* c, double* f64_host, int32_t* i32_host, double* w_host, void* stream) {
  REQUIRE(c && c->have_chains, "bnn_chains_read: call bnn_chains_init first");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (f64_host) CUDA_TRY(cudaMemcpyAsync(f64_host, c->sf.p, sizeof(double) * (size_t)c->C * BNN_F_STRIDE, cudaMemcpyDeviceToHost, st));
  if (i32_host) CUDA_TRY(cudaMemcpyAsync(i32_host, c->si.p, sizeof(int) * (size_t)c->C * BNN_I_STRIDE, cudaMemcpyDeviceToHost, st));
  if (w_host) CUDA_TRY(cudaMemcpyAsync(w_host, c->w_cur.p, sizeof(double) * (size_t)c->C * c->g.P, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

// ---- asynchronous snapshots (include/npbnn_b200.h) ----------------------------------------------------------
// a slot holds the f64 rows, the i32 rows, the weights, then the current weight / feature indicators of chains that
// carry them (doubles; counts returned in n_ind, n_fi)
static size_t snap_bytes(const bnn_ctx* c, size_t* n_ind = nullptr, size_t* n_fi = nullptr) {
  const size_t ni = c->cfg.use_indicators ? (size_t)c->C * c->g.l[0].out * (c->g.l[0].in + c->g.l[0].bias) : 0;
  const size_t nf = c->cfg.use_feature_indicators ? (size_t)c->C * c->g.F : 0;
  if (n_ind) *n_ind = ni;
  if (n_fi) *n_fi = nf;
  return (size_t)c->C * (sizeof(double) * BNN_F_STRIDE + sizeof(int) * BNN_I_STRIDE + sizeof(double) * c->g.P) +
         sizeof(double) * (ni + nf);
}

int bnn_chains_snapshot(bnn_ctx* c, int32_t slot, void* stream) {
  REQUIRE(c && c->have_chains, "bnn_chains_snapshot: call bnn_chains_init first");
  REQUIRE(slot >= 0 && slot < bnn_ctx::kSnapSlots, "bnn_chains_snapshot: slot must be in [0, 64)");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  bnn_ctx::Snap& sn = c->snaps[slot];
  REQUIRE(!sn.pending, "bnn_chains_snapshot: slot still holds an unread snapshot");
  const size_t nb = snap_bytes(c);
  if (!c->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  if (!sn.staged) {
    CUDA_TRY(cudaEventCreateWithFlags(&sn.staged, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&sn.done, cudaEventDisableTiming));
  }
  if (sn.bytes < nb) {
    if (sn.host) CUDA_TRY(cudaFreeHost(sn.host));
    sn.host = nullptr;
    CUDA_TRY(cudaMallocHost(&sn.host, nb));
    sn.bytes = nb;
  }
  CUDA_TRY(sn.dev.ensure(nb, false, st));
  // device-to-device on the chains' stream (the next launches queue right behind it) ...
  char* d = sn.dev.as<char>();
  const size_t nf = sizeof(double) * (size_t)c->C * BNN_F_STRIDE, ni = sizeof(int) * (size_t)c->C * BNN_I_STRIDE;
  const size_t nw = sizeof(double) * (size_t)c->C * c->g.P;
  CUDA_TRY(cudaMemcpyAsync(d, c->sf.p, nf, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(d + nf, c->si.p, ni, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(d + nf + ni, c->w_cur.p, nw, cudaMemcpyDeviceToDevice, st));
  size_t n_ind, n_fi;
  snap_bytes(c, &n_ind, &n_fi);
  if (n_ind) CUDA_TRY(cudaMemcpyAsync(d + nf + ni + nw, c->ind_cur.p, sizeof(double) * n_ind, cudaMemcpyDeviceToDevice, st));
  if (n_fi)
    CUDA_TRY(cudaMemcpyAsync(d + nf + ni + nw + sizeof(double) * n_ind, c->fi_cur.p, sizeof(double) * n_fi,
                             cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(cudaEventRecord(sn.staged, st));
  // ... device-to-host on the copy stream, off the chains' critical path
  CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, sn.staged, 0));
  CUDA_TRY(cudaMemcpyAsync(sn.host, d, nb, cudaMemcpyDeviceToHost, c->copy_stream));
  CUDA_TRY(cudaEventRecord(sn.done, c->copy_stream));
  sn.pending = true;
  return 0;
}

int bnn_snapshot_ready(bnn_ctx* c, int32_t slot) {
  if (!c || slot < 0 || slot >= bnn_ctx::kSnapSlots || !c->snaps[slot].pending) return -1;
  cudaError_t e = cudaEventQuery(c->snaps[slot].done);
  if (e == cudaSuccess) return 1;
  if (e == cudaErrorNotReady) return 0;
  g_last_error = std::string("bnn_snapshot_ready: ") + cudaGetErrorString(e);
  return -1;
}

int bnn_snapshot_read(bnn_ctx* c, int32_t slot, double* f64_host, int32_t* i32_host, double* w_host) {
  REQUIRE(c && slot >= 0 && slot < bnn_ctx::kSnapSlots && c->snaps[slot].pending,
          "bnn_snapshot_read: no snapshot pending in this slot");
  CUDA_TRY(cudaSetDevice(c->device));
  bnn_ctx::Snap& sn = c->snaps[slot];
  CUDA_TRY(cudaEventSynchronize(sn.done));
  const char* h = static_cast<const char*>(sn.host);
  const size_t nf = sizeof(double) * (size_t)c->C * BNN_F_STRIDE, ni = sizeof(int) * (size_t)c->C * BNN_I_STRIDE;
  const size_t nw = sizeof(double) * (size_t)c->C * c->g.P;
  if (f64_host) memcpy(f64_host, h, nf);
  if (i32_host) memcpy(i32_host, h + nf, ni);
  if (w_host) memcpy(w_host, h + nf + ni, nw);
  sn.pending = false;
  return 0;
}

int bnn_snapshot_read_indicators(bnn_ctx* c, int32_t slot, double* ind_host, double* fi_host) {
  REQUIRE(c && slot >= 0 && slot < bnn_ctx::kSnapSlots && c->snaps[slot].pending,
          "bnn_snapshot_read_indicators: no snapshot pending in this slot");
  REQUIRE(!ind_host || c->cfg.use_indicators, "bnn_snapshot_read_indicators: the chains have no weight indicators");
  REQUIRE(!fi_host || c->cfg.use_feature_indicators, "bnn_snapshot_read_indicators: the chains have no feature indicators");
  CUDA_TRY(cudaSetDevice(c->device));
  bnn_ctx::Snap& sn = c->snaps[slot];
  CUDA_TRY(cudaEventSynchronize(sn.done));
  size_t n_ind, n_fi;
  const size_t nb = snap_bytes(c, &n_ind, &n_fi);
  const char* h = static_cast<const char*>(sn.host) + nb - sizeof(double) * (n_ind + n_fi);
  if (ind_host) memcpy(ind_host, h, sizeof(double) * n_ind);
  if (fi_host) memcpy(fi_host, h + sizeof(double) * n_ind, sizeof(double) * n_fi);
  return 0;
}

int bnn_set_feature_means(bnn_ctx* c, const double* mean_host, void* stream) {
  REQUIRE(c && c->have_net && mean_host, "bnn_set_feature_means: call bnn_set_net first");
  invalidate_graphs(c);
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (upload(c->feat_mean, mean_host, (size_t)c->g.F, st)) return 1;
  CUDA_TRY(cudaStreamSynchronize(st));
  c->have_feat_mean = true;
  return 0;
}

int bnn_chains_read_indicators(bnn_ctx* c, double* ind_host, double* fi_host, void* stream) {
  REQUIRE(c && c->have_chains, "bnn_chains_read_indicators: call bnn_chains_init first");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t P0 = (size_t)c->g.l[0].out * (c->g.l[0].in + c->g.l[0].bias);
  if (ind_host) {
    REQUIRE(c->cfg.use_indicators, "bnn_chains_read_indicators: the chains have no weight indicators");
    CUDA_TRY(cudaMemcpyAsync(ind_host, c->ind_cur.p, sizeof(double) * (size_t)c->C * P0, cudaMemcpyDeviceToHost, st));
  }
  if (fi_host) {
    REQUIRE(c->cfg.use_feature_indicators, "bnn_chains_read_indicators: the chains have no feature indicators");
    CUDA_TRY(cudaMemcpyAsync(fi_host, c->fi_cur.p, sizeof(double) * (size_t)c->C * c->g.F, cudaMemcpyDeviceToHost, st));
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

int bnn_chains_write_indicators(bnn_ctx* c, const double* ind_host, const double* fi_host, void* stream) {
  REQUIRE(c && c->have_chains, "bnn_chains_write_indicators: call bnn_chains_init first");
  REQUIRE(!ind_host || c->cfg.use_indicators, "bnn_chains_write_indicators: the chains have no weight indicators");
  REQUIRE(!fi_host || c->cfg.use_feature_indicators, "bnn_chains_write_indicators: the chains have no feature indicators");
  const NetGeom& g = c->g;
  const size_t P0 = (size_t)g.l[0].out * (g.l[0].in + g.l[0].bias);
  for (size_t i = 0; ind_host && i < (size_t)c->C * P0; ++i)
    REQUIRE(ind_host[i] == 0.0 || ind_host[i] == 1.0, "bnn_chains_write_indicators: weight indicators must be 0 or 1");
  for (size_t i = 0; fi_host && i < (size_t)c->C * g.F; ++i)
    REQUIRE(fi_host[i] == 0.0 || fi_host[i] == 1.0, "bnn_chains_write_indicators: feature indicators must be 0 or 1");
  if (!ind_host && !fi_host) return 0;
  invalidate_graphs(c);              // the captured sequences read the indicators
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (ind_host) CUDA_TRY(cudaMemcpyAsync(c->ind_cur.p, ind_host, sizeof(double) * (size_t)c->C * P0, cudaMemcpyHostToDevice, st));
  if (fi_host) CUDA_TRY(cudaMemcpyAsync(c->fi_cur.p, fi_host, sizeof(double) * (size_t)c->C * g.F, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaStreamSynchronize(st));   // the caller's arrays are free on return
  // the current weights are scored again under the new indicators, as bnn_chains_init scores w0 (the proposal step
  // copies ind_cur / fi_cur into the proposal buffers)
  ChainDev d = chain_dev(c);
  CUDA_TRY(bnn_launch_mh_update(d, 0, 2, 0, st));
  c->launches++;
  if (int rc = chains_forward(c, st)) return rc;
  if (c->rowshard) return 0;          // the caller reduces over the ranks first, then bnn_rowshard_update(accept = 2)
  CUDA_TRY(bnn_launch_mh_update(d, 2, 0, 0, st));
  c->launches++;
  return 0;
}

int bnn_chains_write(bnn_ctx* c, const double* f64_host, const int32_t* i32_host, void* stream) {
  REQUIRE(c && c->have_chains, "bnn_chains_write: call bnn_chains_init first");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (f64_host) CUDA_TRY(cudaMemcpyAsync(c->sf.p, f64_host, sizeof(double) * (size_t)c->C * BNN_F_STRIDE, cudaMemcpyHostToDevice, st));
  if (i32_host) CUDA_TRY(cudaMemcpyAsync(c->si.p, i32_host, sizeof(int) * (size_t)c->C * BNN_I_STRIDE, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

int bnn_chains_set_prior_scales(bnn_ctx* c, const double* entry_scale_host, void* stream) {
  REQUIRE(c && c->have_chains, "bnn_chains_set_prior_scales: call bnn_chains_init first");
  invalidate_graphs(c);
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (entry_scale_host) {
    if (int rc = upload_entry_scales(c->ps_entry, c->pls_entry, entry_scale_host, (size_t)c->C * c->g.P, st,
                                     "bnn_chains_set_prior_scales")) return rc;
    c->have_ps_entry = true;
  } else {
    c->have_ps_entry = false;
  }
  ChainDev d = chain_dev(c);
  CUDA_TRY(bnn_launch_prior_refresh(d, st));
  c->launches++;
  return 0;
}

int bnn_chains_set_additional_prob(bnn_ctx* c, const double* per_chain_host, void* stream) {
  REQUIRE(c && c->have_chains, "bnn_chains_set_additional_prob: call bnn_chains_init first");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (!per_chain_host) {
    if (c->have_add_prob) invalidate_graphs(c);      // the captured sequences read the buffer
    c->have_add_prob = false;
    return 0;
  }
  for (int ch = 0; ch < c->C; ++ch)
    REQUIRE(std::isfinite(per_chain_host[ch]), "bnn_chains_set_additional_prob: values must be finite");
  if (!c->have_add_prob) {
    // the first value after bnn_chains_init: the proposal step starts reading the buffer, the captured sequences did not
    invalidate_graphs(c);
    CUDA_TRY(c->add_prob.ensure(sizeof(double) * (size_t)c->C, false, st));
  }
  // in stream order: the steps queued before this call use the old value, the ones after it (a graph replay too) the new
  CUDA_TRY(cudaMemcpyAsync(c->add_prob.p, per_chain_host, sizeof(double) * (size_t)c->C, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaStreamSynchronize(st));   // the caller's array is free on return
  c->have_add_prob = true;
  return 0;
}

int bnn_chains_state_dev(bnn_ctx* c, double** f64_dev, int32_t** i32_dev, double** w_dev) {
  REQUIRE(c && c->have_chains, "bnn_chains_state_dev: call bnn_chains_init first");
  if (f64_dev) *f64_dev = c->sf.as<double>();
  if (i32_dev) *i32_dev = c->si.as<int>();
  if (w_dev) *w_dev = c->w_cur.as<double>();
  return 0;
}

int bnn_chains_gather(bnn_ctx* c, int32_t slot, double* out_dev, void* stream) {
  REQUIRE(c && c->have_chains && out_dev, "bnn_chains_gather: bad arguments");
  REQUIRE(slot >= 0 && slot < BNN_F_STRIDE, "bnn_chains_gather: slot out of range");
  CUDA_TRY(cudaSetDevice(c->device));
  CUDA_TRY(cudaMemcpy2DAsync(out_dev, sizeof(double), c->sf.as<double>() + slot, sizeof(double) * BNN_F_STRIDE,
                             sizeof(double), c->C, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int bnn_forward_time(bnn_ctx* c, double* total_ms, int64_t* n_launches, int32_t reset) {
  REQUIRE(c, "bnn_forward_time: null context");
  CUDA_TRY(cudaSetDevice(c->device));
  for (size_t i = 0; i + 1 < c->ev_used; i += 2) {
    CUDA_TRY(cudaEventSynchronize(c->ev[i + 1]));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, c->ev[i], c->ev[i + 1]));
    c->fwd_ms_sum += ms;
    c->fwd_count++;
  }
  c->ev_used = 0;
  if (total_ms) *total_ms = c->fwd_ms_sum;
  if (n_launches) *n_launches = c->fwd_count;
  if (reset) { c->fwd_ms_sum = 0.0; c->fwd_count = 0; }
  return 0;
}

int bnn_measure_fp64_peak(bnn_ctx* c, double* tflops) {
  REQUIRE(c && tflops, "bnn_measure_fp64_peak: bad arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  CUDA_TRY(bnn_measure_dmma_peak(c->n_sms, tflops));
  return 0;
}

int bnn_chains_set_temperature(bnn_ctx* c, const double* temperature_host, void* stream) {
  REQUIRE(c && c->have_chains && temperature_host, "bnn_chains_set_temperature: bad arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(cudaMemcpy2DAsync(c->sf.as<double>() + BNN_F_TEMPERATURE, sizeof(double) * BNN_F_STRIDE, temperature_host,
                             sizeof(double), sizeof(double), c->C, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

static int predict_impl(bnn_ctx* c, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                        const double* alpha_dev, const int32_t* override_cols, const double* override_vals,
                        int32_t n_override, double* mean_dev, double* votes_dev, double* dense_dev, const double* u_dev,
                        int32_t* class_counts_dev, double* post_pred_dev, void* stream, bool samp_philox = false,
                        uint64_t samp_seed = 0, int64_t samp_row0 = 0, int32_t samp_set0 = 0) {
  REQUIRE(c && c->have_net, "bnn_predict: call bnn_set_net first");
  REQUIRE(x_dev && w_dev && n >= 1 && n_sets >= 1, "bnn_predict: bad arguments");
  REQUIRE(mean_dev || votes_dev || dense_dev, "bnn_predict: no output requested");
  REQUIRE(n_override >= 0 && (n_override == 0 || (override_cols && override_vals)), "bnn_predict: bad override arguments");
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const NetGeom g = geom_for_rows(c->g_base, n);      // prediction picks its padding from ITS row count
  REQUIRE(!(votes_dev && g.lik != BNN_LIK_CATEGORICAL), "bnn_predict: vote summary needs the categorical likelihood");
  const long long n_pad = (n + 15) / 16 * 16;
  CUDA_TRY(c->xs_pred.ensure(sizeof(double) * (size_t)n_pad * g.F_pad, false, st));
  const int* ovc = nullptr;
  const double* ovv = nullptr;
  if (n_override > 0) {
    for (int k = 0; k < n_override; ++k) REQUIRE(override_cols[k] >= 0 && override_cols[k] < g.F, "bnn_predict: override column out of range");
    if (upload(c->ov_cols, override_cols, n_override, st)) return 1;
    if (upload(c->ov_vals, override_vals, n_override, st)) return 1;
    CUDA_TRY(cudaStreamSynchronize(st));
    ovc = c->ov_cols.as<int>();
    ovv = c->ov_vals.as<double>();
  }
  CUDA_TRY(bnn_launch_pack_x(x_dev, c->xs_pred.as<double>(), n, n_pad, g.F, g.F_pad, g.x_swz, ovc, ovv, n_override, st));
  if (int rc = ensure_wp_scratch(c, g, (size_t)n_sets, st)) return rc;
  CUDA_TRY(bnn_launch_pack_w(g, w_dev, c->wp_scratch.as<double>(), n_sets, st));
  FwdParams p = fwd_params(c, g, c->xs_pred.as<double>(), n, n);
  p.wp = c->wp_scratch.as<double>();
  p.alpha = alpha_dev;
  p.C = n_sets;
  p.mean_out = mean_dev; p.votes_out = votes_dev; p.dense_out = dense_dev;
  p.inv_sets = (double)n_sets;   // divisor (np.mean and the vote share divide, BNN_lib.py:390-392)
  p.samp_u = u_dev; p.samp_counts = class_counts_dev; p.samp_dense = post_pred_dev;
  p.samp_philox = samp_philox ? 1 : 0; p.samp_seed = samp_seed;
  p.samp_row0 = samp_row0; p.samp_set0 = samp_set0;
  if (class_counts_dev) CUDA_TRY(cudaMemsetAsync(class_counts_dev, 0, sizeof(int32_t) * (size_t)n_sets * g.K, st));
  if (c->opt_pred_tf32 && !c->force_generic && bnn_pred_tf32_fits(p)) {
    // opt-in reduced precision (stated tolerance: class probabilities to ~1e-6 absolute); summaries only
    CUDA_TRY(bnn_launch_pred_tf32(p, c->n_sms, c->opt_pred_tf32 >= 2 ? 1 : 3, st, &c->last_kernel));
    c->launches += 3;
    return 0;
  }
  CUDA_TRY(timed_forward(c, p, true, st));
  c->launches += 3;
  return 0;
}

int bnn_predict(bnn_ctx* c, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                const double* alpha_dev, const int32_t* override_cols, const double* override_vals,
                int32_t n_override, double* mean_dev, double* votes_dev, double* dense_dev, void* stream) {
  return predict_impl(c, x_dev, n, w_dev, n_sets, alpha_dev, override_cols, override_vals, n_override, mean_dev,
                      votes_dev, dense_dev, nullptr, nullptr, nullptr, stream);
}

int bnn_predict_sample_philox_at(bnn_ctx* c, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                                 const double* alpha_dev, uint64_t seed, int64_t row0, int32_t set0, double* est_dev,
                                 int32_t* class_counts_dev, double* post_pred_dev, void* stream) {
  REQUIRE(c && c->have_net && c->g.lik == BNN_LIK_CATEGORICAL, "bnn_predict_sample_philox: needs the categorical likelihood");
  REQUIRE(est_dev, "bnn_predict_sample_philox: est_dev is required");
  REQUIRE(row0 >= 0 && set0 >= 0, "bnn_predict_sample_philox_at: negative offset");
  return predict_impl(c, x_dev, n, w_dev, n_sets, alpha_dev, nullptr, nullptr, 0, nullptr, est_dev, nullptr, nullptr,
                      class_counts_dev, post_pred_dev, stream, true, seed, row0, set0);
}

int bnn_predict_sample_philox(bnn_ctx* c, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                              const double* alpha_dev, uint64_t seed, double* est_dev, int32_t* class_counts_dev,
                              double* post_pred_dev, void* stream) {
  return bnn_predict_sample_philox_at(c, x_dev, n, w_dev, n_sets, alpha_dev, seed, 0, 0, est_dev, class_counts_dev,
                                      post_pred_dev, stream);
}

int bnn_predict_sample(bnn_ctx* c, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                       const double* alpha_dev, const double* u_dev, double* est_dev, int32_t* class_counts_dev,
                       double* post_pred_dev, void* stream) {
  REQUIRE(c && c->have_net && c->g.lik == BNN_LIK_CATEGORICAL, "bnn_predict_sample: needs the categorical likelihood");
  REQUIRE(u_dev && est_dev, "bnn_predict_sample: u_dev and est_dev are required");
  // the per-row shares of the drawn classes use the vote accumulator of the prediction kernels
  return predict_impl(c, x_dev, n, w_dev, n_sets, alpha_dev, nullptr, nullptr, 0, nullptr, est_dev, nullptr, u_dev,
                      class_counts_dev, post_pred_dev, stream);
}

}  // extern "C"
