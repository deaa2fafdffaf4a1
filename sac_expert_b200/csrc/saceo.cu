// libsaceo: C ABI + launch orchestration of the SAC-EO gradient-update hot path on B200 (sm_100a).
// See include/saceo.h for the contract and the reference call sites each entry point replaces.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstdarg>
#include <string>
#include <vector>
#include <map>
#include <algorithm>

#include "../../include/saceo.h"
#include "gemm_simt.cuh"
#include "gemm_skinny.cuh"
#include "elem.cuh"
#include "fvp.cuh"
#include "trpo.cuh"
#include "tc_gemm.cuh"
#include "mlp_ws.cuh"
#include "model_term.cuh"
#include "model_fit.cuh"
#include "policy.cuh"

using namespace saceo;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
  return code;
}
#define CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) \
  return fail(SACEO_E_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); } while (0)

static inline long long rup(long long x, long long m) { return (x + m - 1) / m * m; }
static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
constexpr int MAXH = SACEO_POLICY_MAX_HIDDEN;

struct NetD {            // one (population of) MLP(s) in the flat Keras layout: nh hidden layers, then the linear output layer
  const float* theta; long long sa, sn; int nnet;
  int in, out, nh;
  int hw[MAXH], ha[MAXH];  // width and activation of each hidden layer
  const uint8_t* planes = nullptr; long long pa = 0, pn = 0;   // fp16 hi/lo weight-plane images (mlp_ws.cuh), bytes per agent / net
  // layer l in [0, nh]: fan-in, width, activation, and the offsets of its weight [K x N] and bias [N] in theta
  int K(int l) const { return l == 0 ? in : hw[l - 1]; }
  int N(int l) const { return l == nh ? out : hw[l]; }
  int act(int l) const { return l == nh ? ACT_LINEAR : ha[l]; }
  long long oW(int l) const { return l == 0 ? 0 : ob(l - 1) + N(l - 1); }
  long long ob(int l) const { return oW(l) + (long long)K(l) * N(l); }
  long long n() const { return ob(nh) + N(nh); }                                      // parameters
  int widest(int l0) const { return l0 == nh ? N(nh) : std::max(N(l0), widest(l0 + 1)); }   // of layers l0 ... nh
  // the warp-specialised fused kernels (mlp_ws.cuh) take this net in both directions: two FW_H-wide hidden layers,
  // 1 to WS_MAXOUT outputs, 16-byte aligned parameters.  Every other net runs on the per-layer GEMM chain.
  bool ws() const {
    return nh == 2 && mlp_fwd_ws_eligible(N(0), N(1), out, in, theta, sa, sn) &&
           mlp_bwd_ws_eligible(N(0), N(1), out, out, false, 0, theta, sa, sn);
  }
};
static NetD net_desc(const float* theta, long long sa, long long sn, int nnet, int in, int out, int nh, const int* hw,
                     const int* ha) {
  NetD d{theta, sa, sn, nnet, in, out, nh};
  for (int l = 0; l < nh; ++l) { d.hw[l] = hw[l]; d.ha[l] = ha[l]; }
  return d;
}
// The nets of a config, shape only: fill_layout and carve size from them, actor_net / critic_net / model_net bind them.
static NetD actor_desc(const saceo_config& c) {
  return net_desc(nullptr, 0, 0, 1, c.S, c.per_state_std ? 2 * c.A : c.A, 2, c.actor_hidden, c.actor_act);
}
static NetD critic_desc(const saceo_config& c) {
  return net_desc(nullptr, 0, 0, 2, c.S + c.A, 1, 2, c.critic_hidden, c.critic_act);
}
static NetD model_desc(const saceo_config& c) {
  return net_desc(nullptr, 0, 0, c.num_models, c.S + c.A, c.separate_reward_nn ? c.S : c.S + 1, c.model_layers,
                  c.model_hidden, c.model_act);
}
// an actor's parameters: its layers, then without a per-state std its logstd variable (continuous_actors.py:56-57)
static long long actor_params(const NetD& d, bool per_state_std) { return d.n() + (per_state_std ? 0 : d.out); }

struct saceo_ctx {
  saceo_config cfg;
  // engine switches, decoded once from cfg.gemm_mode and the cfg.reserved tuning switches (include/saceo.h)
  bool tc = false;                     // tcgen05 bf16x3 GEMM engine
  int tc_variant = 0;                  // its tile variant
  bool fuse_fwd = false, fuse_bwd = false;   // fused forward / backward-chain kernel (needs ws_kernels)
  bool ws_kernels = false;             // weight-plane images for the warp-specialised fused kernels (tcgen05 engine only)
  bool fork = false;                   // side streams: the concurrent actor-phase branch and the weight-gradient fan-out
  saceo_layout L;
  KCtx k;                 // device-visible view (tables + workspace)
  FvpWs f;
  bool bound = false;
  void* ws = nullptr;
  long long ws_bytes = 0;
  std::map<std::string, std::pair<void*, long long>> names;
  long long* idx_stage = nullptr;
  float* dbpart = nullptr;             // per-tile bias-gradient partials of the fused backward kernel
  long long dbpart_cap = 0;            // floats; a launch that needs more falls back to the ones-row bias path
  // weight-plane images maintained by k_adam / k_planes_build (warp-specialised fused kernels, mlp_ws.cuh)
  uint8_t *pl_actor = nullptr, *pl_q = nullptr, *pl_qt = nullptr;
  int planes_dirty = 3;                // bit 0: actor image stale, bit 1: critic / target images stale
  // actor-phase buffers of their own (input operands, head outputs, neglogp, critic input with pi(s)), so that the
  // critic-independent half of the actor phase can run on a second stream next to the critic phase
  float *Xpi2 = nullptr, *aOut2 = nullptr, *nlp2 = nullptr, *Xc3 = nullptr;
  // bf16 hi/lo plane images of h1 / dH2 (actor: Rs rows, critics: B rows per net): operands of k_dw_planes
  uint8_t *aH1p = nullptr, *adH2p = nullptr, *cH1p = nullptr, *cdH2p = nullptr, *adH1p = nullptr, *cdH1p = nullptr;
  long long a_img = 0, c_img = 0;      // bytes per (agent, net) image
  // activations of each hidden layer and their gradients, [agent][net][rows][width]: actor, critics, models (evaluation,
  // expert term) and the actor on the fvp_rows states (with its input fX and the tangent fT of J x)
  float *aH[MAXH] = {}, *daH[MAXH] = {}, *cH[MAXH] = {}, *cdH[MAXH] = {}, *mH[MAXH] = {}, *mdH[MAXH] = {};
  float *fX = nullptr, *fH[MAXH] = {}, *fdH[MAXH] = {}, *fT[MAXH] = {};
  cudaStream_t s2 = nullptr, s3 = nullptr, s4 = nullptr;      // s3 / s4: the three independent weight-gradient GEMMs of a backward pass side by side
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_g = nullptr, ev_g3 = nullptr, ev_g4 = nullptr;
  // saceo_update_host_async: the H2D copies of step t+1 ride a copy stream into one of two device staging sets while step
  // t computes; the update stream then only does device-to-device copies into the bound tables
  cudaStream_t sc = nullptr;
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
  char* hstage[2] = {nullptr, nullptr};
  bool hstage_used[2] = {false, false};
  int hslot = 0;
  FitCtx fit;             // dynamics-model fitting (saceo_fit_bind)
  NetD fit_rnet{};        // its reward nets (separate_reward_nn)
  float *fit_H[MAXH] = {}, *fit_dH[MAXH] = {}, *fit_rH[MAXH] = {}, *fit_rdH[MAXH] = {};   // per-layer H / dH of both
  bool fit_bound = false;
  void* fit_ws = nullptr;
  long long launches = 0;
  // per-launch CUDA-event profile of one un-graphed step (saceo_profile_step)
  bool prof = false;
  std::vector<cudaEvent_t> prof_ev;
  std::vector<const char*> prof_name;
  size_t prof_n = 0;
  BwdVariant bwd_variant{-1, -1, -1};   // profiling mode: the k_mlp_bwd_ws instantiation of the last fused backward launch
  cudaGraphExec_t graph[3][2] = {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}};   // [rng mode][polyak]
  long long graph_nodes[3][2] = {{0, 0}, {0, 0}, {0, 0}};
};

// every kernel launch site reports here: launch counter + (profiling mode) an event right after the launch
static inline void count_launch(saceo_ctx* x, const char* name, cudaStream_t st) {
  x->launches++;
  if (!x->prof) return;
  if (x->prof_n == x->prof_ev.size()) {
    cudaEvent_t e; cudaEventCreate(&e);
    x->prof_ev.push_back(e); x->prof_name.push_back(name);
  }
  x->prof_name[x->prof_n] = name;
  cudaEventRecord(x->prof_ev[x->prof_n++], st);
}
#define LAUNCH(ctx, kern, grid, block, smem, st, ...) do { \
  kern<<<grid, block, smem, st>>>(__VA_ARGS__); count_launch((ctx), #kern, st); } while (0)

// ------------------------------------------------------------------------------------------
// layout
// ------------------------------------------------------------------------------------------
static int validate(const saceo_config* c) {
  if (!c) return fail(SACEO_E_INVALID, "null config");
  if (c->abi_version != SACEO_ABI_VERSION) return fail(SACEO_E_INVALID, "abi_version %d != %d", c->abi_version, SACEO_ABI_VERSION);
  if (c->n_agents < 1 || c->n_agents > 32000) return fail(SACEO_E_INVALID, "n_agents out of range");
  if (c->S < 1 || c->A < 1 || c->B < 1) return fail(SACEO_E_INVALID, "S, A, B must be positive");
  if (c->model_layers < 1 || c->model_layers > MAXH)
    return fail(SACEO_E_INVALID, "model_layers must be in [1, %d] (got %d)", MAXH, c->model_layers);
  for (int i = 0; i < 2; ++i) {
    if (c->actor_hidden[i] < 1 || c->critic_hidden[i] < 1) return fail(SACEO_E_INVALID, "hidden sizes must be positive");
    if (c->actor_act[i] < 0 || c->actor_act[i] > 2 || c->critic_act[i] < 0 || c->critic_act[i] > 2)
      return fail(SACEO_E_INVALID, "activations must be tanh, relu or elu");   // nn_utils.py:18
  }
  for (int i = 0; i < c->model_layers; ++i)
    if (c->model_act[i] < 0 || c->model_act[i] > 2) return fail(SACEO_E_INVALID, "activations must be tanh, relu or elu");
  if (c->num_models < 0 || c->num_models > 2) return fail(SACEO_E_INVALID, "num_models must be 0, 1 or 2 (only models[0..1] are used, SAC_expert.py:325-326)");
  if (c->num_models > 0) {
    if (c->E < 1) return fail(SACEO_E_INVALID, "E must be positive for SAC-EO");
    if (c->num_models == 2 && (c->E & 1)) return fail(SACEO_E_INVALID, "E must be even with two models (unequal array_split halves cannot be added, SAC_expert.py:329-332)");
    for (int i = 0; i < c->model_layers; ++i)
      if (c->model_hidden[i] < 1) return fail(SACEO_E_INVALID, "model hidden sizes must be positive (layer %d: %d)", i, c->model_hidden[i]);
  }
  if (c->target_update_int < 1) return fail(SACEO_E_INVALID, "target_update_int must be >= 1");
  if (c->replay_capacity < 1) return fail(SACEO_E_INVALID, "replay_capacity must be >= 1");
  if (c->gemm_mode != SACEO_GEMM_FP32_SIMT && c->gemm_mode != SACEO_GEMM_TCGEN05_BF16X3)
    return fail(SACEO_E_INVALID, "unknown gemm_mode");
  if (c->reserved[3] || c->reserved[4] || c->reserved[7]) return fail(SACEO_E_INVALID, "reserved[3], [4] and [7] must be 0");
  return 0;
}

struct Bump {   // workspace carver (also used dry to size it)
  char* base; long long off = 0;
  std::map<std::string, std::pair<void*, long long>>* names;
  template <typename T> T* get(const char* name, long long count) {
    off = rup(off, 256);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    long long bytes = count * (long long)sizeof(T);
    if (names && base) (*names)[name] = {p, bytes};
    off += bytes;
    return p;
  }
  // one buffer of `rows` rows per hidden layer l of net n, named <name><l+1>; down: from the last layer to the first
  void layers(float** H, const char* name, const NetD& n, long long rows, bool down = false) {
    char nm[24];
    for (int i = 0; i < n.nh; ++i) {
      const int l = down ? n.nh - 1 - i : i;
      snprintf(nm, sizeof(nm), "%s%d", name, l + 1);
      H[l] = get<float>(nm, rows * n.N(l));
    }
  }
};

static void fill_layout(const saceo_config* c, saceo_layout* L) {
  memset(L, 0, sizeof(*L));
  const int S = c->S, A = c->A;
  const NetD an = actor_desc(*c), mn = model_desc(*c);
  L->Ao = an.out;
  L->model_out = mn.out;
  L->na = actor_params(an, c->per_state_std);
  L->nc = critic_desc(*c).n();
  L->nm = c->num_models > 0 ? mn.n() : 0;
  L->na_stride = rup(L->na + 1, 32);   // last padded word carries g_alpha in the grad buffer
  L->nc_stride = rup(L->nc, 32);
  L->nm_stride = rup(L->nm > 0 ? L->nm : 1, 32);
  L->off_s = 0; L->off_a = S; L->off_sp = S + A; L->off_r = 2 * S + A;
  L->off_d = (int)rup(2 * S + A + 1, 2);
  L->row_words = (int)rup(L->off_d + 2, 4);
  int o = 0;
  L->off_s_mean = o; o += S; L->off_s_std = o; o += S;
  L->off_a_mean = o; o += A; L->off_a_std = o; o += A;
  L->off_ret_std = o; o += 1;
  L->off_m_s_mean = o; o += S; L->off_m_s_std = o; o += S;
  L->off_m_a_mean = o; o += A; L->off_m_a_std = o; o += A;
  L->off_m_d_mean = o; o += S; L->off_m_d_std = o; o += S;
  L->off_act_limit = o; o += A;
  L->norm_stride = (int)rup(o, 4);
  L->hyper_stride = 8;
  L->n_losses = 8;
}

static void decode_switches(saceo_ctx* x) {
  const saceo_config& c = x->cfg;
  x->tc = c.gemm_mode == SACEO_GEMM_TCGEN05_BF16X3;
  x->tc_variant = c.reserved[0];
  x->fuse_fwd = x->tc && c.reserved[1] == 0;
  x->fuse_bwd = x->tc && c.reserved[2] == 0;
  x->ws_kernels = x->tc && c.reserved[5] == 0;
  x->fork = c.reserved[6] == 0;
}

static void carve(saceo_ctx* x, char* base) {
  const saceo_config& c = x->cfg; const saceo_layout& L = x->L;
  KCtx& k = x->k;
  Bump b{base, 0, base ? &x->names : nullptr};
  const long long n = c.n_agents;
  const int S = c.S, A = c.A, B = c.B, E = c.num_models > 0 ? c.E : 0, R = (int)rup(B + E, 32);   // padded row stride
  const int SA = S + A;
  const NetD an = actor_desc(c), cn = critic_desc(c);
  NetD mn = model_desc(c);
  if (c.num_models == 0) for (int l = 0; l < mn.nh; ++l) mn.hw[l] = 1;   // no models: one-float placeholders
  k.idx = b.get<long long>("idx", n * B);
  k.noise = b.get<float>("noise", n * (3LL * B + E) * A);
  k.perm = b.get<int>("perm", n * (E > 0 ? E : 1));
  k.mb_s = b.get<float>("mb_s", n * B * S);   k.mb_a = b.get<float>("mb_a", n * B * A);
  k.mb_sp = b.get<float>("mb_sp", n * B * S); k.mb_r = b.get<float>("mb_r", n * B);
  k.mb_omd = b.get<float>("mb_omd", n * B);
  k.Xpi = b.get<float>("Xpi", n * R * rup(S, 4));
  b.layers(x->aH, "aH", an, n * R);
  k.aOut = b.get<float>("aOut", n * R * L.Ao);             k.daOut = b.get<float>("daOut", n * R * L.Ao);
  b.layers(x->daH, "daH", an, n * R, true);
  k.dls = b.get<float>("dls", n * R * A);
  k.Xc = b.get<float>("Xc", n * B * rup(SA, 4));
  k.Xc2 = b.get<float>("Xc2", n * B * rup(SA, 4));
  x->Xc3 = k.Xc3 = b.get<float>("Xc3", n * B * rup(SA, 4));
  x->Xpi2 = b.get<float>("Xpi2", n * R * rup(S, 4));
  x->aOut2 = b.get<float>("aOut2", n * R * L.Ao);
  x->nlp2 = b.get<float>("nlp2", n * R);
  b.layers(x->cH, "cH", cn, n * 2 * B);
  k.cQ = b.get<float>("cQ", n * 2 * B);                          k.cdQ = b.get<float>("cdQ", n * 2 * B);
  b.layers(x->cdH, "cdH", cn, n * 2 * B, true);
  k.cdXa = b.get<float>("cdXa", n * 2 * B * A);
  const long long e1 = E > 0 ? E : 1;
  k.Xm = b.get<float>("Xm", n * 2 * e1 * SA);
  b.layers(x->mH, "mH", mn, n * 2 * e1);
  k.mOut = b.get<float>("mOut", n * 2 * e1 * L.model_out); k.mdOut = b.get<float>("mdOut", n * 2 * e1 * S);
  b.layers(x->mdH, "mdH", mn, n * 2 * e1, true);
  k.mdXa = b.get<float>("mdXa", n * 2 * e1 * A);
  k.y = b.get<float>("y", n * B);  k.nlp = b.get<float>("nlp", n * R);
  k.g_q = b.get<float>("g_q", n * 2 * L.nc_stride);
  k.g_actor = b.get<float>("g_actor", n * L.na_stride);
  k.lrt = b.get<float>("lrt", n * 4);
  k.losses = b.get<float>("losses", n * L.n_losses);
  k.mse_part = b.get<float>("mse_part", n * 2);
  {   // sized for the largest fused-backward caller: the update (R rows) and the Fisher-vector / TRPO / PPO paths (fvp_rows)
    long long rmax = R > B ? R : B;
    if (c.fvp_rows > rmax) rmax = c.fvp_rows;
    x->dbpart_cap = n * 2 * cdiv(rmax, TC_BM) * 2 * FW_H;
    x->dbpart = b.get<float>("dbpart", x->dbpart_cap);
  }
  k.step_ctr = b.get<unsigned long long>("step_ctr", 2);
  x->pl_actor = x->pl_q = x->pl_qt = nullptr;
  x->aH1p = x->adH2p = x->cH1p = x->cdH2p = x->adH1p = x->cdH1p = nullptr;
  x->a_img = (long long)(R / 32) * WS_STAGE; x->c_img = (long long)(rup(B, 32) / 32) * WS_STAGE;
  if (x->ws_kernels) {   // plane images only for the nets the fused kernels take
    if (an.ws()) {
      x->pl_actor = b.get<uint8_t>("pl_actor", n * ws_image_bytes(S, L.Ao));
      x->aH1p = b.get<uint8_t>("aH1p", n * x->a_img); x->adH2p = b.get<uint8_t>("adH2p", n * x->a_img);
      x->adH1p = b.get<uint8_t>("adH1p", n * x->a_img);
    }
    if (cn.ws()) {
      x->pl_q = b.get<uint8_t>("pl_q", n * 2 * ws_image_bytes(SA, 1));
      x->pl_qt = b.get<uint8_t>("pl_qt", n * 2 * ws_image_bytes(SA, 1));
      x->cH1p = b.get<uint8_t>("cH1p", n * 2 * x->c_img); x->cdH2p = b.get<uint8_t>("cdH2p", n * 2 * x->c_img);
      x->cdH1p = b.get<uint8_t>("cdH1p", n * 2 * x->c_img);
    }
  }
  x->idx_stage = b.get<long long>("idx_stage", n * B);
  // Fisher-vector / CG workspace
  FvpWs& f = x->f;
  const long long N = c.fvp_rows;
  f.N = (int)N;
  if (N > 0) {
    x->fX = b.get<float>("fX", n * N * S);
    b.layers(x->fH, "fH", an, n * N);
    f.Out = b.get<float>("fOut", n * N * L.Ao);
    b.layers(x->fT, "fT", an, n * N);
    f.Tmp = b.get<float>("fTmp", n * N * an.widest(1));   // T[l-1].W_l of every layer l >= 1 (fvp_apply)
    f.TOut = b.get<float>("fTOut", n * N * L.Ao);
    f.G = b.get<float>("fG", n * N * L.Ao);
    b.layers(x->fdH, "fdH", an, n * N, true);
    f.gls = b.get<float>("fgls", n * N * A);
    f.p = b.get<float>("cg_p", n * L.na_stride); f.r = b.get<float>("cg_r", n * L.na_stride);
    f.z = b.get<float>("cg_z", n * L.na_stride); f.x = b.get<float>("cg_x", n * L.na_stride);
    f.sc = b.get<float>("cg_sc", n * 8);
  }
  x->ws_bytes = rup(b.off, 256);
}

extern "C" int saceo_query_layout(const saceo_config* cfg, saceo_layout* out) {
  int rc = validate(cfg); if (rc) return rc;
  if (!out) return fail(SACEO_E_INVALID, "null out");
  fill_layout(cfg, out);
  saceo_ctx tmp; tmp.cfg = *cfg; tmp.L = *out;
  decode_switches(&tmp);
  carve(&tmp, nullptr);
  out->workspace_bytes = tmp.ws_bytes;
  return 0;
}

extern "C" int saceo_abi_version(void) { return SACEO_ABI_VERSION; }
extern "C" const char* saceo_last_error(void) { return g_err; }

static int create_fill(saceo_ctx* x, const saceo_config* cfg);
extern "C" int saceo_destroy(saceo_ctx* x);

extern "C" int saceo_create(const saceo_config* cfg, saceo_ctx** out) {
  int rc = validate(cfg); if (rc) return rc;
  if (!out) return fail(SACEO_E_INVALID, "null out");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(SACEO_E_NODEVICE, "no CUDA device: libsaceo has no CPU fallback");
  }
  if (cfg->device < 0 || cfg->device >= ndev) return fail(SACEO_E_INVALID, "device %d out of range", cfg->device);
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return fail(SACEO_E_NODEVICE, "device %d is sm_%d%d; libsaceo is built for sm_100a only", cfg->device, prop.major, prop.minor);
  CU(cudaSetDevice(cfg->device));
  saceo_ctx* x = new saceo_ctx();
  rc = create_fill(x, cfg);
  if (rc) { saceo_destroy(x); return rc; }     // nothing of a half-built context leaks
  *out = x;
  return 0;
}

static int create_fill(saceo_ctx* x, const saceo_config* cfg) {
  x->cfg = *cfg;
  decode_switches(x);
  fill_layout(cfg, &x->L);
  memset(&x->k, 0, sizeof(KCtx)); memset(&x->f, 0, sizeof(FvpWs)); memset(&x->fit, 0, sizeof(FitCtx));
  carve(x, nullptr);
  x->L.workspace_bytes = x->ws_bytes;
  if (cudaMalloc(&x->ws, (size_t)x->ws_bytes) != cudaSuccess) {
    cudaGetLastError(); x->ws = nullptr;
    return fail(SACEO_E_NOMEM, "cudaMalloc of %lld workspace bytes failed", (long long)x->ws_bytes);
  }
  CU(cudaMemset(x->ws, 0, (size_t)x->ws_bytes));
  carve(x, (char*)x->ws);
  KCtx& k = x->k;
  k.n_agents = cfg->n_agents; k.S = cfg->S; k.A = cfg->A; k.Ao = x->L.Ao; k.mo = x->L.model_out;
  k.B = cfg->B; k.E = cfg->num_models > 0 ? cfg->E : 0; k.R = k.B + k.E; k.Rs = (int)rup(k.R, 32); k.nmod = cfg->num_models;
  k.ldXc = (int)rup(cfg->S + cfg->A, 4); k.ldXp = (int)rup(cfg->S, 4);
  k.per_state_std = cfg->per_state_std; k.sep_reward = cfg->separate_reward_nn;
  k.mnh = cfg->model_layers; k.mh1 = cfg->model_hidden[0]; k.mh2 = cfg->model_hidden[1];
  k.mact0 = cfg->model_act[0]; k.mact1 = cfg->model_act[1];
  k.delta_clip = cfg->delta_clip_pred; k.cap = cfg->replay_capacity; k.L = x->L; k.eps_force = -1.f;
  // identity expert permutation until draws are injected / generated
  if (k.E > 0) {
    std::vector<int> pm((size_t)cfg->n_agents * k.E);
    for (int a = 0; a < cfg->n_agents; ++a) for (int i = 0; i < k.E; ++i) pm[(size_t)a * k.E + i] = i;
    CU(cudaMemcpy(k.perm, pm.data(), pm.size() * sizeof(int), cudaMemcpyHostToDevice));
  }
  CU(cudaStreamCreateWithFlags(&x->s2, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&x->ev_fork, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&x->ev_join, cudaEventDisableTiming));
  CU(cudaStreamCreateWithFlags(&x->s3, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&x->s4, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&x->ev_g, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&x->ev_g3, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&x->ev_g4, cudaEventDisableTiming));
  CU(tc_gemm_init());
  CU(mlp_ws_init());
  CU(model_term_init());
  return 0;
}

extern "C" int saceo_destroy(saceo_ctx* x) {
  if (!x) return 0;
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 2; ++j) if (x->graph[i][j]) cudaGraphExecDestroy(x->graph[i][j]);
  if (x->ws) cudaFree(x->ws);
  if (x->fit_ws) cudaFree(x->fit_ws);
  if (x->s2) cudaStreamDestroy(x->s2);
  if (x->ev_fork) cudaEventDestroy(x->ev_fork);
  if (x->ev_join) cudaEventDestroy(x->ev_join);
  if (x->s3) cudaStreamDestroy(x->s3);
  if (x->s4) cudaStreamDestroy(x->s4);
  if (x->sc) cudaStreamDestroy(x->sc);
  for (int i = 0; i < 2; ++i) {
    if (x->ev_h2d[i]) cudaEventDestroy(x->ev_h2d[i]);
    if (x->ev_free[i]) cudaEventDestroy(x->ev_free[i]);
    if (x->hstage[i]) cudaFree(x->hstage[i]);
  }
  for (cudaEvent_t e : {x->ev_g, x->ev_g3, x->ev_g4}) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : x->prof_ev) cudaEventDestroy(e);
  delete x;
  return 0;
}

extern "C" int saceo_bind(saceo_ctx* x, const saceo_tables* t) {
  if (!x || !t) return fail(SACEO_E_INVALID, "null argument");
  if (!t->actor || !t->actor_m || !t->actor_v || !t->q || !t->q_m || !t->q_v || !t->qt || !t->alpha ||
      !t->alpha_m || !t->alpha_v || !t->adam_t || !t->norm || !t->hyper)
    return fail(SACEO_E_INVALID, "a required table pointer is NULL");
  if (x->cfg.num_models > 0 && (!t->model || !t->expert_s || !t->expert_sp))
    return fail(SACEO_E_INVALID, "SAC-EO needs model, expert_s and expert_sp tables");
  x->k.T = *t;
  x->k.expert_s = t->expert_s; x->k.expert_sp = t->expert_sp;
  x->bound = true;
  x->planes_dirty = 3;
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 2; ++j)
    if (x->graph[i][j]) { cudaGraphExecDestroy(x->graph[i][j]); x->graph[i][j] = nullptr; }
  return 0;
}

extern "C" void* saceo_debug_ptr(saceo_ctx* x, const char* name, int64_t* bytes_out) {
  if (!x || !name) return nullptr;
  auto it = x->names.find(name);
  if (it == x->names.end()) return nullptr;
  if (bytes_out) *bytes_out = it->second.second;
  return it->second.first;
}
extern "C" int64_t saceo_launch_count(const saceo_ctx* x) { return x ? x->launches : 0; }

// The fp16 hi/lo weight-plane images follow the fp32 tables: k_adam keeps them current for everything the library
// itself updates; after a bind or an external write (saceo_weights_changed) they are rebuilt before the next use.
extern "C" int saceo_weights_changed(saceo_ctx* x) {
  if (!x) return fail(SACEO_E_INVALID, "null ctx");
  x->planes_dirty = 3;
  return 0;
}
// the images of `nets` consecutive nets with K0 inputs and nout outputs, net i's fp32 table at theta + i * stride
// (maintenance: not counted as a launch of the step)
static void planes_build(const float* theta, long long stride, uint8_t* img, int K0, int nout, int nets, cudaStream_t st) {
  const int items = (((K0 + 31) / 32) * 32 + 256 + ws_w2_rows(nout)) * 32;
  k_planes_build<<<dim3(cdiv(items, 256), nets), 256, 0, st>>>(theta, stride, img, K0, nout);
}
static int ensure_planes(saceo_ctx* x, cudaStream_t st) {
  if (!x->planes_dirty || !x->bound) return 0;
  const saceo_config& c = x->cfg; const int n = c.n_agents;
  if (x->pl_actor && (x->planes_dirty & 1)) planes_build(x->k.T.actor, x->L.na_stride, x->pl_actor, c.S, x->L.Ao, n, st);
  if (x->pl_q && (x->planes_dirty & 2)) {
    planes_build(x->k.T.q, x->L.nc_stride, x->pl_q, c.S + c.A, 1, 2 * n, st);
    planes_build(x->k.T.qt, x->L.nc_stride, x->pl_qt, c.S + c.A, 1, 2 * n, st);
  }
  x->planes_dirty = 0;
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) return fail(SACEO_E_CUDA, "plane build failed: %s", cudaGetErrorString(e));
  return 0;
}

static unsigned long long* g_ws_dbg = nullptr;
static int g_ws_sel = 0, g_ws_count = 0;      // test-only: which warp-specialised launch (ordinal since the last set) stamps its phases

// ------------------------------------------------------------------------------------------
// GEMM dispatch
// ------------------------------------------------------------------------------------------
static void simt_launch(bool TA, bool TB, bool ONES, const GemmP& p, int nagents, cudaStream_t st) {
  dim3 grid(cdiv(p.N, SG_BN), cdiv(p.M - p.m_off, SG_BM), nagents * p.nnet), block(SG_THREADS);
  if (!TA && !TB) k_gemm_simt<false, false, false><<<grid, block, 0, st>>>(p);
  else if (!TA && TB) k_gemm_simt<false, true, false><<<grid, block, 0, st>>>(p);
  else if (TA && !TB && ONES) k_gemm_simt<true, false, true><<<grid, block, 0, st>>>(p);
  else if (TA && !TB) k_gemm_simt<true, false, false><<<grid, block, 0, st>>>(p);
  else k_gemm_simt<true, true, false><<<grid, block, 0, st>>>(p);
}

// Engine choice per GEMM: tensor cores for 128-row tiles of wide layers, the skinny kernel when one
// output dimension is <= 32 (expert rows, heads, bias rows, row tails), the tiled SIMT kernel otherwise.
static int gemm(saceo_ctx* x, bool TA, bool TB, bool ONES, const GemmP& p, int nagents, cudaStream_t st) {
  if (p.M <= 0 || p.N <= 0 || p.K <= 0) return 0;
  int row0 = 0;
  if (x->tc && tc_gemm_eligible(TA, TB, ONES, p)) {
    if (tc_gemm_launch(TA, TB, ONES, p, nagents, x->tc_variant, st) < 0) return fail(SACEO_E_CUDA, "tcgen05 gemm launch failed");
    count_launch(x, "k_gemm_tc", st);
    row0 = tc_rows(ONES, p);
    if (row0 >= p.M) return 0;
  }
  if (p.M - row0 <= 32) {
    skinny_launch(skinny_rows(TA, TB, ONES, p, row0), nagents, st);
  } else if (p.M - row0 <= 64 && p.N > 32) {          // e.g. [dW0; db0] with S+A+1 = 36 rows: two 32-row passes
    SkinnyP s1 = skinny_rows(TA, TB, ONES, p, row0); s1.Ms = row0 + 32;
    skinny_launch(s1, nagents, st);
    count_launch(x, "k_gemm_skinny", st);
    skinny_launch(skinny_rows(TA, TB, ONES, p, row0 + 32), nagents, st);
  } else if (row0 == 0 && p.N <= 32) {
    skinny_launch(skinny_cols(TA, TB, ONES, p), nagents, st);
  } else {
    GemmP t = p; t.m_off = row0;
    simt_launch(TA, TB, ONES, t, nagents, st);
    count_launch(x, "k_gemm_simt", st);
    return 0;
  }
  count_launch(x, "k_gemm_skinny", st);
  return 0;
}

// One pass of one net population: what its forward and its backward call share.  The plane images are set only
// when the backward pass takes the plane path (fused chain + column-sum biases + k_dw_planes); the forward pass then
// writes h1 ONLY as a plane image, so both calls must see the same pass.
struct Pass {
  NetD n;
  const float* X; int ldx; long long sXa, sXn;        // input rows
  int rows; long long rowsAllocH;                      // rows of the pass / rows per net allocated in H, dH
  float* const* H;                                     // saved activation of each hidden layer
  float* const* dH;                                    // its gradient (backward)
  // bf16 hi/lo plane images of h1 / dH2 / dH1, rup(rows, 32) rows each.  The kernels write rows [0, rows) only, while
  // k_dw_planes / k_dw0_planes contract over whole 32-row slabs: rows [rows, rup(rows, 32)) must hold zeros (the
  // workspace is cleared at creation and nothing writes those rows afterwards).  A pass with images keeps h1 only as
  // its image, so its backward must be one the fused kernel takes: mlp_backward refuses any other
  uint8_t *H1p = nullptr, *dH2p = nullptr, *dH1p = nullptr;
  long long sQa = 0, sQn = 0;                          // their bytes per agent / net
  // the caller guarantees that rows [rows, rowsAllocH) of X, H, dOut, dH are zero, so the
  // weight-gradient contractions may run over a row count rounded up to the 32-row slabs of the streaming kernel
  bool kpad = false;
  int hnets = 0;        // nets per agent the activation buffers H, dH are laid out for (0: n.nnet)
  int dout_cols = 0;    // columns of dOut that flow back into the last hidden layer's dH (0: n.out)
  bool fwd_f16 = true;  // forward operands are O(1): the GEMM chain splits them into fp16 planes (tc_gemm.cuh split8), else bf16
  long long sHa(int w) const { return (long long)(hnets ? hnets : n.nnet) * rowsAllocH * w; }   // agent / net strides of
  long long sHn(int w) const { return rowsAllocH * w; }                                          // a w-wide activation
  int kout() const { return dout_cols ? dout_cols : n.out; }
};

// forward through one population of MLPs (nn_utils.py:101-136), unfused: one GEMM per layer
static int mlp_forward_unfused(saceo_ctx* x, const Pass& ps, float* Out, int ldo, long long sOa, long long sOn, cudaStream_t st) {
  const NetD& n = ps.n;
  const float* A = ps.X; int lda = ps.ldx; long long sAa = ps.sXa, sAn = ps.sXn;
  for (int l = 0; l <= n.nh; ++l) {
    GemmP p{}; p.nnet = n.nnet; p.f16 = ps.fwd_f16;
    p.A = A; p.lda = lda; p.sAa = sAa; p.sAn = sAn;
    p.B = n.theta + n.oW(l); p.ldb = n.N(l); p.sBa = n.sa; p.sBn = n.sn;
    p.bias = n.theta + n.ob(l); p.sba = n.sa; p.sbn = n.sn;
    if (l < n.nh) { p.C = ps.H[l]; p.ldc = n.N(l); p.sCa = ps.sHa(n.N(l)); p.sCn = ps.sHn(n.N(l)); }
    else { p.C = Out; p.ldc = ldo; p.sCa = sOa; p.sCn = sOn; }
    p.M = ps.rows; p.N = n.N(l); p.K = n.K(l); p.epi = l < n.nh ? EPI_ACT : EPI_NONE; p.act = n.act(l);
    int rc = gemm(x, false, false, false, p, x->cfg.n_agents, st); if (rc) return rc;
    A = p.C; lda = p.ldc; sAa = p.sCa; sAn = p.sCn;
  }
  return 0;
}

// whether mlp_forward runs net n in k_mlp_fwd_ws, which writes no hidden activation unless asked to (save_h)
static bool fwd_ws(const saceo_ctx* x, const NetD& n) { return n.planes && x->fuse_fwd && n.ws(); }

// Forward pass dispatcher: nets with a weight-plane image go through the warp-specialised fused kernel (activations
// stay in TMEM between layers; h1/h2 reach HBM only when save_h), every other net through the GEMM chain.
static int mlp_forward(saceo_ctx* x, const Pass& ps, float* Out, int ldo, long long sOa, long long sOn, cudaStream_t st,
                       bool save_h = true) {
  const NetD& n = ps.n;
  if (fwd_ws(x, n)) {
    // warp-specialised kernel on the TMA-fed weight planes: every row (partial tiles are masked)
    FwdW f{};
    f.X = ps.X; f.ldx = ps.ldx; f.sXa = ps.sXa; f.sXn = ps.sXn;
    f.theta = n.theta; f.sTa = n.sa; f.sTn = n.sn;
    f.planes = n.planes; f.sPa = n.pa; f.sPn = n.pn;
    f.H1 = save_h ? ps.H[0] : nullptr; f.H2 = save_h ? ps.H[1] : nullptr; f.sHa = ps.sHa(n.N(0)); f.sHn = ps.sHn(n.N(0));
    f.H1p = save_h ? ps.H1p : nullptr; f.sQa = ps.sQa; f.sQn = ps.sQn;
    f.Out = Out; f.ldo = ldo; f.sOa = sOa; f.sOn = sOn;
    f.rows = ps.rows; f.K0 = n.in; f.nout = n.out; f.nnet = n.nnet; f.act0 = n.act(0); f.act1 = n.act(1);
    f.dbg = (g_ws_dbg && g_ws_count++ == g_ws_sel) ? g_ws_dbg : nullptr;
    if (mlp_fwd_ws_launch(f, x->cfg.n_agents, st) != cudaSuccess) return fail(SACEO_E_CUDA, "fused forward launch failed");
    count_launch(x, "k_mlp_fwd_ws", st);
    return 0;
  }
  return mlp_forward_unfused(x, ps, Out, ldo, sOa, sOn, st);
}

// The fused backward kernels index dbpart as [agent*nnet+net][tile][2][256]: callers with more row tiles than the
// workspace was sized for (e.g. model fitting with 256-wide models and a large minibatch) take the ones-row bias path.
static bool dbpart_fits(const saceo_ctx* x, const NetD& n, int rows) {
  return x->dbpart && (long long)x->cfg.n_agents * n.nnet * cdiv(rows, TC_BM) * 2 * FW_H <= x->dbpart_cap;
}

// What a fused backward kernel has done before the per-layer loop runs.
struct BwdFused {
  bool chain = false;        // dH2, dH1 and dXa
  bool bias = false;         // db1 and db0, from the kernel's column sums (k_bias_finish)
  bool dw1_planes = false;   // dH2 left as planes only: dW1 from the plane images (k_dw_planes)
  bool dw0_planes = false;   // dH1 left as planes only: dW0 from the dH1 plane image (k_dw0_planes)
};

// Backward through the layers, from the output layer down to layer 0, of whatever the fused chain left: per layer the
// weight gradient (grads) and, without the fused chain, the input gradient (the hidden layers' dH, then the dXa columns).
static int mlp_backward_layers(saceo_ctx* x, const Pass& ps, const float* dOut, int ldd, long long sDa, long long sDn,
                               float* grads, float* dXa, int A_cols, long long sXaA, long long sXaN, const BwdFused& fz,
                               cudaStream_t st) {
  const NetD& n = ps.n;
  const int na = x->cfg.n_agents, nh = n.nh;
  const int krows = (ps.kpad && rup(ps.rows, 32) <= ps.rowsAllocH) ? (int)rup(ps.rows, 32) : ps.rows;
  // activation i (X, then the hidden layers' H) and its gradient D[i] (the hidden layers' dH, then dOut for i = nh + 1);
  // H_i and dH_i share ld and strides
  const float* Act[MAXH + 1]; const float* D[MAXH + 2]; float* dH[MAXH + 1];
  int ld[MAXH + 2]; long long sa[MAXH + 2], sn[MAXH + 2];
  Act[0] = ps.X; D[0] = nullptr; dH[0] = nullptr; ld[0] = ps.ldx; sa[0] = ps.sXa; sn[0] = ps.sXn;
  for (int i = 1; i <= nh; ++i) {
    Act[i] = ps.H[i - 1]; D[i] = dH[i] = ps.dH[i - 1];
    ld[i] = n.N(i - 1); sa[i] = ps.sHa(ld[i]); sn[i] = ps.sHn(ld[i]);
  }
  D[nh + 1] = dOut; ld[nh + 1] = ldd; sa[nh + 1] = sDa; sn[nh + 1] = sDn;
  // the three weight-gradient GEMMs are independent of each other: with the fused chain they fan out over three streams
  // (captured into the graph as parallel branches) - at small populations each is one under-filled, latency-bound wave
  const bool fan = fz.chain && grads && x->fork && !x->prof && x->s3 && x->s4;
  cudaStream_t wst[MAXH + 1];            // stream of each layer's dW
  for (int l = 0; l <= nh; ++l) wst[l] = st;
  if (fan) {                             // fz.chain: two hidden layers
    CU(cudaEventRecord(x->ev_g, st));
    CU(cudaStreamWaitEvent(x->s3, x->ev_g, 0)); CU(cudaStreamWaitEvent(x->s4, x->ev_g, 0));
    wst[2] = x->s3; wst[0] = x->s4;
  }
  int rc;
  for (int l = nh; l >= 0; --l) {
    if (grads && l == 1 && fz.dw1_planes) {   // dW1 = H1^T . dH2 from the plane images
      DwP d{};
      d.Ap = ps.H1p; d.sAa = ps.sQa; d.sAn = ps.sQn; d.Bp = ps.dH2p; d.sBa = ps.sQa; d.sBn = ps.sQn;
      d.G = grads + n.oW(l); d.sGa = n.sa; d.sGn = n.sn; d.rows = ps.rows; d.nnet = n.nnet;
      k_dw_planes<<<na * n.nnet, WS_NT, DW_BYTES, wst[1]>>>(d);
      count_launch(x, "k_dw_planes", wst[1]);
    } else if (grads && l == 0 && fz.dw0_planes) {   // dW0 = X^T . dH1 from the plane image
      Dw0P d{};
      d.X = ps.X; d.ldx = ps.ldx; d.sXa = ps.sXa; d.sXn = ps.sXn; d.Bp = ps.dH1p; d.sBa = ps.sQa; d.sBn = ps.sQn;
      d.G = grads + n.oW(l); d.sGa = n.sa; d.sGn = n.sn; d.rows = ps.rows; d.in = n.in; d.nnet = n.nnet;
      k_dw0_planes<<<na * n.nnet, WS_NT, DW0_BYTES, wst[0]>>>(d);
      count_launch(x, "k_dw0_planes", wst[0]);
    } else if (grads) {   // [dW_l; db_l] = [Act_l, 1]^T . D_l+1, without the ones row where the fused kernel formed db_l
      const bool ones = l == nh || !fz.bias;
      GemmP p{}; p.nnet = n.nnet;
      p.A = Act[l]; p.lda = ld[l]; p.sAa = sa[l]; p.sAn = sn[l];
      p.B = D[l + 1]; p.ldb = ld[l + 1]; p.sBa = sa[l + 1]; p.sBn = sn[l + 1];
      p.C = grads + n.oW(l); p.ldc = n.N(l); p.sCa = n.sa; p.sCn = n.sn;
      p.M = ones ? n.K(l) + 1 : n.K(l); p.N = n.N(l); p.K = krows; p.epi = EPI_NONE;
      rc = gemm(x, true, false, ones, p, na, wst[l]); if (rc) return rc;
    }
    if (l == 0 && fan) {
      CU(cudaEventRecord(x->ev_g3, x->s3)); CU(cudaEventRecord(x->ev_g4, x->s4));
      CU(cudaStreamWaitEvent(st, x->ev_g3, 0)); CU(cudaStreamWaitEvent(st, x->ev_g4, 0));
    }
    if (fz.chain || (l == 0 && !dXa)) continue;
    // l > 0: dH_l = (D_l+1 . W_l^T) * act_l-1'(H_l);  l = 0: dX[:, S:S+A] = D_1 . W0[S:S+A, :]^T
    GemmP p{}; p.nnet = n.nnet;
    p.A = D[l + 1]; p.lda = ld[l + 1]; p.sAa = sa[l + 1]; p.sAn = sn[l + 1];
    p.B = n.theta + n.oW(l); p.ldb = n.N(l); p.sBa = n.sa; p.sBn = n.sn;
    if (l > 0) {
      p.C = dH[l]; p.ldc = ld[l]; p.sCa = sa[l]; p.sCn = sn[l]; p.aux = Act[l];
      p.N = n.K(l); p.epi = EPI_MUL_DACT; p.act = n.act(l - 1);
    } else {
      p.B += (long long)(n.in - A_cols) * n.N(l);
      p.C = dXa; p.ldc = A_cols; p.sCa = sXaA; p.sCn = sXaN; p.N = A_cols; p.epi = EPI_NONE;
    }
    p.M = ps.rows; p.K = l == nh ? ps.kout() : n.N(l);
    rc = gemm(x, false, true, false, p, na, st); if (rc) return rc;
  }
  return 0;
}

// backward through the same MLPs.  grads (nullable): flat [W|b] blocks in the layout of theta, via the ones-row trick.
// dXa (nullable): gradient w.r.t. the last A_cols (action) columns of the input only (their rows of W0).
// The fused gradient chain (dH2, dH1, dXa) runs on tensor cores with the tile resident in TMEM where the warp-specialised
// kernel takes the pass; the per-layer loop does the rest.
static int mlp_backward(saceo_ctx* x, const Pass& ps, const float* dOut, int ldd, long long sDa, long long sDn,
                        float* grads, float* dXa, int A_cols, long long sXaA, long long sXaN, cudaStream_t st) {
  const NetD& n = ps.n;
  const int na = x->cfg.n_agents, rows = ps.rows, tiles = cdiv(rows, TC_BM);
  BwdFused fz;
  if (n.planes && x->fuse_bwd && n.ws() &&   // and the kernel has a variant for this pass's dOut width and dXa columns
      mlp_bwd_ws_eligible(n.N(0), n.N(1), ps.kout(), n.out, dXa != nullptr, A_cols, n.theta, n.sa, n.sn)) {
    float* dbpart = grads && dbpart_fits(x, n, rows) ? x->dbpart : nullptr;
    BwdW f{};
    f.dOut = dOut; f.ldd = ldd; f.sDa = sDa; f.sDn = sDn; f.kout = ps.kout();
    f.theta = n.theta; f.sTa = n.sa; f.sTn = n.sn; f.K0 = n.in; f.nout = n.out;
    f.planes = n.planes; f.sPa = n.pa; f.sPn = n.pn;
    f.H1 = ps.H[0]; f.H2 = ps.H[1]; f.sHa = ps.sHa(n.N(0)); f.sHn = ps.sHn(n.N(0));
    f.dH2 = grads ? ps.dH[1] : nullptr; f.dH1 = grads ? ps.dH[0] : nullptr;
    f.dXa = dXa; f.s_cols = n.in - A_cols; f.a_cols = A_cols; f.sXa = sXaA; f.sXn = sXaN;
    f.rows = rows; f.nnet = n.nnet; f.act0 = n.act(0); f.act1 = n.act(1); f.dbpart = dbpart;
    // on the plane path mlp_forward left h1 as its plane image only: read it there, with or without grads
    if (ps.H1p) { f.H1p = ps.H1p; f.sQa = ps.sQa; f.sQn = ps.sQn; }
    // hidden-to-hidden weight gradient from bf16 plane images (k_dw_planes): dH2 then leaves the kernel as planes only
    fz.dw1_planes = dbpart && ps.H1p;
    if (fz.dw1_planes) { f.dH2 = nullptr; f.dH2p = ps.dH2p; }
    // first-layer weight gradient from the dH1 plane image (k_dw0_planes): dH1 then leaves the kernel as planes only
    fz.dw0_planes = fz.dw1_planes && ps.dH1p && dw0_planes_eligible(n.in, rows, ps.ldx, ps.X, ps.sXa, ps.sXn);
    if (fz.dw0_planes) { f.dH1 = nullptr; f.dH1p = ps.dH1p; }
    f.dbg = (g_ws_dbg && g_ws_count++ == g_ws_sel) ? g_ws_dbg : nullptr;
    if (mlp_bwd_ws_launch(f, na, st) != cudaSuccess) return fail(SACEO_E_CUDA, "fused backward launch failed");
    count_launch(x, "k_mlp_bwd_ws", st);
    if (x->prof) x->bwd_variant = mlp_bwd_ws_variant(f);
    fz.chain = true;
    if (dbpart) {     // bias gradients of the two hidden layers come from the kernel's column sums
      k_bias_finish<<<na * n.nnet, 2 * FW_H, 0, st>>>(dbpart, tiles, grads, n.sa, n.sn, n.nnet, n.ob(1), n.ob(0));
      count_launch(x, "k_bias_finish", st);
      fz.bias = true;
    }
  }
  if (ps.H1p && !fz.chain)
    return fail(SACEO_E_INVALID, "pass on the plane path needs the fused backward (the GEMM chain cannot read the h1 image)");
  return mlp_backward_layers(x, ps, dOut, ldd, sDa, sDn, grads, dXa, A_cols, sXaA, sXaN, fz, st);
}

static NetD actor_net(const saceo_ctx* x) {
  NetD d = actor_desc(x->cfg);
  d.theta = x->k.T.actor; d.sa = x->L.na_stride;
  d.planes = x->pl_actor; d.pa = ws_image_bytes(d.in, d.out);
  return d;
}
static NetD critic_net(const saceo_ctx* x, bool target) {
  NetD d = critic_desc(x->cfg);
  d.theta = target ? x->k.T.qt : x->k.T.q; d.sa = 2 * x->L.nc_stride; d.sn = x->L.nc_stride;
  d.planes = target ? x->pl_qt : x->pl_q; d.pn = ws_image_bytes(d.in, 1); d.pa = 2 * d.pn;
  return d;
}
// the dynamics models (model_layers hidden layers) with parameters theta: the bound table, or the one being fitted
static NetD model_net(const saceo_ctx* x, const float* theta, int nnet) {
  NetD d = model_desc(x->cfg);
  d.theta = theta; d.sa = 2 * x->L.nm_stride; d.sn = x->L.nm_stride; d.nnet = nnet;
  return d;
}

// Gives a pass the plane images if mlp_backward(grads) of it takes the plane path (fused chain + column-sum biases +
// k_dw_planes); decided once, so that its forward and backward calls cannot disagree.  The images' rows
// [ps.rows, rup(ps.rows, 32)) must be zero (see Pass::H1p).
static void plane_path(const saceo_ctx* x, Pass& ps, uint8_t* H1p, uint8_t* dH2p, uint8_t* dH1p, long long sQa, long long sQn) {
  const NetD& n = ps.n;
  if (!n.planes || !x->fuse_bwd || !x->fuse_fwd || !H1p || !dH2p || !dbpart_fits(x, n, ps.rows) || !n.ws()) return;
  ps.H1p = H1p; ps.dH2p = dH2p; ps.dH1p = dH1p; ps.sQa = sQa; ps.sQn = sQn;
}

// the actor on the staged observation rows Xpi of view k: <= B rows (TD target, temperature, acting) or the E expert
// rows of the on-policy expert gradient
static Pass actor_pass(const saceo_ctx* x, const KCtx& k, int rows) {
  return Pass{actor_net(x), k.Xpi, k.ldXp, (long long)k.Rs * k.ldXp, 0, rows, k.Rs, x->aH, x->daH};
}
// the actor update over its R = B + E rows
static Pass actor_update_pass(const saceo_ctx* x, const KCtx& k) {
  Pass ps = actor_pass(x, k, k.R);
  ps.kpad = true;
  plane_path(x, ps, x->aH1p, x->adH2p, x->adH1p, x->a_img, 0);
  return ps;
}
// twin critics (or their targets) on the first `rows` of B critic input rows X (Xc, Xc2 or Xc3)
static Pass critic_pass(const saceo_ctx* x, bool target, const float* X, int rows) {
  const KCtx& k = x->k;
  return Pass{critic_net(x, target), X, k.ldXc, (long long)k.B * k.ldXc, 0, rows, k.B, x->cH, x->cdH};
}
// the critic update over the B minibatch rows
static Pass critic_update_pass(const saceo_ctx* x) {
  Pass ps = critic_pass(x, false, x->k.Xc2, x->k.B);
  plane_path(x, ps, x->cH1p, x->cdH2p, x->cdH1p, 2 * x->c_img, x->c_img);
  return ps;
}
// the actor on the fvp_rows states (Fisher-vector product, CG, TRPO / PPO surrogate)
static Pass fvp_pass(const saceo_ctx* x) {
  const KCtx& k = x->k; const FvpWs& f = x->f;
  return Pass{actor_net(x), x->fX, k.S, (long long)f.N * k.S, 0, f.N, f.N, x->fH, x->fdH};
}
// the models on the first `rows` of the E staged rows of Xm; every model reads net 0's block (zero net stride)
static Pass model_eval_pass(const saceo_ctx* x, int rows) {
  const KCtx& k = x->k; const int SA = k.S + k.A;
  return Pass{model_net(x, k.T.model, k.nmod), k.Xm, SA, 2LL * k.E * SA, 0, rows, k.E, x->mH, x->mdH};
}
// the k.nmod frozen models of view k, each on its share of the E staged expert rows of Xm (expert-observation term)
static Pass model_term_pass(const saceo_ctx* x, const KCtx& k) {
  const int SA = k.S + k.A;
  Pass ps{model_net(x, k.T.model, k.nmod), k.Xm, SA, 2LL * k.E * SA, (long long)k.E * SA, k.nmod == 2 ? k.E / 2 : k.E, k.E,
          x->mH, x->mdH};
  ps.hnets = 2;         // the model buffers are carved [agent][2][E rows] whatever nmod, as k_model_loss reads mOut / mdOut
  ps.dout_cols = k.S;   // k_model_loss writes the S state columns of mdOut: the reward output column gets no gradient
  ps.fwd_f16 = false;   // the expert term's forward keeps the bf16 planes it has always used and been tested with
  return ps;
}
// a model or reward net being fitted on the staged minibatch rows
static Pass fit_pass(const saceo_ctx* x, const NetD& n, float* const* H, float* const* dH) {
  const FitCtx& f = x->fit; const int SA = x->cfg.S + x->cfg.A;
  return Pass{n, f.X, SA, 2LL * f.mbs * SA, (long long)f.mbs * SA, f.mb, f.mbs, H, dH};
}

// ------------------------------------------------------------------------------------------
// update phases
// ------------------------------------------------------------------------------------------
static int check_launch() {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) return fail(SACEO_E_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
  return 0;
}

static int phase_gather(saceo_ctx* x, cudaStream_t st) {
  const KCtx& k = x->k;
  LAUNCH(x, k_gather, dim3(cdiv(k.B, 8), k.n_agents), 256, 0, st, k, k.idx, k.mb_s, k.mb_a, k.mb_sp, k.mb_r,
         (double*)nullptr, k.mb_omd, 1);      // + normalised critic-phase inputs (Xpi, Xc[:, :S], Xc2)
  return check_launch();
}

// phase 0: TD target + critic gradients
static int phase_critic_grads(saceo_ctx* x, cudaStream_t st) {
  const KCtx& k = x->k; const int n = k.n_agents, B = k.B, A = k.A;
  int rc;
  // inputs were staged by the gather: Xpi = N_s(sp), Xc = [N_s(sp) | .], Xc2 = [N_s(s) | N_a(a)]
  rc = mlp_forward(x, actor_pass(x, k, B), k.aOut, k.Ao, (long long)k.Rs * k.Ao, 0, st, false); if (rc) return rc;
  LAUNCH(x, k_head_fwd, dim3(cdiv(B, 128), n), 128, 0, st, k, B, B, k.noise, (3LL * B + k.E) * A, 0, 1,
         (float*)nullptr, (float*)nullptr, 0LL, 0);
  rc = mlp_forward(x, critic_pass(x, true, k.Xc, B), k.cQ, 1, 2LL * B, B, st, false); if (rc) return rc;
  LAUNCH(x, k_td_target, dim3(cdiv(B, 128), n), 128, 0, st, k);
  const Pass qp = critic_update_pass(x);
  rc = mlp_forward(x, qp, k.cQ, 1, 2LL * B, B, st); if (rc) return rc;
  LAUNCH(x, k_critic_loss, dim3(2, n), 256, 0, st, k);
  rc = mlp_backward(x, qp, k.cdQ, 1, 2LL * B, B, k.g_q, nullptr, 0, 0, 0, st);
  if (rc) return rc;
  return check_launch();
}

static int phase_critic_apply(saceo_ctx* x, int do_polyak, cudaStream_t st) {
  const KCtx& k = x->k;
  LAUNCH(x, k_adam, dim3(cdiv(cdiv(x->L.nc, 4), 256), 2, k.n_agents), 256, 0, st, k.T.q, k.T.q_m, k.T.q_v, k.g_q, k.T.qt,
         k.lrt, k.T.hyper, x->L.hyper_stride, 0, x->L.nc, x->L.nc_stride, 2, do_polyak, x->pl_q, x->pl_qt, k.S + k.A, 1);
  return check_launch();
}

// The actor phase works on buffers of its own (Xpi2 = [N_s(s); N_s(sE)], aOut2, nlp2, Xc3 = [N_s(s) | N_a(pi(s))]), so
// that its critic-independent half (actor forward, head, expert-observation term through the frozen models) can run on
// a second stream next to the critic phase: only pi(s) -> Q(s, pi(s)) needs the UPDATED critics (SAC_expert.py:312-317).
static KCtx actor_view(const saceo_ctx* x, bool bc = false) {
  KCtx kk = x->k;
  kk.Xpi = x->Xpi2; kk.aOut = x->aOut2; kk.nlp = x->nlp2; kk.Xc2 = x->Xc3;
  if (bc) kk.eps_force = 1.f;
  return kk;
}

// Expert-observation term on the staged model inputs Xm: forward through the frozen model(s), MSE against s'E, backward
// to the action columns (mdXa, mse_part).  Shared by the SAC-EO / BC actor phase and the on-policy expert gradient.
static int model_term_phase(saceo_ctx* x, const KCtx& k, cudaStream_t st) {
  const int n = k.n_agents, S = k.S, A = k.A, E = k.E, mo = x->L.model_out;
  if (k.nmod == 0) return 0;
  if (model_term_eligible(k)) {
    // fused expert-observation term: model forward, MSE, backward to the action columns in one kernel
    if (model_term_launch(k, k.mse_part, st) != cudaSuccess) return fail(SACEO_E_CUDA, "model-term launch failed");
    count_launch(x, "k_model_term", st);
    return 0;
  }
  // the GEMM chain: the models have no weight-plane image
  const Pass mp = model_term_pass(x, k);
  int rc = mlp_forward_unfused(x, mp, k.mOut, mo, 2LL * E * mo, (long long)E * mo, st); if (rc) return rc;
  LAUNCH(x, k_model_loss, dim3(n), 256, 0, st, k);
  // backward to the action columns (weights frozen)
  return mlp_backward_layers(x, mp, k.mdOut, S, 2LL * E * S, (long long)E * S, nullptr, k.mdXa, A,
                             2LL * E * A, (long long)E * A, BwdFused{}, st);
}

// phase 2a: everything of the actor step that does not depend on the critics
static int phase_actor_pre(saceo_ctx* x, cudaStream_t st, bool bc = false) {
  const KCtx kk = actor_view(x, bc);
  const KCtx& k = kk; const int n = k.n_agents, B = k.B, S = k.S, A = k.A, R = k.R, E = k.E;
  int rc;
  LAUNCH(x, k_stage, dim3(cdiv((long long)R * S, 256), n), 256, 0, st, k);
  rc = mlp_forward(x, actor_update_pass(x, k), k.aOut, k.Ao, (long long)k.Rs * k.Ao, 0, st); if (rc) return rc;
  LAUNCH(x, k_head_fwd, dim3(cdiv(R, 128), n), 128, 0, st, k, R, B, k.noise, (3LL * B + E) * A, B, 2,
         (float*)nullptr, (float*)nullptr, 0LL, 0);      // pi(s) -> the action columns of Xc3
  rc = model_term_phase(x, k, st); if (rc) return rc;
  return check_launch();
}

// phase 2b: policy loss through the UPDATED critics, head backward, actor backward and weight gradients
// bc: behaviour cloning (BC.py:309-363) - the expert weight is forced to 1 and the policy-loss half (critic forward /
// backward-to-action on the B minibatch rows) is skipped: those rows then carry exactly-zero output gradients.
static int phase_actor_post(saceo_ctx* x, cudaStream_t st, bool bc = false) {
  const KCtx kk = actor_view(x, bc);
  const KCtx& k = kk; const int n = k.n_agents, B = k.B, A = k.A, R = k.R;
  int rc;
  if (!bc) {
    const Pass qp = critic_pass(x, false, k.Xc2, B);
    rc = mlp_forward(x, qp, k.cQ, 1, 2LL * B, B, st); if (rc) return rc;
    LAUNCH(x, k_actor_q, dim3(n), 256, 0, st, k);
    rc = mlp_backward(x, qp, k.cdQ, 1, 2LL * B, B, nullptr, k.cdXa, A, 2LL * B * A, (long long)B * A, st);
    if (rc) return rc;
  } else {
    CU(cudaMemsetAsync(k.cdXa, 0, sizeof(float) * (size_t)n * 2 * B * A, st));
  }
  LAUNCH(x, k_head_bwd, dim3(cdiv(R, 128), n), 128, 0, st, k, R);
  rc = mlp_backward(x, actor_update_pass(x, k), k.daOut, k.Ao, (long long)k.Rs * k.Ao, 0, k.g_actor, nullptr, 0, 0, 0,
                    st);
  if (rc) return rc;
  if (!k.per_state_std) LAUNCH(x, k_lsv_reduce, dim3(n), 32 * cdiv(A, 32), 0, st, k, R);
  return check_launch();
}
static int phase_actor_grads(saceo_ctx* x, cudaStream_t st, bool bc = false) {
  int rc = phase_actor_pre(x, st, bc); if (rc) return rc;
  return phase_actor_post(x, st, bc);
}

// one Keras-Adam step of the actor optimiser with gradient g; k_adam also keeps the actor's weight planes current
static int actor_adam(saceo_ctx* x, const float* g, cudaStream_t st) {
  const KCtx& k = x->k;
  LAUNCH(x, k_adam, dim3(cdiv(cdiv(x->L.na, 4), 256), 1, k.n_agents), 256, 0, st, k.T.actor, k.T.actor_m, k.T.actor_v,
         g, (float*)nullptr, k.lrt, k.T.hyper, x->L.hyper_stride, 2, x->L.na, x->L.na_stride, 1, 0,
         x->pl_actor, (uint8_t*)nullptr, k.S, k.Ao);
  return check_launch();
}

// phase 4/5: temperature (forward of the UPDATED actor on s with fresh noise u5)
static int phase_alpha(saceo_ctx* x, int apply, cudaStream_t st) {
  const KCtx kk = actor_view(x);          // Xpi2 still holds N_s(s) from the actor phase
  const KCtx& k = kk; const int n = k.n_agents, B = k.B, A = k.A;
  int rc = mlp_forward(x, actor_pass(x, k, B), k.aOut, k.Ao, (long long)k.Rs * k.Ao, 0, st, false); if (rc) return rc;
  LAUNCH(x, k_head_fwd, dim3(cdiv(B, 128), n), 128, 0, st, k, B, B, k.noise, (3LL * B + k.E) * A, 2 * B + k.E, 0,
         (float*)nullptr, (float*)nullptr, 0LL, 0);
  LAUNCH(x, k_alpha_step, dim3(n), 256, 0, st, k, apply);
  return check_launch();
}

static int step_once(saceo_ctx* x, int use_rng, int do_polyak, cudaStream_t st) {
  const KCtx& k = x->k;
  int rc;
  LAUNCH(x, k_step_begin, dim3(cdiv(k.n_agents * 4, 128)), 128, 0, st, k, use_rng);
  if (use_rng) {
    const int items = ((3 * k.B + k.E) * k.A + 3) / 4;
    LAUNCH(x, k_rng_fill, dim3(cdiv(items > k.B ? items : k.B, 256), k.n_agents), 256, 0, st, k, use_rng == 2 ? 1 : 0);
  }
  if ((rc = phase_gather(x, st))) return rc;
  // fork: the critic-independent half of the actor phase on the second stream (captured into the same graph).
  // Off on a single-stream context and in the per-kernel profile.
  // Only when the TD-target actor pass runs in k_mlp_fwd_ws, which then writes no hidden activation: the GEMM chain
  // would write them into the buffers the actor phase saves into.
  const bool fork = x->fork && !x->prof && x->s2 != nullptr && fwd_ws(x, actor_net(x)) && x->pl_q != nullptr;
  if (fork) {
    CU(cudaEventRecord(x->ev_fork, st));
    CU(cudaStreamWaitEvent(x->s2, x->ev_fork, 0));
    if ((rc = phase_actor_pre(x, x->s2))) return rc;
    CU(cudaEventRecord(x->ev_join, x->s2));
  }
  if ((rc = phase_critic_grads(x, st))) return rc;
  if ((rc = phase_critic_apply(x, do_polyak, st))) return rc;
  if (fork) { CU(cudaStreamWaitEvent(st, x->ev_join, 0)); }
  else if ((rc = phase_actor_pre(x, st))) return rc;
  if ((rc = phase_actor_post(x, st))) return rc;
  if ((rc = actor_adam(x, x->k.g_actor, st))) return rc;
  if ((rc = phase_alpha(x, 1, st))) return rc;
  return 0;
}

extern "C" int saceo_set_draws(saceo_ctx* x, const int64_t* idx, const float* noise, const int32_t* perm, void* stream) {
  if (!x) return fail(SACEO_E_INVALID, "null ctx");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k;
  if (idx) CU(cudaMemcpyAsync(k.idx, idx, sizeof(long long) * k.n_agents * k.B, cudaMemcpyDeviceToDevice, st));
  if (noise) CU(cudaMemcpyAsync(k.noise, noise, sizeof(float) * k.n_agents * (3LL * k.B + k.E) * k.A, cudaMemcpyDeviceToDevice, st));
  if (perm && k.E > 0) CU(cudaMemcpyAsync(k.perm, perm, sizeof(int) * k.n_agents * k.E, cudaMemcpyDeviceToDevice, st));
  return 0;
}

extern "C" int saceo_update(saceo_ctx* x, int32_t n_steps, int64_t num_timesteps, int32_t use_device_rng,
                            uint64_t seed, float* losses_out, void* stream) {
  if (!x) return fail(SACEO_E_INVALID, "null ctx");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  if (!x->k.T.replay || !x->k.T.replay_size) return fail(SACEO_E_UNBOUND, "replay tables are not bound");
  if (n_steps < 1) return fail(SACEO_E_INVALID, "n_steps must be >= 1");
  cudaStream_t st = (cudaStream_t)stream;
  const int rng = use_device_rng == 2 ? 2 : (use_device_rng ? 1 : 0);   // 2: device noise/permutation, indices already in place
  { int rcp = ensure_planes(x, st); if (rcp) return rcp; }
  if (rng) LAUNCH(x, k_set_seed, 1, 1, 0, st, x->k, (unsigned long long)seed);
  for (int i = 0; i < n_steps; ++i) {
    const int pol = ((num_timesteps + i) % x->cfg.target_update_int) == 0 ? 1 : 0;
    if (x->cfg.use_graph) {
      if (!x->graph[rng][pol]) {
        cudaGraph_t g;
        CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        const long long before = x->launches;
        int rc = step_once(x, rng, pol, st);
        cudaError_t e = cudaStreamEndCapture(st, &g);
        x->graph_nodes[rng][pol] = x->launches - before;
        x->launches = before;
        if (rc) return rc;
        if (e != cudaSuccess) return fail(SACEO_E_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
        CU(cudaGraphInstantiate(&x->graph[rng][pol], g, 0));
        cudaGraphDestroy(g);
      }
      CU(cudaGraphLaunch(x->graph[rng][pol], st));
      x->launches += x->graph_nodes[rng][pol];
    } else {
      int rc = step_once(x, rng, pol, st); if (rc) return rc;
    }
  }
  if (losses_out)
    CU(cudaMemcpyAsync(losses_out, x->k.losses, sizeof(float) * x->k.n_agents * x->L.n_losses, cudaMemcpyDeviceToDevice, st));
  return 0;
}

// Behaviour cloning from expert observations: BC._update_actor (BC.py:309-363) = the expert-observation term alone
// (epsilon = 1), one Adam step on the actor; critics, temperature, targets and their optimisers are not touched.
extern "C" int saceo_bc_update(saceo_ctx* x, int32_t n_steps, int32_t use_device_rng, uint64_t seed, float* losses_out,
                               void* stream) {
  if (!x) return fail(SACEO_E_INVALID, "null ctx");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  if (x->cfg.num_models < 1) return fail(SACEO_E_INVALID, "behaviour cloning needs num_models >= 1");
  if (n_steps < 1) return fail(SACEO_E_INVALID, "n_steps must be >= 1");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k;
  { int rcp = ensure_planes(x, st); if (rcp) return rcp; }
  if (use_device_rng) LAUNCH(x, k_set_seed, 1, 1, 0, st, k, (unsigned long long)seed);
  for (int i = 0; i < n_steps; ++i) {
    LAUNCH(x, k_bc_begin, cdiv(k.n_agents, 128), 128, 0, st, k, use_device_rng ? 1 : 0);
    if (use_device_rng) {
      const int items = ((3 * k.B + k.E) * k.A + 3) / 4;
      LAUNCH(x, k_rng_fill, dim3(cdiv(items > k.B ? items : k.B, 256), k.n_agents), 256, 0, st, k, 1);
    }
    int rc = phase_actor_grads(x, st, true); if (rc) return rc;
    if ((rc = actor_adam(x, x->k.g_actor, st))) return rc;
    LAUNCH(x, k_bc_loss, cdiv(k.n_agents, 128), 128, 0, st, k);
  }
  if (losses_out)
    CU(cudaMemcpyAsync(losses_out, k.losses, sizeof(float) * k.n_agents * x->L.n_losses, cudaMemcpyDeviceToDevice, st));
  return check_launch();
}

// One update WITHOUT the CUDA graph, an event after every kernel launch: per-launch device times measured live
// (bench.py's per-kernel roofline).  names_out: max_n x 32 chars, us_out: max_n floats; synchronises the stream.
extern "C" int saceo_profile_step(saceo_ctx* x, int64_t num_timesteps, int32_t use_device_rng, uint64_t seed,
                                  char* names_out, float* us_out, int32_t max_n, int32_t* n_out, void* stream) {
  if (!x || !names_out || !us_out || !n_out || max_n < 1) return fail(SACEO_E_INVALID, "bad argument");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  cudaStream_t st = (cudaStream_t)stream;
  const int rng = use_device_rng == 2 ? 2 : (use_device_rng ? 1 : 0);
  const int pol = (num_timesteps % x->cfg.target_update_int) == 0 ? 1 : 0;
  { int rcp = ensure_planes(x, st); if (rcp) return rcp; }
  if (rng) LAUNCH(x, k_set_seed, 1, 1, 0, st, x->k, (unsigned long long)seed);
  cudaEvent_t e0; CU(cudaEventCreate(&e0));
  x->prof = true; x->prof_n = 0;
  CU(cudaEventRecord(e0, st));
  int rc = step_once(x, rng, pol, st);
  x->prof = false;
  if (rc) { cudaEventDestroy(e0); return rc; }
  CU(cudaStreamSynchronize(st));
  const int n = (int)x->prof_n < max_n ? (int)x->prof_n : max_n;
  cudaEvent_t prev = e0;
  for (int i = 0; i < n; ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, prev, x->prof_ev[i]);
    us_out[i] = ms * 1000.f;
    strncpy(names_out + (size_t)i * 32, x->prof_name[i], 31);
    names_out[(size_t)i * 32 + 31] = 0;
    prev = x->prof_ev[i];
  }
  *n_out = n;
  cudaEventDestroy(e0);
  return 0;
}

static int update_host_impl(saceo_ctx* x, int64_t num_timesteps, uint64_t seed, const int64_t* idx_host,
                            const float* expert_host, float* losses_host, void* stream, bool sync) {
  if (!x) return fail(SACEO_E_INVALID, "null ctx");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  cudaStream_t st = (cudaStream_t)stream; KCtx& k = x->k;
  const bool want_e = expert_host && k.E > 0;
  const long long ne = (long long)k.n_agents * k.E * k.S;
  const size_t idx_bytes = sizeof(long long) * (size_t)k.n_agents * k.B, exp_bytes = sizeof(float) * 2 * (size_t)ne;
  int rc;
  if (!sync && (want_e || idx_host)) {
    // pipelined host path: H2D on the copy stream into staging set `s` (overlaps the previous step, which still reads the
    // bound tables), then stream-ordered device-to-device copies into the bound tables / the index buffer
    if (!x->sc) {
      CU(cudaStreamCreateWithFlags(&x->sc, cudaStreamNonBlocking));
      for (int i = 0; i < 2; ++i) {
        CU(cudaEventCreateWithFlags(&x->ev_h2d[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&x->ev_free[i], cudaEventDisableTiming));
        CU(cudaMalloc(&x->hstage[i], idx_bytes + exp_bytes + 256));
      }
    }
    const int s = x->hslot; x->hslot ^= 1;
    char* sidx = x->hstage[s]; char* sexp = x->hstage[s] + ((idx_bytes + 255) & ~(size_t)255);
    if (x->hstage_used[s]) CU(cudaStreamWaitEvent(x->sc, x->ev_free[s], 0));     // its last consumer has copied out of it
    if (want_e) CU(cudaMemcpyAsync(sexp, expert_host, exp_bytes, cudaMemcpyHostToDevice, x->sc));
    if (idx_host) CU(cudaMemcpyAsync(sidx, idx_host, idx_bytes, cudaMemcpyHostToDevice, x->sc));
    CU(cudaEventRecord(x->ev_h2d[s], x->sc));
    CU(cudaStreamWaitEvent(st, x->ev_h2d[s], 0));
    if (want_e) {
      CU(cudaMemcpyAsync(k.T.expert_s, sexp, sizeof(float) * ne, cudaMemcpyDeviceToDevice, st));
      CU(cudaMemcpyAsync(k.T.expert_sp, sexp + sizeof(float) * ne, sizeof(float) * ne, cudaMemcpyDeviceToDevice, st));
    }
    if (idx_host) CU(cudaMemcpyAsync(k.idx, sidx, idx_bytes, cudaMemcpyDeviceToDevice, st));
    CU(cudaEventRecord(x->ev_free[s], st));
    x->hstage_used[s] = true;
  } else {
    if (want_e) {
      // host layout [2, n, E, S] (all sE rows, then all s'E rows) -> the BOUND expert tables (like Population.set_expert
      // followed by an update): the kernels and the captured graphs keep reading the tables saceo_bind() gave them
      CU(cudaMemcpyAsync(k.T.expert_s, expert_host, sizeof(float) * ne, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(k.T.expert_sp, expert_host + ne, sizeof(float) * ne, cudaMemcpyHostToDevice, st));
    }
    if (idx_host) CU(cudaMemcpyAsync(k.idx, idx_host, idx_bytes, cudaMemcpyHostToDevice, st));
  }
  if (idx_host) {
    // host indices (np.random.randint, buffers.py:135) + device noise / expert shuffle
    rc = saceo_update(x, 1, num_timesteps, 2, seed, nullptr, stream); if (rc) return rc;
  } else {
    rc = saceo_update(x, 1, num_timesteps, 1, seed, nullptr, stream); if (rc) return rc;
  }
  if (losses_host)
    CU(cudaMemcpyAsync(losses_host, k.losses, sizeof(float) * k.n_agents * x->L.n_losses, cudaMemcpyDeviceToHost, st));
  if (sync) CU(cudaStreamSynchronize(st));
  return 0;
}
extern "C" int saceo_update_host(saceo_ctx* x, int64_t num_timesteps, uint64_t seed, const int64_t* idx_host,
                                 const float* expert_host, float* losses_host, void* stream) {
  return update_host_impl(x, num_timesteps, seed, idx_host, expert_host, losses_host, stream, true);
}
extern "C" int saceo_update_host_async(saceo_ctx* x, int64_t num_timesteps, uint64_t seed, const int64_t* idx_host,
                                       const float* expert_host, float* losses_host, void* stream) {
  return update_host_impl(x, num_timesteps, seed, idx_host, expert_host, losses_host, stream, false);
}

extern "C" int saceo_update_phase(saceo_ctx* x, int32_t phase, int64_t num_timesteps, void* stream) {
  if (!x) return fail(SACEO_E_INVALID, "null ctx");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k;
  int rc;
  { int rcp = ensure_planes(x, st); if (rcp) return rcp; }
  switch (phase) {
    case 0:
      LAUNCH(x, k_step_begin, dim3(cdiv(k.n_agents * 4, 128)), 128, 0, st, k, 0);
      if ((rc = phase_gather(x, st))) return rc;
      return phase_critic_grads(x, st);
    case 1: return phase_critic_apply(x, (num_timesteps % x->cfg.target_update_int) == 0 ? 1 : 0, st);
    case 2: return phase_actor_grads(x, st);
    case 3: return actor_adam(x, x->k.g_actor, st);
    case 4: return phase_alpha(x, 0, st);
    case 5: LAUNCH(x, k_alpha_apply, dim3(cdiv(k.n_agents, 128)), 128, 0, st, k); return check_launch();
    default: return fail(SACEO_E_INVALID, "phase must be 0..5");
  }
}

// ------------------------------------------------------------------------------------------
// gather / inference entry points
// ------------------------------------------------------------------------------------------
extern "C" int saceo_gather(saceo_ctx* x, const int64_t* idx, float* out_s, float* out_a, float* out_sp,
                            float* out_r, double* out_d, void* stream) {
  if (!x || !idx) return fail(SACEO_E_INVALID, "null argument");
  if (!x->bound || !x->k.T.replay) return fail(SACEO_E_UNBOUND, "replay table is not bound");
  const KCtx& k = x->k;
  LAUNCH(x, k_gather, dim3(cdiv(k.B, 8), k.n_agents), 256, 0, (cudaStream_t)stream, k, (const long long*)idx,
         out_s, out_a, out_sp, out_r, out_d, (float*)nullptr, 0);
  return check_launch();
}

// TrajectoryBuffer.add for the whole population in one call (buffers.py:41-71, SAC_expert.py:793-801): k packed AoS rows
// per agent (device, [n_agents, k, row_words]) appended to every agent's ring, ring arithmetic on the device.
extern "C" int saceo_replay_append(saceo_ctx* x, const float* rows, int32_t k, void* stream) {
  if (!x || !rows) return fail(SACEO_E_INVALID, "null argument");
  if (!x->bound || !x->k.T.replay || !x->k.T.replay_size || !x->k.T.replay_start)
    return fail(SACEO_E_UNBOUND, "replay, replay_size and replay_start tables must be bound");
  if (k < 1 || k > x->cfg.replay_capacity) return fail(SACEO_E_INVALID, "k must be in [1, replay_capacity]");
  if (reinterpret_cast<uintptr_t>(rows) & 15) return fail(SACEO_E_INVALID, "rows must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& kc = x->k;
  const int items = k * (x->L.row_words >> 2);
  LAUNCH(x, k_replay_append_rows, dim3(cdiv(items, 256), kc.n_agents), 256, 0, st, kc, rows, k, const_cast<float*>(kc.T.replay),
         kc.T.replay_size, kc.T.replay_start);
  LAUNCH(x, k_replay_append_commit, dim3(cdiv(kc.n_agents, 128)), 128, 0, st, kc, k, const_cast<int*>(kc.T.replay_size),
         const_cast<int*>(kc.T.replay_start));
  return check_launch();
}

extern "C" int saceo_actor_forward(saceo_ctx* x, const float* obs, int32_t rows, const float* noise,
                                   float* act_out, float* neglogp_out, void* stream) {
  if (!x || !obs || rows < 1) return fail(SACEO_E_INVALID, "bad argument");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k; const int n = k.n_agents;
  { int rcp = ensure_planes(x, st); if (rcp) return rcp; }
  // expert rows would be routed to the model input: use only the first B ("main") rows per chunk
  for (int r0 = 0; r0 < rows; r0 += k.B) {
    const int nr = rows - r0 < k.B ? rows - r0 : k.B;
    LAUNCH(x, k_stage_obs, dim3(cdiv((long long)nr * k.S, 256), n), 256, 0, st, k, obs, rows, r0, nr, k.Xpi, k.ldXp,
           (long long)k.Rs * k.ldXp, 0);
    int rc = mlp_forward(x, actor_pass(x, k, nr), k.aOut, k.Ao, (long long)k.Rs * k.Ao, 0, st, false); if (rc) return rc;
    LAUNCH(x, k_head_fwd, dim3(cdiv(nr, 128), n), 128, 0, st, k, nr, nr, noise, (long long)rows * k.A, r0, 0,
           act_out, neglogp_out, (long long)rows, r0);
  }
  return check_launch();
}

extern "C" int saceo_critic_forward(saceo_ctx* x, int32_t which, const float* obs, const float* act, int32_t rows,
                                    int32_t scale_ret, float* q_out, void* stream) {
  if (!x || !obs || !act || !q_out || rows < 1) return fail(SACEO_E_INVALID, "bad argument");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k; const int n = k.n_agents;
  { int rcp = ensure_planes(x, st); if (rcp) return rcp; }
  for (int r0 = 0; r0 < rows; r0 += k.B) {
    const int nr = rows - r0 < k.B ? rows - r0 : k.B;
    LAUNCH(x, k_stage_obs, dim3(cdiv((long long)nr * k.S, 256), n), 256, 0, st, k, obs, rows, r0, nr, k.Xc, k.ldXc,
           (long long)k.B * k.ldXc, 0);
    LAUNCH(x, k_stage_act, dim3(cdiv((long long)nr * k.A, 256), n), 256, 0, st, k, act, rows, r0, nr, k.Xc, k.ldXc,
           (long long)k.B * k.ldXc, 0);
    int rc = mlp_forward(x, critic_pass(x, which != 0, k.Xc, nr), q_out + r0, 1, 2LL * rows, rows, st, false); if (rc) return rc;
  }
  if (scale_ret) LAUNCH(x, k_scale_ret, dim3(cdiv(2LL * rows, 256), n), 256, 0, st, k, q_out, rows);
  return check_launch();
}

extern "C" int saceo_model_eval(saceo_ctx* x, const float* obs, const float* act, int32_t rows, float* sp_out,
                                void* stream) {
  if (!x || !obs || !act || !sp_out || rows < 1) return fail(SACEO_E_INVALID, "bad argument");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  if (x->cfg.num_models < 1) return fail(SACEO_E_INVALID, "no models configured");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k; const int n = k.n_agents, SA = k.S + k.A, E = k.E;
  for (int r0 = 0; r0 < rows; r0 += E) {
    const int nr = rows - r0 < E ? rows - r0 : E;
    // every model sees the same rows: stage them into net 0's block and read it with a zero net stride
    LAUNCH(x, k_stage_obs, dim3(cdiv((long long)nr * k.S, 256), n), 256, 0, st, k, obs, rows, r0, nr, k.Xm, SA,
           2LL * E * SA, 1);
    LAUNCH(x, k_stage_act, dim3(cdiv((long long)nr * k.A, 256), n), 256, 0, st, k, act, rows, r0, nr, k.Xm, SA,
           2LL * E * SA, 1);
    const int mo = x->L.model_out;
    int rc = mlp_forward(x, model_eval_pass(x, nr), k.mOut, mo, 2LL * E * mo, (long long)E * mo, st); if (rc) return rc;
    LAUNCH(x, k_model_out, dim3(cdiv((long long)nr * k.S, 256), n, k.nmod), 256, 0, st, k, obs, rows, r0, nr, sp_out);
  }
  return check_launch();
}

// ------------------------------------------------------------------------------------------
// dynamics-model fitting (mbrl_onpolicy_alg.py:301-319; SAC_expert.py:480-556)
// ------------------------------------------------------------------------------------------
extern "C" int saceo_fit_bind(saceo_ctx* x, const saceo_fit_tables* t, int32_t model_batch, int32_t use_grad_clip) {
  if (!x || !t) return fail(SACEO_E_INVALID, "null argument");
  if (x->cfg.num_models < 1) return fail(SACEO_E_INVALID, "model fitting needs num_models >= 1");
  const bool sep = x->cfg.separate_reward_nn != 0;
  NetD rn{};             // the reward nets
  if (sep) {
    if (!t->reward || !t->reward_m || !t->reward_v) return fail(SACEO_E_INVALID, "separate_reward_nn: the reward tables of saceo_fit_tables are required");
    if (t->reward_hidden[0] < 1 || t->reward_hidden[1] < 1) return fail(SACEO_E_INVALID, "reward_hidden must be positive");
    for (int i = 0; i < 2; ++i)
      if (t->reward_act[i] < 0 || t->reward_act[i] > SACEO_ACT_ELU) return fail(SACEO_E_INVALID, "bad reward activation");
    rn = net_desc(t->reward, 2 * t->reward_stride, t->reward_stride, x->cfg.num_models, x->cfg.S + x->cfg.A, 1, 2,
                  t->reward_hidden, t->reward_act);
    if (t->reward_stride < rn.n() || (t->reward_stride % 32) != 0) return fail(SACEO_E_INVALID, "reward_stride must be a multiple of 32 and >= %lld", rn.n());
  }
  if (model_batch < 1) return fail(SACEO_E_INVALID, "model_batch must be >= 1");
  if (!t->model || !t->model_m || !t->model_v || !t->model_t || !t->fit_hyper)
    return fail(SACEO_E_INVALID, "a required fit table pointer is NULL");
  const int nls = (t->model_logstd != nullptr) + (t->model_logstd_m != nullptr) + (t->model_logstd_v != nullptr);
  if (nls != 0 && nls != 3) return fail(SACEO_E_INVALID, "model_logstd, model_logstd_m and model_logstd_v must be given together");
  if (x->cfg.S > 512) return fail(SACEO_E_INVALID, "model fitting supports S <= 512 (per-column weights of the loss kernel live in shared memory)");
  CU(cudaSetDevice(x->cfg.device));
  if (x->fit_ws) { CU(cudaDeviceSynchronize()); cudaFree(x->fit_ws); x->fit_ws = nullptr; x->fit_bound = false; }
  const saceo_config& c = x->cfg;
  FitCtx& f = x->fit;
  memset(&f, 0, sizeof(f));
  f.model = t->model; f.m = t->model_m; f.v = t->model_v; f.t = t->model_t; f.hyper = t->fit_hyper;
  f.ls = t->model_logstd; f.ls_m = t->model_logstd_m; f.ls_v = t->model_logstd_v; f.S = c.S;
  f.mb = model_batch; f.mbs = (int)rup(model_batch, 32); f.nmod = c.num_models; f.use_clip = use_grad_clip;
  f.nm = x->L.nm; f.nm_stride = x->L.nm_stride;
  if (sep) {
    f.rw = t->reward; f.rw_m = t->reward_m; f.rw_v = t->reward_v;
    f.nr_stride = t->reward_stride; f.nr = rn.n();
  }
  x->fit_rnet = rn;
  const NetD mn = model_desc(c);
  const long long n2 = 2LL * c.n_agents, mb = f.mbs, SA = c.S + c.A, mo = x->L.model_out;
  for (int pass = 0; pass < 2; ++pass) {
    Bump b{pass ? (char*)x->fit_ws : nullptr, 0, pass ? &x->names : nullptr};
    f.X = b.get<float>("fit_X", n2 * mb * SA);        f.T = b.get<float>("fit_T", n2 * mb * (c.S + 1));
    b.layers(x->fit_H, "fit_H", mn, n2 * mb);
    f.Out = b.get<float>("fit_Out", n2 * mb * mo);    f.dOut = b.get<float>("fit_dOut", n2 * mb * mo);
    b.layers(x->fit_dH, "fit_dH", mn, n2 * mb, true);
    f.g = b.get<float>("g_model", n2 * x->L.nm_stride);
    f.loss_part = b.get<float>("fit_loss", n2);
    f.g_ls = b.get<float>("g_model_logstd", n2 * c.S);
    f.gscale = b.get<float>("fit_gscale", c.n_agents); f.gnorm = b.get<float>("fit_gnorm", c.n_agents);
    f.lrt = b.get<float>("fit_lrt", c.n_agents);
    if (sep) {
      b.layers(x->fit_rH, "fit_rH", rn, n2 * mb);
      f.rOut = b.get<float>("fit_rOut", n2 * mb);       f.rdOut = b.get<float>("fit_rdOut", n2 * mb);
      b.layers(x->fit_rdH, "fit_rdH", rn, n2 * mb, true);
      f.g_r = b.get<float>("g_reward", n2 * f.nr_stride);
    }
    if (!pass) {
      const long long bytes = rup(b.off, 256);
      if (cudaMalloc(&x->fit_ws, (size_t)bytes) != cudaSuccess) {
        cudaGetLastError(); x->fit_ws = nullptr;
        return fail(SACEO_E_NOMEM, "cudaMalloc of %lld model-fit workspace bytes failed", bytes);
      }
      CU(cudaMemset(x->fit_ws, 0, (size_t)bytes));
    }
  }
  x->fit_bound = true;
  return 0;
}

// One joint gradient step on every agent's models per entry of idx ([n_steps, n_agents, num_models, model_batch]
// logical replay rows).  losses_out (nullable): [n_steps, n_agents, num_models] per-model minibatch losses.
extern "C" int saceo_model_fit(saceo_ctx* x, int32_t n_steps, const int64_t* idx, float* losses_out, void* stream) {
  if (!x) return fail(SACEO_E_INVALID, "null context");
  if (!x->bound || !x->fit_bound) return fail(SACEO_E_UNBOUND, "saceo_bind and saceo_fit_bind must precede saceo_model_fit");
  if (!idx || n_steps < 0) return fail(SACEO_E_INVALID, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const KCtx& k = x->k; const FitCtx& f = x->fit;
  const int n = k.n_agents, mb = f.mb, ms = f.mbs, SA = k.S + k.A, mo = x->L.model_out;
  const Pass mp = fit_pass(x, model_net(x, f.model, f.nmod), x->fit_H, x->fit_dH);
  const Pass rp = fit_pass(x, x->fit_rnet, x->fit_rH, x->fit_rdH);
  for (int s = 0; s < n_steps; ++s) {
    const long long* ix = reinterpret_cast<const long long*>(idx) + (long long)s * n * f.nmod * mb;
    LAUNCH(x, k_fit_begin, cdiv(n, 128), 128, 0, st, f, n);
    LAUNCH(x, k_fit_stage, dim3(cdiv((long long)mb * (SA + k.S + 1), 256), f.nmod, n), 256, 0, st, k, f, ix);
    int rc = mlp_forward(x, mp, f.Out, mo, 2LL * ms * mo, (long long)ms * mo, st);
    if (rc) return rc;
    if (f.rw) {      // the reward network sees the same normalised input (base_world_model.py:72-74)
      rc = mlp_forward(x, rp, f.rOut, 1, 2LL * ms, (long long)ms, st);
      if (rc) return rc;
    }
    LAUNCH(x, k_fit_loss, dim3(f.nmod, n), 256, 0, st, k, f,
           losses_out ? losses_out + (long long)s * n * f.nmod : (float*)nullptr);
    // no kpad: K = 200 on the register-staged kernel beats K = 224 streamed (measured)
    rc = mlp_backward(x, mp, f.dOut, mo, 2LL * ms * mo, (long long)ms * mo, f.g, nullptr, 0, 0, 0, st);
    if (rc) return rc;
    if (f.rw) {
      rc = mlp_backward(x, rp, f.rdOut, 1, 2LL * ms, (long long)ms, f.g_r, nullptr, 0, 0, 0, st);
      if (rc) return rc;
    }
    if (f.use_clip) LAUNCH(x, k_fit_gnorm, n, 1024, 0, st, f);
    LAUNCH(x, k_fit_adam, dim3(cdiv(cdiv(f.nm, 4), 256), f.nmod, n), 256, 0, st, f, 0);
    if (f.rw) LAUNCH(x, k_fit_adam, dim3(cdiv(cdiv(f.nr, 4), 256), f.nmod, n), 256, 0, st, f, 1);
  }
  return check_launch();
}

// ------------------------------------------------------------------------------------------
// Fisher-vector product and conjugate gradient (trpo.py:200-227, update_utils.py:4-24)
// ------------------------------------------------------------------------------------------
static int fvp_prepare(saceo_ctx* x, cudaStream_t st) {
  { int rcp = ensure_planes(x, st); if (rcp) return rcp; }
  const KCtx& k = x->k; const FvpWs& f = x->f; const int n = k.n_agents, N = f.N;
  LAUNCH(x, k_stage_obs, dim3(cdiv((long long)N * k.S, 256), n), 256, 0, st, k, k.T.fvp_states, N, 0, N, x->fX, k.S,
         (long long)N * k.S, 0);
  return mlp_forward(x, fvp_pass(x), f.Out, k.Ao, (long long)N * k.Ao, 0, st);
}

// Fx = J^T M J x / N + damp x, with the activations of fvp_prepare() resident
static int fvp_apply(saceo_ctx* x, const float* xin, float damp, float* Fx, cudaStream_t st) {
  const KCtx& k = x->k; const FvpWs& f = x->f; const int n = k.n_agents, N = f.N;
  NetD an = actor_net(x);
  NetD tn = an; tn.theta = xin;                       // tangent "network": same flat layout
  const long long sO = (long long)N * k.Ao;
  int rc;
  // J x layer by layer: T[0] = (X.P0 + c0) * act0'(H[0]);  T[l] = (H[l-1].P_l + c_l + Tmp) * act_l'(H[l]) with
  // Tmp = T[l-1].W_l;  the output layer writes TOut, without the activation factor
  for (int l = 0; l <= an.nh; ++l) {
    const int K = an.K(l), W = an.N(l);
    const long long sK = (long long)N * K, sW = (long long)N * W;
    GemmP p{};
    if (l > 0) {
      p.nnet = 1; p.A = x->fT[l - 1]; p.lda = K; p.sAa = sK; p.B = an.theta + an.oW(l); p.ldb = W; p.sBa = an.sa;
      p.C = f.Tmp; p.ldc = W; p.sCa = sW; p.M = N; p.N = W; p.K = K; p.epi = EPI_NONE;
      rc = gemm(x, false, false, false, p, n, st); if (rc) return rc;
      p = GemmP{}; p.addend = f.Tmp;
    }
    p.nnet = 1; p.A = l > 0 ? x->fH[l - 1] : x->fX; p.lda = K; p.sAa = sK; p.B = tn.theta + tn.oW(l); p.ldb = W; p.sBa = an.sa;
    p.bias = tn.theta + tn.ob(l); p.sba = an.sa;
    p.C = l < an.nh ? x->fT[l] : f.TOut; p.ldc = W; p.sCa = sW; p.M = N; p.N = W; p.K = K; p.epi = EPI_NONE;
    if (l < an.nh) { p.aux = x->fH[l]; p.epi = EPI_MUL_DACT; p.act = an.act(l); }
    rc = gemm(x, false, false, false, p, n, st); if (rc) return rc;
  }
  // metric: G = M . J x / N   (per row), plus per-row logstd_var contribution
  LAUNCH(x, k_fvp_metric, dim3(cdiv(N, 128), n), 128, 0, st, k, f, xin, x->cfg.std_mult);
  // J^T G  -> Fx (flat layout), then + damp x
  rc = mlp_backward(x, fvp_pass(x), f.G, k.Ao, sO, 0, Fx, nullptr, 0, 0, 0, st); if (rc) return rc;
  LAUNCH(x, k_fvp_finish, dim3(cdiv(x->L.na, 256), n), 256, 0, st, k, f, xin, damp, Fx);
  return check_launch();
}

extern "C" int saceo_fvp(saceo_ctx* x, const float* xin, float damp, float* Fx, void* stream) {
  if (!x || !xin || !Fx) return fail(SACEO_E_INVALID, "null argument");
  if (!x->bound || !x->k.T.fvp_states || x->f.N < 1) return fail(SACEO_E_UNBOUND, "fvp_states not bound / fvp_rows == 0");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = fvp_prepare(x, st); if (rc) return rc;
  return fvp_apply(x, xin, damp, Fx, st);
}

extern "C" int saceo_cg_solve(saceo_ctx* x, const float* b, int32_t iters, float tol, float damp, float* x_out,
                              float* vFv_out, void* stream) {
  if (!x || !b || !x_out) return fail(SACEO_E_INVALID, "null argument");
  if (!x->bound || !x->k.T.fvp_states || x->f.N < 1) return fail(SACEO_E_UNBOUND, "fvp_states not bound / fvp_rows == 0");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k; const FvpWs& f = x->f; const int n = k.n_agents;
  int rc = fvp_prepare(x, st); if (rc) return rc;
  LAUNCH(x, k_cg_init, dim3(n), 256, 0, st, k, f, b);                 // p = r = b, x = 0, rr = r.r, active = 1
  for (int it = 0; it < iters; ++it) {
    rc = fvp_apply(x, f.p, damp, f.z, st); if (rc) return rc;         // z = F(p)
    LAUNCH(x, k_cg_step, dim3(n), 256, 0, st, k, f, tol);             // v, x, r, rr', mu, p, early-exit latch
  }
  CU(cudaMemcpyAsync(x_out, f.x, sizeof(float) * n * x->L.na_stride, cudaMemcpyDeviceToDevice, st));
  if (vFv_out) {
    rc = fvp_apply(x, f.x, damp, f.z, st); if (rc) return rc;         // vFv = x . F(x)   (trpo.py:185)
    LAUNCH(x, k_cg_vfv, dim3(n), 256, 0, st, k, f, vFv_out);
  }
  return check_launch();
}

// ------------------------------------------------------------------------------------------
// TRPO surrogate gradient and line-search statistics (trpo.py:36-63, :229-317) on the fvp_states rows
// ------------------------------------------------------------------------------------------
static int trpo_check(saceo_ctx* x) {
  if (!x) return fail(SACEO_E_INVALID, "null ctx");
  if (!x->bound || !x->k.T.fvp_states || x->f.N < 1) return fail(SACEO_E_UNBOUND, "fvp_states not bound / fvp_rows == 0");
  // the four per-row statistics live in the Tmp scratch of the Fisher-vector workspace, [N, widest layer past the first]
  if (actor_net(x).widest(1) < 4) return fail(SACEO_E_INVALID, "TRPO / PPO entry points need actor_hidden[1] >= 4");
  return 0;
}

static int surrogate_grad(saceo_ctx* x, const float* act, const float* adv, const float* nlp_old, const float* alpha,
                          float clip_eps, float max_grad_norm, bool want_norm, float* grad_out, float* stats_out,
                          cudaStream_t st) {
  int rc = trpo_check(x); if (rc) return rc;
  if (!act || !adv || !grad_out) return fail(SACEO_E_INVALID, "act, adv and grad_out are required");
  const KCtx& k = x->k; const FvpWs& f = x->f; const int n = k.n_agents, N = f.N;
  rc = fvp_prepare(x, st); if (rc) return rc;
  LAUNCH(x, k_trpo_rows, dim3(cdiv(N, 128), n), 128, 0, st, k, f, act, adv, nlp_old, (const float*)nullptr, alpha,
         x->cfg.std_mult, 1, clip_eps, (float*)nullptr, (float*)nullptr);
  if (stats_out) LAUNCH(x, k_trpo_reduce, dim3(n), 256, 0, st, f, stats_out);
  rc = mlp_backward(x, fvp_pass(x), f.G, k.Ao, (long long)N * k.Ao, 0, grad_out, nullptr, 0, 0, 0, st);
  if (rc) return rc;
  // logstd-variable entries = fixed-order column sums of the per-row terms (damp 0: the x operand is only a finite filler)
  LAUNCH(x, k_fvp_finish, dim3(cdiv(x->L.na, 256), n), 256, 0, st, k, f, (const float*)k.T.actor, 0.f, grad_out);
  if (want_norm) LAUNCH(x, k_grad_clip, dim3(n), 256, 0, st, k, grad_out, max_grad_norm, stats_out);
  return check_launch();
}

extern "C" int saceo_trpo_grad(saceo_ctx* x, const float* act, const float* adv, const float* nlp_old, const float* alpha,
                               float* grad_out, float* stats_out, void* stream) {
  return surrogate_grad(x, act, adv, nlp_old, alpha, -1.f, 0.f, false, grad_out, stats_out, (cudaStream_t)stream);
}

extern "C" int saceo_ppo_grad(saceo_ctx* x, const float* act, const float* adv, const float* nlp_old, const float* alpha,
                              float eps_clip, float max_grad_norm, float* grad_out, float* stats_out, void* stream) {
  if (!(eps_clip >= 0.f)) return fail(SACEO_E_INVALID, "eps_clip must be >= 0");
  if (!nlp_old) return fail(SACEO_E_INVALID, "nlp_old is required");
  return surrogate_grad(x, act, adv, nlp_old, alpha, eps_clip, max_grad_norm, true, grad_out, stats_out, (cudaStream_t)stream);
}

// Expert-observation gradient of the on-policy classes (trpo.py:92-158, ppo.py:176-213): see trpo.cuh.  Draws (noise
// rows [2B, 2B+E), expert permutation) are the ones last injected with saceo_set_draws.
extern "C" int saceo_onpolicy_expert_grad(saceo_ctx* x, int32_t n_models, int32_t clip_actions, float* grad_out,
                                          float* stats_out, void* stream) {
  if (!x || !grad_out) return fail(SACEO_E_INVALID, "null argument");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  if (n_models < 1 || n_models > x->cfg.num_models) return fail(SACEO_E_INVALID, "n_models must be in [1, num_models]");
  if (x->k.E < 1 || (n_models == 2 && (x->k.E & 1))) return fail(SACEO_E_INVALID, "needs E >= 1 expert rows (even for two models)");
  if (reinterpret_cast<uintptr_t>(grad_out) & 15) return fail(SACEO_E_INVALID, "grad_out must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  { int rcp = ensure_planes(x, st); if (rcp) return rcp; }
  KCtx kk = actor_view(x, true);            // expert weight forced to 1: the blend is applied by saceo_grad_blend
  kk.nmod = n_models; kk.g_actor = grad_out;
  const KCtx& k = kk; const int n = k.n_agents, E = k.E, Rs = k.Rs;
  const Pass ap = actor_pass(x, k, E);
  int rc;
  CU(cudaMemsetAsync(grad_out, 0, sizeof(float) * (size_t)n * x->L.na_stride, st));
  LAUNCH(x, k_exp_stage, dim3(cdiv((long long)E * k.S, 256), n), 256, 0, st, k);
  rc = mlp_forward(x, ap, k.aOut, k.Ao, (long long)Rs * k.Ao, 0, st);
  if (rc) return rc;
  LAUNCH(x, k_ghead, dim3(cdiv(E, 128), n), 128, 0, st, k, x->cfg.std_mult, clip_actions, 0);
  rc = model_term_phase(x, k, st); if (rc) return rc;
  LAUNCH(x, k_ghead, dim3(cdiv(E, 128), n), 128, 0, st, k, x->cfg.std_mult, clip_actions, 1);
  rc = mlp_backward(x, ap, k.daOut, k.Ao, (long long)Rs * k.Ao, 0, grad_out, nullptr, 0, 0, 0, st);
  if (rc) return rc;
  if (!k.per_state_std) LAUNCH(x, k_lsv_reduce, dim3(n), 32 * cdiv(k.A, 32), 0, st, k, E);
  if (stats_out) LAUNCH(x, k_exp_stats, dim3(cdiv(n, 128)), 128, 0, st, k, stats_out);
  return check_launch();
}

// grad_final = (1 - eps) neg_pg + eps mse_grad per agent, the reference's logged norms, and (max_grad_norm > 0, PPO)
// tf.clip_by_global_norm of the result.  out may alias neg_pg.
extern "C" int saceo_grad_blend(saceo_ctx* x, const float* neg_pg, const float* mse_grad, const float* eps, float max_grad_norm,
                                float* out, float* stats_out, void* stream) {
  if (!x || !neg_pg || !mse_grad || !eps || !out) return fail(SACEO_E_INVALID, "null argument");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k;
  const NetD an = actor_net(x);
  BlendSeg sg{};                                   // the bounds of every weight and bias tensor
  for (int l = 0; l <= an.nh; ++l) { sg.b[sg.nseg++] = an.oW(l); sg.b[sg.nseg++] = an.ob(l); }
  sg.b[sg.nseg] = an.n();
  if (x->L.na > an.n()) sg.b[++sg.nseg] = x->L.na;  // + the state-independent logstd variable
  LAUNCH(x, k_grad_blend, dim3(k.n_agents), 256, 0, st, k, sg, neg_pg, mse_grad, eps, out, stats_out);
  if (max_grad_norm > 0.f || stats_out) LAUNCH(x, k_grad_clip, dim3(k.n_agents), 256, 0, st, k, out, max_grad_norm, stats_out);
  return check_launch();
}

// One Keras-Adam step of the actor optimiser with a caller-supplied gradient (ppo.py:234): only the actor's step
// counter advances; the learning rate is hyper[3] (actor_lr), read at launch time.
extern "C" int saceo_actor_adam(saceo_ctx* x, const float* grad, void* stream) {
  if (!x || !grad) return fail(SACEO_E_INVALID, "null argument");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  if (reinterpret_cast<uintptr_t>(grad) & 15) return fail(SACEO_E_INVALID, "grad must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k;
  LAUNCH(x, k_bc_begin, dim3(cdiv(k.n_agents, 128)), 128, 0, st, k, 0);
  return actor_adam(x, grad, st);
}

extern "C" int saceo_trpo_eval(saceo_ctx* x, const float* act, const float* adv, const float* nlp_old, const float* kl_ref,
                               float* nlp_out, float* kl_info_out, float* stats_out, void* stream) {
  int rc = trpo_check(x); if (rc) return rc;
  if ((nlp_out || nlp_old) && !act) return fail(SACEO_E_INVALID, "act is required for neglogp / the ratio");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k; const FvpWs& f = x->f; const int n = k.n_agents, N = f.N;
  rc = fvp_prepare(x, st); if (rc) return rc;
  LAUNCH(x, k_trpo_rows, dim3(cdiv(N, 128), n), 128, 0, st, k, f, act, adv, nlp_old, kl_ref, (const float*)nullptr,
         x->cfg.std_mult, 0, -1.f, nlp_out, kl_info_out);
  if (stats_out) LAUNCH(x, k_trpo_reduce, dim3(n), 256, 0, st, f, stats_out);
  return check_launch();
}

extern "C" int saceo_actor_step(saceo_ctx* x, const float* theta_ref, const float* dir, const float* scale, void* stream) {
  if (!x || !theta_ref || !dir || !scale) return fail(SACEO_E_INVALID, "null argument");
  if (!x->bound) return fail(SACEO_E_UNBOUND, "saceo_bind() has not been called");
  cudaStream_t st = (cudaStream_t)stream; const KCtx& k = x->k;
  LAUNCH(x, k_actor_step, dim3(cdiv(x->L.na, 256), k.n_agents), 256, 0, st, k, theta_ref, dir, scale);
  x->planes_dirty |= 1;        // theta written outside k_adam: the weight planes are rebuilt before their next use
  return check_launch();
}

// ------------------------------------------------------------------------------------------
// policy acting for any depth (policy.cuh)
// ------------------------------------------------------------------------------------------
static int policy_validate(const saceo_policy_config* c) {
  if (!c) return fail(SACEO_E_INVALID, "null policy config");
  if (c->abi_version != SACEO_ABI_VERSION) return fail(SACEO_E_INVALID, "abi_version %d != %d", c->abi_version, SACEO_ABI_VERSION);
  if (c->n_policies < 1 || c->n_policies > 65535) return fail(SACEO_E_INVALID, "n_policies must be in [1, 65535]");
  if (c->S < 1 || c->A < 1) return fail(SACEO_E_INVALID, "S and A must be positive");
  if (c->n_hidden < 1 || c->n_hidden > SACEO_POLICY_MAX_HIDDEN)
    return fail(SACEO_E_INVALID, "n_hidden must be in [1, %d] (got %d)", SACEO_POLICY_MAX_HIDDEN, c->n_hidden);
  for (int l = 0; l < c->n_hidden; ++l) {
    if (c->hidden[l] < 1 || c->hidden[l] > POL_MAX_WIDTH)
      return fail(SACEO_E_INVALID, "hidden width %d of layer %d outside [1, %d]", c->hidden[l], l, POL_MAX_WIDTH);
    if (c->act[l] < SACEO_ACT_RELU || c->act[l] > SACEO_ACT_ELU)
      return fail(SACEO_E_INVALID, "activations must be tanh, relu or elu (layer %d: %d)", l, c->act[l]);
  }
  if (!(c->std_mult > 0.f)) return fail(SACEO_E_INVALID, "std_mult must be positive");
  return 0;
}

static void policy_layout(const saceo_policy_config* c, long long* n, long long* stride, int* nstride, long long* off) {
  const NetD d = net_desc(nullptr, 0, 0, 1, c->S, c->per_state_std ? 2 * c->A : c->A, c->n_hidden, c->hidden, c->act);
  if (off) {
    for (int l = 0; l <= d.nh; ++l) off[l] = d.oW(l);
    off[d.nh + 1] = d.n();
  }
  *n = actor_params(d, c->per_state_std); *stride = rup(*n, 32); *nstride = (int)rup(2LL * c->S + c->A, 4);
}

extern "C" int saceo_policy_layout(const saceo_policy_config* cfg, int64_t* n_params, int64_t* param_stride,
                                   int32_t* norm_stride) {
  int rc = policy_validate(cfg); if (rc) return rc;
  long long n, s; int ns;
  policy_layout(cfg, &n, &s, &ns, nullptr);
  if (n_params) *n_params = n;
  if (param_stride) *param_stride = s;
  if (norm_stride) *norm_stride = ns;
  return 0;
}

static constexpr int kPolMaxSmem = 200 * 1024;
static int policy_device_ready(int dev) {      // sm_100 check + shared-memory opt-in, once per device
  static int ready[64] = {0};
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(SACEO_E_NODEVICE, "no CUDA device: libsaceo has no CPU fallback");
  }
  if (dev < 0 || dev >= ndev || dev >= 64) return fail(SACEO_E_INVALID, "device %d out of range", dev);
  if (ready[dev]) return 0;
  int major = 0, minor = 0;
  CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  CU(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  if (major != 10) return fail(SACEO_E_NODEVICE, "device %d is sm_%d%d; libsaceo is built for sm_100a only", dev, major, minor);
  int prev = 0;
  CU(cudaGetDevice(&prev));
  if (prev != dev) CU(cudaSetDevice(dev));
  const cudaError_t e = cudaFuncSetAttribute(k_policy_forward, cudaFuncAttributeMaxDynamicSharedMemorySize, kPolMaxSmem);
  if (prev != dev) cudaSetDevice(prev);
  CU(e);
  ready[dev] = 1;
  return 0;
}

extern "C" int saceo_policy_act(const saceo_policy_config* cfg, const float* params, const float* norm, const float* obs,
                                int32_t rows, const float* noise, float* act_out, void* stream) {
  int rc = policy_validate(cfg); if (rc) return rc;
  if (rows < 1) return fail(SACEO_E_INVALID, "rows must be positive");
  if (!params || !norm || !obs || !act_out) return fail(SACEO_E_INVALID, "null argument");
  PolicyP p{};
  long long n; int ns;
  policy_layout(cfg, &n, &p.pstride, &ns, p.off);
  p.params = params; p.norm = norm; p.obs = obs; p.noise = noise; p.out = act_out;
  p.nstride = ns; p.rows = rows; p.S = cfg->S; p.A = cfg->A; p.Ao = cfg->per_state_std ? 2 * cfg->A : cfg->A;
  p.nl = cfg->n_hidden + 1;
  p.width[0] = cfg->S;
  int w = cfg->S > p.Ao ? cfg->S : p.Ao;
  for (int l = 0; l < cfg->n_hidden; ++l) {
    p.width[l + 1] = cfg->hidden[l]; p.act[l] = cfg->act[l];
    if (cfg->hidden[l] > w) w = cfg->hidden[l];
  }
  p.width[p.nl] = p.Ao; p.act[cfg->n_hidden] = ACT_LINEAR;
  p.squash = cfg->squash != 0; p.per_state_std = cfg->per_state_std != 0;
  p.ls_add = cfg->per_state_std ? (float)(log((double)cfg->std_mult) - log(log(2.0))) : (float)log((double)cfg->std_mult);
  p.ld = (int)rup(w, 4);
  // row tile: as many rows as ~96 KB of ping-pong buffers hold (weight reuse), at least one 4-row block
  int rt = (96 * 1024 / 4) / (2 * p.ld);
  rt = rt < POL_RB ? POL_RB : rt > 32 ? 32 : rt / POL_RB * POL_RB;
  if (rt > rup(rows, POL_RB)) rt = (int)rup(rows, POL_RB);
  p.rt = rt;
  const size_t smem = (size_t)2 * rt * p.ld * sizeof(float);
  if (smem > (size_t)kPolMaxSmem) return fail(SACEO_E_INVALID, "S = %d too wide for the shared-memory activation buffers", cfg->S);
  rc = policy_device_ready(cfg->device); if (rc) return rc;
  int prev = 0;
  CU(cudaGetDevice(&prev));
  if (prev != cfg->device) CU(cudaSetDevice(cfg->device));
  k_policy_forward<<<dim3(cdiv(rows, rt), cfg->n_policies), POL_THREADS, smem, (cudaStream_t)stream>>>(p);
  rc = check_launch();
  if (prev != cfg->device) cudaSetDevice(prev);
  return rc;
}

// ------------------------------------------------------------------------------------------
// standalone GEMM self-test surface
// ------------------------------------------------------------------------------------------
// test-only: per-CTA phase timestamps of the tcgen05 streaming kernel (dbg = device buffer, 8 u64 per CTA)
extern "C" int saceo_test_set_tc_debug(void* dbg) { g_tc_dbg = (unsigned long long*)dbg; return 0; }
// test-only: 8 phase stamps per CTA of the tensor-core expert-term kernel
extern "C" int saceo_test_set_mt_debug(void* dbg) { g_mt_dbg = (unsigned long long*)dbg; return 0; }
// test-only: on != 0 runs the expert term on the fp32 CUDA-core kernel (k_model_term) wherever it is eligible
extern "C" int saceo_test_set_mt_fp32(int32_t on) { g_mt_fp32 = on != 0; return 0; }
// test-only: the sel-th warp-specialised fused launch from now on writes 16 phase stamps per CTA into dbg
extern "C" int saceo_test_set_ws_debug(void* dbg, int32_t sel) { g_ws_dbg = (unsigned long long*)dbg; g_ws_sel = sel; g_ws_count = 0; return 0; }

extern "C" int saceo_test_gemm(int32_t gemm_mode, int32_t batch, int32_t M, int32_t N, int32_t K, int32_t transA,
                               int32_t transB, const float* A, const float* Bm, float* C, void* stream) {
  if (!A || !Bm || !C || batch < 1) return fail(SACEO_E_INVALID, "bad argument");
  GemmP p{}; p.nnet = 1; p.A = A; p.B = Bm; p.C = C; p.M = M; p.N = N; p.K = K;
  p.lda = transA ? M : K; p.ldb = transB ? K : N; p.ldc = N;
  p.sAa = (long long)M * K; p.sBa = (long long)K * N; p.sCa = (long long)M * N; p.epi = EPI_NONE;
  saceo_ctx tmp; tmp.tc = (gemm_mode & 0xff) == SACEO_GEMM_TCGEN05_BF16X3; tmp.tc_variant = (gemm_mode >> 8) & 0xff;
  if (tmp.tc) {
    CU(tc_gemm_init());
    if (!tc_gemm_eligible(transA != 0, transB != 0, false, p))
      return fail(SACEO_E_INVALID, "shape not eligible for the tcgen05 engine");
  }
  int rc = gemm(&tmp, transA != 0, transB != 0, false, p, batch, (cudaStream_t)stream); if (rc) return rc;
  return check_launch();
}

extern "C" int saceo_test_gemm_ex(const saceo_gemm_args* a, saceo_gemm_route* route, void* stream) {
  if (!a || !route || !a->A || !a->B || !a->C || a->n_agents < 1 || a->nnet < 1) return fail(SACEO_E_INVALID, "bad argument");
  if (a->ones && !a->transA) return fail(SACEO_E_INVALID, "the ones row needs transA");
  const bool TA = a->transA != 0, TB = a->transB != 0, ONES = a->ones != 0;
  GemmP p{};
  p.A = a->A; p.B = a->B; p.C = a->C; p.bias = a->bias; p.addend = a->addend; p.aux = a->aux;
  p.M = a->M; p.N = a->N; p.K = a->K; p.lda = a->lda; p.ldb = a->ldb; p.ldc = a->ldc;
  p.sAa = a->sAa; p.sAn = a->sAn; p.sBa = a->sBa; p.sBn = a->sBn; p.sCa = a->sCa; p.sCn = a->sCn; p.sba = a->sba; p.sbn = a->sbn;
  p.nnet = a->nnet; p.epi = a->epi; p.act = a->act; p.f16 = a->f16;
  saceo_ctx tmp; tmp.tc = (a->gemm_mode & 0xff) == SACEO_GEMM_TCGEN05_BF16X3; tmp.tc_variant = (a->gemm_mode >> 8) & 0xff;
  tmp.prof = true;        // count_launch records each launch's name: the route report
  if (tmp.tc) CU(tc_gemm_init());
  *route = saceo_gemm_route{};
  const bool tc = tmp.tc && p.M > 0 && p.N > 0 && p.K > 0 && tc_gemm_eligible(TA, TB, ONES, p);
  if (tc) {
    const TcRoute r = tc_route(TA, TB, p, tmp.tc_variant);
    route->tc_rows = tc_rows(ONES, p);
    route->tc_stream = r.stream; route->tc_akc = r.akc; route->tc_bkc = r.bkc;
    route->tc_bn = r.bn; route->tc_stages = r.stages; route->tc_threads = r.threads;
  }
  int rc = gemm(&tmp, TA, TB, ONES, p, a->n_agents, (cudaStream_t)stream);
  for (size_t i = 0; i < tmp.prof_n; ++i) {
    const std::string name = tmp.prof_name[i];
    if (name == "k_gemm_tc") route->n_tc++;
    else if (name == "k_gemm_skinny") route->n_skinny++;
    else if (name == "k_gemm_simt") route->n_simt++;
  }
  for (cudaEvent_t e : tmp.prof_ev) cudaEventDestroy(e);
  if (rc) return rc;
  return check_launch();
}

extern "C" int saceo_test_mlp_ws(const saceo_mlp_ws_args* a, saceo_mlp_ws_route* route, void* stream) {
  if (!a || !route || !a->theta || !a->X || !a->H[0] || !a->H[1] || a->n_agents < 1 || a->nnet < 1 || a->rows < 1 ||
      a->rowsAllocH < a->rows || a->hnets < a->nnet || a->in < 1 || a->nout < 1 || (!a->out && !a->dout))
    return fail(SACEO_E_INVALID, "bad argument");
  for (int l = 0; l < 2; ++l)
    if (a->hidden[l] < 1 || a->act[l] < 0 || a->act[l] > 2) return fail(SACEO_E_INVALID, "bad hidden layer %d", l);
  if (a->dout && (!a->dH[0] || !a->dH[1] || a->kout < 1 || a->kout > a->nout || (a->dXa && (a->A_cols < 1 || a->A_cols > a->in))))
    return fail(SACEO_E_INVALID, "bad backward argument");
  if (a->planes && a->nnet > 1 && a->sTa != a->nnet * a->sTn)
    return fail(SACEO_E_INVALID, "the plane image needs the nets of an agent at consecutive theta strides");
  const cudaStream_t st = (cudaStream_t)stream;
  saceo_ctx tmp;
  tmp.cfg.n_agents = a->n_agents;
  tmp.tc = tmp.fuse_fwd = tmp.fuse_bwd = tmp.ws_kernels = true;
  tmp.prof = true;        // count_launch records each launch's name: the route report
  tmp.dbpart = a->dbpart; tmp.dbpart_cap = a->dbpart_cap;
  CU(tc_gemm_init());
  CU(mlp_ws_init());
  NetD n = net_desc(a->theta, a->sTa, a->sTn, a->nnet, a->in, a->nout, 2, a->hidden, a->act);
  if (a->planes && n.ws()) {   // the image, built by the launch ensure_planes uses, for nets the fused kernels take
    n.planes = a->planes; n.pn = ws_image_bytes(a->in, a->nout); n.pa = a->nnet * n.pn;
    planes_build(a->theta, a->nnet > 1 ? a->sTn : a->sTa, a->planes, a->in, a->nout, a->n_agents * a->nnet, st);
  }
  float* H[2] = {a->H[0], a->H[1]};
  float* dH[2] = {a->dH[0], a->dH[1]};
  Pass ps{n, a->X, a->ldx, a->sXa, a->sXn, a->rows, a->rowsAllocH, H, dH};
  ps.hnets = a->hnets; ps.dout_cols = a->kout;
  plane_path(&tmp, ps, a->H1p, a->dH2p, a->dH1p, a->sQa, a->sQn);
  *route = saceo_mlp_ws_route{};
  route->plane_path = ps.H1p != nullptr;
  int rc = 0;
  if (a->out) rc = mlp_forward(&tmp, ps, a->out, a->ldo, a->sOa, a->sOn, st, a->save_h != 0);
  if (!rc && a->dout)
    rc = mlp_backward(&tmp, ps, a->dout, a->ldd, a->sDa, a->sDn, a->grads, a->dXa, a->A_cols, a->sXaA, a->sXaN, st);
  route->bwd_ng = tmp.bwd_variant.ng; route->bwd_na = tmp.bwd_variant.na; route->bwd_mode = tmp.bwd_variant.mode;
  for (size_t i = 0; i < tmp.prof_n; ++i) {
    const std::string name = tmp.prof_name[i];
    if (name == "k_mlp_fwd_ws") route->n_fwd_ws++;
    else if (name == "k_mlp_bwd_ws") route->n_bwd_ws++;
    else if (name == "k_dw_planes") route->n_dw_planes++;
    else if (name == "k_dw0_planes") route->n_dw0_planes++;
    else if (name == "k_bias_finish") route->n_bias_finish++;
    else if (name == "k_gemm_tc") route->n_tc++;
    else if (name == "k_gemm_skinny") route->n_skinny++;
    else if (name == "k_gemm_simt") route->n_simt++;
  }
  for (cudaEvent_t e : tmp.prof_ev) cudaEventDestroy(e);
  if (rc) return rc;
  return check_launch();
}
