// engine.cu -- host side of libmcmcgpu.so: the C ABI of include/mcmcgpu.h (contexts, models, runs).
// No CPU fallback exists: every compute entry point needs a CUDA device and fails with
// MCMCGPU_E_CUDA otherwise.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "common.cuh"
#include "fused_chain.h"
#include "k1_regress.h"
#include "nccl_dyn.h"
#include "population.h"
#include "stats.h"
#include "transition.h"
#include "zv.h"

using namespace mg;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(x)                                                                                      \
  do {                                                                                             \
    cudaError_t e__ = (x);                                                                         \
    if (e__ != cudaSuccess)                                                                        \
      return fail(MCMCGPU_E_CUDA, std::string("CUDA: ") + cudaGetErrorString(e__) + " at " + __FILE__ + ":" + std::to_string(__LINE__)); \
  } while (0)

struct mcmcgpu_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  NcclComm comm = nullptr;
  int rank = 0, nranks = 1;
  int64_t time_eval = 0;      // option: time every likelihood launch with events
  int64_t poll_every = 0;     // option: waves between completion polls (HMCDA / NUTS / tuned HMC); 0 = automatic
  int64_t force_splits = 0;   // option: override K1 row splits
  int64_t k1_debug = 0;       // option (experiments): see K1Args::debug
  int64_t use_graphs = 1;     // option: replay fixed-length wave loops from a CUDA graph
  int64_t fuse_leap = 1;      // option: interior leapfrog updates inside the likelihood kernel when it runs unsplit
  int32_t* h_remaining = nullptr;  // pinned
  cudaMemPool_t pool = nullptr;    // this context's own stream-ordered pool (the device's default pool is left alone)
};

struct mcmcgpu_model {
  mcmcgpu_ctx* ctx = nullptr;
  int family = 0;
  int64_t N = 0, d = 0;
  double hyper[4] = {0, 0, 0, 0};
  double k1_hyper[4] = {0, 0, 0, 0};
  double* d_series = nullptr;
  K1Pack pack;
  bool is_regression = false;
  bool row_sharded = false;
  ModelDev dev() const {
    ModelDev M; M.family = family; M.N = N; M.d = d;
    for (int i = 0; i < 4; i++) M.hyper[i] = hyper[i];
    M.series = d_series;
    return M;
  }
};

// Run and temporary buffers come from a stream-ordered memory pool owned by the context (cudaMemPoolCreate;
// cudaMallocFromPoolAsync / cudaFreeAsync on the context's stream): with a release threshold the pool keeps freed blocks, so
// creating, fetching and destroying a run costs no cudaMalloc / cudaFree round trips to the driver (measured on a 5-step
// cfg3 run: fetch 6..400 ms -> a few ms).  The pool is private: other users of the device's default pool in the same
// process (e.g. PyTorch's cudaMallocAsync backend) keep their own threshold and cached blocks.
// t_stream / t_pool belong to the context the current API call works on (set by use_ctx at every entry point).
static thread_local cudaStream_t t_stream = nullptr;
static thread_local cudaMemPool_t t_pool = nullptr;
static cudaError_t use_ctx(const mcmcgpu_ctx* c);
template <typename T>
static cudaError_t dalloc(T** p, size_t n) { return cudaMallocFromPoolAsync((void**)p, sizeof(T) * (n ? n : 1), t_pool, t_stream); }
static void dfree(void* p) { if (p) cudaFreeAsync(p, t_stream); }

struct mcmcgpu_run {
  mcmcgpu_model* m = nullptr;
  mcmcgpu_sampler_cfg s;
  mcmcgpu_runner_cfg r;
  int engine = 0;
  int64_t C = 0, Cp = 0, S = 0, d = 0;
  bool executed = false;     // at least one execute call has run
  bool started = false;      // the init wave has run
  bool has_diag = false;
  int64_t step0 = 0;         // chains start at step step0 + 1 (mcmcgpu_run_set_state)
  int64_t step_limit = 0;    // last step the chains have been allowed to run so far
  bool restore_da = false;
  // inputs
  double *init = nullptr, *scale = nullptr, *inj_normals = nullptr, *inj_uniforms = nullptr;
  // outputs
  double *samples = nullptr, *grads = nullptr, *logtarget = nullptr, *eps = nullptr, *final_eps = nullptr;
  uint8_t* accept = nullptr;
  int32_t *nleaps = nullptr, *status = nullptr;
  unsigned long long* n_evals = nullptr;
  // wave state
  double *rb = nullptr, *rb_acc = nullptr;
  double *stream = nullptr, *stream_accept = nullptr;   // streamed summaries (stream_stats) instead of stored draws
  double* init_lt = nullptr;   // log-target at the initial point (the `reset` evaluation of the population runners)
  const int64_t* chain_ids = nullptr;   // per-chain Philox keys (population runners that regroup replicas); not owned
  double *ram_S = nullptr, *ram_al = nullptr, *ram_Sb = nullptr, *ram_scratch = nullptr;
  uint8_t* ram_pending = nullptr;
  double *q = nullptr, *part = nullptr, *red = nullptr, *cur_pars = nullptr, *cur_grad = nullptr, *cur_lt = nullptr,
         *mom = nullptr, *H0 = nullptr, *eps_cur = nullptr, *da_leapstep = nullptr, *da_dual = nullptr, *da_dualH = nullptr,
         *tn_step = nullptr;
  int32_t *phase = nullptr, *leap = nullptr, *nleaps_cur = nullptr, *remaining = nullptr;
  int64_t *istep = nullptr, *kept = nullptr, *tn_nleaps = nullptr, *tn_acc = nullptr, *tn_prop = nullptr;
  uint8_t *need_ll = nullptr, *k1_done = nullptr;
  NutsState nuts{};          // NUTS runs only
  bool adapt_metric = false; // NUTS: mcmcgpu_run_set_metric_adaptation was called
  bool nuts_multinomial = false;   // NUTS: mcmcgpu_run_set_nuts_transition(MCMCGPU_NUTS_MULTINOMIAL)
  int nsplit = 1;
  std::vector<void*> owned, owned_big;
  template <typename T>
  cudaError_t alloc(T** p, size_t n, bool zero = true) {
    // the pool for the many small state arrays; plain cudaMalloc for the few large output arrays (growing the pool by
    // gigabytes costs more than cudaMalloc: cfg2's 3.7 GB of kept draws, 0.11 s -> 0.22 s end to end when pooled)
    const bool big = sizeof(T) * n >= (256ull << 20);
    cudaError_t e = big ? cudaMalloc((void**)p, sizeof(T) * n) : dalloc(p, n);
    if (e != cudaSuccess) return e;
    (big ? owned_big : owned).push_back((void*)*p);
    if (zero) return cudaMemsetAsync(*p, 0, sizeof(T) * (n ? n : 1), m->ctx->stream);
    return cudaSuccess;
  }
};

static cudaError_t use_ctx(const mcmcgpu_ctx* c) { t_stream = c->stream; t_pool = c->pool; return cudaSetDevice(c->device); }

// ------------------------------------------------------------------------------------------------
struct Events {    // CUDA events destroyed on scope exit (every return path of the CU() macro included)
  std::vector<cudaEvent_t> v;
  ~Events() { for (cudaEvent_t e : v) cudaEventDestroy(e); }
  cudaError_t make(cudaEvent_t* e) {
    cudaError_t rc = cudaEventCreate(e);
    if (rc == cudaSuccess) v.push_back(*e);
    return rc;
  }
};
struct DevBufs {   // frees everything on scope exit
  std::vector<void*> v;
  ~DevBufs() { for (void* p : v) dfree(p); }
  template <typename T> cudaError_t get(T** p, size_t n, cudaStream_t st, bool zero = true) {
    cudaError_t e = dalloc(p, n);
    if (e != cudaSuccess) return e;
    v.push_back((void*)*p);
    return zero ? cudaMemsetAsync(*p, 0, sizeof(T) * (n ? n : 1), st) : cudaSuccess;
  }
  template <typename T> cudaError_t up(T** p, const T* host, size_t n, cudaStream_t st) {
    cudaError_t e = get(p, n, st, false);
    if (e != cudaSuccess) return e;
    return cudaMemcpyAsync(*p, host, sizeof(T) * n, cudaMemcpyHostToDevice, st);
  }
};


extern "C" {

int32_t mcmcgpu_abi_version(void) { return MCMCGPU_ABI_VERSION; }
const char* mcmcgpu_last_error(void) { return g_err.c_str(); }

int32_t mcmcgpu_destroy(mcmcgpu_ctx* c);
int32_t mcmcgpu_init(int32_t device_id, mcmcgpu_ctx** out) {
  if (!out) return fail(MCMCGPU_E_ARG, "out is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(MCMCGPU_E_CUDA, std::string("no CUDA device available (libmcmcgpu has no CPU fallback): ") +
                                    (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
  if (device_id < 0) CU(cudaGetDevice(&device_id));
  if (device_id >= n) return fail(MCMCGPU_E_ARG, "device_id out of range");
  CU(cudaSetDevice(device_id));
  mcmcgpu_ctx* c = new mcmcgpu_ctx();
  c->device = device_id;
  cudaError_t e2 = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (e2 == cudaSuccess) e2 = cudaMallocHost((void**)&c->h_remaining, sizeof(int32_t));
  if (e2 == cudaSuccess) {
    // a private pool that keeps up to 2 GB of freed run / temporary buffers (dalloc / dfree above)
    cudaMemPoolProps props;
    memset(&props, 0, sizeof(props));
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device_id;
    e2 = cudaMemPoolCreate(&c->pool, &props);
    uint64_t keep = 2ull << 30;
    if (e2 == cudaSuccess) e2 = cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  if (e2 != cudaSuccess) {
    mcmcgpu_destroy(c);
    return fail(MCMCGPU_E_CUDA, std::string("CUDA: ") + cudaGetErrorString(e2) + " in mcmcgpu_init");
  }
  *out = c;
  return MCMCGPU_OK;
}

int32_t mcmcgpu_destroy(mcmcgpu_ctx* c) {
  if (!c) return MCMCGPU_OK;
  use_ctx(c);
  if (c->comm) { const NcclApi* api = nccl_api(nullptr); if (api) api->CommDestroy(c->comm); }
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->pool) cudaMemPoolDestroy(c->pool);              // cached blocks back to the driver
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  if (c->h_remaining) cudaFreeHost(c->h_remaining);
  delete c;
  return MCMCGPU_OK;
}

int32_t mcmcgpu_set_stream(mcmcgpu_ctx* c, void* cuda_stream) {
  if (!c) return fail(MCMCGPU_E_ARG, "ctx is NULL");
  CU(use_ctx(c));
  if (c->stream) cudaStreamSynchronize(c->stream);      // everything allocated / queued in the old stream's order is complete
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  if (cuda_stream) { c->stream = (cudaStream_t)cuda_stream; c->own_stream = false; }
  else { CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)); c->own_stream = true; }
  t_stream = c->stream;
  return MCMCGPU_OK;
}

int32_t mcmcgpu_set_option(mcmcgpu_ctx* c, const char* key, int64_t value) {
  if (!c || !key) return fail(MCMCGPU_E_ARG, "ctx/key is NULL");
  std::string k(key);
  if (k == "time_eval") c->time_eval = value;
  else if (k == "poll_every") c->poll_every = value < 0 ? 0 : value;
  else if (k == "force_splits") c->force_splits = value;
  else if (k == "k1_debug") c->k1_debug = value;
  else if (k == "use_graphs") c->use_graphs = value;
  else if (k == "fuse_leap") c->fuse_leap = value;
  else return fail(MCMCGPU_E_ARG, "unknown option " + k);
  return MCMCGPU_OK;
}

int32_t mcmcgpu_comm_unique_id(void* out128) {
  if (!out128) return fail(MCMCGPU_E_ARG, "out128 is NULL");
  const char* err = nullptr;
  const NcclApi* api = nccl_api(&err);
  if (!api) return fail(MCMCGPU_E_COMM, err ? err : "NCCL unavailable");
  NcclUniqueId id;
  int rc = api->GetUniqueId(&id);
  if (rc != 0) return fail(MCMCGPU_E_COMM, std::string("ncclGetUniqueId: ") + (api->GetErrorString ? api->GetErrorString(rc) : "error"));
  memcpy(out128, &id, sizeof(id));
  return MCMCGPU_OK;
}

int32_t mcmcgpu_comm_init(mcmcgpu_ctx* c, int32_t rank, int32_t nranks, const void* unique_id128) {
  if (!c || !unique_id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(MCMCGPU_E_ARG, "bad comm arguments");
  const char* err = nullptr;
  const NcclApi* api = nccl_api(&err);
  if (!api) return fail(MCMCGPU_E_COMM, err ? err : "NCCL unavailable");
  CU(use_ctx(c));
  NcclUniqueId id;
  memcpy(&id, unique_id128, sizeof(id));
  int rc = api->CommInitRank(&c->comm, nranks, id, rank);
  if (rc != 0) return fail(MCMCGPU_E_COMM, std::string("ncclCommInitRank: ") + (api->GetErrorString ? api->GetErrorString(rc) : "error"));
  c->rank = rank; c->nranks = nranks;
  return MCMCGPU_OK;
}

// ---- model ---------------------------------------------------------------------------------------
static int model_create_impl(mcmcgpu_ctx* c, int32_t family, int64_t N, int64_t d, const double* X, const double* y,
                             const double* hyper, int32_t nhyper, int32_t row_sharded, bool on_device, mcmcgpu_model** out) {
  if (!c || !out) return fail(MCMCGPU_E_ARG, "ctx/out is NULL");
  if (d < 1) return fail(MCMCGPU_E_ARG, "d must be >= 1");
  if (nhyper < 0 || nhyper > 4 || (nhyper > 0 && !hyper)) return fail(MCMCGPU_E_ARG, "bad hyper");
  CU(use_ctx(c));
  mcmcgpu_model* m = new mcmcgpu_model();
  // released on every failing return below (validation errors and failing CUDA calls alike)
  struct Guard { mcmcgpu_model* m; ~Guard() { if (m) { k1_free(m->pack); if (m->d_series) dfree(m->d_series); delete m; } } } guard{m};
  m->ctx = c; m->family = family; m->N = N; m->d = d;
  for (int i = 0; i < nhyper; i++) m->hyper[i] = hyper[i];
  switch (family) {
    case MCMCGPU_FAM_NORMAL_FN: m->N = 0; break;
    case MCMCGPU_FAM_ABS_NORMAL:
    case MCMCGPU_FAM_NORMAL_DSL:
      m->N = 0;
      if (nhyper < 2) { m->hyper[0] = 0.0; m->hyper[1] = 1.0; }
      if (!(m->hyper[1] > 0)) { return fail(MCMCGPU_E_ARG, "Normal sigma must be > 0"); }
      break;
    case MCMCGPU_FAM_LINEAR:
      if (nhyper < 1) m->hyper[0] = 1.0;
      if (nhyper < 2) m->hyper[1] = 1.0;
      m->is_regression = true; break;
    case MCMCGPU_FAM_LOGISTIC:
      if (nhyper < 1) m->hyper[0] = 1.0;
      if (nhyper < 2) m->hyper[1] = -1.0;
      // the two conventions of the reference: exp(-X*vars) (examples/logistic_regression.jl:18) and exp(X*vars)
      // (test/test_syntax.jl:18); K1 folds this sign into beta, which is exact only for +-1
      if (m->hyper[1] != 1.0 && m->hyper[1] != -1.0) { return fail(MCMCGPU_E_ARG, "logistic sign must be +1 or -1"); }
      m->is_regression = true; break;
    case MCMCGPU_FAM_PROBIT:
      if (nhyper < 1) m->hyper[0] = 10.0;
      m->is_regression = true; break;
    case MCMCGPU_FAM_OU:
      if (d != 3) { return fail(MCMCGPU_E_ARG, "Ornstein-Uhlenbeck has 3 parameters (tau, sigma, mu)"); }
      if (nhyper < 3) { m->hyper[0] = 100.0; m->hyper[1] = 2.0; m->hyper[2] = 20.0; }
      if (!y || N < 2) { return fail(MCMCGPU_E_ARG, "OU needs a series of length >= 2 in y"); }
      break;
    default: return fail(MCMCGPU_E_ARG, "unknown family");
  }
  if (m->is_regression) {
    if (!X || !y || N < 1) { return fail(MCMCGPU_E_ARG, "regression families need X (N x d) and y (N)"); }
    if (!(m->hyper[0] > 0)) { return fail(MCMCGPU_E_ARG, "prior sd must be > 0"); }
    if (!k1_supported(d)) { return fail(MCMCGPU_E_ARG, "regression families support 1 <= d <= 200 in this build"); }
    if (row_sharded && !c->comm) { return fail(MCMCGPU_E_COMM, "row_sharded model needs mcmcgpu_comm_init first"); }
    m->row_sharded = row_sharded != 0;
    if (on_device) {
      CU(k1_pack(m->pack, X, y, N, d, c->stream));
      CU(cudaStreamSynchronize(c->stream));
    } else {
      double *dX = nullptr, *dy = nullptr;
      DevBufs staging;                       // the column-major upload lives only until the tile images are packed
      CU(staging.up(&dX, X, (size_t)(N * d), c->stream));
      CU(staging.up(&dy, y, (size_t)N, c->stream));
      CU(k1_pack(m->pack, dX, dy, N, d, c->stream));
      CU(cudaStreamSynchronize(c->stream));
    }
    for (int i = 0; i < 4; i++) m->k1_hyper[i] = m->hyper[i];
    if (family == MCMCGPU_FAM_LINEAR) m->k1_hyper[3] = std::log(m->hyper[1]);
  }
  if (family == MCMCGPU_FAM_OU) {
    CU(dalloc(&m->d_series, (size_t)N));
    CU(cudaMemcpyAsync(m->d_series, y, sizeof(double) * (size_t)N, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  guard.m = nullptr;
  *out = m;
  return MCMCGPU_OK;
}

int32_t mcmcgpu_model_create(mcmcgpu_ctx* c, int32_t family, int64_t N, int64_t d, const double* X, const double* y,
                             const double* hyper, int32_t nhyper, int32_t row_sharded, mcmcgpu_model** out) {
  return model_create_impl(c, family, N, d, X, y, hyper, nhyper, row_sharded, false, out);
}

int32_t mcmcgpu_model_create_device(mcmcgpu_ctx* c, int32_t family, int64_t N, int64_t d, const double* X_dev,
                                    const double* y_dev, const double* hyper, int32_t nhyper, int32_t row_sharded,
                                    mcmcgpu_model** out) {
  return model_create_impl(c, family, N, d, X_dev, y_dev, hyper, nhyper, row_sharded, true, out);
}

int32_t mcmcgpu_model_destroy(mcmcgpu_model* m) {
  if (!m) return MCMCGPU_OK;
  use_ctx(m->ctx);
  k1_free(m->pack);
  if (m->d_series) dfree(m->d_series);
  delete m;
  return MCMCGPU_OK;
}

}  // extern "C"

// one evaluation of every chain at q -> part (and the all-reduce for row-sharded models)
static int eval_wave(mcmcgpu_model* m, const double* q, double* part, double* red, int nsplit, int64_t C, int64_t Cp,
                     bool need_grad, const uint8_t* need_ll, const int32_t* phase, const int32_t* remaining,
                     const double** part_out, int* nsplit_out, cudaEvent_t ev_k1_done = nullptr, const mcmcgpu_run* fuse = nullptr) {
  cudaStream_t st = m->ctx->stream;
  *part_out = part; *nsplit_out = nsplit;
  if (m->is_regression) {
    K1Args a;
    a.P = m->pack; a.family = m->family;
    for (int i = 0; i < 4; i++) a.hyper[i] = m->k1_hyper[i];
    a.q = q; a.part = part; a.Cp = Cp; a.nsplit = nsplit; a.need_grad = need_grad ? 1 : 0;
    a.need_ll = need_ll; a.phase = phase; a.remaining = remaining; a.debug = (int32_t)m->ctx->k1_debug;
    a.fuse_leap = 0; a.leap = nullptr; a.nleaps_cur = nullptr; a.eps_cur = nullptr; a.mom = nullptr; a.q_rw = nullptr;
    a.need_ll_rw = nullptr; a.k1_done = nullptr; a.n_evals = nullptr;
    if (fuse) {      // interior leapfrogs made by the likelihood kernel itself (run_fuses_leap)
      a.fuse_leap = 1; a.leap = fuse->leap; a.nleaps_cur = fuse->nleaps_cur; a.eps_cur = fuse->eps_cur; a.mom = fuse->mom; a.q_rw = fuse->q;
      a.need_ll_rw = fuse->need_ll; a.k1_done = fuse->k1_done; a.n_evals = fuse->n_evals;
    }
    CU(k1_launch(a, st));
    if (ev_k1_done) CU(cudaEventRecord(ev_k1_done, st));   // what follows (split fold, all-reduce) is timed apart: run_info.comm_ms
    if (!m->row_sharded && nsplit > 4 && red) {
      // many row splits (small problems spread over the whole machine): fold them with a parallel pass, in split order,
      // so the per-chain transition thread does not walk nsplit partial buffers serially
      CU(launch_reduce_splits(part, nsplit, m->d + 2, Cp, red, st));
      *part_out = red; *nsplit_out = 1;
    }
    if (m->row_sharded) {
      const NcclApi* api = nccl_api(nullptr);
      if (!api || !m->ctx->comm) return fail(MCMCGPU_E_COMM, "communicator not initialised");
      CU(launch_reduce_splits(part, nsplit, m->d + 2, Cp, red, st));
      int rc = api->AllReduce(red, red, (size_t)((m->d + 2) * Cp), NCCL_FLOAT64, NCCL_SUM, m->ctx->comm, st);
      if (rc != 0) return fail(MCMCGPU_E_COMM, std::string("ncclAllReduce: ") + (api->GetErrorString ? api->GetErrorString(rc) : "error"));
      *part_out = red; *nsplit_out = 1;
    }
  } else {
    CU(launch_eval_closed(m->dev(), q, part, C, Cp, phase, remaining, st));
    if (ev_k1_done) CU(cudaEventRecord(ev_k1_done, st));
    *nsplit_out = 1;
  }
  return MCMCGPU_OK;
}

static int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

extern "C" {

int32_t mcmcgpu_logtarget_grad(mcmcgpu_model* m, const double* B, int64_t C, double* out_lt, double* out_grad) {
  if (!m || !B || !out_lt || C < 1) return fail(MCMCGPU_E_ARG, "bad arguments");
  mcmcgpu_ctx* c = m->ctx;
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  const int64_t d = m->d, Cp = round_up(C, K1_CHAINS);
  int nsplit = m->is_regression ? (c->force_splits > 0 ? (int)c->force_splits : k1_choose_splits(m->pack, Cp, -1, m->family)) : 1;
  double *hB = nullptr, *q = nullptr, *part = nullptr, *red = nullptr, *lt = nullptr, *grad = nullptr, *gout = nullptr;
  struct Freer { double** p[7]; ~Freer() { for (auto pp : p) if (*pp) { dfree(*pp); *pp = nullptr; } } } freer{{&hB, &q, &part, &red, &lt, &grad, &gout}};
  CU(dalloc(&hB, (size_t)(C * d)));
  CU(dalloc(&q, (size_t)(d * Cp)));
  CU(dalloc(&part, (size_t)(nsplit * (d + 2) * Cp)));
  CU(dalloc(&red, (size_t)((d + 2) * Cp)));
  CU(dalloc(&lt, (size_t)Cp));
  CU(dalloc(&grad, (size_t)(d * Cp)));
  CU(dalloc(&gout, (size_t)(C * d)));
  CU(cudaMemsetAsync(q, 0, sizeof(double) * (size_t)(d * Cp), st));
  CU(cudaMemcpyAsync(hB, B, sizeof(double) * (size_t)(C * d), cudaMemcpyHostToDevice, st));
  CU(transpose_to_chain_minor(hB, q, C, d, Cp, st));
  const double* pp; int ns;
  int rc = eval_wave(m, q, part, red, nsplit, C, Cp, out_grad != nullptr, nullptr, nullptr, nullptr, &pp, &ns);
  if (rc != MCMCGPU_OK) return rc;
  CU(launch_finalize(m->dev(), q, pp, ns, C, Cp, lt, out_grad ? grad : nullptr, st));
  CU(cudaMemcpyAsync(out_lt, lt, sizeof(double) * (size_t)C, cudaMemcpyDeviceToHost, st));
  if (out_grad) {
    CU(transpose_to_chain_major(grad, gout, 0, C, d, Cp, st));
    CU(cudaMemcpyAsync(out_grad, gout, sizeof(double) * (size_t)(C * d), cudaMemcpyDeviceToHost, st));
  }
  CU(cudaStreamSynchronize(st));
  return MCMCGPU_OK;   // temporaries are released by `freer` on every path
}

// ---- run -----------------------------------------------------------------------------------------
static int check_cfg(const mcmcgpu_model* m, const mcmcgpu_sampler_cfg* s, const mcmcgpu_runner_cfg* r) {
  // SerialMC.jl:25-27
  if (r->first - 1 < 0) return fail(MCMCGPU_E_ARG, "Burnin rounds should be >= 0");
  if (r->last <= r->first - 1) return fail(MCMCGPU_E_ARG, "Total MCMC length should be > to burnin");
  if (r->step < 1) return fail(MCMCGPU_E_ARG, "Thinning should be >= 1");
  if (r->nchains < 1) return fail(MCMCGPU_E_ARG, "nchains must be >= 1");
  if (r->last >= (1LL << 32) - 1) return fail(MCMCGPU_E_ARG, "at most 2^32-2 steps");
  switch (s->kind) {
    case MCMCGPU_RWM: if (!(s->scale > 0)) return fail(MCMCGPU_E_ARG, "scale should be > 0"); break;             // RWM.jl:29
    case MCMCGPU_MALA: if (!(s->scale > 0)) return fail(MCMCGPU_E_ARG, "MALA drift step should be > 0"); break;   // MALA.jl:55
    case MCMCGPU_HMC:
      if (s->nleaps <= 0) return fail(MCMCGPU_E_ARG, "inner steps should be > 0");                                // HMC.jl:60
      if (!(s->scale > 0)) return fail(MCMCGPU_E_ARG, "inner steps scaling should be > 0");                       // HMC.jl:61
      break;
    case MCMCGPU_RAM:                                                                                             // RAM.jl:29-30
      if (!(s->scale > 0)) return fail(MCMCGPU_E_ARG, "scale should be > 0");
      if (!(s->rate > 0 && s->rate < 1)) return fail(MCMCGPU_E_ARG, "target acceptance rate should be between 0 and 1");
      break;
    case MCMCGPU_HMCDA:                                                                                           // HMCDA.jl:33-36
      if (!(s->rate > 0 && s->rate < 1)) return fail(MCMCGPU_E_ARG, "Target acceptance rate should be between 0 and 1");
      if (!(s->len > 0)) return fail(MCMCGPU_E_ARG, "len parameter of HMCDA sampler must be non-negative");
      if (!(s->shrinkage > 0)) return fail(MCMCGPU_E_ARG, "shrinkage parameter of HMCDA sampler must be positive");
      if (!(s->t0 >= 0)) return fail(MCMCGPU_E_ARG, "t0 parameter of HMCDA sampler must be non-negative");
      break;
    case MCMCGPU_NUTS:                                                                                            // HMCDA's rules
      if (!(s->rate > 0 && s->rate < 1)) return fail(MCMCGPU_E_ARG, "Target acceptance rate should be between 0 and 1");
      if (!(s->shrinkage > 0)) return fail(MCMCGPU_E_ARG, "shrinkage parameter of NUTS sampler must be positive");
      if (!(s->t0 >= 0)) return fail(MCMCGPU_E_ARG, "t0 parameter of NUTS sampler must be non-negative");
      if (s->nleaps < 1 || s->nleaps > NUTS_MAX_DOUBLINGS) return fail(MCMCGPU_E_ARG, "NUTS maxdoublings should be in 1..10");
      break;
    default: return fail(MCMCGPU_E_ARG, "unknown sampler kind");
  }
  if (s->tuner_on) {
    if (s->kind != MCMCGPU_MALA && s->kind != MCMCGPU_HMC) return fail(MCMCGPU_E_ARG, "EmpMCTuner applies to MALA and HMC");
    if (s->adapt_step <= 0 || s->max_step <= 0 || !(s->target_rate > 0 && s->target_rate < 1))   // samplers.jl:40-43
      return fail(MCMCGPU_E_ARG, "bad EmpMCTuner parameters");
  }
  (void)m;
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_destroy(mcmcgpu_run* run) {
  if (!run) return MCMCGPU_OK;
  use_ctx(run->m->ctx);
  cudaStreamSynchronize(run->m->ctx->stream);
  for (void* p : run->owned) dfree(p);
  for (void* p : run->owned_big) cudaFree(p);          // synchronises: pending work on the buffers is complete
  delete run;
  return MCMCGPU_OK;
}

}  // extern "C"

// init_dev_cm: initial points already on the device, chain-minor [d][Cp] (population runners); overrides `init`
static int run_create_impl(mcmcgpu_model* m, const mcmcgpu_sampler_cfg* s, const mcmcgpu_runner_cfg* r, const double* init,
                           const double* init_dev_cm, const double* scale, const double* inj_normals, const double* inj_uniforms,
                           mcmcgpu_run** out) {
  if (!m || !s || !r || (!init && !init_dev_cm) || !out) return fail(MCMCGPU_E_ARG, "NULL argument");
  int rc = check_cfg(m, s, r);
  if (rc != MCMCGPU_OK) return rc;
  if ((inj_normals == nullptr) != (inj_uniforms == nullptr)) return fail(MCMCGPU_E_ARG, "inject both normals and uniforms or neither");
  mcmcgpu_ctx* c = m->ctx;
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  mcmcgpu_run* R = new mcmcgpu_run();
  R->m = m; R->s = *s; R->r = *r;
  if (init_dev_cm) R->r.init_per_chain = 1;
  r = &R->r;
  if (R->s.max_leaps <= 0) R->s.max_leaps = 1LL << 20;
  const int64_t d = m->d, C = r->nchains, Cp = round_up(C, K1_CHAINS);
  const int64_t S = (r->last - r->first) / r->step + 1;
  R->C = C; R->Cp = Cp; R->S = S; R->d = d;
  int engine = r->engine;
  const bool can_fuse = fused_supported(m->family, d, m->N);
  const bool nuts = s->kind == MCMCGPU_NUTS;
  if (nuts) {
    const char* why = engine == MCMCGPU_ENGINE_FUSED ? "NUTS runs on engine WAVE only (engine FUSED has no NUTS)"
                      : inj_normals ? "NUTS draws its own Philox numbers: injected normals / uniforms are not supported"
                      : r->store_rb ? "storeLeaps applies to HMC / HMCDA" : m->row_sharded ? "NUTS does not support row-sharded models" : nullptr;
    if (why) { delete R; return fail(MCMCGPU_E_ARG, why); }
    engine = MCMCGPU_ENGINE_WAVE;
  }
  if (engine == MCMCGPU_ENGINE_AUTO) engine = can_fuse ? MCMCGPU_ENGINE_FUSED : MCMCGPU_ENGINE_WAVE;
  if (engine == MCMCGPU_ENGINE_FUSED && !can_fuse) { delete R; return fail(MCMCGPU_E_ARG, "engine FUSED supports the closed-form families with d <= 8"); }
  if (engine != MCMCGPU_ENGINE_FUSED && engine != MCMCGPU_ENGINE_WAVE) { delete R; return fail(MCMCGPU_E_ARG, "unknown engine"); }
  R->engine = engine;
  R->has_diag = (s->kind == MCMCGPU_HMCDA) || (s->kind == MCMCGPU_RAM) || nuts || s->tuner_on;
  if (s->kind == MCMCGPU_RAM && engine == MCMCGPU_ENGINE_WAVE && d > RAM_BIG_MAX_D) { delete R; return fail(MCMCGPU_E_ARG, "RAM supports d <= 128"); }
#define RCU(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) { std::string msg = std::string("CUDA: ") + cudaGetErrorString(e__) + " at " + __FILE__ + ":" + std::to_string(__LINE__); mcmcgpu_run_destroy(R); return fail(MCMCGPU_E_CUDA, msg); } } while (0)
  // inputs
  if (init_dev_cm) {
    RCU(R->alloc(&R->init, (size_t)(d * Cp), false));
    RCU(cudaMemcpyAsync(R->init, init_dev_cm, sizeof(double) * (size_t)(d * Cp), cudaMemcpyDeviceToDevice, st));
  } else if (r->init_per_chain) {
    double* tmp = nullptr;
    DevBufs staging;                        // released on every path, the failing ones of RCU included
    RCU(staging.up(&tmp, init, (size_t)(C * d), st));
    RCU(R->alloc(&R->init, (size_t)(d * Cp)));
    RCU(transpose_to_chain_minor(tmp, R->init, C, d, Cp, st));
    RCU(cudaStreamSynchronize(st));
  } else {
    RCU(R->alloc(&R->init, (size_t)d));
    RCU(cudaMemcpyAsync(R->init, init, sizeof(double) * (size_t)d, cudaMemcpyHostToDevice, st));
  }
  {
    std::vector<double> sc((size_t)d, 1.0);
    if (scale) for (int64_t j = 0; j < d; j++) sc[(size_t)j] = scale[j];
    RCU(R->alloc(&R->scale, (size_t)d));
    RCU(cudaMemcpyAsync(R->scale, sc.data(), sizeof(double) * (size_t)d, cudaMemcpyHostToDevice, st));
    RCU(cudaStreamSynchronize(st));
  }
  if (inj_normals) {
    const int64_t K = (r->last + 1) * d, Ku = r->last + 1;
    double *tmp = nullptr, *tmpu = nullptr;
    DevBufs staging;
    RCU(staging.up(&tmp, inj_normals, (size_t)(C * K), st));
    RCU(R->alloc(&R->inj_normals, (size_t)(K * Cp)));
    RCU(transpose_to_chain_minor(tmp, R->inj_normals, C, K, Cp, st));
    RCU(staging.up(&tmpu, inj_uniforms, (size_t)(C * Ku), st));
    RCU(R->alloc(&R->inj_uniforms, (size_t)(Ku * Cp)));
    RCU(transpose_to_chain_minor(tmpu, R->inj_uniforms, C, Ku, Cp, st));
    RCU(cudaStreamSynchronize(st));
  }
  // outputs
  if (r->stream_stats) {
    if (engine != MCMCGPU_ENGINE_FUSED || r->store_grad || r->store_logtarget || r->store_rb || S < 2) {
      mcmcgpu_run_destroy(R);
      return fail(MCMCGPU_E_ARG, "stream_stats needs engine FUSED, at least 2 kept steps and no stored gradients / log-targets / leaps");
    }
    if (R->r.stream_batchlen <= 0) R->r.stream_batchlen = 100;
    RCU(R->alloc(&R->stream, (size_t)(FUSED_STREAM_ROWS * d * Cp)));
    RCU(R->alloc(&R->stream_accept, (size_t)Cp));
  } else {
    RCU(R->alloc(&R->samples, (size_t)(S * d * Cp), false));
    RCU(R->alloc(&R->accept, (size_t)(S * Cp)));
  }
  if (r->store_grad) RCU(R->alloc(&R->grads, (size_t)(S * d * Cp), false));
  if (r->store_logtarget) RCU(R->alloc(&R->logtarget, (size_t)(S * Cp), false));
  if (r->store_rb) {
    if (s->kind != MCMCGPU_HMC && s->kind != MCMCGPU_HMCDA) { mcmcgpu_run_destroy(R); return fail(MCMCGPU_E_ARG, "storeLeaps applies to HMC / HMCDA"); }
    RCU(R->alloc(&R->rb, (size_t)(S * d * Cp), false));
  }
  if (R->has_diag) {
    RCU(R->alloc(&R->eps, (size_t)(S * Cp)));
    RCU(R->alloc(&R->nleaps, (size_t)(S * Cp)));
  }
  RCU(R->alloc(&R->final_eps, (size_t)Cp));
  RCU(R->alloc(&R->status, (size_t)Cp));
  RCU(R->alloc(&R->n_evals, 1));
  if (engine == MCMCGPU_ENGINE_WAVE) {
    R->nsplit = m->is_regression ? (c->force_splits > 0 ? (int)c->force_splits : k1_choose_splits(m->pack, Cp, -1, m->family)) : 1;
    RCU(R->alloc(&R->q, (size_t)(d * Cp)));
    RCU(R->alloc(&R->part, (size_t)(R->nsplit * (d + 2) * Cp)));
    if (m->row_sharded || R->nsplit > 4) RCU(R->alloc(&R->red, (size_t)((d + 2) * Cp)));
    RCU(R->alloc(&R->cur_pars, (size_t)(d * Cp)));
    RCU(R->alloc(&R->cur_grad, (size_t)(d * Cp)));
    RCU(R->alloc(&R->cur_lt, (size_t)Cp));
    RCU(R->alloc(&R->mom, (size_t)(d * Cp)));
    RCU(R->alloc(&R->H0, (size_t)Cp));
    RCU(R->alloc(&R->eps_cur, (size_t)Cp));
    RCU(R->alloc(&R->da_leapstep, (size_t)Cp));
    RCU(R->alloc(&R->da_dual, (size_t)Cp));
    RCU(R->alloc(&R->da_dualH, (size_t)Cp));
    RCU(R->alloc(&R->tn_step, (size_t)Cp));
    RCU(R->alloc(&R->phase, (size_t)Cp));
    RCU(R->alloc(&R->leap, (size_t)Cp));
    RCU(R->alloc(&R->nleaps_cur, (size_t)Cp));
    RCU(R->alloc(&R->remaining, 1));
    RCU(R->alloc(&R->istep, (size_t)Cp));
    RCU(R->alloc(&R->kept, (size_t)Cp));
    RCU(R->alloc(&R->tn_nleaps, (size_t)Cp));
    RCU(R->alloc(&R->tn_acc, (size_t)Cp));
    RCU(R->alloc(&R->tn_prop, (size_t)Cp));
    RCU(R->alloc(&R->need_ll, (size_t)Cp));
    RCU(R->alloc(&R->k1_done, (size_t)Cp));
    RCU(R->alloc(&R->init_lt, (size_t)Cp));
    if (r->store_rb) RCU(R->alloc(&R->rb_acc, (size_t)(d * Cp)));
    if (s->kind == MCMCGPU_RAM && d > RAM_WAVE_MAX_D) {      // one CTA per chain: chain-major factor + 3 work matrices per chain
      RCU(R->alloc(&R->ram_Sb, (size_t)(C * d * d)));
      RCU(R->alloc(&R->ram_scratch, (size_t)(3 * C * d * d), false));
      RCU(R->alloc(&R->ram_al, (size_t)Cp));
      RCU(R->alloc(&R->ram_pending, (size_t)Cp));
    } else if (s->kind == MCMCGPU_RAM) {
      RCU(R->alloc(&R->ram_S, (size_t)(d * d * Cp)));
      RCU(R->alloc(&R->ram_al, (size_t)Cp));
      RCU(R->alloc(&R->ram_pending, (size_t)Cp));
    }
    if (nuts) {      // (8 + 2 (maxdoublings - 1)) d doubles and 10 scalars per chain
      NutsState& T = R->nuts;
      for (int sd = 0; sd < 2; sd++) {
        RCU(R->alloc(&T.th[sd], (size_t)(d * Cp), false));
        RCU(R->alloc(&T.p[sd], (size_t)(d * Cp), false));
        RCU(R->alloc(&T.g[sd], (size_t)(d * Cp), false));
      }
      RCU(R->alloc(&T.sub_pars, (size_t)(d * Cp), false));
      RCU(R->alloc(&T.sub_grad, (size_t)(d * Cp), false));
      RCU(R->alloc(&T.sub_lt, (size_t)Cp));
      RCU(R->alloc(&T.ck_th, (size_t)((s->nleaps - 1) * d * Cp), false));
      RCU(R->alloc(&T.ck_p, (size_t)((s->nleaps - 1) * d * Cp), false));
      RCU(R->alloc(&T.log_u0, (size_t)Cp));
      RCU(R->alloc(&T.alpha, (size_t)Cp));
      RCU(R->alloc(&T.j, (size_t)Cp));
      RCU(R->alloc(&T.leaf, (size_t)Cp));
      RCU(R->alloc(&T.leaps, (size_t)Cp));
      RCU(R->alloc(&T.n, (size_t)Cp));
      RCU(R->alloc(&T.n_sub, (size_t)Cp));
      RCU(R->alloc(&T.dir, (size_t)Cp));
      RCU(R->alloc(&T.moved, (size_t)Cp));
    }
  }
  RCU(cudaStreamSynchronize(st));
  *out = R;
  return MCMCGPU_OK;
}

extern "C" {
int32_t mcmcgpu_run_create(mcmcgpu_model* m, const mcmcgpu_sampler_cfg* s, const mcmcgpu_runner_cfg* r, const double* init,
                           const double* scale, const double* inj_normals, const double* inj_uniforms, mcmcgpu_run** out) {
  if (!init) return fail(MCMCGPU_E_ARG, "NULL argument");
  return run_create_impl(m, s, r, init, nullptr, scale, inj_normals, inj_uniforms, out);
}

static RunnerDev runner_dev(const mcmcgpu_run* R) {
  RunnerDev D;
  D.first = R->r.first; D.step = R->r.step; D.last = R->r.last; D.S = R->S; D.C = R->C; D.Cp = R->Cp;
  D.chain_offset = R->r.chain_offset; D.seed = R->r.seed; D.init_per_chain = R->r.init_per_chain;
  D.store_grad = R->r.store_grad; D.store_lt = R->r.store_logtarget; D.store_rb = R->r.store_rb;
  return D;
}
static SamplerDev sampler_dev(const mcmcgpu_run* R) {
  SamplerDev D;
  const mcmcgpu_sampler_cfg& s = R->s;
  D.kind = s.kind; D.nleaps = s.nleaps; D.scale = s.scale; D.rate = s.rate; D.len = s.len; D.shrinkage = s.shrinkage;
  D.t0 = s.t0; D.step = s.step; D.max_leaps = s.max_leaps; D.tuner_on = s.tuner_on; D.adapt_step = s.adapt_step;
  D.max_step = s.max_step; D.target_path = s.target_path; D.target_rate = s.target_rate;
  return D;
}

__global__ void wave_init_kernel(int32_t* phase, int32_t* remaining, double* q, const double* init, int init_per_chain,
                                 int64_t C, int64_t Cp, int64_t d) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0) *remaining = (int32_t)C;
  if (c >= Cp) return;
  phase[c] = (c < C) ? PH_INIT : PH_DONE;
  for (int64_t j = 0; j < d; j++) q[j * Cp + c] = (c < C) ? (init_per_chain ? init[j * Cp + c] : init[j]) : 0.0;
}

// the multinomial transition's tree state and per-step outputs, at the first execute (when the metric is known)
static int alloc_multinomial(mcmcgpu_run* R) {
  NutsState& T = R->nuts;
  const size_t Cp = (size_t)R->Cp, rec = (size_t)R->s.nleaps * (size_t)R->d * Cp, lev = (size_t)R->s.nleaps * Cp;
  double** recs[] = {&T.mn_rho, &T.mn_pb, &T.mn_pe, &T.mn_th, &T.mn_g};
  for (double** a : recs) CU(R->alloc(a, rec, false));
  if (T.A) {
    CU(R->alloc(&T.mn_vb, rec, false));
    CU(R->alloc(&T.mn_ve, rec, false));
    CU(R->alloc(&T.mn_vin, (size_t)R->d * Cp, false));
  }
  CU(R->alloc(&T.mn_lsw, lev, false)); CU(R->alloc(&T.mn_lt, lev, false)); CU(R->alloc(&T.mn_h, lev, false));
  CU(R->alloc(&T.mn_trho, (size_t)R->d * Cp, false)); CU(R->alloc(&T.mn_pin, (size_t)R->d * Cp, false));
  CU(R->alloc(&T.mn_tlsw, Cp)); CU(R->alloc(&T.mn_sh, Cp));
  CU(R->alloc(&T.st_accept_stat, (size_t)R->S * Cp)); CU(R->alloc(&T.st_energy, (size_t)R->S * Cp));
  CU(R->alloc(&T.st_divergent, (size_t)R->S * Cp));
  return MCMCGPU_OK;
}

// the likelihood kernel can make the interior leapfrog updates itself when one CTA sees all rows of its chains
static bool run_fuses_leap(const mcmcgpu_run* R) {
  const mcmcgpu_model* m = R->m;
  return m->is_regression && !m->row_sharded && R->nsplit == 1 && !R->r.store_rb && m->ctx->fuse_leap &&
         (R->s.kind == MCMCGPU_HMC || R->s.kind == MCMCGPU_HMCDA);
}

static int execute_impl(mcmcgpu_run* R, int64_t nsteps, mcmcgpu_run_info* info) {
  mcmcgpu_model* m = R->m;
  mcmcgpu_ctx* c = m->ctx;
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  const int64_t from = R->started ? R->step_limit : R->step0;
  if (from >= R->r.last) return fail(MCMCGPU_E_STATE, "run has already reached its last step");
  int64_t upto = (nsteps < 0 || from + nsteps > R->r.last) ? R->r.last : from + nsteps;
  const int64_t seg = upto - from;
  if (seg <= 0) return fail(MCMCGPU_E_ARG, "nsteps must be >= 1");
  Events events;
  cudaEvent_t e0, e1;
  CU(events.make(&e0)); CU(events.make(&e1));
  int64_t launches = 0, waves = 0;
  double eval_ms = 0.0, comm_ms = 0.0;
  CU(cudaMemsetAsync(R->n_evals, 0, sizeof(unsigned long long), st));
  CU(cudaEventRecord(e0, st));
  if (R->engine == MCMCGPU_ENGINE_FUSED) {
    if (R->started || upto != R->r.last || R->step0 != 0)
      return fail(MCMCGPU_E_STATE, "engine FUSED runs the whole chain in one launch: use mcmcgpu_run_execute, or engine WAVE for stepwise execution");
    FusedArgs A;
    A.M = m->dev(); A.S = sampler_dev(R); A.R = runner_dev(R);
    A.init = R->init; A.scale = R->scale; A.inj_normals = R->inj_normals; A.inj_uniforms = R->inj_uniforms;
    A.samples = R->samples; A.grads = R->grads; A.accept = R->accept; A.logtarget = R->logtarget;
    A.eps = R->eps; A.nleaps = R->nleaps; A.final_eps = R->final_eps; A.final_pars = nullptr; A.rb = R->rb;
    A.status = R->status; A.n_evals = R->n_evals;
    A.stream = R->stream; A.stream_accept = R->stream_accept; A.stream_batchlen = R->r.stream_batchlen;
    CU(launch_fused(A, st));
    launches = 1;
    R->started = true;
  } else {
    if (R->nuts_multinomial && !R->nuts.mn_rho) {
      int rc = alloc_multinomial(R);
      if (rc) return rc;
    }
    WaveArgs W;
    W.M = m->dev(); W.S = sampler_dev(R); W.R = runner_dev(R);
    const mcmcgpu_run* fuse = run_fuses_leap(R) ? R : nullptr;
    W.fused_interior = fuse ? 1 : 0; W.k1_done = R->k1_done;
    // fixed-length HMC with the fused interior leapfrog: all chains of a run move in lockstep (they pause only between
    // steps), so on the waves that evaluate an interior leapfrog -- all but every nleaps-th -- the likelihood kernel does
    // everything and the transition kernel is not launched at all
    const bool lockstep = fuse && R->s.kind == MCMCGPU_HMC && !R->s.tuner_on;
    int64_t leap_pos = 0;                    // evaluations already made in the current step (0 .. nleaps-1)
    W.nsplit = R->nsplit; W.resume = 0; W.restore_da = R->restore_da ? 1 : 0; W.step0 = R->step0; W.step_limit = upto;
    W.q = R->q; W.part = R->part;
    W.cur_pars = R->cur_pars; W.cur_grad = R->cur_grad; W.cur_lt = R->cur_lt; W.mom = R->mom; W.H0 = R->H0;
    W.phase = R->phase; W.leap = R->leap; W.nleaps_cur = R->nleaps_cur; W.istep = R->istep; W.kept = R->kept;
    W.eps_cur = R->eps_cur; W.da_leapstep = R->da_leapstep; W.da_dual = R->da_dual; W.da_dualH = R->da_dualH;
    W.tn_step = R->tn_step; W.tn_nleaps = R->tn_nleaps; W.tn_acc = R->tn_acc; W.tn_prop = R->tn_prop;
    W.ram_S = R->ram_S; W.ram_al = R->ram_al; W.ram_pending = R->ram_pending; W.ram_Sb = R->ram_Sb; W.ram_scratch = R->ram_scratch;
    W.need_ll = R->need_ll; W.status = R->status; W.remaining = R->remaining; W.n_evals = R->n_evals;
    W.init = R->init; W.scale = R->scale; W.inj_normals = R->inj_normals; W.inj_uniforms = R->inj_uniforms;
    W.samples = R->samples; W.grads = R->grads; W.accept = R->accept; W.logtarget = R->logtarget;
    W.eps = R->eps; W.nleaps = R->nleaps; W.final_eps = R->final_eps; W.rb = R->rb; W.rb_acc = R->rb_acc;
    W.init_lt = R->init_lt; W.chain_ids = R->chain_ids; W.nuts = R->nuts;
    const int kind = R->s.kind;
    const bool need_grad = (kind != MCMCGPU_RWM && kind != MCMCGPU_RAM);
    const bool is_ram = (kind == MCMCGPU_RAM);
    // RWM / MALA / RAM / NUTS: every chain needs the log-target on every wave -- tell the likelihood kernel so (null flag array)
    const uint8_t* need_ll_flags = (kind == MCMCGPU_HMC || kind == MCMCGPU_HMCDA) ? R->need_ll : nullptr;
    // number of waves when it is known in advance; otherwise poll the device counter
    int64_t known = -1;
    if (kind == MCMCGPU_RWM || kind == MCMCGPU_MALA || kind == MCMCGPU_RAM) known = seg;
    else if (kind == MCMCGPU_HMC && !R->s.tuner_on) known = seg * (int64_t)R->s.nleaps;
    bool first = false;
    if (!R->started) {
      CU(cudaMemsetAsync(R->kept, 0, sizeof(int64_t) * (size_t)R->Cp, st));
      wave_init_kernel<<<(unsigned)((R->Cp + 127) / 128), 128, 0, st>>>(R->phase, R->remaining, R->q, R->init,
                                                                         R->r.init_per_chain, R->C, R->Cp, R->d);
      CU(cudaGetLastError());
      launches++;
      if (known >= 0) known += 1;   // the wave that evaluates the initial point
      first = true;
      R->started = true;
      if (is_ram) { CU(launch_ram(W, true, st)); launches++; }
    } else {
      W.resume = 1;                  // restart the paused chains: they draw and write their next pending point
      CU(launch_transition(W, st));
      W.resume = 0;
      launches++;
      if (is_ram) { CU(launch_ram(W, false, st)); launches++; }
    }
    // completion polls: when one wave is long (>= ~0.5 ms of likelihood work) poll after every wave, so that no empty
    // wave is ever launched (and none is counted in n_waves / eval_ms); for tiny waves poll every 8
    int64_t poll = c->poll_every;
    if (poll <= 0) poll = (m->is_regression && (double)m->N * (double)m->d * (double)R->Cp >= 5e9) ? 1 : 8;
    std::vector<cudaEvent_t> evs;
    bool graph_done = false;
    for (;;) {
      if (known >= 0 && waves >= known) break;
      // launch-bound regime (small N x C): replay the waves from a CUDA graph (captured once: GW x [likelihood, transition])
      // instead of 2+ stream launches per wave.  With a known wave count the graph is launched todo / GW times; otherwise
      // (HMCDA, tuned HMC: per-chain trajectory lengths) it is launched until the device counter of unfinished chains
      // reads zero -- every kernel of a wave returns at once when it does, so the surplus waves of the last replay cost
      // launch latency only.
      // (measured at N = 256, d = 100, 94 720 chains, 0.5 ms per wave: replay 0.537 ms per wave against 0.500 from the stream, so
      //  graphs are kept for waves of well under 0.1 ms of likelihood work)
      const bool tiny_wave = !m->is_regression || (double)m->N * (double)m->d * (double)R->Cp < 4e8;
      if (!graph_done && !first && !c->time_eval && !m->row_sharded && c->use_graphs && tiny_wave && (known >= 0 || poll > 1)) {
        graph_done = true;
        const int64_t GW = 32;
        const int64_t todo = known >= 0 ? known - waves : GW * 2;
        if (todo >= 2 * GW) {
          cudaGraph_t graph = nullptr; cudaGraphExec_t gexec = nullptr;
          CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
          int crc = MCMCGPU_OK;
          for (int64_t g = 0; g < GW && crc == MCMCGPU_OK; g++) {
            const double* pp; int ns;
            crc = eval_wave(m, R->q, R->part, R->red, R->nsplit, R->C, R->Cp, need_grad, need_ll_flags, R->phase, R->remaining, &pp, &ns, nullptr, fuse);
            W.part = pp; W.nsplit = ns;
            if (crc == MCMCGPU_OK && launch_transition(W, st) != cudaSuccess) crc = MCMCGPU_E_CUDA;
            if (crc == MCMCGPU_OK && is_ram && launch_ram(W, false, st) != cudaSuccess) crc = MCMCGPU_E_CUDA;
          }
          cudaError_t ce = cudaStreamEndCapture(st, &graph);
          if (crc != MCMCGPU_OK || ce != cudaSuccess) { if (graph) cudaGraphDestroy(graph); return fail(MCMCGPU_E_CUDA, "CUDA graph capture of the wave loop failed"); }
          struct GraphGuard { cudaGraph_t g; cudaGraphExec_t e; ~GraphGuard() { if (e) cudaGraphExecDestroy(e); if (g) cudaGraphDestroy(g); } } gg{graph, nullptr};
          CU(cudaGraphInstantiate(&gexec, graph, 0));
          gg.e = gexec;
          const int64_t per_wave = 2 + (is_ram ? 1 : 0) + ((m->is_regression && R->nsplit > 4 && R->red) ? 1 : 0);
          if (known >= 0) {
            const int64_t reps = todo / GW;
            for (int64_t rp = 0; rp < reps; rp++) CU(cudaGraphLaunch(gexec, st));
            waves += reps * GW;
            launches += reps * GW * per_wave;
            if (lockstep) leap_pos = (leap_pos + reps * GW) % (int64_t)R->s.nleaps;   // the replayed waves ran the transition kernel every time
            CU(cudaStreamSynchronize(st));
          } else {
            for (;;) {
              CU(cudaGraphLaunch(gexec, st));
              waves += GW; launches += GW * per_wave;
              CU(cudaMemcpyAsync(c->h_remaining, R->remaining, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
              CU(cudaStreamSynchronize(st));
              if (*c->h_remaining == 0) break;
            }
            break;      // every chain has finished (or paused at the step limit)
          }
        }
      }
      if (known >= 0 && waves >= known) break;
      const double* pp; int ns;
      cudaEvent_t a0 = nullptr, am = nullptr, a1 = nullptr;
      if (c->time_eval) { CU(events.make(&a0)); CU(events.make(&am)); CU(events.make(&a1)); CU(cudaEventRecord(a0, st)); }
      int rc = eval_wave(m, R->q, R->part, R->red, R->nsplit, R->C, R->Cp, need_grad || first,
                         first ? nullptr : need_ll_flags, R->phase, R->remaining, &pp, &ns, am, fuse);
      if (rc != MCMCGPU_OK) return rc;
      if (c->time_eval) { CU(cudaEventRecord(a1, st)); evs.push_back(a0); evs.push_back(am); evs.push_back(a1); }
      W.part = pp; W.nsplit = ns;
      bool interior_wave = false;
      if (lockstep && !first) { interior_wave = (leap_pos + 1 < (int64_t)R->s.nleaps); leap_pos = (leap_pos + 1) % (int64_t)R->s.nleaps; }
      if (!interior_wave) { CU(launch_transition(W, st)); launches++; }
      if (is_ram) { CU(launch_ram(W, false, st)); launches++; }
      launches += 1 + (m->row_sharded ? 1 : 0);
      waves++;
      first = false;
      if (known >= 0) { if (waves >= known) break; }
      else if (waves % poll == 0) {
        CU(cudaMemcpyAsync(c->h_remaining, R->remaining, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (*c->h_remaining == 0) break;
      }
    }
    if (c->time_eval) {
      CU(cudaStreamSynchronize(st));
      for (size_t k = 0; k + 2 < evs.size(); k += 3) {
        float ms = 0;
        cudaEventElapsedTime(&ms, evs[k], evs[k + 1]); eval_ms += ms;        // the likelihood kernel
        cudaEventElapsedTime(&ms, evs[k + 1], evs[k + 2]); comm_ms += ms;    // split fold + all-reduce (row-sharded models)
      }
    }
  }
  CU(cudaEventRecord(e1, st));
  CU(cudaStreamSynchronize(st));
  float ms = 0;
  CU(cudaEventElapsedTime(&ms, e0, e1));
  R->executed = true;
  R->step_limit = upto;
  unsigned long long nev = 0;
  CU(cudaMemcpy(&nev, R->n_evals, sizeof(nev), cudaMemcpyDeviceToHost));
  if (info) { info->gpu_ms = ms; info->n_grad_evals = (int64_t)nev; info->n_waves = waves; info->n_launches = launches; info->eval_ms = eval_ms; info->comm_ms = comm_ms; }
  // initial-support check (RWM.jl:55, MALA.jl:85, HMC.jl:121, HMCDA.jl:88)
  std::vector<int32_t> stt((size_t)R->C);
  CU(cudaMemcpy(stt.data(), R->status, sizeof(int32_t) * (size_t)R->C, cudaMemcpyDeviceToHost));
  int64_t nbad = 0;
  for (int32_t v : stt) nbad += (v != 0);
  if (nbad) return fail(MCMCGPU_E_SUPPORT, "Initial values out of model support, try other values (" + std::to_string(nbad) + " chain(s))");
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_execute(mcmcgpu_run* R, mcmcgpu_run_info* info) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  return execute_impl(R, -1, info);
}

int32_t mcmcgpu_run_execute_steps(mcmcgpu_run* R, int64_t nsteps, mcmcgpu_run_info* info) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (nsteps < 1) return fail(MCMCGPU_E_ARG, "nsteps must be >= 1");
  return execute_impl(R, nsteps, info);
}

// metric adaptation needs the whole warm-up: a run may start at step0 = 0 or after the warm-up
static bool step0_in_warmup(const mcmcgpu_run* R, int64_t step0) { return step0 > 0 && step0 < R->r.first - 2; }

static int upload_chain_vec(mcmcgpu_run* R, double* dst, const double* src) {
  return cudaMemcpyAsync(dst, src, sizeof(double) * (size_t)R->C, cudaMemcpyHostToDevice, R->m->ctx->stream) == cudaSuccess
             ? MCMCGPU_OK : fail(MCMCGPU_E_CUDA, "CUDA: state upload failed");
}

int32_t mcmcgpu_run_set_state(mcmcgpu_run* R, int64_t step0, const double* leapstep, const double* dual_leapstep,
                              const double* dualH) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (R->started) return fail(MCMCGPU_E_STATE, "state must be set before the first execute");
  if (R->engine != MCMCGPU_ENGINE_WAVE) return fail(MCMCGPU_E_STATE, "mcmcgpu_run_set_state needs engine WAVE");
  if (step0 < 0 || step0 >= R->r.last) return fail(MCMCGPU_E_ARG, "step0 must be in [0, last)");
  if (R->r.first <= step0) return fail(MCMCGPU_E_ARG, "the kept range must start after step0");
  if (R->adapt_metric && step0_in_warmup(R, step0)) return fail(MCMCGPU_E_ARG, "metric adaptation cannot start inside the warm-up (set_state step0)");
  CU(use_ctx(R->m->ctx));
  R->step0 = step0;
  if (leapstep || dual_leapstep || dualH) {
    if (R->s.kind != MCMCGPU_HMCDA && R->s.kind != MCMCGPU_NUTS) return fail(MCMCGPU_E_ARG, "step-size state applies to HMCDA and NUTS");
    if (!leapstep || !dual_leapstep || !dualH) return fail(MCMCGPU_E_ARG, "give leapstep, dual_leapstep and dualH together");
    int rc;
    if ((rc = upload_chain_vec(R, R->da_leapstep, leapstep))) return rc;
    if ((rc = upload_chain_vec(R, R->da_dual, dual_leapstep))) return rc;
    if ((rc = upload_chain_vec(R, R->da_dualH, dualH))) return rc;
    CU(cudaStreamSynchronize(R->m->ctx->stream));
    R->restore_da = true;
  }
  return MCMCGPU_OK;
}

// Stan's adaptation windows (windowed_adaptation.hpp) over the W = first - 2 warm-up steps on which the dual averaging
// adapts; the window counter of step i is k = i - 1.  Returns the window-end steps and the steps lo..hi whose samples
// enter the variance estimate (none when W < 20).
static std::vector<int64_t> metric_windows(int64_t W, int64_t init, int64_t term, int64_t window, int64_t* lo, int64_t* hi) {
  std::vector<int64_t> ends;
  *lo = 1; *hi = 0;
  if (W < 20) return ends;
  if (init > W || term > W || window > W || init + window + term > W) {
    init = (int64_t)(0.15 * (double)W); term = (int64_t)(0.1 * (double)W); window = W - (init + term);
  }
  const int64_t last = W - term - 1;       // the last window ends here
  int64_t size = window, next = init + window - 1;
  for (;;) {                               // at the end of the window that ends at k = next:
    ends.push_back(next + 1);
    if (next == last) break;
    size *= 2;
    next += size;
    if (next != last && next + 2 * size >= W - term) next = last;
  }
  *lo = init + 1; *hi = W - term;
  return ends;
}

// the starting metric of every chain from a host array of C x d (chain-major), allocated on first use
static int upload_metric(mcmcgpu_run* R, const double* host) {
  cudaStream_t st = R->m->ctx->stream;
  if (!R->nuts.minv) CU(R->alloc(&R->nuts.minv, (size_t)(R->d * R->Cp)));
  double* tmp = nullptr;
  DevBufs staging;
  CU(staging.up(&tmp, host, (size_t)(R->C * R->d), st));
  CU(transpose_to_chain_minor(tmp, R->nuts.minv, R->C, R->d, R->Cp, st));
  CU(cudaStreamSynchronize(st));
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_set_metric(mcmcgpu_run* R, const double* inv_metric, int32_t per_chain) {
  if (!R || !inv_metric) return fail(MCMCGPU_E_ARG, "NULL argument");
  if (R->s.kind != MCMCGPU_NUTS) return fail(MCMCGPU_E_ARG, "a metric applies to NUTS");
  if (R->started) return fail(MCMCGPU_E_STATE, "the metric must be set before the first execute");
  if (R->nuts.A) return fail(MCMCGPU_E_ARG, "the run has a dense metric (mcmcgpu_run_set_dense_metric)");
  const int64_t C = R->C, d = R->d, n = per_chain ? C * d : d;
  for (int64_t k = 0; k < n; k++)
    if (!(std::isfinite(inv_metric[k]) && inv_metric[k] > 0)) return fail(MCMCGPU_E_ARG, "every inverse metric entry must be finite and > 0");
  CU(use_ctx(R->m->ctx));
  if (per_chain) return upload_metric(R, inv_metric);
  std::vector<double> all((size_t)(C * d));
  for (int64_t c = 0; c < C; c++) std::copy(inv_metric, inv_metric + d, all.begin() + c * d);
  return upload_metric(R, all.data());
}

int32_t mcmcgpu_run_set_metric_adaptation(mcmcgpu_run* R, int64_t init_buffer, int64_t term_buffer, int64_t window) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (R->s.kind != MCMCGPU_NUTS) return fail(MCMCGPU_E_ARG, "metric adaptation applies to NUTS");
  if (R->started) return fail(MCMCGPU_E_STATE, "metric adaptation must be set before the first execute");
  if (init_buffer < 0 || term_buffer < 0 || window < 1) return fail(MCMCGPU_E_ARG, "adaptation buffers must be >= 0 and the window >= 1");
  if (step0_in_warmup(R, R->step0)) return fail(MCMCGPU_E_ARG, "metric adaptation cannot start inside the warm-up (set_state step0)");
  CU(use_ctx(R->m->ctx));
  NutsState& T = R->nuts;
  const bool dense = T.A != nullptr;
  const int64_t dd = R->d * R->d;
  if (!dense && !T.minv) {
    std::vector<double> ones((size_t)(R->C * R->d), 1.0);
    int rc = upload_metric(R, ones.data());
    if (rc) return rc;
  }
  if (dense && T.a_ld == 1) {      // every chain adapts its own copy of the shared starting matrix and its factor
    double *A = nullptr, *L = nullptr;
    CU(R->alloc(&A, (size_t)(dd * R->Cp), false));
    CU(R->alloc(&L, (size_t)(dd * R->Cp), false));
    CU(broadcast_to_chain_minor(T.A, A, dd, R->C, R->Cp, R->m->ctx->stream));
    CU(broadcast_to_chain_minor(T.L, L, dd, R->C, R->Cp, R->m->ctx->stream));
    T.A = A; T.L = L; T.a_ld = R->Cp;
  }
  int64_t lo, hi;
  const std::vector<int64_t> ends = metric_windows(R->r.first - 2, init_buffer, term_buffer, window, &lo, &hi);
  if (!T.wf_mean) {
    CU(R->alloc(&T.wf_mean, (size_t)(R->d * R->Cp)));
    CU(R->alloc(&T.wf_m2, (size_t)((dense ? dd : R->d) * R->Cp)));
    CU(R->alloc(&T.wf_n, (size_t)R->Cp));
    CU(R->alloc(&T.da_eps0, (size_t)R->Cp));
    CU(R->alloc(&T.da_i0, (size_t)R->Cp));
  }
  int64_t* win_end = nullptr;
  CU(R->alloc(&win_end, ends.size()));
  T.win_end = win_end;
  if (!ends.empty()) CU(cudaMemcpyAsync(win_end, ends.data(), sizeof(int64_t) * ends.size(), cudaMemcpyHostToDevice, R->m->ctx->stream));
  CU(cudaStreamSynchronize(R->m->ctx->stream));
  T.n_win = (int32_t)ends.size(); T.win_lo = lo; T.win_hi = hi;
  R->adapt_metric = true;
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_get_metric(mcmcgpu_run* R, double* out_inv_metric) {
  if (!R || !out_inv_metric) return fail(MCMCGPU_E_ARG, "NULL argument");
  if (R->s.kind != MCMCGPU_NUTS) return fail(MCMCGPU_E_ARG, "a metric applies to NUTS");
  if (R->nuts.A) return fail(MCMCGPU_E_ARG, "the run has a dense metric: use mcmcgpu_run_get_dense_metric");
  if (!R->nuts.minv) {
    std::fill(out_inv_metric, out_inv_metric + R->C * R->d, 1.0);
    return MCMCGPU_OK;
  }
  CU(use_ctx(R->m->ctx));
  cudaStream_t st = R->m->ctx->stream;
  double* tmp = nullptr;
  DevBufs bufs;
  CU(bufs.get(&tmp, (size_t)(R->C * R->d), st, false));
  CU(transpose_to_chain_major(R->nuts.minv, tmp, 0, R->C, R->d, R->Cp, st));
  CU(cudaMemcpyAsync(out_inv_metric, tmp, sizeof(double) * (size_t)(R->C * R->d), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return MCMCGPU_OK;
}

// A dense metric: every matrix finite and exactly symmetric on the host, then positive definite by the device Cholesky
// that nuts_kernel uses (the factor it leaves is the run's L).  Being symmetric, a chain's column-major d x d block is also
// its row-major one, which is the device layout.  A shared matrix is stored once (a_ld = 1) and read by every chain.
int32_t mcmcgpu_run_set_dense_metric(mcmcgpu_run* R, const double* inv_metric, int32_t per_chain) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (R->s.kind != MCMCGPU_NUTS) return fail(MCMCGPU_E_ARG, "a metric applies to NUTS");
  if (R->started) return fail(MCMCGPU_E_STATE, "the metric must be set before the first execute");
  if (R->adapt_metric) return fail(MCMCGPU_E_ARG, "set the dense metric before mcmcgpu_run_set_metric_adaptation");
  if (R->nuts.minv) return fail(MCMCGPU_E_ARG, "the run has a diagonal metric (mcmcgpu_run_set_metric)");
  const int64_t d = R->d, dd = d * d, Cp = R->Cp;
  std::vector<double> ident;
  if (!inv_metric) {
    ident.assign((size_t)dd, 0.0);
    for (int64_t j = 0; j < d; j++) ident[(size_t)(j * d + j)] = 1.0;
    inv_metric = ident.data(); per_chain = 0;
  }
  const int64_t nm = per_chain ? R->C : 1, ld = per_chain ? Cp : 1;
  for (int64_t c = 0; c < nm; c++)
    for (int64_t j = 0; j < d; j++)
      for (int64_t i = 0; i < d; i++) {
        const double x = inv_metric[c * dd + j * d + i];
        if (!std::isfinite(x)) return fail(MCMCGPU_E_ARG, "every dense inverse metric entry must be finite");
        if (x != inv_metric[c * dd + i * d + j]) return fail(MCMCGPU_E_ARG, "every dense inverse metric must be exactly symmetric");
      }
  CU(use_ctx(R->m->ctx));
  cudaStream_t st = R->m->ctx->stream;
  double *A = nullptr, *L = nullptr, *tmp = nullptr;
  int32_t* bad = nullptr;
  DevBufs bufs;
  CU(R->alloc(&A, (size_t)(dd * ld), false));
  CU(R->alloc(&L, (size_t)(dd * ld)));
  if (per_chain) {
    CU(bufs.up(&tmp, inv_metric, (size_t)(nm * dd), st));
    CU(transpose_to_chain_minor(tmp, A, nm, dd, Cp, st));
  } else {
    CU(cudaMemcpyAsync(A, inv_metric, sizeof(double) * (size_t)dd, cudaMemcpyHostToDevice, st));
  }
  CU(bufs.get(&bad, (size_t)nm, st, false));
  CU(launch_dense_factor(A, L, d, nm, ld, bad, st));
  std::vector<int32_t> hbad((size_t)nm);
  CU(cudaMemcpyAsync(hbad.data(), bad, sizeof(int32_t) * (size_t)nm, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  for (int32_t b : hbad)
    if (b) return fail(MCMCGPU_E_ARG, "every dense inverse metric must be positive definite (its Cholesky factorisation failed)");
  NutsState& T = R->nuts;
  if (!T.v[0]) {
    CU(R->alloc(&T.v[0], (size_t)(d * Cp), false));
    CU(R->alloc(&T.v[1], (size_t)(d * Cp), false));
  }
  T.A = A; T.L = L; T.a_ld = ld;
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_get_dense_metric(mcmcgpu_run* R, double* out) {
  if (!R || !out) return fail(MCMCGPU_E_ARG, "NULL argument");
  if (R->s.kind != MCMCGPU_NUTS || !R->nuts.A) return fail(MCMCGPU_E_ARG, "the run has no dense metric");
  CU(use_ctx(R->m->ctx));
  cudaStream_t st = R->m->ctx->stream;
  const NutsState& T = R->nuts;
  const int64_t C = R->C, d = R->d, dd = d * d;
  if (T.a_ld == 1) {
    CU(cudaMemcpyAsync(out, T.A, sizeof(double) * (size_t)dd, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int64_t c = 1; c < C; c++) std::copy(out, out + dd, out + c * dd);
  } else {
    double* tmp = nullptr;
    DevBufs bufs;
    CU(bufs.get(&tmp, (size_t)(C * dd), st, false));
    CU(transpose_to_chain_major(T.A, tmp, 0, C, dd, R->Cp, st));
    CU(cudaMemcpyAsync(out, tmp, sizeof(double) * (size_t)(C * dd), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  for (int64_t c = 0; c < C; c++)            // row-major (device) to column-major: an adapted A is not exactly symmetric
    for (int64_t j = 0; j < d; j++)
      for (int64_t k = j + 1; k < d; k++) std::swap(out[c * dd + j * d + k], out[c * dd + k * d + j]);
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_set_nuts_transition(mcmcgpu_run* R, int32_t transition) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (R->s.kind != MCMCGPU_NUTS) return fail(MCMCGPU_E_ARG, "the NUTS transition applies to NUTS");
  if (transition != MCMCGPU_NUTS_SLICE && transition != MCMCGPU_NUTS_MULTINOMIAL) return fail(MCMCGPU_E_ARG, "unknown NUTS transition");
  if (R->started) return fail(MCMCGPU_E_STATE, "the NUTS transition must be set before the first execute");
  R->nuts_multinomial = transition == MCMCGPU_NUTS_MULTINOMIAL;
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_get_state(mcmcgpu_run* R, double* pars, double* leapstep, double* dual_leapstep, double* dualH) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (!R->executed) return fail(MCMCGPU_E_STATE, "run has not been executed");
  if (R->engine != MCMCGPU_ENGINE_WAVE) return fail(MCMCGPU_E_STATE, "mcmcgpu_run_get_state needs engine WAVE");
  CU(use_ctx(R->m->ctx));
  cudaStream_t st = R->m->ctx->stream;
  if (pars) {
    double* tmp = nullptr;
    DevBufs bufs;
    CU(bufs.get(&tmp, (size_t)(R->C * R->d), st, false));
    CU(transpose_to_chain_major(R->cur_pars, tmp, 0, R->C, R->d, R->Cp, st));
    CU(cudaMemcpyAsync(pars, tmp, sizeof(double) * (size_t)(R->C * R->d), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  const double* src[3] = {R->da_leapstep, R->da_dual, R->da_dualH};
  double* dst[3] = {leapstep, dual_leapstep, dualH};
  for (int k = 0; k < 3; k++)
    if (dst[k]) CU(cudaMemcpyAsync(dst[k], src[k], sizeof(double) * (size_t)R->C, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return MCMCGPU_OK;
}

static int fetch_chunked(mcmcgpu_run* R, const double* dev, int64_t K, double* host) {
  // device [K][Cp] chain-minor -> host [C][K], in chain chunks through two staging buffers
  cudaStream_t st = R->m->ctx->stream;
  const int64_t C = R->C, Cp = R->Cp;
  int64_t chunk = (int64_t)(32.0 * 1024 * 1024 / (8.0 * (double)K));     // 32 MB staging buffers: long enough copies, cheap to allocate
  if (chunk < 64) chunk = 64;
  if (chunk > C) chunk = C;
  double* stage[2] = {nullptr, nullptr};
  cudaEvent_t done[2];
  DevBufs bufs; Events events;
  CU(bufs.get(&stage[0], (size_t)(chunk * K), st, false));
  CU(bufs.get(&stage[1], (size_t)(chunk * K), st, false));
  CU(events.make(&done[0])); CU(events.make(&done[1]));
  int b = 0; bool used[2] = {false, false};
  for (int64_t c0 = 0; c0 < C; c0 += chunk, b ^= 1) {
    int64_t nc = (C - c0 < chunk) ? C - c0 : chunk;
    if (used[b]) CU(cudaEventSynchronize(done[b]));
    CU(transpose_to_chain_major(dev, stage[b], c0, nc, K, Cp, st));
    CU(cudaMemcpyAsync(host + c0 * K, stage[b], sizeof(double) * (size_t)(nc * K), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(done[b], st));
    used[b] = true;
  }
  CU(cudaStreamSynchronize(st));
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_fetch(mcmcgpu_run* R, double* out_samples, double* out_grads, uint8_t* out_accept, double* out_logtarget) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (!R->executed) return fail(MCMCGPU_E_STATE, "run has not been executed");
  if (R->stream) return fail(MCMCGPU_E_STATE, "the run streamed its summaries (stream_stats): no draws were stored; use mcmcgpu_run_stats");
  CU(use_ctx(R->m->ctx));
  cudaStream_t st = R->m->ctx->stream;
  int rc;
  if (out_samples) { rc = fetch_chunked(R, R->samples, R->S * R->d, out_samples); if (rc) return rc; }
  if (out_grads) {
    if (!R->grads) return fail(MCMCGPU_E_STATE, "gradients were not stored (store_grad = 0)");
    rc = fetch_chunked(R, R->grads, R->S * R->d, out_grads); if (rc) return rc;
  }
  if (out_logtarget) {
    if (!R->logtarget) return fail(MCMCGPU_E_STATE, "log-targets were not stored (store_logtarget = 0)");
    rc = fetch_chunked(R, R->logtarget, R->S, out_logtarget); if (rc) return rc;
  }
  if (out_accept) {
    uint8_t* tmp = nullptr;
    DevBufs bufs;
    CU(bufs.get(&tmp, (size_t)(R->C * R->S), st, false));
    CU(transpose_to_chain_major_u8(R->accept, tmp, 0, R->C, R->S, R->Cp, st));
    CU(cudaMemcpyAsync(out_accept, tmp, (size_t)(R->C * R->S), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return MCMCGPU_OK;
}

__global__ void i32_to_i64_kernel(const int32_t* in, int64_t* out, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i];
}

int32_t mcmcgpu_run_fetch_rb(mcmcgpu_run* R, double* out_rb) {
  if (!R || !out_rb) return fail(MCMCGPU_E_ARG, "NULL argument");
  if (!R->executed) return fail(MCMCGPU_E_STATE, "run has not been executed");
  if (!R->rb) return fail(MCMCGPU_E_STATE, "Rao-Blackwell sums were not stored (store_rb = 0)");
  CU(use_ctx(R->m->ctx));
  return fetch_chunked(R, R->rb, R->S * R->d, out_rb);
}

int32_t mcmcgpu_run_fetch_diag(mcmcgpu_run* R, double* out_eps, int64_t* out_nleaps) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (!R->executed) return fail(MCMCGPU_E_STATE, "run has not been executed");
  if (!R->has_diag) return fail(MCMCGPU_E_STATE, "sampler has no step-size diagnostics");
  CU(use_ctx(R->m->ctx));
  cudaStream_t st = R->m->ctx->stream;
  if (out_eps) { int rc = fetch_chunked(R, R->eps, R->S, out_eps); if (rc) return rc; }
  if (out_nleaps) {
    // widen to double-sized lanes so the same transposer can be used
    int64_t n = R->S * R->Cp;
    int64_t* wide = nullptr;
    DevBufs bufs;
    CU(bufs.get(&wide, (size_t)n, st, false));
    i32_to_i64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(R->nleaps, wide, n);
    CU(cudaGetLastError());
    int rc = fetch_chunked(R, reinterpret_cast<const double*>(wide), R->S, reinterpret_cast<double*>(out_nleaps));
    if (rc) return rc;
  }
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_fetch_nuts_stats(mcmcgpu_run* R, double* accept_stat, double* energy, uint8_t* divergent) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (R->s.kind != MCMCGPU_NUTS || !R->nuts_multinomial) return fail(MCMCGPU_E_ARG, "NUTS statistics are kept by multinomial NUTS runs");
  if (!R->executed) return fail(MCMCGPU_E_STATE, "run has not been executed");
  CU(use_ctx(R->m->ctx));
  const NutsState& T = R->nuts;
  int rc;
  if (accept_stat && (rc = fetch_chunked(R, T.st_accept_stat, R->S, accept_stat))) return rc;
  if (energy && (rc = fetch_chunked(R, T.st_energy, R->S, energy))) return rc;
  if (divergent) {
    cudaStream_t st = R->m->ctx->stream;
    uint8_t* tmp = nullptr;
    DevBufs bufs;
    CU(bufs.get(&tmp, (size_t)(R->C * R->S), st, false));
    CU(transpose_to_chain_major_u8(T.st_divergent, tmp, 0, R->C, R->S, R->Cp, st));
    CU(cudaMemcpyAsync(divergent, tmp, (size_t)(R->C * R->S), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return MCMCGPU_OK;
}

static int stats_common(mcmcgpu_ctx* c, const double* samples, const uint8_t* accept, int64_t S, int64_t d, int64_t C, int64_t Cp,
                        int32_t vtype, int64_t maxlag, int64_t batchlen, double* out_mean, double* out_var_iid, double* out_var,
                        double* out_ess, double* out_actime, double* out_accept_rate) {
  cudaStream_t st = c->stream;
  if (vtype < MCMCGPU_VAR_IID || vtype > MCMCGPU_VAR_IPSE) return fail(MCMCGPU_E_ARG, "Unknown variance type");   // var.jl:138
  if ((out_ess || out_actime) && vtype == MCMCGPU_VAR_IID) return fail(MCMCGPU_E_ARG, "Unknown ESS type iid");      // ess.jl:4,7
  if (S < 2) return fail(MCMCGPU_E_ARG, "need at least 2 kept draws");
  if (maxlag < 0) maxlag = S - 1;
  if (maxlag > S - 1) maxlag = S - 1;
  if (batchlen <= 0) batchlen = 100;
  if (vtype == MCMCGPU_VAR_BM && S / batchlen <= 1)
    return fail(MCMCGPU_E_ARG, "Choose batch size such that the number of batches is greather than one");           // var.jl:22
  double* outs[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  double* hosts[5] = {out_mean, out_var_iid, out_var, out_ess, out_actime};
  DevBufs bufs;                              // every temporary below is released on every return path
  for (int k = 0; k < 5; k++) if (hosts[k] || k == 0) CU(bufs.get(&outs[k], (size_t)(d * Cp), st, false));   // the mean is always formed (pass 2 reads it)
  double* bmean = nullptr;      // scratch of the stats kernels: batch-mean means, or the state of unfinished Geyer scans
  if (vtype == MCMCGPU_VAR_BM) CU(bufs.get(&bmean, (size_t)(d * Cp), st, false));
  else if (vtype != MCMCGPU_VAR_IID) CU(bufs.get(&bmean, (size_t)(STATS_SCRATCH_PLANES * d * Cp + 2), st, false));
  unsigned int unfinished = 0;
  CU(launch_stats(samples, S, d, C, Cp, vtype, maxlag, batchlen, outs[0], outs[1], outs[2], outs[3], outs[4], bmean, &unfinished, st));
  if (unfinished) {
    // few unfinished Geyer scans: finish them on a compact time-contiguous copy (one warp per series); many (slowly mixing
    // chains) or a copy that would not fit comfortably: one thread per series on the strided draws
    double* gather = nullptr;
    const double need = (double)unfinished * (double)S * 8.0;
    if ((double)unfinished <= 0.25 * (double)(C * d) && need <= 8e9) {
      if (dalloc(&gather, (size_t)unfinished * (size_t)S) == cudaSuccess) bufs.v.push_back(gather); else { gather = nullptr; cudaGetLastError(); }
    }
    CU(launch_stats_more(samples, S, d, C, Cp, vtype, maxlag, outs[0], outs[1], outs[2], outs[3], outs[4], bmean, unfinished, gather, st));
  }
  // all results are laid out chain-major on the device first, then copied out back to back: one synchronisation
  double* tmp = nullptr;
  CU(bufs.get(&tmp, (size_t)(5 * C * d), st, false));
  for (int k = 0; k < 5; k++) if (hosts[k]) {
    CU(transpose_to_chain_major(outs[k], tmp + (size_t)k * (size_t)(C * d), 0, C, d, Cp, st));
    CU(cudaMemcpyAsync(hosts[k], tmp + (size_t)k * (size_t)(C * d), sizeof(double) * (size_t)(C * d), cudaMemcpyDeviceToHost, st));
  }
  if (out_accept_rate && accept) {
    double* rate = nullptr;
    CU(bufs.get(&rate, (size_t)Cp, st, false));
    CU(launch_accept_rate(accept, S, C, Cp, rate, st));
    CU(cudaMemcpyAsync(out_accept_rate, rate, sizeof(double) * (size_t)C, cudaMemcpyDeviceToHost, st));
  }
  CU(cudaStreamSynchronize(st));
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_stats(mcmcgpu_run* R, int32_t vtype, int64_t maxlag, int64_t batchlen, double* out_mean, double* out_var_iid,
                          double* out_var, double* out_ess, double* out_actime, double* out_accept_rate) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (!R->executed) return fail(MCMCGPU_E_STATE, "run has not been executed");
  CU(use_ctx(R->m->ctx));
  if (R->stream) {      // summaries accumulated while sampling: rows mean, var_iid, var_bm, ess, actime
    if (vtype != MCMCGPU_VAR_IID && vtype != MCMCGPU_VAR_BM) return fail(MCMCGPU_E_ARG, "a streamed run (stream_stats) offers vtype iid and bm");
    if ((out_ess || out_actime) && vtype == MCMCGPU_VAR_IID) return fail(MCMCGPU_E_ARG, "Unknown ESS type iid");
    if (vtype == MCMCGPU_VAR_BM && batchlen > 0 && batchlen != R->r.stream_batchlen)
      return fail(MCMCGPU_E_ARG, "the batch length of a streamed run is fixed at run creation (stream_batchlen)");
    if (vtype == MCMCGPU_VAR_BM && R->S / R->r.stream_batchlen <= 1)
      return fail(MCMCGPU_E_ARG, "Choose batch size such that the number of batches is greather than one");        // var.jl:22
    cudaStream_t st = R->m->ctx->stream;
    const int64_t C = R->C, d = R->d, Cp = R->Cp, P = d * Cp;
    double* hosts[5] = {out_mean, out_var_iid, out_var, out_ess, out_actime};
    const int rows[5] = {0, 1, vtype == MCMCGPU_VAR_BM ? 2 : 1, 3, 4};
    DevBufs bufs;
    double* tmp = nullptr;
    CU(bufs.get(&tmp, (size_t)(5 * C * d), st, false));
    for (int k = 0; k < 5; k++) if (hosts[k]) {
      CU(transpose_to_chain_major(R->stream + rows[k] * P, tmp + (size_t)k * (size_t)(C * d), 0, C, d, Cp, st));
      CU(cudaMemcpyAsync(hosts[k], tmp + (size_t)k * (size_t)(C * d), sizeof(double) * (size_t)(C * d), cudaMemcpyDeviceToHost, st));
    }
    if (out_accept_rate) CU(cudaMemcpyAsync(out_accept_rate, R->stream_accept, sizeof(double) * (size_t)C, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return MCMCGPU_OK;
  }
  return stats_common(R->m->ctx, R->samples, R->accept, R->S, R->d, R->C, R->Cp, vtype, maxlag, batchlen, out_mean, out_var_iid,
                      out_var, out_ess, out_actime, out_accept_rate);
}

int32_t mcmcgpu_stats(mcmcgpu_ctx* c, const double* samples, int64_t S, int64_t d, int64_t C, int32_t vtype, int64_t maxlag,
                      int64_t batchlen, double* out_mean, double* out_var_iid, double* out_var, double* out_ess, double* out_actime) {
  if (!c || !samples || S < 1 || d < 1 || C < 1) return fail(MCMCGPU_E_ARG, "bad arguments");
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  const int64_t Cp = round_up(C, K1_CHAINS), K = S * d;
  double *tmp = nullptr, *dev = nullptr;
  DevBufs bufs;
  CU(bufs.up(&tmp, samples, (size_t)(C * K), st));
  CU(bufs.get(&dev, (size_t)(K * Cp), st, false));
  CU(transpose_to_chain_minor(tmp, dev, C, K, Cp, st));
  int rc = stats_common(c, dev, nullptr, S, d, C, Cp, vtype, maxlag, batchlen, out_mean, out_var_iid, out_var, out_ess, out_actime, nullptr);
  cudaStreamSynchronize(st);
  return rc;
}

static int zv_common(mcmcgpu_ctx* c, const double* samples, const double* grads, int64_t S, int64_t d, int64_t C, int64_t Cp,
                     int32_t order, double* out_zv, double* out_a) {
  cudaStream_t st = c->stream;
  if (!out_a) return fail(MCMCGPU_E_ARG, "out_a is NULL");
  if (S < 2) return fail(MCMCGPU_E_ARG, "need at least 2 kept draws");
  if (!zv_supported(d, order)) return fail(MCMCGPU_E_ARG, "ZV: order must be 1 or 2 and the k x (k+d) covariance must fit in shared memory (order 1: d <= 110; order 2: d <= 13)");
  const int64_t k = zv_features(d, order);
  DevBufs B;
  double *zv = nullptr, *a = nullptr, *tmp = nullptr;
  int32_t* status = nullptr;
  if (out_zv) CU(B.get(&zv, (size_t)(S * d * Cp), st, false));
  CU(B.get(&a, (size_t)(k * d * Cp), st));
  CU(B.get(&status, (size_t)Cp, st));
  CU(launch_zv(samples, grads, S, d, C, Cp, order, zv, a, status, st));
  CU(B.get(&tmp, (size_t)(C * k * d), st, false));
  CU(transpose_to_chain_major(a, tmp, 0, C, k * d, Cp, st));
  CU(cudaMemcpyAsync(out_a, tmp, sizeof(double) * (size_t)(C * k * d), cudaMemcpyDeviceToHost, st));
  if (out_zv) {
    double* t2 = nullptr;
    CU(B.get(&t2, (size_t)(C * S * d), st, false));
    CU(transpose_to_chain_major(zv, t2, 0, C, S * d, Cp, st));
    CU(cudaMemcpyAsync(out_zv, t2, sizeof(double) * (size_t)(C * S * d), cudaMemcpyDeviceToHost, st));
  }
  std::vector<int32_t> stt((size_t)C);
  CU(cudaMemcpyAsync(stt.data(), status, sizeof(int32_t) * (size_t)C, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  for (int32_t v : stt) if (v) return fail(MCMCGPU_E_ARG, "ZV: singular feature covariance (SingularException in the reference's inv)");
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_zv(mcmcgpu_run* R, int32_t order, double* out_zv, double* out_a) {
  if (!R) return fail(MCMCGPU_E_ARG, "run is NULL");
  if (!R->executed) return fail(MCMCGPU_E_STATE, "run has not been executed");
  if (!R->grads) return fail(MCMCGPU_E_STATE, "ZV needs the stored gradients (store_grad = 1)");
  CU(use_ctx(R->m->ctx));
  return zv_common(R->m->ctx, R->samples, R->grads, R->S, R->d, R->C, R->Cp, order, out_zv, out_a);
}

int32_t mcmcgpu_zv(mcmcgpu_ctx* c, const double* samples, const double* grads, int64_t S, int64_t d, int64_t C, int32_t order,
                   double* out_zv, double* out_a) {
  if (!c || !samples || !grads || S < 1 || d < 1 || C < 1) return fail(MCMCGPU_E_ARG, "bad arguments");
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  const int64_t Cp = round_up(C, K1_CHAINS), K = S * d;
  DevBufs B;
  double *tmp = nullptr, *ds = nullptr, *dg = nullptr;
  CU(B.get(&tmp, (size_t)(C * K), st, false));
  CU(B.get(&ds, (size_t)(K * Cp), st)); CU(B.get(&dg, (size_t)(K * Cp), st));
  CU(cudaMemcpyAsync(tmp, samples, sizeof(double) * (size_t)(C * K), cudaMemcpyHostToDevice, st));
  CU(transpose_to_chain_minor(tmp, ds, C, K, Cp, st));
  CU(cudaMemcpyAsync(tmp, grads, sizeof(double) * (size_t)(C * K), cudaMemcpyHostToDevice, st));
  CU(transpose_to_chain_minor(tmp, dg, C, K, Cp, st));
  return zv_common(c, ds, dg, S, d, C, Cp, order, out_zv, out_a);
}

int32_t mcmcgpu_run_chains(mcmcgpu_model* m, const mcmcgpu_sampler_cfg* s, const mcmcgpu_runner_cfg* r, const double* init,
                           const double* scale, const double* inj_normals, const double* inj_uniforms, double* out_samples,
                           double* out_grads, uint8_t* out_accept, double* out_logtarget, mcmcgpu_run_info* info) {
  if (!r) return fail(MCMCGPU_E_ARG, "NULL argument");
  mcmcgpu_runner_cfg rr = *r;
  rr.store_grad = out_grads ? 1 : 0;
  rr.store_logtarget = out_logtarget ? 1 : 0;
  rr.store_rb = 0;
  mcmcgpu_run* R = nullptr;
  int rc = mcmcgpu_run_create(m, s, &rr, init, scale, inj_normals, inj_uniforms, &R);
  if (rc != MCMCGPU_OK) return rc;
  rc = mcmcgpu_run_execute(R, info);
  // "Initial values out of model support" is an assertion in the reference (RWM.jl:55, ...): no chain is produced, so
  // nothing is fetched (the kept-draw arrays of a chain that never started are not initialised)
  if (rc == MCMCGPU_OK) rc = mcmcgpu_run_fetch(R, out_samples, out_grads, out_accept, out_logtarget);
  mcmcgpu_run_destroy(R);
  return rc;
}

int32_t mcmcgpu_philox_draws(mcmcgpu_ctx* c, uint64_t seed, int64_t chain_offset, int64_t nchains, int64_t d, int64_t last,
                             double* out_normals, double* out_uniforms) {
  if (!c || !out_normals || !out_uniforms || nchains < 1 || d < 1 || last < 0) return fail(MCMCGPU_E_ARG, "bad arguments");
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  double *zn = nullptr, *un = nullptr;
  const int64_t n = nchains * (last + 1);
  DevBufs bufs;
  CU(bufs.get(&zn, (size_t)(n * d), st, false));
  CU(bufs.get(&un, (size_t)n, st, false));
  CU(launch_philox_dump(seed, chain_offset, nchains, d, last, zn, un, st));
  CU(cudaMemcpyAsync(out_normals, zn, sizeof(double) * (size_t)(n * d), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out_uniforms, un, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return MCMCGPU_OK;
}

// ---- population runners (SURVEY.md 8f.1) ----------------------------------------------------------------
static int fill_tasks(PopTasks& T, int32_t family, int64_t d, int32_t nt, const double* hypers, const mcmcgpu_sampler_cfg* samplers) {
  if (!pop_supported(family, d)) return fail(MCMCGPU_E_ARG, "population runners support the closed-form families (normal, normal_dsl, abs_normal) with d <= 8");
  if (nt < 1 || nt > POP_MAX_TASKS) return fail(MCMCGPU_E_ARG, "between 1 and 64 tasks");
  if (!hypers || !samplers) return fail(MCMCGPU_E_ARG, "NULL argument");
  T.nt = nt; T.family = family; T.d = (int32_t)d;
  for (int t = 0; t < nt; t++) {
    T.hyper[t][0] = hypers[4 * t]; T.hyper[t][1] = hypers[4 * t + 1];
    const mcmcgpu_sampler_cfg& s = samplers[t];
    if (s.tuner_on || (s.kind != MCMCGPU_RWM && s.kind != MCMCGPU_MALA && s.kind != MCMCGPU_HMC))
      return fail(MCMCGPU_E_ARG, "population runners take RWM, MALA or HMC tasks without tuner");
    if (!(s.scale > 0) || (s.kind == MCMCGPU_HMC && s.nleaps <= 0)) return fail(MCMCGPU_E_ARG, "bad sampler parameters");
    if ((family == MCMCGPU_FAM_NORMAL_DSL || family == MCMCGPU_FAM_ABS_NORMAL) && !(T.hyper[t][1] > 0)) return fail(MCMCGPU_E_ARG, "sigma must be > 0");
    T.kind[t] = s.kind; T.nleaps[t] = s.nleaps; T.scale[t] = s.scale;
  }
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_seqmc(mcmcgpu_ctx* c, int32_t family, int64_t d, int32_t nt, const double* hypers,
                          const mcmcgpu_sampler_cfg* samplers, int64_t steps, int64_t burnin, double trigger, int64_t npart,
                          const double* particles, uint64_t seed, const double* inj_normals, const double* inj_uniforms,
                          const double* inj_res_uniforms, double* out_samples, double* out_weights, int64_t* out_nresamples,
                          mcmcgpu_run_info* info) {
  if (!c || !particles || !out_samples || !out_weights) return fail(MCMCGPU_E_ARG, "NULL argument");
  if (burnin < 0) return fail(MCMCGPU_E_ARG, "Burnin rounds should be >= 0");                   // SeqMC.jl:29
  if (steps <= burnin) return fail(MCMCGPU_E_ARG, "Steps should be > to burnin");               // SeqMC.jl:30
  if (npart < 2) return fail(MCMCGPU_E_ARG, "at least 2 particles");
  const bool inj = inj_normals != nullptr;
  if (inj != (inj_uniforms != nullptr) || inj != (inj_res_uniforms != nullptr)) return fail(MCMCGPU_E_ARG, "inject all three draw arrays or none");
  SeqArgs A;
  int rc = fill_tasks(A.T, family, d, nt, hypers, samplers);
  if (rc != MCMCGPU_OK) return rc;
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  DevBufs B;
  const int64_t Np = round_up(npart, 64), S = (steps - burnin) * npart, K = steps * nt * npart * (c->comm ? c->nranks : 1);
  A.npart = npart; A.Np = Np; A.steps = steps; A.burnin = burnin; A.seed = seed; A.trigger = trigger;
  // particles sharded over the ranks of the context's communicator: npart is THIS rank's share (equal on all ranks);
  // per target the ranks exchange (pars, logtarget, logW) with one ncclAllGather and resample their own slots
  A.rank = c->comm ? c->rank : 0; A.nranks = c->comm ? c->nranks : 1;
  A.gpart = npart * A.nranks; A.sendbuf = nullptr; A.gathered = nullptr;
  const NcclApi* api = nullptr;
  if (A.nranks > 1) {
    api = nccl_api(nullptr);
    if (!api) return fail(MCMCGPU_E_COMM, "NCCL unavailable");
    double* gb = nullptr;
    CU(B.get(&A.sendbuf, (size_t)((d + 2) * Np), st));
    CU(B.get(&gb, (size_t)(A.nranks * (d + 2) * Np), st));
    A.gathered = gb;
  }
  double* hp = nullptr;
  CU(B.up(&hp, particles, (size_t)(npart * d), st));
  CU(B.get(&A.pars, (size_t)(d * Np), st));
  CU(transpose_to_chain_minor(hp, A.pars, npart, d, Np, st));
  CU(B.get(&A.pars_tmp, (size_t)(d * Np), st));
  CU(B.get(&A.logW, (size_t)Np, st)); CU(B.get(&A.logtarget, (size_t)Np, st)); CU(B.get(&A.lt_tmp, (size_t)Np, st));
  CU(B.get(&A.W, (size_t)(Np * (c->comm ? c->nranks : 1)), st)); CU(B.get(&A.cp, (size_t)(Np * (c->comm ? c->nranks : 1)), st));
  CU(B.get(&A.samples, (size_t)(S * d), st, false)); CU(B.get(&A.weights, (size_t)S, st, false));
  CU(B.get(&A.nres, 1, st)); CU(B.get(&A.nevals, 1, st));
  A.inj_normals = A.inj_uniforms = A.inj_res = nullptr;
  if (inj) {
    double *a = nullptr, *b = nullptr, *r = nullptr;
    CU(B.up(&a, inj_normals, (size_t)(K * d), st)); CU(B.up(&b, inj_uniforms, (size_t)K, st)); CU(B.up(&r, inj_res_uniforms, (size_t)K, st));
    A.inj_normals = a; A.inj_uniforms = b; A.inj_res = r;
  }
  Events events;
  cudaEvent_t e0, e1;
  CU(events.make(&e0)); CU(events.make(&e1));
  CU(cudaEventRecord(e0, st));
  int64_t launches = 0;
  for (int64_t i = 1; i <= steps; i++) {                                                        // SeqMC.jl:62
    A.iter = i;
    for (int t = 0; t < nt; t++) {                                                              // :64
      A.target = t;
      CU(launch_seqmc_mutate(A, st));
      if (A.nranks > 1) {
        CU(launch_seqmc_pack(A, st));
        int nrc = api->AllGather(A.sendbuf, (void*)A.gathered, (size_t)((d + 2) * Np), NCCL_FLOAT64, c->comm, st);
        if (nrc != 0) return fail(MCMCGPU_E_COMM, std::string("ncclAllGather: ") + (api->GetErrorString ? api->GetErrorString(nrc) : "error"));
        launches++;
      }
      CU(launch_seqmc_resample(A, st));
      launches += 2;
    }
    CU(launch_seqmc_store(A, st));
    launches++;
  }
  CU(cudaEventRecord(e1, st));
  CU(cudaMemcpyAsync(out_samples, A.samples, sizeof(double) * (size_t)(S * d), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out_weights, A.weights, sizeof(double) * (size_t)S, cudaMemcpyDeviceToHost, st));
  unsigned long long nres = 0, nev = 0;
  CU(cudaMemcpyAsync(&nres, A.nres, sizeof(nres), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(&nev, A.nevals, sizeof(nev), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
  if (out_nresamples) *out_nresamples = (int64_t)nres;
  if (info) { info->gpu_ms = ms; info->n_grad_evals = (int64_t)nev; info->n_waves = steps * nt; info->n_launches = launches; info->eval_ms = 0; info->comm_ms = 0; }
  return MCMCGPU_OK;
}

// SeqMC over arbitrary models (regression families through K1; SURVEY.md 8f.1 "reuses K1"): the mutation of every particle
// by task t -- reset(task, particle) + one sampler step (SeqMC.jl:66-72) -- is a one-step run of the wave engine on model t
// started at the particles (its initial evaluation is the `reset` evaluation), so particles are chains: K1 evaluates all
// of them at once.  Weights, trigger, cumulative sum, resampling and the multi-GPU all-gather are the kernels of
// population.cu.  Draw conventions as mcmcgpu_run_seqmc (Philox key = global particle id, step = (iter-1) nt + t + 1).
int32_t mcmcgpu_run_seqmc_models(mcmcgpu_ctx* c, int32_t nt, mcmcgpu_model* const* models, const mcmcgpu_sampler_cfg* samplers,
                                 int64_t steps, int64_t burnin, double trigger, int64_t npart, const double* particles,
                                 uint64_t seed, const double* inj_normals, const double* inj_uniforms,
                                 const double* inj_res_uniforms, double* out_samples, double* out_weights,
                                 int64_t* out_nresamples, mcmcgpu_run_info* info) {
  if (!c || !models || !samplers || !particles || !out_samples || !out_weights) return fail(MCMCGPU_E_ARG, "NULL argument");
  if (burnin < 0) return fail(MCMCGPU_E_ARG, "Burnin rounds should be >= 0");                   // SeqMC.jl:29
  if (steps <= burnin) return fail(MCMCGPU_E_ARG, "Steps should be > to burnin");               // SeqMC.jl:30
  if (npart < 2 || nt < 1 || nt > POP_MAX_TASKS) return fail(MCMCGPU_E_ARG, "at least 2 particles and between 1 and 64 tasks");
  const bool inj = inj_normals != nullptr;
  if (inj != (inj_uniforms != nullptr) || inj != (inj_res_uniforms != nullptr)) return fail(MCMCGPU_E_ARG, "inject all three draw arrays or none");
  for (int t = 0; t < nt; t++) {
    if (!models[t] || models[t]->ctx != c) return fail(MCMCGPU_E_ARG, "every model must belong to this context");
    if (models[t]->d != models[0]->d) return fail(MCMCGPU_E_ARG, "Models do not have the same parameter vector size");   // SeqMC.jl:47
    const mcmcgpu_sampler_cfg& sc = samplers[t];
    if (sc.tuner_on || (sc.kind != MCMCGPU_RWM && sc.kind != MCMCGPU_MALA && sc.kind != MCMCGPU_HMC))
      return fail(MCMCGPU_E_ARG, "population runners take RWM, MALA or HMC tasks without tuner");
  }
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  const int64_t d = models[0]->d;
  SeqArgs A;
  A.T.nt = nt; A.T.family = models[0]->family; A.T.d = (int32_t)d;
  DevBufs B;
  const int nranks = c->comm ? c->nranks : 1;
  const int64_t Np = round_up(npart, K1_CHAINS), S = (steps - burnin) * npart;
  A.npart = npart; A.Np = Np; A.steps = steps; A.burnin = burnin; A.seed = seed; A.trigger = trigger;
  A.rank = c->comm ? c->rank : 0; A.nranks = nranks;
  A.gpart = npart * nranks; A.sendbuf = nullptr; A.gathered = nullptr;
  const NcclApi* api = nullptr;
  if (nranks > 1) {
    api = nccl_api(nullptr);
    if (!api) return fail(MCMCGPU_E_COMM, "NCCL unavailable");
    double* gb = nullptr;
    CU(B.get(&A.sendbuf, (size_t)((d + 2) * Np), st));
    CU(B.get(&gb, (size_t)(nranks * (d + 2) * Np), st));
    A.gathered = gb;
  }
  double* hp = nullptr;
  CU(B.up(&hp, particles, (size_t)(npart * d), st));
  CU(B.get(&A.pars, (size_t)(d * Np), st));
  CU(transpose_to_chain_minor(hp, A.pars, npart, d, Np, st));
  CU(B.get(&A.pars_tmp, (size_t)(d * Np), st));
  CU(B.get(&A.logW, (size_t)Np, st)); CU(B.get(&A.logtarget, (size_t)Np, st)); CU(B.get(&A.lt_tmp, (size_t)Np, st));
  CU(B.get(&A.W, (size_t)(Np * nranks), st)); CU(B.get(&A.cp, (size_t)(Np * nranks), st));
  CU(B.get(&A.samples, (size_t)(S * d), st, false)); CU(B.get(&A.weights, (size_t)S, st, false));
  CU(B.get(&A.nres, 1, st)); CU(B.get(&A.nevals, 1, st));
  A.inj_normals = A.inj_uniforms = A.inj_res = nullptr;
  if (inj) {      // only the resampling uniforms are read by a population kernel; the sampler draws go through the runs
    double* r = nullptr;
    CU(B.up(&r, inj_res_uniforms, (size_t)(steps * nt * A.gpart), st));
    A.inj_res = r;
  }
  std::vector<double> zst, ust;      // injected sampler draws of one (iteration, target) in the run layout [particle][2][d]
  if (inj) { zst.assign((size_t)(npart * 2 * d), 0.0); ust.assign((size_t)(npart * 2), 0.0); }
  Events events;
  cudaEvent_t e0, e1;
  CU(events.make(&e0)); CU(events.make(&e1));
  CU(cudaEventRecord(e0, st));
  int64_t launches = 0, nev_total = 0, waves = 0;
  const int64_t time_eval_saved = c->time_eval;
  c->time_eval = 0;
  struct Restore { mcmcgpu_ctx* c; int64_t v; ~Restore() { c->time_eval = v; } } restore{c, time_eval_saved};
  for (int64_t i = 1; i <= steps; i++) {                                                        // SeqMC.jl:62
    A.iter = i;
    for (int t = 0; t < nt; t++) {                                                              // :64
      A.target = t;
      const int64_t pstep = (i - 1) * nt + t + 1;
      mcmcgpu_runner_cfg rc;
      memset(&rc, 0, sizeof(rc));
      rc.step = 1; rc.nchains = npart; rc.chain_offset = (int64_t)A.rank * npart; rc.seed = seed;
      rc.init_per_chain = 1; rc.store_grad = 0; rc.store_logtarget = 1; rc.engine = MCMCGPU_ENGINE_WAVE; rc.store_rb = 0;
      const double *zn = nullptr, *un = nullptr;
      if (inj) {
        rc.first = 1; rc.last = 1;
        const int64_t kbase = ((i - 1) * nt + t) * A.gpart + (int64_t)A.rank * npart;
        for (int64_t n = 0; n < npart; n++) {
          memcpy(&zst[(size_t)((n * 2 + 1) * d)], inj_normals + (kbase + n) * d, sizeof(double) * (size_t)d);
          ust[(size_t)(n * 2 + 1)] = inj_uniforms[kbase + n];
        }
        zn = zst.data(); un = ust.data();
      } else {
        rc.first = pstep; rc.last = pstep;
      }
      mcmcgpu_run* R = nullptr;
      int rcode = run_create_impl(models[t], &samplers[t], &rc, nullptr, A.pars, nullptr, zn, un, &R);
      if (rcode != MCMCGPU_OK) return rcode;
      struct RunGuard { mcmcgpu_run* r; ~RunGuard() { mcmcgpu_run_destroy(r); } } guard{R};
      if (!inj) R->step0 = pstep - 1;              // the step's Philox counter is (iter-1) nt + t + 1, as in the closed-form runner
      mcmcgpu_run_info ri;
      rcode = execute_impl(R, -1, &ri);
      if (rcode != MCMCGPU_OK) return rcode;
      nev_total += ri.n_grad_evals; launches += ri.n_launches; waves += ri.n_waves;
      CU(launch_seqmc_apply(A, R->samples, R->logtarget, R->init_lt, st));
      if (nranks > 1) {
        CU(launch_seqmc_pack(A, st));
        int nrc = api->AllGather(A.sendbuf, (void*)A.gathered, (size_t)((d + 2) * Np), NCCL_FLOAT64, c->comm, st);
        if (nrc != 0) return fail(MCMCGPU_E_COMM, std::string("ncclAllGather: ") + (api->GetErrorString ? api->GetErrorString(nrc) : "error"));
        launches++;
      }
      CU(launch_seqmc_resample(A, st));
      launches += 2;
      CU(cudaStreamSynchronize(st));               // the run's buffers are released by `guard` right after
    }
    CU(launch_seqmc_store(A, st));
    launches++;
  }
  CU(cudaEventRecord(e1, st));
  CU(cudaMemcpyAsync(out_samples, A.samples, sizeof(double) * (size_t)(S * d), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out_weights, A.weights, sizeof(double) * (size_t)S, cudaMemcpyDeviceToHost, st));
  unsigned long long nres = 0;
  CU(cudaMemcpyAsync(&nres, A.nres, sizeof(nres), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
  if (out_nresamples) *out_nresamples = (int64_t)nres;
  if (info) { info->gpu_ms = ms; info->n_grad_evals = nev_total; info->n_waves = waves; info->n_launches = launches; info->eval_ms = 0; info->comm_ms = 0; }
  return MCMCGPU_OK;
}

// SerialTempMC over arbitrary models (regression families through K1): at every iteration a replica consumes ONE task --
// its own, or at a swap attempt the candidate task, restarted at s.pars (SerialTempMC.jl:57-71) -- so the replicas are
// regrouped by task and each group is a one-step run of the wave engine on that task's model (particles = chains, as in
// mcmcgpu_run_seqmc_models); per-chain Philox keys keep a replica's draws independent of its position in the group.
// Draw conventions as mcmcgpu_run_serialtemp (key = global replica id, sampler step = column + 1, pick / swap blocks).
int32_t mcmcgpu_run_serialtemp_models(mcmcgpu_ctx* c, int32_t nt, mcmcgpu_model* const* models, const mcmcgpu_sampler_cfg* samplers,
                                      int64_t steps, int64_t burnin, int64_t swap_period, int64_t nrep, int64_t rep_offset,
                                      const double* inits, uint64_t seed, const double* inj_normals, const double* inj_uniforms,
                                      const double* inj_pick, const double* inj_swap, double* out_samples, int32_t* out_at,
                                      mcmcgpu_run_info* info) {
  if (!c || !models || !samplers || !inits || !out_samples) return fail(MCMCGPU_E_ARG, "NULL argument");
  if (burnin < 0) return fail(MCMCGPU_E_ARG, "Burnin rounds should be >= 0");                   // SerialTempMC.jl:22
  if (steps <= burnin) return fail(MCMCGPU_E_ARG, "Steps should be > to burnin");               // SerialTempMC.jl:23
  if (nt < 2 || nt > POP_MAX_TASKS || swap_period < 1 || nrep < 1) return fail(MCMCGPU_E_ARG, "need 2..64 tasks, swapPeriod >= 1, nrep >= 1");
  const bool inj = inj_normals != nullptr;
  if (inj != (inj_uniforms != nullptr) || inj != (inj_pick != nullptr) || inj != (inj_swap != nullptr))
    return fail(MCMCGPU_E_ARG, "inject all four draw arrays or none");
  for (int t = 0; t < nt; t++) {
    if (!models[t] || models[t]->ctx != c) return fail(MCMCGPU_E_ARG, "every model must belong to this context");
    if (models[t]->d != models[0]->d) return fail(MCMCGPU_E_ARG, "Models do not have the same parameter vector size");   // SerialTempMC.jl:39
    const mcmcgpu_sampler_cfg& sc = samplers[t];
    if (sc.tuner_on || (sc.kind != MCMCGPU_RWM && sc.kind != MCMCGPU_MALA && sc.kind != MCMCGPU_HMC))
      return fail(MCMCGPU_E_ARG, "population runners take RWM, MALA or HMC tasks without tuner");
  }
  const int64_t d = models[0]->d;
  for (int t = 0; t < nt; t++) {          // every task is started from its model.init (:44): the samplers' support assertion
    double lt = 0.0;
    int rc0 = mcmcgpu_logtarget_grad(models[t], inits + t * d, 1, &lt, nullptr);
    if (rc0 != MCMCGPU_OK) return rc0;
    if (!std::isfinite(lt)) return fail(MCMCGPU_E_SUPPORT, "Initial values out of model support, try other values");
  }
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  DevBufs B;
  const int64_t Rp = round_up(nrep, K1_CHAINS), S = steps - burnin;
  TempMArgs A;
  A.nt = nt; A.d = (int32_t)d; A.nrep = nrep; A.Rp = Rp; A.rep_offset = rep_offset; A.steps = steps; A.burnin = burnin; A.seed = seed;
  CU(B.get(&A.state, (size_t)(d * Rp), st)); CU(B.get(&A.pars, (size_t)(d * Rp), st)); CU(B.get(&A.ppars, (size_t)(d * Rp), st));
  CU(B.get(&A.res_pp, (size_t)(d * Rp), st)); CU(B.get(&A.res_lt0, (size_t)Rp, st)); CU(B.get(&A.logtarget, (size_t)Rp, st));
  CU(B.get(&A.at, (size_t)Rp, st)); CU(B.get(&A.sel, (size_t)Rp, st));
  CU(B.get(&A.samples, (size_t)(nrep * S * d), st, false));
  A.at_out = nullptr;
  if (out_at) CU(B.get(&A.at_out, (size_t)(nrep * S), st));
  A.inj_pick = A.inj_swap = nullptr;
  if (inj) {
    double *p = nullptr, *w = nullptr;
    CU(B.up(&p, inj_pick, (size_t)(nrep * (steps + 1)), st)); CU(B.up(&w, inj_swap, (size_t)(nrep * (steps + 1)), st));
    A.inj_pick = p; A.inj_swap = w;
  }
  int64_t launches = 0, nev_total = 0, waves = 0;
  const int64_t time_eval_saved = c->time_eval;
  c->time_eval = 0;
  struct Restore { mcmcgpu_ctx* c; int64_t v; ~Restore() { c->time_eval = v; } } restore{c, time_eval_saved};
  std::vector<double> zst, ust;
  // one group: the replicas idx consume task t with the draws of column col, started at A.pars; results -> A.res_pp / A.res_lt0
  auto group = [&](int t, const std::vector<int64_t>& idx, int64_t col) -> int {
    const int64_t n = (int64_t)idx.size(), Cp = round_up(n, K1_CHAINS);
    DevBufs G;
    int64_t *idx_dev = nullptr, *ids = nullptr;
    double* start = nullptr;
    CU(G.up(&idx_dev, idx.data(), (size_t)n, st));
    CU(G.get(&start, (size_t)(d * Cp), st, false)); CU(G.get(&ids, (size_t)Cp, st, false));
    CU(launch_temp_gather(A, idx_dev, n, Cp, start, ids, st));
    mcmcgpu_runner_cfg rc;
    memset(&rc, 0, sizeof(rc));
    rc.step = 1; rc.nchains = n; rc.chain_offset = 0; rc.seed = seed; rc.init_per_chain = 1; rc.store_logtarget = 1; rc.engine = MCMCGPU_ENGINE_WAVE;
    const double *zn = nullptr, *un = nullptr;
    if (inj) {
      rc.first = 1; rc.last = 1;
      zst.assign((size_t)(n * 2 * d), 0.0); ust.assign((size_t)(n * 2), 0.0);
      for (int64_t k = 0; k < n; k++) {
        const int64_t r = idx[(size_t)k];
        memcpy(&zst[(size_t)((k * 2 + 1) * d)], inj_normals + (r * (steps + 2) + col) * d, sizeof(double) * (size_t)d);
        ust[(size_t)(k * 2 + 1)] = inj_uniforms[r * (steps + 2) + col];
      }
      zn = zst.data(); un = ust.data();
    } else {
      rc.first = col + 1; rc.last = col + 1;
    }
    mcmcgpu_run* R = nullptr;
    int rcode = run_create_impl(models[t], &samplers[t], &rc, nullptr, start, nullptr, zn, un, &R);
    if (rcode != MCMCGPU_OK) return rcode;
    struct RunGuard { mcmcgpu_run* r; ~RunGuard() { mcmcgpu_run_destroy(r); } } guard{R};
    if (!inj) R->step0 = col;
    R->chain_ids = ids;
    mcmcgpu_run_info ri;
    rcode = execute_impl(R, -1, &ri);
    if (rcode != MCMCGPU_OK) return rcode;
    nev_total += ri.n_grad_evals; launches += ri.n_launches + 2; waves += ri.n_waves;
    CU(launch_temp_scatter(A, idx_dev, n, Cp, R->samples, R->init_lt, st));
    CU(cudaStreamSynchronize(st));
    return MCMCGPU_OK;
  };
  Events events;
  cudaEvent_t e0, e1;
  CU(events.make(&e0)); CU(events.make(&e1));
  CU(cudaEventRecord(e0, st));
  std::vector<int64_t> all((size_t)nrep);
  for (int64_t r = 0; r < nrep; r++) all[(size_t)r] = r;
  const size_t plane = sizeof(double) * (size_t)(d * Rp);
  // :44 the first consume of task 1 from its model.init (column 0), :51 its second step from its own state (column 1)
  for (int64_t j = 0; j < d; j++) CU(launch_fill(A.pars + j * Rp, inits[j], Rp, st));
  int rcode = group(0, all, 0);
  if (rcode != MCMCGPU_OK) return rcode;
  CU(cudaMemcpyAsync(A.state, A.res_pp, plane, cudaMemcpyDeviceToDevice, st));
  CU(cudaMemcpyAsync(A.pars, A.state, plane, cudaMemcpyDeviceToDevice, st));
  rcode = group(0, all, 1);
  if (rcode != MCMCGPU_OK) return rcode;
  CU(cudaMemcpyAsync(A.ppars, A.res_pp, plane, cudaMemcpyDeviceToDevice, st));
  CU(cudaMemcpyAsync(A.state, A.res_pp, plane, cudaMemcpyDeviceToDevice, st));
  CU(cudaMemcpyAsync(A.logtarget, A.res_lt0, sizeof(double) * (size_t)Rp, cudaMemcpyDeviceToDevice, st));   // s.logtarget (:53)
  std::vector<int32_t> sel((size_t)nrep);
  std::vector<std::vector<int64_t>> groups((size_t)nt);
  for (int64_t i = 1; i <= steps; i++) {
    const bool swap_step = (i % swap_period) == 0;                                              // :57
    CU(launch_temp_plan(A, i, swap_step, st));
    CU(cudaMemcpyAsync(sel.data(), A.sel, sizeof(int32_t) * (size_t)nrep, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (auto& g : groups) g.clear();
    for (int64_t r = 0; r < nrep; r++) groups[(size_t)sel[(size_t)r]].push_back(r);
    for (int t = 0; t < nt; t++) {
      if (groups[(size_t)t].empty()) continue;
      rcode = group(t, groups[(size_t)t], i + 1);
      if (rcode != MCMCGPU_OK) return rcode;
    }
    CU(launch_temp_update(A, i, swap_step, st));
    launches += 2;
  }
  CU(cudaEventRecord(e1, st));
  CU(cudaMemcpyAsync(out_samples, A.samples, sizeof(double) * (size_t)(nrep * S * d), cudaMemcpyDeviceToHost, st));
  if (out_at) CU(cudaMemcpyAsync(out_at, A.at_out, sizeof(int32_t) * (size_t)(nrep * S), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
  if (info) { info->gpu_ms = ms; info->n_grad_evals = nev_total; info->n_waves = waves; info->n_launches = launches; info->eval_ms = 0; info->comm_ms = 0; }
  return MCMCGPU_OK;
}

int32_t mcmcgpu_run_serialtemp(mcmcgpu_ctx* c, int32_t family, int64_t d, int32_t nt, const double* hypers,
                               const mcmcgpu_sampler_cfg* samplers, int64_t steps, int64_t burnin, int64_t swap_period, int64_t nrep,
                               const double* inits, uint64_t seed, const double* inj_normals, const double* inj_uniforms,
                               const double* inj_pick, const double* inj_swap, double* out_samples, int32_t* out_at,
                               mcmcgpu_run_info* info) {
  if (!c || !inits || !out_samples) return fail(MCMCGPU_E_ARG, "NULL argument");
  if (burnin < 0) return fail(MCMCGPU_E_ARG, "Burnin rounds should be >= 0");                   // SerialTempMC.jl:22
  if (steps <= burnin) return fail(MCMCGPU_E_ARG, "Steps should be > to burnin");               // SerialTempMC.jl:23
  if (nt < 2 || swap_period < 1 || nrep < 1) return fail(MCMCGPU_E_ARG, "need >= 2 tasks, swapPeriod >= 1, nrep >= 1");
  const bool inj = inj_normals != nullptr;
  if (inj != (inj_uniforms != nullptr) || inj != (inj_pick != nullptr) || inj != (inj_swap != nullptr))
    return fail(MCMCGPU_E_ARG, "inject all four draw arrays or none");
  TempArgs A;
  int rc = fill_tasks(A.T, family, d, nt, hypers, samplers);
  if (rc != MCMCGPU_OK) return rc;
  CU(use_ctx(c));
  cudaStream_t st = c->stream;
  DevBufs B;
  const int64_t S = steps - burnin;
  A.nrep = nrep; A.steps = steps; A.burnin = burnin; A.swap_period = swap_period; A.seed = seed;
  double* di = nullptr;
  CU(B.up(&di, inits, (size_t)(d * nt), st));
  A.inits = di;
  A.inj_normals = A.inj_uniforms = A.inj_pick = A.inj_swap = nullptr;
  if (inj) {
    double *a = nullptr, *b = nullptr, *p = nullptr, *w = nullptr;
    CU(B.up(&a, inj_normals, (size_t)(nrep * (steps + 2) * d), st)); CU(B.up(&b, inj_uniforms, (size_t)(nrep * (steps + 2)), st));
    CU(B.up(&p, inj_pick, (size_t)(nrep * (steps + 1)), st)); CU(B.up(&w, inj_swap, (size_t)(nrep * (steps + 1)), st));
    A.inj_normals = a; A.inj_uniforms = b; A.inj_pick = p; A.inj_swap = w;
  }
  CU(B.get(&A.samples, (size_t)(nrep * S * d), st, false));
  A.at = nullptr;
  if (out_at) CU(B.get(&A.at, (size_t)(nrep * S), st));
  CU(B.get(&A.status, (size_t)nrep, st)); CU(B.get(&A.nevals, 1, st));
  Events events;
  cudaEvent_t e0, e1;
  CU(events.make(&e0)); CU(events.make(&e1));
  CU(cudaEventRecord(e0, st));
  CU(launch_serialtemp(A, st));
  CU(cudaEventRecord(e1, st));
  CU(cudaMemcpyAsync(out_samples, A.samples, sizeof(double) * (size_t)(nrep * S * d), cudaMemcpyDeviceToHost, st));
  if (out_at) CU(cudaMemcpyAsync(out_at, A.at, sizeof(int32_t) * (size_t)(nrep * S), cudaMemcpyDeviceToHost, st));
  std::vector<int32_t> stt((size_t)nrep);
  unsigned long long nev = 0;
  CU(cudaMemcpyAsync(stt.data(), A.status, sizeof(int32_t) * (size_t)nrep, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(&nev, A.nevals, sizeof(nev), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
  if (info) { info->gpu_ms = ms; info->n_grad_evals = (int64_t)nev; info->n_waves = 0; info->n_launches = 1; info->eval_ms = 0; info->comm_ms = 0; }
  for (int32_t v : stt) if (v) return fail(MCMCGPU_E_SUPPORT, "Initial values out of model support, try other values");
  return MCMCGPU_OK;
}

}  // extern "C"
