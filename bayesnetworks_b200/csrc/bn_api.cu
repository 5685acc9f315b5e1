// The extern "C" layer of libbn_b200.so (include/bn_b200.h): context management,
// host<->device marshalling, kernel launches.  No compute happens on the host.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/bn_b200.h"
#include "gram.h"
#include "kernels.h"

using namespace bn;

// bn_run copies the leading bn_best_graph out of each chain's BestTrack
static_assert(offsetof(BestTrack, log_post) == offsetof(bn_best_graph, log_post) &&
              offsetof(BestTrack, log_lik) == offsetof(bn_best_graph, log_lik) &&
              offsetof(BestTrack, log_prior) == offsetof(bn_best_graph, log_prior) &&
              offsetof(BestTrack, iter) == offsetof(bn_best_graph, iter) &&
              offsetof(BestTrack, total_edges) == offsetof(bn_best_graph, total_edges) &&
              offsetof(BestTrack, found) == offsetof(bn_best_graph, found) &&
              sizeof(bn_best_graph) <= sizeof(BestTrack), "BestTrack must start with bn_best_graph");

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU_TRY(expr)                                                                        \
  do {                                                                                      \
    cudaError_t e_ = (expr);                                                                \
    if (e_ != cudaSuccess)                                                                  \
      return fail(e_ == cudaErrorMemoryAllocation ? BN_ERR_OOM : BN_ERR_CUDA, "%s: %s (%s:%d)", \
                  #expr, cudaGetErrorString(e_), __FILE__, __LINE__);                       \
  } while (0)

static thread_local cudaStream_t g_default_stream = nullptr;

extern "C" const char* bn_last_error(void) { return g_err; }
extern "C" int bn_set_default_stream(void* s) { g_default_stream = (cudaStream_t)s; return BN_OK; }
extern "C" int bn_abi_version(void) { return BN_B200_ABI_VERSION; }
extern "C" int bn_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// ---------------------------------------------------------------------------
// device workspace pool: cudaMalloc/cudaFree of the 100 MB..GB scratch buffers (centred
// copy of X, split-K partials, per-chain state) costs far more than the kernels that use
// them, so freed blocks are kept per device and handed out again.  bn_trim_pool() or
// BN_B200_POOL=0 returns the memory to the driver.
// ---------------------------------------------------------------------------
#include <mutex>
namespace {
struct PoolBlock { void* p; size_t n; int dev; bool used; };
std::mutex g_pool_mu;
std::vector<PoolBlock> g_pool;
const size_t kPoolMaxBlock = (size_t)8 << 30;

bool pool_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("BN_B200_POOL"); on = (e && e[0] == '0') ? 0 : 1; }
  return on == 1;
}

cudaError_t pool_alloc(void** out, size_t n) {
  if (n == 0) n = 1;
  int dev = 0;
  cudaGetDevice(&dev);
  if (pool_enabled()) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    int best = -1;
    for (int i = 0; i < (int)g_pool.size(); i++) {
      PoolBlock& b = g_pool[i];
      if (!b.used && b.dev == dev && b.n >= n && b.n <= 2 * n + (1 << 20) &&
          (best < 0 || b.n < g_pool[best].n))
        best = i;
    }
    if (best >= 0) { g_pool[best].used = true; *out = g_pool[best].p; return cudaSuccess; }
  }
  cudaError_t e = cudaMalloc(out, n);
  if (e != cudaSuccess && pool_enabled()) {
    // out of memory: drop the cached blocks of this device and retry once
    std::lock_guard<std::mutex> lk(g_pool_mu);
    cudaGetLastError();
    for (auto it = g_pool.begin(); it != g_pool.end();)
      if (!it->used && it->dev == dev) { cudaFree(it->p); it = g_pool.erase(it); } else ++it;
    e = cudaMalloc(out, n);
  }
  if (e == cudaSuccess && pool_enabled() && n <= kPoolMaxBlock) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    g_pool.push_back({*out, n, dev, true});
  }
  return e;
}

void pool_free(void* p) {
  if (!p) return;
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    for (PoolBlock& b : g_pool)
      if (b.p == p) { b.used = false; return; }
  }
  cudaFree(p);
}
}  // namespace

extern "C" int bn_trim_pool(void) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  for (auto it = g_pool.begin(); it != g_pool.end();)
    if (!it->used) { cudaSetDevice(it->dev); cudaFree(it->p); it = g_pool.erase(it); } else ++it;
  return BN_OK;
}

// BN_B200_TIMING=1: host wall-clock of the stages of bn_create*/bn_run on stderr
#include <chrono>
namespace {
struct StageTimer {
  bool on;
  std::chrono::steady_clock::time_point t;
  const char* fn;
  explicit StageTimer(const char* f) : fn(f) {
    static int env = -1;
    if (env < 0) { const char* e = getenv("BN_B200_TIMING"); env = (e && e[0] == '1') ? 1 : 0; }
    on = env == 1;
    if (on) t = std::chrono::steady_clock::now();
  }
  void lap(const char* what) {
    if (!on) return;
    const auto n = std::chrono::steady_clock::now();
    fprintf(stderr, "[bn timing] %s: %s %.3f ms\n", fn, what, std::chrono::duration<double, std::milli>(n - t).count());
    t = n;
  }
};
}  // namespace

__global__ void colsum_from_mean_kernel(const double* __restrict__ mean, int n_samples, int P,
                                        double* __restrict__ colsum) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < P) colsum[p] = mean[p] * (double)n_samples;
}

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
struct bn_ctx {
  int device = 0;
  int n_sms = 148;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  int n_samples = 0, P = 0, max_par = 0, n_sim_edges = 0;
  double phi = 1, omega = 6.9;
  double* d_C = nullptr;       // centred Gram [P][P]
  double* d_diag = nullptr;    // [P]
  double* d_mean = nullptr;    // [P]
  double* d_colsum = nullptr;  // [P]
  uint8_t* d_node_type = nullptr;
  uint8_t* d_sim_edge = nullptr;  // [parent + child*P]
  int* d_prior_par = nullptr;     // [P][prior_stride]
  int* d_prior_npar = nullptr;    // [P]
  int prior_stride = 1;           // largest in-degree of the supplied graph (>= 1)
  float gram_ms = 0.f;
  int64_t launches = 0;
  std::vector<void*> owned;  // device allocations freed by bn_destroy
};

template <typename T>
static cudaError_t dalloc(bn_ctx* c, T** p, size_t n) {
  cudaError_t e = pool_alloc((void**)p, n * sizeof(T));
  if (e == cudaSuccess && c) c->owned.push_back((void*)*p);
  return e;
}

extern "C" void bn_destroy(bn_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  for (void* p : c->owned) pool_free(p);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

static int check_graph_args(int n_samples, int P, const int* src, const int* tgt, int n_edges,
                            const int* node_type, int max_par) {
  if (n_samples < 3) return fail(BN_ERR_BAD_ARG, "n_samples must be >= 3 (got %d)", n_samples);
  if (P < 2 || P > 65535) return fail(BN_ERR_BAD_ARG, "n_nodes must be in [2, 65535] (got %d)", P);
  if (max_par < 1) return fail(BN_ERR_BAD_ARG, "max_par must be >= 1 (got %d)", max_par);
  if (max_par > 64) return fail(BN_ERR_UNSUPPORTED, "max_par > 64 is not supported (got %d)", max_par);
  if (n_edges < 0 || (n_edges > 0 && (!src || !tgt))) return fail(BN_ERR_BAD_ARG, "bad edge list");
  if (!node_type) return fail(BN_ERR_BAD_ARG, "node_type is NULL");
  for (int p = 0; p < P; p++)
    if (node_type[p] < 0 || node_type[p] > 2)
      return fail(BN_ERR_BAD_ARG, "node_type[%d] = %d is not 0/1/2", p, node_type[p]);
  for (int e = 0; e < n_edges; e++)
    if (src[e] < 1 || src[e] > P || tgt[e] < 1 || tgt[e] > P)
      return fail(BN_ERR_BAD_ARG, "edge %d (%d -> %d) out of range 1..%d", e, src[e], tgt[e], P);
  return BN_OK;
}

// device selection + graph/prior upload shared by the three constructors
static int ctx_begin(int n_samples, int P, const int* src, const int* tgt, int n_edges, const int* node_type,
                     int max_par, double phi, double omega, int device, bn_ctx** out) {
  if (!out) return fail(BN_ERR_BAD_ARG, "out is NULL");
  *out = nullptr;
  StageTimer tm("ctx_begin");
  int rc = check_graph_args(n_samples, P, src, tgt, n_edges, node_type, max_par);
  if (rc) return rc;
  int ndev = bn_device_count();
  if (ndev <= 0) return fail(BN_ERR_NO_DEVICE, "no CUDA device available (libbn_b200 has no CPU path)");
  if (device < 0 || device >= ndev) return fail(BN_ERR_NO_DEVICE, "device %d out of range (0..%d)", device, ndev - 1);
  CU_TRY(cudaSetDevice(device));
  bn_ctx* c = new bn_ctx();
  c->device = device;
  c->n_samples = n_samples; c->P = P; c->max_par = max_par; c->phi = phi; c->omega = omega;
  tm.lap("args+device");
  // (cudaGetDeviceProperties costs 3-25 ms per call; one attribute is microseconds)
  int n_sms = 0;
  if (cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && n_sms > 0) c->n_sms = n_sms;
  tm.lap("device attributes");
  *out = c;  // from here on the caller destroys on failure
  CU_TRY(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  tm.lap("stream create");
  c->stream = g_default_stream ? g_default_stream : c->own_stream;

  // parent lists edges[tgt-1].push_back(src-1), src/network.h:117-120.  The supplied graph may
  // give a node more than max_par parents: with InitialNetwork = 2 (the default) it only feeds
  // simEdge / NsimEdges (:138-146,164-169), so the lists keep their own stride and the limit is
  // checked by bn_run for InitialNetwork = 0 only.
  std::vector<int> npar(P, 0);
  for (int e = 0; e < n_edges; e++) npar[tgt[e] - 1]++;
  int stride = 1;
  for (int p = 0; p < P; p++) if (npar[p] > stride) stride = npar[p];
  c->prior_stride = stride;
  std::fill(npar.begin(), npar.end(), 0);
  std::vector<int> par((size_t)P * stride, -1);
  std::vector<uint8_t> sim((size_t)P * P, 0), types(P);
  for (int e = 0; e < n_edges; e++) {
    const int child = tgt[e] - 1, parent = src[e] - 1;
    par[(size_t)child * stride + npar[child]++] = parent;
    // simEdge(parent, child) = 1; NsimEdges counts list entries, src/network.h:140-145
    sim[(size_t)parent + (size_t)child * P] = 1;
    c->n_sim_edges++;
  }
  for (int p = 0; p < P; p++) types[p] = (uint8_t)node_type[p];
  tm.lap("host graph arrays");
  CU_TRY(dalloc(c, &c->d_prior_par, par.size()));
  CU_TRY(dalloc(c, &c->d_prior_npar, npar.size()));
  CU_TRY(dalloc(c, &c->d_sim_edge, sim.size()));
  CU_TRY(dalloc(c, &c->d_node_type, types.size()));
  CU_TRY(dalloc(c, &c->d_C, (size_t)P * P));
  CU_TRY(dalloc(c, &c->d_diag, (size_t)P));
  CU_TRY(dalloc(c, &c->d_mean, (size_t)P));
  CU_TRY(dalloc(c, &c->d_colsum, (size_t)P));
  tm.lap("device allocations");
  CU_TRY(cudaMemcpy(c->d_prior_par, par.data(), par.size() * sizeof(int), cudaMemcpyHostToDevice));
  CU_TRY(cudaMemcpy(c->d_prior_npar, npar.data(), npar.size() * sizeof(int), cudaMemcpyHostToDevice));
  CU_TRY(cudaMemcpy(c->d_sim_edge, sim.data(), sim.size(), cudaMemcpyHostToDevice));
  CU_TRY(cudaMemcpy(c->d_node_type, types.data(), types.size(), cudaMemcpyHostToDevice));
  tm.lap("graph upload");
  return BN_OK;
}

// X on the device (dX, ldx) -> d_C.  If inplace, dX is the context's padded buffer.
// hX != NULL: X is still in host memory; its H2D copy into dXc is pipelined with the build
// (gram_build_from_host), one block of 128 columns at a time on a second stream.
static int ctx_build_gram(bn_ctx* c, const double* dX, int64_t ldx, double* dXc, const GramPlan& pl,
                          const double* hX = nullptr) {
  double *d_partial = nullptr, *d_scratch = nullptr;
  int* d_flag = nullptr;
  StageTimer tm("ctx_build_gram");
  CU_TRY(pool_alloc((void**)&d_partial, (size_t)pl.workspace_bytes));
  cudaError_t e1 = pool_alloc((void**)&d_scratch, (size_t)c->P * GRAM_MEAN_MAX_CHUNKS * sizeof(double));
  cudaError_t e2 = pool_alloc((void**)&d_flag, sizeof(int));
  int rc = BN_OK;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (e1 != cudaSuccess || e2 != cudaSuccess) rc = fail(BN_ERR_OOM, "gram scratch allocation failed");
  tm.lap("workspace");
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> arrived;
  if (!rc) {
    cudaEventCreate(&ev0); cudaEventCreate(&ev1);
    cudaEventRecord(ev0, c->stream);
    const char* msg;
    if (hX) {
      if (cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
        rc = fail(BN_ERR_CUDA, "cannot create the copy stream");
      } else {
        arrived.resize(pl.n_tiles);
        for (auto& e : arrived) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
        // the copy stream must not start before whatever the compute stream was asked to do first
        cudaEvent_t start;
        cudaEventCreateWithFlags(&start, cudaEventDisableTiming);
        cudaEventRecord(start, c->stream);
        cudaStreamWaitEvent(copy_stream, start, 0);
        cudaEventDestroy(start);
        msg = gram_build_from_host(hX, c->n_samples, c->P, dXc, pl.ld_centered, d_partial, pl, c->d_colsum,
                                   c->d_mean, c->d_C, c->P, d_scratch, d_flag, c->stream, copy_stream,
                                   arrived.data(), &c->launches);
        if (msg) rc = fail(BN_ERR_CUDA, "gram_build_from_host: %s", msg);
      }
    } else {
      msg = gram_build(dX, ldx, c->n_samples, c->P, dXc, pl.ld_centered, d_partial, pl, c->d_colsum,
                       c->d_mean, c->d_C, c->P, d_scratch, d_flag, c->stream, &c->launches);
      if (msg) rc = fail(BN_ERR_CUDA, "gram_build: %s", msg);
    }
  }
  if (!rc) {
    launch_diag(c->d_C, c->P, c->P, c->d_diag, c->stream);
    c->launches++;
    cudaEventRecord(ev1, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) rc = fail(BN_ERR_CUDA, "gram kernels: %s", cudaGetErrorString(e));
  }
  if (!rc) {
    cudaEventElapsedTime(&c->gram_ms, ev0, ev1);
    int flag = 0;
    cudaMemcpy(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost);
    if (flag) rc = fail(BN_ERR_CUDA, "gram_dmma_kernel: TMA pipeline timed out (flag %d)", flag);
  }
  if (ev0) cudaEventDestroy(ev0);
  if (ev1) cudaEventDestroy(ev1);
  if (copy_stream) { cudaStreamSynchronize(copy_stream); cudaStreamDestroy(copy_stream); }
  for (auto& e : arrived) cudaEventDestroy(e);
  pool_free(d_partial); pool_free(d_scratch); pool_free(d_flag);
  tm.lap("launch + sync (incl. pending H2D)");
  return rc;
}

extern "C" int bn_create(const double* X, int n_samples, int P, const int* src, const int* tgt, int n_edges,
                         const int* node_type, int max_par, double phi, double omega, int device,
                         bn_ctx** out) {
  if (!X) return fail(BN_ERR_BAD_ARG, "X is NULL");
  int rc = ctx_begin(n_samples, P, src, tgt, n_edges, node_type, max_par, phi, omega, device, out);
  if (rc) { if (out && *out) { bn_destroy(*out); *out = nullptr; } return rc; }
  bn_ctx* c = *out;
  StageTimer tm("bn_create");
  const GramPlan pl = gram_plan(n_samples, P, c->n_sms);
  double* dXc = nullptr;
  cudaError_t e = pool_alloc((void**)&dXc, (size_t)pl.ld_centered * P * sizeof(double));
  if (e != cudaSuccess) { bn_destroy(c); *out = nullptr; return fail(BN_ERR_OOM, "cannot allocate the device copy of X"); }
  tm.lap("alloc device copy of X");
  // column p of the R matrix is contiguous: the copy into the padded buffer goes block of
  // columns by block of columns, overlapped with the build (centred in place)
  if (!rc) rc = ctx_build_gram(c, dXc, pl.ld_centered, dXc, pl, X);
  pool_free(dXc);
  if (rc) { bn_destroy(c); *out = nullptr; }
  return rc;
}

extern "C" int bn_create_from_device(const double* dX, int64_t ld, int n_samples, int P, const int* src,
                                     const int* tgt, int n_edges, const int* node_type, int max_par,
                                     double phi, double omega, int device, bn_ctx** out) {
  if (!dX) return fail(BN_ERR_BAD_ARG, "dX is NULL");
  if (ld < n_samples) return fail(BN_ERR_BAD_ARG, "ld < n_samples");
  int rc = ctx_begin(n_samples, P, src, tgt, n_edges, node_type, max_par, phi, omega, device, out);
  if (rc) { if (out && *out) { bn_destroy(*out); *out = nullptr; } return rc; }
  bn_ctx* c = *out;
  const GramPlan pl = gram_plan(n_samples, P, c->n_sms);
  double* dXc = nullptr;
  cudaError_t e = pool_alloc((void**)&dXc, (size_t)pl.ld_centered * P * sizeof(double));
  if (e != cudaSuccess) { bn_destroy(c); *out = nullptr; return fail(BN_ERR_OOM, "cannot allocate the centred copy of X"); }
  rc = ctx_build_gram(c, dX, ld, dXc, pl);
  pool_free(dXc);
  if (rc) { bn_destroy(c); *out = nullptr; }
  return rc;
}

extern "C" int bn_create_from_stats(int n_samples, int P, const double* mean, const double* centered,
                                    const int* src, const int* tgt, int n_edges, const int* node_type,
                                    int max_par, double phi, double omega, int device, bn_ctx** out) {
  if (!mean || !centered) return fail(BN_ERR_BAD_ARG, "mean/centered_gram is NULL");
  int rc = ctx_begin(n_samples, P, src, tgt, n_edges, node_type, max_par, phi, omega, device, out);
  if (rc) { if (out && *out) { bn_destroy(*out); *out = nullptr; } return rc; }
  bn_ctx* c = *out;
  std::vector<double> colsum(P);
  for (int p = 0; p < P; p++) colsum[p] = mean[p] * (double)n_samples;
  cudaError_t e = cudaMemcpy(c->d_C, centered, (size_t)P * P * 8, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(c->d_mean, mean, (size_t)P * 8, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(c->d_colsum, colsum.data(), (size_t)P * 8, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    launch_diag(c->d_C, P, P, c->d_diag, c->stream);
    c->launches++;
    e = cudaStreamSynchronize(c->stream);
  }
  if (e != cudaSuccess) {
    rc = fail(BN_ERR_CUDA, "upload of sufficient statistics: %s", cudaGetErrorString(e));
    bn_destroy(c); *out = nullptr;
  }
  return rc;
}

// ---------------------------------------------------------------------------
// row-sharded sufficient statistics (SURVEY.md 8e: config 5)
// ---------------------------------------------------------------------------
extern "C" int bn_block_colsum_device(const double* dX, int64_t ld, int n_rows, int P, double* d_out_sum,
                                      int device, void* stream) {
  if (!dX || !d_out_sum) return fail(BN_ERR_BAD_ARG, "NULL argument");
  if (n_rows < 1 || P < 1 || ld < n_rows) return fail(BN_ERR_BAD_ARG, "bad block shape");
  int ndev = bn_device_count();
  if (ndev <= 0) return fail(BN_ERR_NO_DEVICE, "no CUDA device available (libbn_b200 has no CPU path)");
  if (device < 0 || device >= ndev) return fail(BN_ERR_NO_DEVICE, "device %d out of range", device);
  CU_TRY(cudaSetDevice(device));
  cudaStream_t st = stream ? (cudaStream_t)stream : g_default_stream;
  double *d_part = nullptr, *d_mean = nullptr;
  CU_TRY(pool_alloc((void**)&d_part, (size_t)P * GRAM_MEAN_MAX_CHUNKS * sizeof(double)));
  cudaError_t e = pool_alloc((void**)&d_mean, (size_t)P * sizeof(double));
  if (e == cudaSuccess) {
    gram_column_sums(dX, ld, n_rows, P, d_part, d_out_sum, d_mean, st);
    e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
  }
  pool_free(d_part); pool_free(d_mean);
  if (e != cudaSuccess) return fail(BN_ERR_CUDA, "block column sums: %s", cudaGetErrorString(e));
  return BN_OK;
}

extern "C" int bn_block_gram_device(const double* dX, int64_t ld, int n_rows, int P, const double* d_mean,
                                    double* d_out_gram, int device, void* stream, float* ms) {
  if (!dX || !d_mean || !d_out_gram) return fail(BN_ERR_BAD_ARG, "NULL argument");
  if (n_rows < 1 || P < 2 || ld < n_rows) return fail(BN_ERR_BAD_ARG, "bad block shape");
  int ndev = bn_device_count();
  if (ndev <= 0) return fail(BN_ERR_NO_DEVICE, "no CUDA device available (libbn_b200 has no CPU path)");
  if (device < 0 || device >= ndev) return fail(BN_ERR_NO_DEVICE, "device %d out of range", device);
  CU_TRY(cudaSetDevice(device));
  cudaStream_t st = stream ? (cudaStream_t)stream : g_default_stream;
  int n_sms = 148;
  cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, device);
  const GramPlan pl = gram_plan(n_rows, P, n_sms);
  double *dXc = nullptr, *d_partial = nullptr;
  int* d_flag = nullptr;
  cudaError_t e = pool_alloc((void**)&dXc, (size_t)pl.ld_centered * P * sizeof(double));
  if (e == cudaSuccess) e = pool_alloc((void**)&d_partial, (size_t)pl.workspace_bytes);
  if (e == cudaSuccess) e = pool_alloc((void**)&d_flag, sizeof(int));
  int rc = BN_OK;
  if (e != cudaSuccess) rc = fail(BN_ERR_OOM, "block gram workspace allocation failed");
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (!rc) {
    cudaEventCreate(&ev0); cudaEventCreate(&ev1);
    cudaEventRecord(ev0, st);
    const char* msg = gram_build(dX, ld, n_rows, P, dXc, pl.ld_centered, d_partial, pl, nullptr,
                                 const_cast<double*>(d_mean), d_out_gram, P, nullptr, d_flag, st, nullptr, true);
    if (msg) rc = fail(BN_ERR_CUDA, "gram_build: %s", msg);
  }
  if (!rc) {
    cudaEventRecord(ev1, st);
    e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) rc = fail(BN_ERR_CUDA, "block gram kernels: %s", cudaGetErrorString(e));
  }
  if (!rc) {
    float t = 0.f;
    cudaEventElapsedTime(&t, ev0, ev1);
    if (ms) *ms = t;
    int flag = 0;
    cudaMemcpy(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost);
    if (flag) rc = fail(BN_ERR_CUDA, "gram_dmma_kernel: TMA pipeline timed out (flag %d)", flag);
  }
  if (ev0) cudaEventDestroy(ev0);
  if (ev1) cudaEventDestroy(ev1);
  pool_free(dXc); pool_free(d_partial); pool_free(d_flag);
  return rc;
}

extern "C" int bn_create_from_stats_device(int n_samples, int P, const double* d_mean, const double* d_centered,
                                           const int* src, const int* tgt, int n_edges, const int* node_type,
                                           int max_par, double phi, double omega, int device, bn_ctx** out) {
  if (!d_mean || !d_centered) return fail(BN_ERR_BAD_ARG, "mean/centered_gram is NULL");
  int rc = ctx_begin(n_samples, P, src, tgt, n_edges, node_type, max_par, phi, omega, device, out);
  if (rc) { if (out && *out) { bn_destroy(*out); *out = nullptr; } return rc; }
  bn_ctx* c = *out;
  cudaError_t e = cudaMemcpyAsync(c->d_C, d_centered, (size_t)P * P * 8, cudaMemcpyDeviceToDevice, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_mean, d_mean, (size_t)P * 8, cudaMemcpyDeviceToDevice, c->stream);
  if (e == cudaSuccess) {
    colsum_from_mean_kernel<<<(P + 127) / 128, 128, 0, c->stream>>>(c->d_mean, n_samples, P, c->d_colsum);
    launch_diag(c->d_C, P, P, c->d_diag, c->stream);
    c->launches += 2;
    e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
  }
  if (e != cudaSuccess) {
    rc = fail(BN_ERR_CUDA, "device sufficient statistics: %s", cudaGetErrorString(e));
    bn_destroy(c); *out = nullptr;
  }
  return rc;
}

extern "C" int bn_set_stream(bn_ctx* c, void* s) {
  if (!c) return fail(BN_ERR_BAD_ARG, "ctx is NULL");
  c->stream = s ? (cudaStream_t)s : c->own_stream;
  return BN_OK;
}

extern "C" int bn_get_gram_ms(bn_ctx* c, float* ms) {
  if (!c || !ms) return fail(BN_ERR_BAD_ARG, "NULL argument");
  *ms = c->gram_ms;
  return BN_OK;
}

extern "C" int64_t bn_get_launch_count(bn_ctx* c) { return c ? c->launches : 0; }

extern "C" int bn_get_stats(bn_ctx* c, double* sum_x, double* sum_xx, double* mean, double* centered) {
  if (!c) return fail(BN_ERR_BAD_ARG, "ctx is NULL");
  CU_TRY(cudaSetDevice(c->device));
  const int P = c->P;
  std::vector<double> C((size_t)P * P), cs(P), mu(P);
  CU_TRY(cudaMemcpy(C.data(), c->d_C, C.size() * 8, cudaMemcpyDeviceToHost));
  CU_TRY(cudaMemcpy(cs.data(), c->d_colsum, (size_t)P * 8, cudaMemcpyDeviceToHost));
  CU_TRY(cudaMemcpy(mu.data(), c->d_mean, (size_t)P * 8, cudaMemcpyDeviceToHost));
  if (sum_x) memcpy(sum_x, cs.data(), (size_t)P * 8);
  if (mean) memcpy(mean, mu.data(), (size_t)P * 8);
  if (centered) memcpy(centered, C.data(), C.size() * 8);
  if (sum_xx) {
    // marshalling only: sum x_i x_j = C_ij + N mean_i mean_j (C is about the computed means)
    const double n = (double)c->n_samples;
    for (int a = 0; a < P; a++)
      for (int b = 0; b < P; b++) sum_xx[(size_t)a + (size_t)b * P] = C[(size_t)a * P + b] + n * mu[a] * mu[b];
  }
  return BN_OK;
}

// ---------------------------------------------------------------------------
// scoring
// ---------------------------------------------------------------------------
extern "C" int bn_score_nodes(bn_ctx* c, int n_items, const int* child, const int* parents, const int* n_par,
                              double* out_ll) {
  if (!c || !child || !parents || !n_par || !out_ll) return fail(BN_ERR_BAD_ARG, "NULL argument");
  if (n_items <= 0) return BN_OK;
  for (int i = 0; i < n_items; i++) {
    if (child[i] < 0 || child[i] >= c->P) return fail(BN_ERR_BAD_ARG, "child[%d] out of range", i);
    if (n_par[i] < 0 || n_par[i] > c->max_par) return fail(BN_ERR_BAD_ARG, "n_par[%d] out of range", i);
    if (c->n_samples - n_par[i] - 1 <= 0) return fail(BN_ERR_BAD_ARG, "n_par[%d] leaves no degrees of freedom", i);
    for (int e = 0; e < n_par[i]; e++) {
      const int q = parents[(size_t)i * c->max_par + e];
      if (q < 0 || q >= c->P) return fail(BN_ERR_BAD_ARG, "parents[%d][%d] out of range", i, e);
    }
  }
  CU_TRY(cudaSetDevice(c->device));
  int *d_child = nullptr, *d_par = nullptr, *d_np = nullptr, *d_npd = nullptr;
  double* d_out = nullptr;
  int rc = BN_OK;
  cudaError_t e = pool_alloc((void**)&d_child, (size_t)n_items * 4);
  if (e == cudaSuccess) e = pool_alloc((void**)&d_par, (size_t)n_items * c->max_par * 4);
  if (e == cudaSuccess) e = pool_alloc((void**)&d_np, (size_t)n_items * 4);
  if (e == cudaSuccess) e = pool_alloc((void**)&d_npd, 4);
  if (e == cudaSuccess) e = pool_alloc((void**)&d_out, (size_t)n_items * 8);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_child, child, (size_t)n_items * 4, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_par, parents, (size_t)n_items * c->max_par * 4, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_np, n_par, (size_t)n_items * 4, cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_npd, 0, 4, c->stream);
  if (e == cudaSuccess) {
    const char* msg = launch_score_nodes(c->d_C, c->P, c->n_samples, c->max_par, n_items, d_child, d_par, d_np,
                                         d_out, d_npd, c->stream);
    c->launches++;
    if (msg) rc = fail(BN_ERR_UNSUPPORTED, "%s", msg);
  }
  if (e == cudaSuccess && !rc) e = cudaMemcpyAsync(out_ll, d_out, (size_t)n_items * 8, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess && !rc) e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess) rc = fail(e == cudaErrorMemoryAllocation ? BN_ERR_OOM : BN_ERR_CUDA, "bn_score_nodes: %s", cudaGetErrorString(e));
  pool_free(d_child); pool_free(d_par); pool_free(d_np); pool_free(d_npd); pool_free(d_out);
  return rc;
}

static int sweep_device(bn_ctx* c, int n_graphs, const int* d_parents, const int* d_npar, double* d_base,
                        double* d_score, double* d_hr, float* kernel_ms) {
  int *d_te = nullptr, *d_ag = nullptr;
  CU_TRY(pool_alloc((void**)&d_te, (size_t)n_graphs * 4));
  cudaError_t e = pool_alloc((void**)&d_ag, (size_t)n_graphs * 4);
  if (e != cudaSuccess) { pool_free(d_te); return fail(BN_ERR_OOM, "sweep scratch"); }
  int* d_order = nullptr;
  {
    const char* so = getenv("BN_B200_SWEEP_ORDER");  // (A/B switch: 0 = natural order)
    if (!(so && so[0] == '0') && (int64_t)n_graphs * c->P < (1ll << 31)) {
      e = pool_alloc((void**)&d_order, (size_t)n_graphs * c->P * 4);
      if (e != cudaSuccess) { pool_free(d_te); pool_free(d_ag); return fail(BN_ERR_OOM, "sweep scratch"); }
    }
  }
  SweepParams sp;
  sp.P = c->P; sp.max_par = c->max_par; sp.n_graphs = n_graphs; sp.n_samples = c->n_samples;
  sp.n_sim_edges = c->n_sim_edges; sp.C = c->d_C; sp.ldc = c->P; sp.diag = c->d_diag;
  sp.node_type = c->d_node_type; sp.sim_edge = c->d_sim_edge; sp.phi = c->phi; sp.omega = c->omega;
  sp.parents = d_parents; sp.n_par = d_npar; sp.te = d_te; sp.agree = d_ag; sp.order = d_order;
  sp.out_base = d_base; sp.out_score = d_score; sp.out_log_hr = d_hr;
  cudaEvent_t ev0, ev1;
  cudaEventCreate(&ev0); cudaEventCreate(&ev1);
  cudaEventRecord(ev0, c->stream);
  const char* msg = launch_sweep(sp, c->stream);
  c->launches += d_order ? 3 : 2;
  cudaEventRecord(ev1, c->stream);
  int rc = BN_OK;
  if (msg) rc = fail(BN_ERR_UNSUPPORTED, "%s", msg);
  e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess && !rc) rc = fail(BN_ERR_CUDA, "sweep kernel: %s", cudaGetErrorString(e));
  if (!rc && kernel_ms) cudaEventElapsedTime(kernel_ms, ev0, ev1);
  cudaEventDestroy(ev0); cudaEventDestroy(ev1);
  pool_free(d_te); pool_free(d_ag);
  if (d_order) pool_free(d_order);
  return rc;
}

extern "C" int bn_score_all_proposals_device(bn_ctx* c, int n_graphs, const int* d_parents, const int* d_npar,
                                             double* d_base, double* d_score, double* d_hr, float* kernel_ms) {
  if (!c || !d_parents || !d_npar) return fail(BN_ERR_BAD_ARG, "NULL argument");
  if (n_graphs <= 0) return fail(BN_ERR_BAD_ARG, "n_graphs <= 0");
  CU_TRY(cudaSetDevice(c->device));
  return sweep_device(c, n_graphs, d_parents, d_npar, d_base, d_score, d_hr, kernel_ms);
}

extern "C" int bn_score_all_proposals(bn_ctx* c, int n_graphs, const int* parents, const int* n_par,
                                      double* out_base, double* out_score, double* out_log_hr) {
  if (!c || !parents || !n_par) return fail(BN_ERR_BAD_ARG, "NULL argument");
  if (n_graphs <= 0) return fail(BN_ERR_BAD_ARG, "n_graphs <= 0");
  const int P = c->P, MP = c->max_par;
  for (int64_t i = 0; i < (int64_t)n_graphs * P; i++) {
    if (n_par[i] < 0 || n_par[i] > MP) return fail(BN_ERR_BAD_ARG, "n_par[%lld] out of range", (long long)i);
    for (int e = 0; e < n_par[i]; e++) {
      const int q = parents[i * MP + e];
      if (q < 0 || q >= P) return fail(BN_ERR_BAD_ARG, "parents[%lld][%d] out of range", (long long)i, e);
    }
  }
  CU_TRY(cudaSetDevice(c->device));
  const size_t npp = (size_t)n_graphs * P * P;
  int *d_par = nullptr, *d_np = nullptr;
  double *d_base = nullptr, *d_score = nullptr, *d_hr = nullptr;
  cudaError_t e = pool_alloc((void**)&d_par, (size_t)n_graphs * P * MP * 4);
  if (e == cudaSuccess) e = pool_alloc((void**)&d_np, (size_t)n_graphs * P * 4);
  if (e == cudaSuccess) e = pool_alloc((void**)&d_base, (size_t)n_graphs * P * 8);
  if (e == cudaSuccess && out_score) e = pool_alloc((void**)&d_score, npp * 8);
  if (e == cudaSuccess && out_log_hr) e = pool_alloc((void**)&d_hr, npp * 8);
  if (e == cudaSuccess) e = cudaMemcpy(d_par, parents, (size_t)n_graphs * P * MP * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d_np, n_par, (size_t)n_graphs * P * 4, cudaMemcpyHostToDevice);
  int rc = BN_OK;
  if (e != cudaSuccess) rc = fail(e == cudaErrorMemoryAllocation ? BN_ERR_OOM : BN_ERR_CUDA, "bn_score_all_proposals: %s", cudaGetErrorString(e));
  if (!rc) rc = sweep_device(c, n_graphs, d_par, d_np, d_base, d_score, d_hr, nullptr);
  if (!rc) {
    if (out_base) e = cudaMemcpy(out_base, d_base, (size_t)n_graphs * P * 8, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && out_score) e = cudaMemcpy(out_score, d_score, npp * 8, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && out_log_hr) e = cudaMemcpy(out_log_hr, d_hr, npp * 8, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = fail(BN_ERR_CUDA, "bn_score_all_proposals D2H: %s", cudaGetErrorString(e));
  }
  pool_free(d_par); pool_free(d_np); pool_free(d_base); pool_free(d_score); pool_free(d_hr);
  return rc;
}

// ---------------------------------------------------------------------------
// chains
// ---------------------------------------------------------------------------
static uint64_t splitmix64(uint64_t& x) {
  uint64_t z = (x += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// R's set.seed() scrambling for the Mersenne-Twister (R sources, src/main/RNG.c: RNG_Init)
static void rmt_seed_state(uint32_t seed, uint32_t* mt) {
  for (int j = 0; j < 50; j++) seed = 69069u * seed + 1u;
  for (int j = 0; j < 625; j++) {
    seed = 69069u * seed + 1u;
    if (j > 0) mt[j - 1] = seed;  // word 0 is the position (forced to 624)
  }
}

// Supplied start graphs (bn_run_args.start_parents): lists in range, -1 padded, without self-loops or
// duplicates, and acyclic (the ancestor bitsets of the chain assume a DAG).
static int check_start_graphs(int nc, int P, int MP, const int* par, const int* npar) {
  std::vector<int> indeg(P), order, kids_n(P), kids_off(P + 1), kids;
  for (int ch = 0; ch < nc; ch++) {
    const int* pc = par + (size_t)ch * P * MP;
    const int* nc_ = npar + (size_t)ch * P;
    std::fill(kids_n.begin(), kids_n.end(), 0);
    for (int c = 0; c < P; c++) {
      const int k = nc_[c];
      if (k < 0 || k > MP) return fail(BN_ERR_BAD_ARG, "start graph of chain %d: node %d has %d parents (max_par = %d)", ch, c, k, MP);
      for (int e = 0; e < MP; e++) {
        const int q = pc[(size_t)c * MP + e];
        if (e >= k) {
          if (q != -1) return fail(BN_ERR_BAD_ARG, "start graph of chain %d: node %d, slot %d beyond its %d parents is not -1", ch, c, e, k);
          continue;
        }
        if (q < 0 || q >= P) return fail(BN_ERR_BAD_ARG, "start graph of chain %d: node %d has parent %d out of range", ch, c, q);
        if (q == c) return fail(BN_ERR_BAD_ARG, "start graph of chain %d: node %d is its own parent", ch, c);
        for (int f = 0; f < e; f++)
          if (pc[(size_t)c * MP + f] == q) return fail(BN_ERR_BAD_ARG, "start graph of chain %d: node %d lists parent %d twice", ch, c, q);
        kids_n[q]++;
      }
    }
    // Kahn: every node must come off the queue
    kids_off[0] = 0;
    for (int c = 0; c < P; c++) kids_off[c + 1] = kids_off[c] + kids_n[c];
    kids.assign(kids_off[P], 0);
    std::fill(kids_n.begin(), kids_n.end(), 0);
    order.clear();
    for (int c = 0; c < P; c++) {
      indeg[c] = nc_[c];
      if (!indeg[c]) order.push_back(c);
      for (int e = 0; e < nc_[c]; e++) { const int q = pc[(size_t)c * MP + e]; kids[kids_off[q] + kids_n[q]++] = c; }
    }
    for (size_t i = 0; i < order.size(); i++)
      for (int t = kids_off[order[i]]; t < kids_off[order[i] + 1]; t++)
        if (--indeg[kids[t]] == 0) order.push_back(kids[t]);
    if ((int)order.size() < P)
      for (int c = 0; c < P; c++)
        if (indeg[c] > 0) return fail(BN_ERR_BAD_ARG, "start graph of chain %d is cyclic: node %d lies on or behind a cycle", ch, c);
  }
  return BN_OK;
}

static int64_t score_state_len(int P, int MP) {
  return (int64_t)P + (MP > 8 ? (int64_t)P * fac_stride(fac_mp(MP)) : 0);
}

extern "C" int bn_score_state_len(bn_ctx* c, int64_t* n) {
  if (!c || !n) return fail(BN_ERR_BAD_ARG, "NULL argument");
  *n = score_state_len(c->P, c->max_par);
  return BN_OK;
}

struct DevBuf {  // frees on scope exit
  std::vector<void*> ptrs;
  ~DevBuf() { for (void* p : ptrs) pool_free(p); }
  template <typename T>
  cudaError_t alloc(T** p, size_t n) {
    cudaError_t e = pool_alloc((void**)p, n * sizeof(T));
    if (e == cudaSuccess) ptrs.push_back((void*)*p);
    return e;
  }
};

extern "C" int bn_run(bn_ctx* c, const bn_run_args* a, bn_trace* trace, int* final_parents, int* final_n_par,
                      bn_chain_stats* stats, float* kernel_ms) {
  if (!c || !a || !trace) return fail(BN_ERR_BAD_ARG, "NULL argument");
  const int nc = a->n_chains;
  if (nc <= 0) return fail(BN_ERR_BAD_ARG, "n_chains <= 0");
  if (a->n_iter < 0 || a->output_every <= 0 || a->drop < 0) return fail(BN_ERR_BAD_ARG, "bad n_iter/output/drop");
  // InitialNetwork: 1 = random start, 2 = empty graph, anything else keeps the supplied graph
  // (src/network.h:148-170)
  const int init_net = (a->initial_network == 1 || a->initial_network == 2) ? a->initial_network : 0;
  if (init_net == 0 && c->prior_stride > c->max_par)
    return fail(BN_ERR_BAD_ARG, "InitialNetwork=%d starts from the supplied graph, in which a node has %d parents (max_par=%d)",
                a->initial_network, c->prior_stride, c->max_par);
  if (a->mt_state_in && a->rng_kind != BN_RNG_RMT) return fail(BN_ERR_BAD_ARG, "mt_state_in needs rng_kind = BN_RNG_RMT");
  if (a->mt_state_out && a->rng_kind != BN_RNG_RMT) return fail(BN_ERR_BAD_ARG, "mt_state_out needs rng_kind = BN_RNG_RMT");
  if (a->rng_kind < BN_RNG_WH || a->rng_kind > BN_RNG_REPLAY) return fail(BN_ERR_BAD_ARG, "bad rng_kind");
  if (a->rng_kind == BN_RNG_REPLAY && (!a->replay || a->replay_len <= 0)) return fail(BN_ERR_BAD_ARG, "replay buffer missing");
  const int need = (a->n_iter + a->output_every - 1) / a->output_every;
  if (trace->capacity < need) return fail(BN_ERR_CAPACITY, "trace capacity %d < %d rows", trace->capacity, need);
  if (!trace->n_rows || !trace->iter || !trace->changed_node || !trace->movetype || !trace->global_ll ||
      !trace->additions || !trace->deletions || !trace->fn || !trace->fp)
    return fail(BN_ERR_BAD_ARG, "trace column pointer is NULL");
  // supplied start graphs and resumed chains
  const bool given = a->start_parents != nullptr, resume = a->state_in != nullptr;
  // (the ancestor and Markov blanket tabulations and the best-graph tracking are compiled into the same
  // kernels only: the default ones stay as they are)
  const bool with_state = given || a->state_out || a->score_state_out || a->anc_freq || a->best || a->mb_freq;
  if (a->best_parents || a->best_n_par || a->best) {
    const char* missing = !a->best_parents ? "best_parents" : !a->best_n_par ? "best_n_par" : !a->best ? "best" : nullptr;
    if (missing) return fail(BN_ERR_BAD_ARG, "the best graph needs best_parents, best_n_par and best: %s is NULL", missing);
  }
  if ((resume || a->score_state_in) && !given) return fail(BN_ERR_BAD_ARG, "state_in / score_state_in need start_parents");
  if (given && !a->start_n_par) return fail(BN_ERR_BAD_ARG, "start_parents needs start_n_par");
  if (resume && a->rng_kind == BN_RNG_RMT && !a->mt_state_in)
    return fail(BN_ERR_BAD_ARG, "resuming an R Mersenne-Twister stream needs mt_state_in");
  if (given) {
    const int rc = check_start_graphs(nc, c->P, c->max_par, a->start_parents, a->start_n_par);
    if (rc) return rc;
  }
  if (resume)
    for (int ch = 0; ch < nc; ch++) {
      const bn_chain_state& st = a->state_in[ch];
      if (st.iter < 0 || st.iter + a->n_iter > 0x7fffffffll)
        return fail(BN_ERR_BAD_ARG, "state_in of chain %d: iteration %lld + n_iter %d is outside 0..INT_MAX", ch,
                    (long long)st.iter, a->n_iter);
      if (st.valid != 0 && st.valid != 1) return fail(BN_ERR_BAD_ARG, "state_in of chain %d: valid = %d (0 or 1)", ch, st.valid);
    }
  CU_TRY(cudaSetDevice(c->device));

  const int64_t P = c->P, MP = c->max_par, W = (P + 31) / 32;
  const int64_t slen = score_state_len((int)P, (int)MP);
  const int64_t cap = trace->capacity > 0 ? trace->capacity : 1;
  StageTimer tm("bn_run");
  DevBuf buf;
  ChainWorkspace w;
  memset(&w, 0, sizeof(w));
  w.scratch_n = scratch_words((int)P, HELPER_WARPS + 1, 32);
  {
    // Two CTAs per chain (chain_pipe_kernel) when every chain can have its SM pair at once: MaxPar <= 8,
    // the whole state fits in shared memory, 2 * n_chains <= SMs.  Opt-in for now: BN_B200_PIPE=1
    // (A/B runs, tests that compare the two forms).
    const char* e = getenv("BN_B200_PIPE");
    int n_sm = 0;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, c->device);
    ChainParams q;
    memset(&q, 0, sizeof(q));
    q.P = (int)P; q.max_par = (int)MP; q.W = (int)W;
    // (its team operations are dealt over the seven helper warps: larger row lists per part)
    const int sn = scratch_words((int)P, HELPER_WARPS, 32) > w.scratch_n ? scratch_words((int)P, HELPER_WARPS, 32) : w.scratch_n;
    w.pipeline = (e && e[0] != '0' && !with_state && MP <= 8 && 2 * nc <= n_sm && chains_can_pipeline(q, sn)) ? 1 : 0;
    if (w.pipeline) w.scratch_n = sn;
    if (w.pipeline && e && (e[0] == '3' || e[0] == '5')) w.pipeline = e[0] - '0';  // (developer switch: the chain's CTA rebuilds every window itself)
  }
  const size_t dscore_n = (size_t)(nc * P * MP) * (w.pipeline ? 2 : 1);
  CU_TRY(buf.alloc(&w.par, (size_t)(nc * P * MP)));
  CU_TRY(buf.alloc(&w.born, (size_t)(nc * P * MP)));
  CU_TRY(buf.alloc(&w.npar, (size_t)(nc * P)));
  CU_TRY(buf.alloc(&w.base, (size_t)(nc * P)));
  CU_TRY(buf.alloc(&w.anc, (size_t)(nc * P * anc_stride((int)W))));
  CU_TRY(buf.alloc(&w.haspar, (size_t)(nc * W)));
  CU_TRY(buf.alloc(&w.hp_list, (size_t)(nc * P)));
  CU_TRY(buf.alloc(&w.scratch, (size_t)nc * w.scratch_n));
  CU_TRY(buf.alloc(&w.dscore, dscore_n));
  if (MP > 8) {  // per-node Cholesky factors + the candidate rows of a round (score_core.cuh)
    CU_TRY(buf.alloc(&w.fac, (size_t)(nc * P * fac_stride(fac_mp((int)MP)))));
    CU_TRY(buf.alloc(&w.rowbuf, (size_t)nc * REPLAY_POS * row_stride(fac_mp((int)MP))));
  }
  CU_TRY(cudaMemsetAsync(w.dscore, 0xff, dscore_n * sizeof(double), c->stream));  // NaN = unknown (tags: -1)
  const bool dev_out = a->device_outputs != 0;
  if (given) {
    int *d_sp = nullptr, *d_sn = nullptr;
    CU_TRY(buf.alloc(&d_sp, (size_t)(nc * P * MP)));
    CU_TRY(buf.alloc(&d_sn, (size_t)(nc * P)));
    CU_TRY(cudaMemcpyAsync(d_sp, a->start_parents, (size_t)(nc * P * MP) * 4, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(cudaMemcpyAsync(d_sn, a->start_n_par, (size_t)(nc * P) * 4, cudaMemcpyHostToDevice, c->stream));
    w.start_par = d_sp; w.start_npar = d_sn;
  }
  std::vector<ChainStart> starts;
  if (resume) {
    starts.resize(nc);
    for (int ch = 0; ch < nc; ch++) {
      const bn_chain_state& st = a->state_in[ch];
      starts[ch].iter = st.iter; starts[ch].valid = st.valid; starts[ch].te_m = st.total_edges_member;
      starts[ch].acc_add = st.additions; starts[ch].acc_del = st.deletions;
    }
    ChainStart* d_st = nullptr;
    CU_TRY(buf.alloc(&d_st, (size_t)nc));
    CU_TRY(cudaMemcpyAsync(d_st, starts.data(), sizeof(ChainStart) * nc, cudaMemcpyHostToDevice, c->stream));
    w.start = d_st;
  }
  // score block [base P | factors P x fac_stride] per chain <-> w.base, w.fac
  const cudaMemcpyKind sc_in = dev_out ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  if (a->score_state_in) {
    CU_TRY(cudaMemcpy2DAsync(w.base, P * 8, a->score_state_in, slen * 8, P * 8, nc, sc_in, c->stream));
    if (MP > 8)
      CU_TRY(cudaMemcpy2DAsync(w.fac, (slen - P) * 8, a->score_state_in + P, slen * 8, (slen - P) * 8, nc, sc_in, c->stream));
    w.scores_in = 1;
  }
  w.scores_out = a->score_state_out ? 1 : 0;
  w.with_state = with_state || a->state_in || a->score_state_in;
  if (dev_out) {
    w.t_iter = trace->iter; w.t_changed = trace->changed_node; w.t_movetype = trace->movetype;
    w.t_gll = trace->global_ll; w.t_add = trace->additions; w.t_del = trace->deletions;
    w.t_fn = trace->fn; w.t_fp = trace->fp;
  } else {
    CU_TRY(buf.alloc(&w.t_iter, (size_t)(nc * cap))); CU_TRY(buf.alloc(&w.t_changed, (size_t)(nc * cap)));
    CU_TRY(buf.alloc(&w.t_movetype, (size_t)(nc * cap))); CU_TRY(buf.alloc(&w.t_gll, (size_t)(nc * cap)));
    CU_TRY(buf.alloc(&w.t_add, (size_t)(nc * cap))); CU_TRY(buf.alloc(&w.t_del, (size_t)(nc * cap)));
    CU_TRY(buf.alloc(&w.t_fn, (size_t)(nc * cap))); CU_TRY(buf.alloc(&w.t_fp, (size_t)(nc * cap)));
  }
  const int mcap = (a->moves && a->moves_capacity > 0) ? a->moves_capacity : 0;
  if (mcap) {
    if (dev_out) w.moves = a->moves;
    else CU_TRY(buf.alloc(&w.moves, (size_t)nc * mcap * 4));
  }
  if (a->edge_freq) {
    if (dev_out) w.edge_freq = a->edge_freq;
    else CU_TRY(buf.alloc(&w.edge_freq, (size_t)(nc * P * P)));
    CU_TRY(cudaMemsetAsync(w.edge_freq, 0, (size_t)(nc * P * P) * 4, c->stream));
  }
  if (a->anc_freq) {
    if (dev_out) w.anc_freq = a->anc_freq;
    else CU_TRY(buf.alloc(&w.anc_freq, (size_t)(nc * P * P)));
    CU_TRY(cudaMemsetAsync(w.anc_freq, 0, (size_t)(nc * P * P) * 4, c->stream));
  }
  int *best_par = nullptr, *best_npar = nullptr;
  std::vector<BestTrack> best_setup;
  if (a->best) {  // per chain: the lists (the output itself with device_outputs), the dirty set, the prior's constants
    if (dev_out) { best_par = a->best_parents; best_npar = a->best_n_par; }
    else { CU_TRY(buf.alloc(&best_par, (size_t)(nc * P * MP))); CU_TRY(buf.alloc(&best_npar, (size_t)(nc * P))); }
    uint32_t* dirty = nullptr;
    int* list = nullptr;
    CU_TRY(buf.alloc(&dirty, (size_t)(nc * W)));
    CU_TRY(buf.alloc(&list, (size_t)(nc * P)));
    best_setup.resize(nc);
    memset(best_setup.data(), 0, sizeof(BestTrack) * nc);
    for (int ch = 0; ch < nc; ch++) {
      BestTrack& b = best_setup[ch];
      b.n_sim = c->n_sim_edges; b.phi = c->phi; b.omega = c->omega;
      b.par = best_par + ch * P * MP; b.npar = best_npar + ch * P; b.dirty = dirty + ch * W; b.list = list + ch * P;
    }
    CU_TRY(buf.alloc(&w.best, (size_t)nc));  // (chain_init fills the rest)
    CU_TRY(cudaMemcpyAsync(w.best, best_setup.data(), sizeof(BestTrack) * nc, cudaMemcpyHostToDevice, c->stream));
  }
  int* mb_freq = nullptr;
  std::vector<MbTrack> mb_setup;
  if (a->mb_freq) {  // per chain: the counts (the output itself with device_outputs) and the witness matrix, both zeroed
    uint16_t* wit = nullptr;
    if (dev_out) mb_freq = a->mb_freq;
    else CU_TRY(buf.alloc(&mb_freq, (size_t)(nc * P * P)));
    CU_TRY(buf.alloc(&wit, (size_t)(nc * P * P)));
    CU_TRY(cudaMemsetAsync(mb_freq, 0, (size_t)(nc * P * P) * 4, c->stream));
    CU_TRY(cudaMemsetAsync(wit, 0, (size_t)(nc * P * P) * 2, c->stream));
    mb_setup.resize(nc);
    for (int ch = 0; ch < nc; ch++) { mb_setup[ch].freq = mb_freq + ch * P * P; mb_setup[ch].wit = wit + ch * P * P; }
    CU_TRY(buf.alloc(&w.mb, (size_t)nc));
    CU_TRY(cudaMemcpyAsync(w.mb, mb_setup.data(), sizeof(MbTrack) * nc, cudaMemcpyHostToDevice, c->stream));
  }
  if (a->npar_freq) {
    if (dev_out) w.npar_freq = a->npar_freq;
    else CU_TRY(buf.alloc(&w.npar_freq, (size_t)(nc * P * (MP + 1))));
    CU_TRY(buf.alloc(&w.npar_since, (size_t)(nc * P)));
    CU_TRY(cudaMemsetAsync(w.npar_freq, 0, (size_t)(nc * P * (MP + 1)) * 4, c->stream));
  }

  // uniform streams
  ChainRngArgs ra;
  memset(&ra, 0, sizeof(ra));
  ra.kind = a->rng_kind;
  std::vector<int> seeds((size_t)3 * nc);
  if (a->seeds) {
    memcpy(seeds.data(), a->seeds, seeds.size() * sizeof(int));
  } else {
    for (int ch = 0; ch < nc; ch++) {
      if (ch == 0) { seeds[0] = 10437; seeds[1] = 13568; seeds[2] = 30524; }  // random4f.h:19-21
      else {
        uint64_t st = 1234ull + (uint64_t)ch;
        seeds[3 * ch + 0] = 1 + (int)(splitmix64(st) % 30268ull);
        seeds[3 * ch + 1] = 1 + (int)(splitmix64(st) % 30306ull);
        seeds[3 * ch + 2] = 1 + (int)(splitmix64(st) % 30322ull);
      }
    }
  }
  if (resume && a->rng_kind == BN_RNG_WH)  // the stream continues from the state the stopped run returned
    for (int ch = 0; ch < nc; ch++) memcpy(&seeds[3 * ch], a->state_in[ch].wh_state, 3 * sizeof(int));
  if (a->rng_kind == BN_RNG_WH) {
    for (int ch = 0; ch < nc; ch++) {
      const int* s = &seeds[3 * ch];
      // the reference's own iz seed (30524, random4f.h:21) exceeds its modulus 30323; the LCG
      // step reduces it, so anything in 1..65535 is a valid starting state
      if (s[0] < 1 || s[0] > 65535 || s[1] < 1 || s[1] > 65535 || s[2] < 1 || s[2] > 65535)
        return fail(BN_ERR_BAD_ARG, "Wichmann-Hill seeds of chain %d out of range 1..65535", ch);
    }
  }
  int* d_seeds = nullptr;
  CU_TRY(buf.alloc(&d_seeds, seeds.size()));
  CU_TRY(cudaMemcpyAsync(d_seeds, seeds.data(), seeds.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  ra.seeds = d_seeds;
  std::vector<uint32_t> mt;
  std::vector<int> mt_pos;
  if (a->rng_kind == BN_RNG_RMT) {
    mt.resize((size_t)624 * nc);
    mt_pos.assign(nc, 624);  // set.seed() leaves the position at 624 = regenerate
    for (int ch = 0; ch < nc; ch++) {
      if (a->mt_state_in) {
        // .Random.seed[2:626] of R: position (dummy[0]) + 624 state words
        const int* st = a->mt_state_in + (size_t)625 * ch;
        mt_pos[ch] = (st[0] < 0 || st[0] > 624) ? 624 : st[0];
        for (int i = 0; i < 624; i++) mt[(size_t)624 * ch + i] = (uint32_t)st[1 + i];
      } else {
        rmt_seed_state((uint32_t)seeds[3 * ch], &mt[(size_t)624 * ch]);
      }
    }
    int* d_pos = nullptr;
    CU_TRY(buf.alloc(&ra.mt_states, mt.size() * (w.pipeline ? 2 : 1)));
    CU_TRY(buf.alloc(&d_pos, (size_t)nc));
    CU_TRY(cudaMemcpyAsync(ra.mt_states, mt.data(), mt.size() * 4, cudaMemcpyHostToDevice, c->stream));
    if (w.pipeline)  // the record builder's own copy of the stream state
      CU_TRY(cudaMemcpyAsync(ra.mt_states + mt.size(), mt.data(), mt.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(cudaMemcpyAsync(d_pos, mt_pos.data(), (size_t)nc * 4, cudaMemcpyHostToDevice, c->stream));
    ra.mt_pos = d_pos;
  }
  if (a->rng_kind == BN_RNG_REPLAY) {
    double* d_rep = nullptr;
    CU_TRY(buf.alloc(&d_rep, (size_t)nc * a->replay_len));
    CU_TRY(cudaMemcpyAsync(d_rep, a->replay, (size_t)nc * a->replay_len * 8, cudaMemcpyHostToDevice, c->stream));
    ra.replay = d_rep;
    ra.replay_len = a->replay_len;
  }

  ChainParams p;
  p.P = (int)P; p.max_par = (int)MP; p.W = (int)W; p.Ws = anc_stride((int)W); p.n_samples = c->n_samples;
  p.C = c->d_C; p.ldc = P; p.diag = c->d_diag; p.node_type = c->d_node_type; p.sim_edge = c->d_sim_edge;
  p.n_sim_edges = c->n_sim_edges; p.phi = c->phi; p.omega = c->omega;
  p.initial_network = init_net; p.drop = a->drop; p.n_iter = a->n_iter;
  p.output_every = a->output_every; p.trace_capacity = (int)cap; p.moves_capacity = mcap;
  p.prior_par = c->d_prior_par; p.prior_npar = c->d_prior_npar; p.prior_stride = c->prior_stride;

  ChainResult* d_res = nullptr;
  CU_TRY(buf.alloc(&d_res, (size_t)nc));
  tm.lap("workspace + seeds");
  cudaEvent_t ev0, ev1;
  cudaEventCreate(&ev0); cudaEventCreate(&ev1);
  cudaEventRecord(ev0, c->stream);
  const char* msg = launch_chains(p, w, ra, d_res, nc, c->stream);
  c->launches++;
  cudaEventRecord(ev1, c->stream);
  cudaError_t e = cudaStreamSynchronize(c->stream);
  if (e == cudaSuccess) e = cudaGetLastError();
  float ms = 0.f;
  if (e == cudaSuccess) cudaEventElapsedTime(&ms, ev0, ev1);
  cudaEventDestroy(ev0); cudaEventDestroy(ev1);
  if (msg) return fail(BN_ERR_UNSUPPORTED, "%s", msg);
  if (e != cudaSuccess) return fail(BN_ERR_CUDA, "chain kernel: %s", cudaGetErrorString(e));
  if (kernel_ms) *kernel_ms = ms;
  tm.lap("chain kernel + sync");

  std::vector<ChainResult> res(nc);
  CU_TRY(cudaMemcpy(res.data(), d_res, sizeof(ChainResult) * nc, cudaMemcpyDeviceToHost));
  int rc = BN_OK;
  if (w.pipeline && getenv("BN_B200_PIPE_STATS"))
    for (int ch = 0; ch < nc && ch < 4; ch++)
      fprintf(stderr, "[bn_b200] chain %d two-CTA: %d windows requested, %d waits for the builder, %d discarded, %d in-place rebuilds, %lld cycles\n",
              ch, res[ch].pipe[0], res[ch].pipe[1], res[ch].pipe[2], res[ch].pipe[3], (long long)res[ch].cyc_total),
      fprintf(stderr, "[bn_b200]   cycles: wait %lld, copy %lld, batch repair %lld, redo after it %lld, stale rebuilds %lld, publish %lld\n",
              res[ch].pipe_cyc[0], res[ch].pipe_cyc[1], res[ch].pipe_cyc[2], res[ch].pipe_cyc[3], res[ch].pipe_cyc[4], res[ch].pipe_cyc[5]);
  std::vector<int> nrows(nc), nmoves(nc);
  for (int ch = 0; ch < nc; ch++) {
    nrows[ch] = res[ch].n_rows;
    nmoves[ch] = res[ch].n_moves < mcap ? res[ch].n_moves : mcap;
    if (stats) {
      bn_chain_stats& s = stats[ch];
      s.uniforms = res[ch].uniforms; s.valid_iters = res[ch].valid_iters;
      for (int t = 0; t < 3; t++) { s.proposed[t] = res[ch].proposed[t]; s.reject[t] = res[ch].reject[t]; }
      s.n_nonpd = res[ch].n_nonpd; s.total_edges = res[ch].total_edges; s.status = res[ch].status;
      s.windows = res[ch].windows;
      s.alg_bytes = res[ch].alg_bytes;
      for (int t = 0; t < 12; t++) s.phase_cycles[t] = res[ch].cyc[t];
      s.slots_simulated = res[ch].slots_sim;
      s.kernel_cycles = res[ch].cyc_total;
    }
    if (res[ch].status == 95 && !rc)
      rc = fail(BN_ERR_CUDA, "chain %d: an accepted move did not fit the graph (two-CTA form: a record escaped its repair)", ch);
    if ((res[ch].status == 91 || res[ch].status == 92) && !rc)
      rc = fail(BN_ERR_CUDA, "chain %d: the two CTAs of the chain lost each other (mailbox watchdog %d)", ch, res[ch].status);
    if (res[ch].status == BN_ERR_NO_LEGAL_PROPOSAL && !rc)
      rc = fail(res[ch].status, "chain %d: no legal proposal exists (every candidate child is a source or full, or every candidate parent a sink / already a parent)", ch);
    if (a->rng_kind == BN_RNG_REPLAY && (res[ch].uniforms > a->replay_len || res[ch].status == BN_ERR_CAPACITY) && !rc)
      rc = fail(BN_ERR_CAPACITY, "chain %d consumed %lld uniforms, the replay buffer holds %lld", ch,
                (long long)res[ch].uniforms, (long long)a->replay_len);
    if (a->mt_state_out && a->rng_kind == BN_RNG_RMT) {
      // stream state after exactly the uniforms the chain consumed (.Random.seed[2:626] layout)
      int pos = mt_pos[ch];
      uint32_t* st = &mt[(size_t)624 * ch];
      rmt_advance(st, pos, res[ch].uniforms);
      int* out = a->mt_state_out + (size_t)625 * ch;
      out[0] = pos;
      for (int i = 0; i < 624; i++) out[1 + i] = (int)st[i];
    }
    if (a->state_out) {
      bn_chain_state& o = a->state_out[ch];
      memset(&o, 0, sizeof(o));
      o.iter = res[ch].end.iter; o.valid = res[ch].end.valid; o.total_edges_member = res[ch].end.te_m;
      o.additions = res[ch].end.acc_add; o.deletions = res[ch].end.acc_del;
      o.uniforms = (resume ? a->state_in[ch].uniforms : 0) + res[ch].uniforms;
      if (a->rng_kind == BN_RNG_WH) wh_advance(&seeds[3 * ch], res[ch].uniforms, o.wh_state);
    }
  }
  if (a->score_state_out) {
    const cudaMemcpyKind k = dev_out ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    CU_TRY(cudaMemcpy2D(a->score_state_out, slen * 8, w.base, P * 8, P * 8, nc, k));
    if (MP > 8) CU_TRY(cudaMemcpy2D(a->score_state_out + P, slen * 8, w.fac, (slen - P) * 8, (slen - P) * 8, nc, k));
  }
  const cudaMemcpyKind out_kind = dev_out ? cudaMemcpyHostToDevice : cudaMemcpyHostToHost;
  CU_TRY(cudaMemcpy(trace->n_rows, nrows.data(), (size_t)nc * 4, out_kind));
  if (a->n_moves) CU_TRY(cudaMemcpy(a->n_moves, nmoves.data(), (size_t)nc * 4, out_kind));
  if (!dev_out) {
    const size_t n = (size_t)(nc * cap);
    CU_TRY(cudaMemcpy(trace->iter, w.t_iter, n * 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(trace->changed_node, w.t_changed, n * 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(trace->movetype, w.t_movetype, n * 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(trace->global_ll, w.t_gll, n * 8, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(trace->additions, w.t_add, n * 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(trace->deletions, w.t_del, n * 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(trace->fn, w.t_fn, n * 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(trace->fp, w.t_fp, n * 4, cudaMemcpyDeviceToHost));
    if (mcap) CU_TRY(cudaMemcpy(a->moves, w.moves, (size_t)nc * mcap * 16, cudaMemcpyDeviceToHost));
    if (a->edge_freq) CU_TRY(cudaMemcpy(a->edge_freq, w.edge_freq, (size_t)(nc * P * P) * 4, cudaMemcpyDeviceToHost));
    if (a->anc_freq) CU_TRY(cudaMemcpy(a->anc_freq, w.anc_freq, (size_t)(nc * P * P) * 4, cudaMemcpyDeviceToHost));
    if (a->mb_freq) CU_TRY(cudaMemcpy(a->mb_freq, mb_freq, (size_t)(nc * P * P) * 4, cudaMemcpyDeviceToHost));
    if (a->npar_freq) CU_TRY(cudaMemcpy(a->npar_freq, w.npar_freq, (size_t)(nc * P * (MP + 1)) * 4, cudaMemcpyDeviceToHost));
    if (a->best) {
      CU_TRY(cudaMemcpy(a->best_parents, best_par, (size_t)(nc * P * MP) * 4, cudaMemcpyDeviceToHost));
      CU_TRY(cudaMemcpy(a->best_n_par, best_npar, (size_t)(nc * P) * 4, cudaMemcpyDeviceToHost));
    }
  }
  if (a->best)  // the leading bn_best_graph of each chain's BestTrack
    CU_TRY(cudaMemcpy2D(a->best, sizeof(bn_best_graph), w.best, sizeof(BestTrack), sizeof(bn_best_graph), nc,
                        dev_out ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost));
  const cudaMemcpyKind fin_kind = dev_out ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  if (final_parents) CU_TRY(cudaMemcpy(final_parents, w.par, (size_t)(nc * P * MP) * 4, fin_kind));
  if (final_n_par) CU_TRY(cudaMemcpy(final_n_par, w.npar, (size_t)(nc * P) * 4, fin_kind));
  tm.lap("results D2H");
  return rc;
}

// ---------------------------------------------------------------------------
// host twin of main_fun (src/bayesnet_mcmc.cpp:27-72)
// ---------------------------------------------------------------------------
extern "C" int bn_main_fun(const double* X, int n_samples, int n_nodes, const int* graph_source,
                           const int* graph_target, int n_edges, const int* graph_node_labels,
                           const int* graph_node_type, int MaxPar, double phi, double omega,
                           int InitialNetwork, int drop, int N, int output, int rng_kind, const int* seeds,
                           int capacity, int* iter, int* ChangedNode, int* movetype, double* globalLL,
                           int* additions, int* deletions, int* FN, int* FP, const int* mt_state_in,
                           int* mt_state_out) {
  (void)graph_node_labels;  // accepted and unused, as in the reference (src/bayesnet_mcmc.cpp:30,42-43)
  bn_ctx* c = nullptr;
  int rc = bn_create(X, n_samples, n_nodes, graph_source, graph_target, n_edges, graph_node_type, MaxPar, phi,
                     omega, 0, &c);
  if (rc) return -rc;
  bn_run_args a;
  memset(&a, 0, sizeof(a));
  a.n_chains = 1; a.rng_kind = rng_kind; a.seeds = seeds; a.initial_network = InitialNetwork;
  a.drop = drop; a.n_iter = N; a.output_every = output;
  a.mt_state_in = mt_state_in; a.mt_state_out = mt_state_out;
  int n_rows = 0;
  bn_trace t;
  t.capacity = capacity; t.n_rows = &n_rows; t.iter = iter; t.changed_node = ChangedNode; t.movetype = movetype;
  t.global_ll = globalLL; t.additions = additions; t.deletions = deletions; t.fn = FN; t.fp = FP;
  rc = bn_run(c, &a, &t, nullptr, nullptr, nullptr, nullptr);
  bn_destroy(c);
  return rc ? -rc : n_rows;
}
