// C-ABI of libapgp (see include/apgp.h): handle bookkeeping, staging copies, launch sequencing.
#include "../../include/apgp.h"
#include "apgp_internal.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

using namespace apgp;

static thread_local std::string g_err;
static int fail(int code, const char* what, cudaError_t ce = cudaSuccess) {
  g_err = what;
  if (ce != cudaSuccess) { g_err += ": "; g_err += cudaGetErrorString(ce); }
  return code;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(APGP_ERR_CUDA, #call, e_); } while (0)
#define CUI(call) do { int e_ = (call); if (e_ != 0) return fail(APGP_ERR_CUDA, #call, (cudaError_t)e_); } while (0)

static const double TINY2 = 1.25e-12 * 1.25e-12;   // george's default yerr^2, added with exp(white_noise)

struct DevBuf {
  void* p = nullptr; size_t cap = 0;
  int reserve_keep(size_t bytes, size_t keep, cudaStream_t st) {     // grow, preserving the first `keep` bytes
    if (bytes <= cap) return 0;
    void* q = nullptr;
    size_t want = bytes + bytes / 2;
    cudaError_t e = cudaMalloc(&q, want);
    if (e != cudaSuccess) return (int)e;
    if (p && keep) { e = cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st); if (e != cudaSuccess) { cudaFree(q); return (int)e; } cudaStreamSynchronize(st); }
    if (p) cudaFree(p);
    p = q; cap = want;
    return 0;
  }
  int reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return (int)e;
    cap = bytes; return 0;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct apgp_handle {
  int device = 0, num_sms = 0;
  cudaStream_t stream = nullptr; bool own_stream = false;
  cudaStream_t copy_in = nullptr, copy_out = nullptr;   // H2D / D2H streams of the pipelined host-buffer predict
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_k[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
  int N = 0, d = 0, Np = 0, Npad = 0;
  int group = -1;        // CTAs per query tile in the variance kernel: 0 = one tile per CTA, -1 = automatic, G = fixed
  bool predict_few = true;   // calls of at most PREDICT_FEW_MAX queries: one CTA per query (APGP_PREDICT_FEW=0: tiled kernels)
  bool var_i8 = true;        // variance engine of grouped calls: int8 tensor cores where they apply (predict_i8.cu), else DMMA
  bool i8_packed = false;    // LinvI8 / i8scale hold the current factorisation's digits
  bool has_training = false, has_hyper = false, factored = false;
  double mean = 0, amp = 1, white_noise = -12;
  double log_metric[APGP_MAX_DIM];
  double logdet = 0, loglik = 0;
  long long launches = 0;
  DevBuf X, y, K, Dinv, r, Linv, work, scal, info, hyper, Xs, alphaA, alpha, LinvF, scratch, qscale;
  DevBuf stage_in, stage_out;          // device staging for on_host calls
  DevBuf ap_k, ap_l, ap_u, ap_x;       // bordered-append work vectors
  double* pin = nullptr;               // pinned host staging for small calls (latency path)
  static constexpr size_t PIN_DOUBLES = 32768;   // 256 KB: [0, PIN/2) inputs, [PIN/2, PIN) outputs
  DevBuf bK, bDinv, br, bscal, binfo, bhyper, bll, bgrad;   // batched log-likelihood workspace
  DevBuf ac_part, ac_f, ac_stage;                            // autocorrelation partial sums, f(t), host-chain staging
  void* comm = nullptr; int comm_rank = 0, comm_world = 1;  // NCCL communicator (apgp_comm_init)
  DevBuf c_hdr, c_send, c_recv;                               // collective staging
  DevBuf gws;                                                // fused cluster-per-restart workspace (chol_group.cuh)
  DevBuf s_p0, s_chain, s_logp, s_blob, s_nacc, s_ri, s_rz, s_rr, s_rl;
  DevBuf o_in, o_x, o_f, o_stats;      // device optimiser staging
  DevBuf g_arrive, g_part, g_plan;     // grouped variance kernel: barrier counters, partial sums, work-split tables
  DevBuf few_ws;                       // few-query predict: per-split partial sums, means, arrival counters
  int plan_Npad = -1, plan_G = -1, plan_d = -1, plan_i8 = -1;   // what g_plan currently holds
  DevBuf LinvI8, i8scale;              // int8 engine operands (pack_linv_i8)
  int last_var_path = 0;               // VarPath of the last variance launch (apgp_debug_last_var_path)
  int last_loglik_path = 0;            // LoglikPath of the last apgp_loglik_batch call (apgp_debug_last_loglik_path)
};

namespace {

__global__ void scale_pad_kernel(const double* __restrict__ a, int N, int Npad, double s, double* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Npad; i += gridDim.x * blockDim.x) out[i] = (i < N) ? s * a[i] : 0.0;
}

struct Guard {  // select the handle's device for the duration of a call
  int prev = -1;
  explicit Guard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~Guard() { if (prev >= 0) cudaSetDevice(prev); }
};

// the tuning knobs' environment overrides, read by apgp_create and apgp_reset
void read_env_knobs(apgp_handle* h) {
  if (const char* gv = getenv("APGP_PREDICT_GROUP")) h->group = atoi(gv);
  if (const char* fv = getenv("APGP_PREDICT_FEW")) h->predict_few = atoi(fv) != 0;
  if (const char* ev = getenv("APGP_PREDICT_VAR_ENGINE")) h->var_i8 = strcmp(ev, "dmma") != 0;
}

void fill_hyper_row(double* row, double mean, double amp, double wn, const double* logM, int d) {
  row[0] = mean; row[1] = amp; row[2] = exp(wn) + TINY2;
  for (int i = 0; i < d; ++i) row[3 + i] = exp(-logM[i]);
}

// apgp_loglik_batch's kernels, as apgp_debug_last_loglik_path reports them
enum LoglikPath { LL_SMALL = 1, LL_GROUP = 2, LL_TILED = 3, LL_GROUP_GRAD = 4 };
// One restart per CTA while the small evaluator fits one CTA's shared memory (N <= ~224), else one CLUSTER per restart
// (fused single launch, chol_group.cuh) -- except a handful of large matrices, which the multi-launch tiled sequence
// spreads over the whole GPU where a cluster is at most 16 SMs (measured, R = 1: N = 1024 0.51 ms fused vs 0.71 ms tiled,
// N = 2048 1.85 vs 1.48 ms; R = 8, N = 2048: 2.87 vs 2.73).  With gradients (grad) everything above the small class takes
// the cluster kernel with gradients, loglik_grad_group_kernel, few large matrices included.  APGP_LOGLIK_PATH = small |
// group | tiled forces a value kernel (small only where it fits); forced group or tiled has no gradients (the caller gets
// APGP_NEEDS_HOST).  APGP_LOGLIK_PATH = group_grad forces the cluster kernel with gradients at any N (group for values).
int choose_loglik_path(const apgp_handle* h, int R, bool grad) {
  const bool fits = loglik_small_smem(h->N, h->d) <= 220 * 1024;
  if (const char* v = getenv("APGP_LOGLIK_PATH")) {
    if (!strcmp(v, "small") && fits) return LL_SMALL;
    if (!strcmp(v, "group")) return LL_GROUP;
    if (!strcmp(v, "tiled")) return LL_TILED;
    if (!strcmp(v, "group_grad")) return grad ? LL_GROUP_GRAD : LL_GROUP;
  }
  if (fits) return LL_SMALL;
  if (grad) return LL_GROUP_GRAD;
  return (h->Np >= 2048 && R <= 8) ? LL_TILED : LL_GROUP;
}

}  // namespace

extern "C" {

const char* apgp_last_error(void) { return g_err.c_str(); }
int apgp_version(void) { return 100; }

int apgp_create(apgp_handle** out, int device) {
  if (!out) return fail(APGP_ERR_ARG, "apgp_create: null out");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(APGP_ERR_CUDA, "apgp_create: no CUDA device (libapgp has no CPU fallback)", e);
  if (device < 0 || device >= ndev) return fail(APGP_ERR_ARG, "apgp_create: bad device index");
  apgp_handle* h = new apgp_handle();
  h->device = device;
  Guard g(device);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { delete h; return fail(APGP_ERR_CUDA, "apgp_create: cudaGetDeviceProperties", e); }
  if (prop.major < 10) { delete h; return fail(APGP_ERR_CUDA, "apgp_create: kernels are built for sm_100a only"); }
  h->num_sms = prop.multiProcessorCount;
  e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { delete h; return fail(APGP_ERR_CUDA, "apgp_create: cudaStreamCreate", e); }
  h->own_stream = true;
  e = cudaHostAlloc((void**)&h->pin, apgp_handle::PIN_DOUBLES * 8, cudaHostAllocDefault);
  if (e != cudaSuccess) { cudaStreamDestroy(h->stream); delete h; return fail(APGP_ERR_CUDA, "apgp_create: cudaHostAlloc", e); }
  read_env_knobs(h);
  *out = h;
  return APGP_OK;
}

int apgp_destroy(apgp_handle* h) {
  if (!h) return APGP_OK;
  Guard g(h->device);
  cudaStreamSynchronize(h->stream);
  DevBuf* bufs[] = {&h->X, &h->y, &h->K, &h->Dinv, &h->r, &h->Linv, &h->work, &h->scal, &h->info, &h->hyper, &h->Xs,
                    &h->alphaA, &h->alpha, &h->LinvF, &h->scratch, &h->qscale, &h->stage_in, &h->stage_out, &h->ap_k, &h->ap_l, &h->ap_u, &h->ap_x, &h->bK,
                    &h->bDinv, &h->br, &h->bscal, &h->binfo, &h->bhyper, &h->bll, &h->bgrad, &h->s_p0, &h->s_chain, &h->s_logp,
                    &h->s_blob, &h->s_nacc, &h->s_ri, &h->s_rz, &h->s_rr, &h->s_rl, &h->o_in, &h->o_x, &h->o_f, &h->o_stats, &h->g_arrive, &h->g_part, &h->g_plan, &h->few_ws, &h->LinvI8, &h->i8scale, &h->gws, &h->ac_part, &h->ac_f, &h->ac_stage, &h->c_hdr, &h->c_send, &h->c_recv};
  for (DevBuf* b : bufs) b->release();
  if (h->comm) comm_destroy(h->comm);
  if (h->pin) cudaFreeHost(h->pin);
  for (int b = 0; b < 2; ++b) {
    if (h->ev_in[b]) cudaEventDestroy(h->ev_in[b]);
    if (h->ev_k[b]) cudaEventDestroy(h->ev_k[b]);
    if (h->ev_out[b]) cudaEventDestroy(h->ev_out[b]);
  }
  if (h->copy_in) cudaStreamDestroy(h->copy_in);
  if (h->copy_out) cudaStreamDestroy(h->copy_out);
  if (h->own_stream) cudaStreamDestroy(h->stream);
  delete h;
  return APGP_OK;
}

int apgp_reset(apgp_handle* h) {
  if (!h) return fail(APGP_ERR_ARG, "null handle");
  Guard g(h->device);
  cudaStreamSynchronize(h->stream);
  if (!h->own_stream) { CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
  h->N = h->d = h->Np = h->Npad = 0;
  h->has_training = h->has_hyper = h->factored = false;
  h->mean = 0; h->amp = 1; h->white_noise = -12; h->logdet = 0; h->loglik = 0;
  h->plan_Npad = h->plan_G = h->plan_d = h->plan_i8 = -1;
  h->i8_packed = false;
  h->last_var_path = 0;
  h->last_loglik_path = 0;
  h->group = -1; h->predict_few = true; h->var_i8 = true;   // tuning knobs back to their defaults (as apgp_create)
  read_env_knobs(h);
  if (h->comm) { comm_destroy(h->comm); h->comm = nullptr; h->comm_rank = 0; h->comm_world = 1; }
  return APGP_OK;
}

int apgp_set_stream(apgp_handle* h, void* s) {
  if (!h) return fail(APGP_ERR_ARG, "null handle");
  Guard g(h->device);
  if (s == nullptr) {
    if (!h->own_stream) { CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    return APGP_OK;
  }
  if (h->own_stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); h->own_stream = false; }
  h->stream = (cudaStream_t)s;
  return APGP_OK;
}

int apgp_synchronize(apgp_handle* h) {
  if (!h) return fail(APGP_ERR_ARG, "null handle");
  Guard g(h->device);
  CU(cudaStreamSynchronize(h->stream));
  return APGP_OK;
}

long long apgp_launch_count(const apgp_handle* h) { return h ? h->launches : 0; }

int apgp_set_group(apgp_handle* h, int group) {
  if (!h || group < -1 || group > 64) return fail(APGP_ERR_ARG, "apgp_set_group");
  h->group = group;
  return APGP_OK;
}

int apgp_set_var_engine(apgp_handle* h, int engine) {
  if (!h || (engine != APGP_VAR_ENGINE_DMMA && engine != APGP_VAR_ENGINE_I8)) return fail(APGP_ERR_ARG, "apgp_set_var_engine");
  h->var_i8 = engine == APGP_VAR_ENGINE_I8;
  return APGP_OK;
}

int apgp_set_predict_few(apgp_handle* h, int enable) {
  if (!h) return fail(APGP_ERR_ARG, "apgp_set_predict_few");
  h->predict_few = enable != 0;
  return APGP_OK;
}

int apgp_set_training(apgp_handle* h, const double* X, const double* y, int N, int d, int on_host) {
  if (!h || !X || !y) return fail(APGP_ERR_ARG, "apgp_set_training: null argument");
  if (N < 1 || d < 1 || d > APGP_MAX_DIM) return fail(APGP_ERR_ARG, "apgp_set_training: need N>=1, 1<=d<=32");
  Guard g(h->device);
  CUI(h->X.reserve((size_t)N * d * 8));
  CUI(h->y.reserve((size_t)N * 8));
  cudaMemcpyKind kind = on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  CU(cudaMemcpyAsync(h->X.p, X, (size_t)N * d * 8, kind, h->stream));
  CU(cudaMemcpyAsync(h->y.p, y, (size_t)N * 8, kind, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->N = N; h->d = d;
  h->Np = (N + 63) / 64 * 64;
  h->has_training = true; h->factored = false;
  return APGP_OK;
}

int apgp_set_hyper(apgp_handle* h, double mean, double amp, const double* log_metric, double white_noise) {
  if (!h || !log_metric) return fail(APGP_ERR_ARG, "apgp_set_hyper: null argument");
  if (!h->has_training) return fail(APGP_ERR_ARG, "apgp_set_hyper: set the training set first (fixes d)");
  h->mean = mean; h->amp = amp; h->white_noise = white_noise;
  for (int i = 0; i < h->d; ++i) h->log_metric[i] = log_metric[i];
  h->has_hyper = true; h->factored = false;
  return APGP_OK;
}

// int8 variance engine: grouped calls from Npad = I8_MIN_NPAD, where it measured 1.5x (N = 1024) to 1.9x (N = 8192)
// faster than the DMMA kernel (profiles/r03_var_engine.jsonl); smaller N, mostly not grouped, stays on DMMA
constexpr int I8_MIN_NPAD = 1024;
static bool i8_applies(const apgp_handle* h) {
  return h->var_i8 && h->group != 0 && h->Npad >= I8_MIN_NPAD && predict_i8_fits(h->Npad, h->d);
}
static int pack_i8_operands(apgp_handle* h, cudaStream_t st, int* nl) {
  CUI(h->LinvI8.reserve(linv_i8_bytes(h->Npad)));
  CUI(h->i8scale.reserve((size_t)h->Npad * 8));
  CUI(launch_pack_linv_i8(h->Linv.as<double>(), h->Np, h->N, h->Npad, h->amp, h->LinvI8.as<unsigned char>(),
                          h->i8scale.as<double>(), st)); ++*nl;
  h->i8_packed = true;
  return APGP_OK;
}

static int pack_predict_operands(apgp_handle* h, int* nl) {
  const int N = h->N, d = h->d, Np = h->Np;
  const int BN = predict_tile_bn(d);
  scale_pad_kernel<<<(h->Npad + 255) / 256, 256, 0, h->stream>>>(h->alpha.as<double>(), N, h->Npad, h->amp,
                                                                 h->alphaA.as<double>()); ++*nl;
  double qs[APGP_MAX_DIM];
  for (int i = 0; i < d; ++i) qs[i] = sqrt(0.5 * exp(-h->log_metric[i]));
  CU(cudaMemcpyAsync(h->qscale.p, qs, d * 8, cudaMemcpyHostToDevice, h->stream));
  CUI(launch_pack_xs(h->X.as<double>(), N, d, h->Npad, h->qscale.as<double>(), h->Xs.as<double>(), h->stream)); ++*nl;
  CUI(launch_pack_linv(h->Linv.as<double>(), Np, N, h->Npad, BN, h->amp, h->LinvF.as<double>(), h->stream)); ++*nl;
  h->i8_packed = false;
  if (i8_applies(h)) { int st_ = pack_i8_operands(h, h->stream, nl); if (st_ != APGP_OK) return st_; }
  return APGP_OK;
}

int apgp_factorize(apgp_handle* h, double* logdet, double* loglik, int* info) {
  if (!h) return fail(APGP_ERR_ARG, "null handle");
  if (!h->has_training || !h->has_hyper) return fail(APGP_ERR_ARG, "apgp_factorize: training set and hyper-parameters required");
  Guard g(h->device);
  const int N = h->N, d = h->d, Np = h->Np;
  const int BN = predict_tile_bn(d);
  h->Npad = (N + BN - 1) / BN * BN;
  h->factored = false;
  if (info) *info = 0;
  bool finite = isfinite(h->mean) && isfinite(h->amp) && isfinite(h->white_noise);
  for (int i = 0; i < d; ++i) finite = finite && isfinite(h->log_metric[i]);
  if (!finite) { if (info) *info = 1; if (loglik) *loglik = -INFINITY; return APGP_NOT_POSDEF; }

  CUI(h->K.reserve((size_t)Np * Np * 8));
  CUI(h->Dinv.reserve((size_t)Np * 64 * 8));
  CUI(h->r.reserve((size_t)Np * 8));
  CUI(h->scal.reserve(4 * 8));
  CUI(h->info.reserve(4));
  CUI(h->hyper.reserve((3 + APGP_MAX_DIM) * 8));
  CUI(h->qscale.reserve(APGP_MAX_DIM * 8));

  double row[3 + APGP_MAX_DIM];
  fill_hyper_row(row, h->mean, h->amp, h->white_noise, h->log_metric, d);
  CU(cudaMemcpyAsync(h->hyper.p, row, (3 + d) * 8, cudaMemcpyHostToDevice, h->stream));
  FactorBatch fb{1, N, Np, h->K.as<double>(), h->Dinv.as<double>(), h->r.as<double>(), h->scal.as<double>(),
                 h->info.as<int>()};
  int nl = 0;
  CUI(launch_build_K(h->X.as<double>(), h->y.as<double>(), N, d, h->hyper.as<double>(), fb, h->stream)); ++nl;
  CUI(launch_cholesky(fb, h->num_sms, h->stream, &nl));
  CUI(launch_loglik_finish(fb, h->scal.as<double>() + 1, h->stream)); ++nl;
  double sc[2]; int inf = 0;
  CU(cudaMemcpyAsync(sc, h->scal.p, 16, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(&inf, h->info.p, 4, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->launches += nl; nl = 0;
  if (inf != 0) {
    if (info) *info = inf;
    if (loglik) *loglik = -INFINITY;
    return APGP_NOT_POSDEF;
  }
  h->logdet = sc[0]; h->loglik = sc[1];
  if (logdet) *logdet = sc[0];
  if (loglik) *loglik = sc[1];

  // explicit inverse, alpha, packed operands for the predict kernels
  CUI(h->Linv.reserve((size_t)Np * Np * 8));
  CUI(h->work.reserve((size_t)Np * Np * 8));
  CUI(h->alpha.reserve((size_t)Np * 8));
  CUI(h->alphaA.reserve((size_t)h->Npad * 8));
  CUI(h->Xs.reserve((size_t)d * h->Npad * 8));
  const size_t lf = (size_t)linvf_total_tiles(h->Npad, BN) * BN * 16 * 8;
  CUI(h->LinvF.reserve(lf));
  CUI(launch_tri_inverse(h->K.as<double>(), h->Dinv.as<double>(), Np, h->Linv.as<double>(), h->work.as<double>(),
                         h->stream, &nl));
  CUI(launch_linvT_matvec(h->Linv.as<double>(), Np, h->r.as<double>(), h->alpha.as<double>(), h->stream)); ++nl;
  if (!getenv("APGP_NO_REFINE")) {
    CUI(h->ap_k.reserve((size_t)Np * 8)); CUI(h->ap_l.reserve((size_t)Np * 8));
    CUI(launch_refine_alpha(h->X.as<double>(), h->y.as<double>(), N, d, Np, h->hyper.as<double>(), h->Linv.as<double>(),
                            h->alpha.as<double>(), h->ap_k.as<double>(), h->ap_l.as<double>(), h->stream, &nl));
  }
  { int st_ = pack_predict_operands(h, &nl); if (st_ != APGP_OK) return st_; }
  CU(cudaStreamSynchronize(h->stream));
  h->launches += nl;
  h->factored = true;
  return APGP_OK;
}

int apgp_append_point(apgp_handle* h, const double* x_new, double y_new, double* logdet, double* loglik) {
  if (!h || !x_new) return fail(APGP_ERR_ARG, "apgp_append_point: null argument");
  if (!h->factored) return fail(APGP_NOT_COMPUTED, "apgp_append_point: GP not computed");
  const int N = h->N, d = h->d, Np = h->Np;
  const int BN = predict_tile_bn(d);
  if (N + 1 > Np || (N + BN) / BN * BN != h->Npad) return APGP_NEEDS_REFACTOR;   // padded buffers are full
  Guard g(h->device);
  CUI(h->X.reserve_keep((size_t)(N + 1) * d * 8, (size_t)N * d * 8, h->stream));
  CUI(h->y.reserve_keep((size_t)(N + 1) * 8, (size_t)N * 8, h->stream));
  CUI(h->ap_k.reserve((size_t)Np * 8)); CUI(h->ap_l.reserve((size_t)Np * 8)); CUI(h->ap_u.reserve((size_t)Np * 8));
  CUI(h->ap_x.reserve(APGP_MAX_DIM * 8));
  CU(cudaMemcpyAsync(h->ap_x.p, x_new, d * 8, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->X.as<double>() + (size_t)N * d, x_new, d * 8, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->y.as<double>() + N, &y_new, 8, cudaMemcpyHostToDevice, h->stream));
  const double kappa = h->amp + exp(h->white_noise) + TINY2;
  int nl = 0;
  CUI(launch_append_point(h->X.as<double>(), N, d, Np, h->ap_x.as<double>(), h->hyper.as<double>(), kappa,
                          y_new - h->mean, h->K.as<double>(), h->Linv.as<double>(), h->r.as<double>(),
                          h->alpha.as<double>(), h->ap_k.as<double>(), h->ap_l.as<double>(), h->ap_u.as<double>(),
                          h->scal.as<double>(), h->info.as<int>(), h->stream, &nl));
  double sc[2]; int status = 0;
  CU(cudaMemcpyAsync(sc, h->scal.p, 16, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(&status, h->info.p, 4, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->launches += nl; nl = 0;
  if (status != 0) return APGP_NOT_POSDEF;      // nothing was written: the N-point factorisation is still valid
  h->N = N + 1;
  h->logdet = sc[0]; h->loglik = sc[1];
  if (logdet) *logdet = sc[0];
  if (loglik) *loglik = sc[1];
  { int st_ = pack_predict_operands(h, &nl); if (st_ != APGP_OK) return st_; }
  CU(cudaStreamSynchronize(h->stream));
  h->launches += nl;
  return APGP_OK;
}

static void fill_predict_params(apgp_handle* h, PredictParams& p) {
  memset(&p, 0, sizeof(p));
  p.d = h->d; p.N = h->N; p.Npad = h->Npad;
  p.Xs = h->Xs.as<double>(); p.alphaA = h->alphaA.as<double>(); p.LinvF = h->LinvF.as<double>();
  for (int i = 0; i < h->d; ++i) p.qscale[i] = sqrt(0.5 * exp(-h->log_metric[i]));
  p.mean = h->mean; p.amp = h->amp;
}

// the variance kernels, as apgp_debug_last_var_path reports them
enum VarPath { VAR_FEW = 1, VAR_TILE = 2, VAR_GROUP_DMMA = 3, VAR_GROUP_I8 = 4 };

// The variance kernel of a call of Qplan queries (of which this launch is p.Q) and its group size G: a handful of
// queries go one CTA per query (APGP_PREDICT_FEW=0 keeps them on the tiled kernels); then the int8 engine where it
// applies and its plan groups the tiles, else the grouped DMMA kernel where its plan does, else one tile per CTA.
static VarPath choose_var_path(const apgp_handle* h, long long Q, long long Qplan, int* G) {
  *G = 1;
  if (Qplan <= PREDICT_FEW_MAX && Q == Qplan && (size_t)h->N * 8 <= 96 * 1024 && h->predict_few) return VAR_FEW;
  if (h->group == 0) return VAR_TILE;
  if (i8_applies(h) && (*G = predict_group_size(h->Npad, h->num_sms, h->group, h->d, Qplan, I8_GROUP_TILE)) > 1)
    return VAR_GROUP_I8;
  if ((*G = predict_group_size(h->Npad, h->num_sms, h->group, h->d, Qplan, DMMA_GROUP_TILE)) > 1) return VAR_GROUP_DMMA;
  *G = 1;
  return VAR_TILE;
}

// one launch of the predict kernels for the queries described by p (device pointers), on stream st
// Qplan: the size of the WHOLE call this launch is a slice of -- the group size (hence the summation order of the mean)
// must not depend on how a host call was sliced
static int predict_launch(apgp_handle* h, PredictParams& p, int want_var, cudaStream_t st, int* nl, long long Qplan) {
  const int d = h->d;
  if (!want_var) { CUI(launch_predict_mean(p, h->num_sms, st, nl)); return APGP_OK; }
  int G = 1;
  VarPath path = choose_var_path(h, p.Q, Qplan, &G);
  if (path == VAR_FEW) {
    if (h->few_ws.cap < predict_few_ws_bytes()) {
      CUI(h->few_ws.reserve(predict_few_ws_bytes()));
      CU(cudaMemsetAsync(h->few_ws.p, 0, predict_few_ws_bytes(), st));
    }
    CUI(launch_predict_few(p, h->Linv.as<double>(), h->Np, h->few_ws.p, st, nl));
  } else if (path != VAR_TILE) {
    const bool i8 = path == VAR_GROUP_I8;
    const GroupTile& tile = i8 ? I8_GROUP_TILE : DMMA_GROUP_TILE;
    if (i8) {
      // packed with the factorisation; here only when the engine was switched to i8 after it
      if (!h->i8_packed) { int st_ = pack_i8_operands(h, st, nl); if (st_ != APGP_OK) return st_; }
      p.LinvI8 = h->LinvI8.as<unsigned char>(); p.i8scale = h->i8scale.as<double>();
    }
    CUI(h->scratch.reserve(predict_group_scratch_bytes(h->Npad, h->num_sms, G, tile)));
    CUI(h->g_arrive.reserve(sizeof(int) * ((h->num_sms + G - 1) / G)));
    CUI(h->g_part.reserve(predict_group_part_bytes(h->Npad, h->num_sms, G)));
    CUI(h->g_plan.reserve(4 * GROUP_MAX_BLOCKS * sizeof(int)));
    p.scratch = h->scratch.as<double>();
    p.grp_arrive = h->g_arrive.as<int>(); p.grp_part = h->g_part.as<double>(); p.grp_plan = h->g_plan.as<int>();
    if (h->plan_Npad != h->Npad || h->plan_G != G || h->plan_d != d || h->plan_i8 != (int)i8) {   // re-plan on a new shape
      int tab[4 * GROUP_MAX_BLOCKS];
      predict_group_plan(h->Npad, h->num_sms, G, d, tab, tile);
      CU(cudaMemcpyAsync(h->g_plan.p, tab, sizeof(tab), cudaMemcpyHostToDevice, st));
      CU(cudaStreamSynchronize(st));
      h->plan_Npad = h->Npad; h->plan_G = G; h->plan_d = d; h->plan_i8 = (int)i8;
    }
    const int ge = i8 ? launch_predict_var_i8(p, h->num_sms, G, st, nl) : launch_predict_var_grouped(p, h->num_sms, G, st, nl);
    if (ge == (int)cudaErrorCooperativeLaunchTooLarge) {
      // the GPU is shared (fewer SMs free than the grid needs for its spin barriers): one tile per CTA instead
      (void)cudaGetLastError();
      --*nl;
      path = VAR_TILE;
    } else {
      CUI(ge);
    }
  }
  if (path == VAR_TILE) {
    CUI(h->scratch.reserve(predict_scratch_bytes(h->Npad, h->num_sms, d)));
    p.scratch = h->scratch.as<double>();
    CUI(launch_predict_var(p, h->num_sms, st, nl));
  }
  h->last_var_path = path;
  return APGP_OK;
}

static int ensure_pipeline(apgp_handle* h) {
  if (h->copy_in) return APGP_OK;
  CU(cudaStreamCreateWithFlags(&h->copy_in, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&h->copy_out, cudaStreamNonBlocking));
  for (int b = 0; b < 2; ++b) {
    CU(cudaEventCreateWithFlags(&h->ev_in[b], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_k[b], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_out[b], cudaEventDisableTiming));
  }
  return APGP_OK;
}

int apgp_predict(apgp_handle* h, const double* Xq, long long Q, double* mu, double* var, double* util,
                 const apgp_predict_opts* o, int on_host) {
  if (!h || !o) return fail(APGP_ERR_ARG, "apgp_predict: null argument");
  if (!h->factored) return fail(APGP_NOT_COMPUTED, "apgp_predict: GP not computed");
  if (Q < 0) return fail(APGP_ERR_ARG, "apgp_predict: Q < 0");
  if (Q == 0) return APGP_OK;
  if (!Xq) return fail(APGP_ERR_ARG, "apgp_predict: null queries");
  if ((var || util) && !o->want_var) return fail(APGP_ERR_ARG, "apgp_predict: var/util outputs need want_var=1");
  if (o->utility < 0 || o->utility > 3) return fail(APGP_ERR_ARG, "apgp_predict: bad utility kind");
  Guard g(h->device);
  const int d = h->d;
  PredictParams p;
  fill_predict_params(h, p);
  p.Q = Q;
  p.has_box = o->has_box; p.utility_kind = o->utility; p.ybest = o->ybest; p.zeta = o->zeta;
  for (int i = 0; i < d; ++i) { p.lo[i] = o->lo[i]; p.hi[i] = o->hi[i]; }
  const int nout = (mu ? 1 : 0) + (var ? 1 : 0) + (util ? 1 : 0);
  int nl = 0;
  if (!on_host) {
    p.Xq = Xq; p.mu = mu; p.var = var; p.util = util;
    { int st_ = predict_launch(h, p, o->want_var, h->stream, &nl, Q); if (st_ != APGP_OK) return st_; }
    h->launches += nl;
    return APGP_OK;
  }
  // small host calls (optimiser rounds: a handful of queries) go through pinned staging: one async H2D,
  // one async D2H, no pageable-memory bounce -- this path is pure latency
  const size_t half = apgp_handle::PIN_DOUBLES / 2;
  const bool small_call = (size_t)Q * d <= half && (size_t)Q * (nout ? nout : 1) <= half;
  // large host calls are cut into slices whose H2D copy, kernel and D2H copies overlap on three streams
  // (double-buffered device staging): end to end the call costs max(kernel, copies) instead of their sum.
  // Slices are whole multiples of one wave of 256-query tiles (num_sms tiles) so no slice ends in a partial wave.
  const long long wave = (long long)h->num_sms * 256;
  const bool pipelined = !small_call && Q >= 4 * wave && !getenv("APGP_NO_PIPELINE");
  if (!pipelined) {
    CUI(h->stage_in.reserve((size_t)Q * d * 8));
    CUI(h->stage_out.reserve((size_t)Q * 8 * (nout ? nout : 1)));
    const double* src = Xq;
    if (small_call) { memcpy(h->pin, Xq, (size_t)Q * d * 8); src = h->pin; }
    CU(cudaMemcpyAsync(h->stage_in.p, src, (size_t)Q * d * 8, cudaMemcpyHostToDevice, h->stream));
    p.Xq = h->stage_in.as<double>();
    double* o0 = h->stage_out.as<double>();
    if (mu) { p.mu = o0; o0 += Q; }
    if (var) { p.var = o0; o0 += Q; }
    if (util) { p.util = o0; o0 += Q; }
    { int st_ = predict_launch(h, p, o->want_var, h->stream, &nl, Q); if (st_ != APGP_OK) return st_; }
    h->launches += nl;
    if (small_call) {
      double* hp = h->pin + half;
      CU(cudaMemcpyAsync(hp, h->stage_out.p, (size_t)Q * 8 * nout, cudaMemcpyDeviceToHost, h->stream));
      CU(cudaStreamSynchronize(h->stream));
      if (mu) { memcpy(mu, hp, (size_t)Q * 8); hp += Q; }
      if (var) { memcpy(var, hp, (size_t)Q * 8); hp += Q; }
      if (util) { memcpy(util, hp, (size_t)Q * 8); hp += Q; }
    } else {
      if (mu) CU(cudaMemcpyAsync(mu, p.mu, (size_t)Q * 8, cudaMemcpyDeviceToHost, h->stream));
      if (var) CU(cudaMemcpyAsync(var, p.var, (size_t)Q * 8, cudaMemcpyDeviceToHost, h->stream));
      if (util) CU(cudaMemcpyAsync(util, p.util, (size_t)Q * 8, cudaMemcpyDeviceToHost, h->stream));
      CU(cudaStreamSynchronize(h->stream));
    }
    return APGP_OK;
  }
  { int st_ = ensure_pipeline(h); if (st_ != APGP_OK) return st_; }
  long long per = (Q / 8) / wave * wave;
  if (per < wave) per = wave;
  const int no = nout ? nout : 1;
  CUI(h->stage_in.reserve((size_t)2 * per * d * 8));
  CUI(h->stage_out.reserve((size_t)2 * per * 8 * no));
  // the copy streams start after everything already queued on the compute stream (e.g. a pending factorisation)
  CU(cudaEventRecord(h->ev_k[0], h->stream)); CU(cudaEventRecord(h->ev_k[1], h->stream));
  CU(cudaEventRecord(h->ev_out[0], h->stream)); CU(cudaEventRecord(h->ev_out[1], h->stream));
  int slice = 0;
  for (long long q0 = 0; q0 < Q; q0 += per, ++slice) {
    const long long qn = (Q - q0 < per) ? (Q - q0) : per;
    const int b = slice & 1;
    double* din = h->stage_in.as<double>() + (size_t)b * per * d;
    double* dout = h->stage_out.as<double>() + (size_t)b * per * no;
    CU(cudaStreamWaitEvent(h->copy_in, h->ev_k[b], 0));                 // the kernel of slice - 2 has read this buffer
    CU(cudaMemcpyAsync(din, Xq + (size_t)q0 * d, (size_t)qn * d * 8, cudaMemcpyHostToDevice, h->copy_in));
    CU(cudaEventRecord(h->ev_in[b], h->copy_in));
    CU(cudaStreamWaitEvent(h->stream, h->ev_in[b], 0));
    CU(cudaStreamWaitEvent(h->stream, h->ev_out[b], 0));                // the D2H of slice - 2 has drained this buffer
    PredictParams ps = p;
    ps.Q = qn; ps.Xq = din;
    double* o0 = dout;
    if (mu) { ps.mu = o0; o0 += qn; }
    if (var) { ps.var = o0; o0 += qn; }
    if (util) { ps.util = o0; o0 += qn; }
    { int st_ = predict_launch(h, ps, o->want_var, h->stream, &nl, Q); if (st_ != APGP_OK) return st_; }
    CU(cudaEventRecord(h->ev_k[b], h->stream));
    CU(cudaStreamWaitEvent(h->copy_out, h->ev_k[b], 0));
    if (mu) CU(cudaMemcpyAsync(mu + q0, ps.mu, (size_t)qn * 8, cudaMemcpyDeviceToHost, h->copy_out));
    if (var) CU(cudaMemcpyAsync(var + q0, ps.var, (size_t)qn * 8, cudaMemcpyDeviceToHost, h->copy_out));
    if (util) CU(cudaMemcpyAsync(util + q0, ps.util, (size_t)qn * 8, cudaMemcpyDeviceToHost, h->copy_out));
    CU(cudaEventRecord(h->ev_out[b], h->copy_out));
  }
  h->launches += nl;
  CU(cudaStreamSynchronize(h->copy_out));
  CU(cudaStreamSynchronize(h->stream));
  return APGP_OK;
}

int apgp_grad_log_likelihood(apgp_handle* h, int fit_amp, double* grad) {
  if (!h || !grad) return fail(APGP_ERR_ARG, "apgp_grad_log_likelihood: null argument");
  const int d = h->d;
  const int P = 1 + (fit_amp ? 1 : 0) + d;
  for (int i = 0; i < P; ++i) grad[i] = 0.0;
  if (!h->factored) return APGP_NOT_COMPUTED;      // george: zeros when quiet and not computed
  Guard g(h->device);
  CUI(h->bscal.reserve(grad_loglik_doubles(h->Np, d) * 8));
  int nl = 0;
  CUI(launch_grad_loglik(h->X.as<double>(), h->N, d, h->Np, h->Linv.as<double>(), h->alpha.as<double>(),
                         h->hyper.as<double>(), fit_amp, h->work.as<double>(), h->bscal.as<double>(), h->stream, &nl));
  double out[2 + APGP_MAX_DIM];
  CU(cudaMemcpyAsync(out, h->bscal.p, (2 + d) * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->launches += nl;
  int k = 0;
  grad[k++] = out[0];
  if (fit_amp) grad[k++] = out[1];
  for (int i = 0; i < d; ++i) grad[k++] = out[2 + i];
  return APGP_OK;
}

int apgp_loglik_batch(apgp_handle* h, const double* P_host, int R, int P, int fit_amp, double white_noise,
                      double* ll_host, double* grad_host) {
  if (!h || !P_host || !ll_host) return fail(APGP_ERR_ARG, "apgp_loglik_batch: null argument");
  if (!h->has_training) return fail(APGP_ERR_ARG, "apgp_loglik_batch: no training set");
  const int d = h->d, N = h->N, Np = h->Np;
  if (P != 1 + (fit_amp ? 1 : 0) + d) return fail(APGP_ERR_ARG, "apgp_loglik_batch: P != 1 + fit_amp + d");
  if (R < 1) return APGP_OK;
  const int path = choose_loglik_path(h, R, grad_host != nullptr);
  // gradients come from the small kernel and the cluster kernel with gradients, not from a forced value-only kernel
  if (grad_host && path != LL_SMALL && path != LL_GROUP_GRAD) return APGP_NEEDS_HOST;
  h->last_loglik_path = path;
  Guard g(h->device);
  const double noise = exp(white_noise) + TINY2;
  // chunk the restart axis so the workspace stays below ~4 GiB (the gradient kernel keeps L and its inverse per restart)
  size_t per = (path == LL_GROUP_GRAD) ? loglik_grad_group_ws_bytes(Np, d, 1) : (size_t)Np * Np * 8;
  int Rc = (path == LL_SMALL) ? R : (int)((4ull << 30) / per); if (Rc < 1) Rc = 1; if (Rc > R) Rc = R;
  if (path == LL_GROUP) {
    CUI(h->gws.reserve(chol_group_ws_bytes(Np, Rc)));
  } else if (path == LL_GROUP_GRAD) {
    CUI(h->gws.reserve(loglik_grad_group_ws_bytes(Np, d, Rc)));
  } else if (path == LL_TILED) {
    CUI(h->bK.reserve(per * Rc));
    CUI(h->bDinv.reserve((size_t)Rc * Np * 64 * 8));
    CUI(h->br.reserve((size_t)Rc * Np * 8));
    CUI(h->binfo.reserve((size_t)Rc * 4));
  }
  CUI(h->bscal.reserve((size_t)(Rc > 2 + APGP_MAXD ? Rc : 2 + APGP_MAXD) * 8));
  CUI(h->bhyper.reserve((size_t)Rc * (3 + d) * 8));
  CUI(h->bll.reserve((size_t)Rc * 8));
  if (grad_host) CUI(h->bgrad.reserve((size_t)Rc * (2 + d) * 8));
  std::vector<double> gtmp(grad_host ? (size_t)Rc * (2 + d) : 0);
  std::vector<double> rows(path == LL_TILED ? (size_t)Rc * (3 + d) : 0);
  for (int r0 = 0; r0 < R; r0 += Rc) {
    const int rc = (R - r0 < Rc) ? (R - r0) : Rc;
    // the small and group kernels take the parameter vectors; the tiled sequence takes hyper rows (a vector that is not
    // finite is set to -inf below)
    const double* src = P_host + (size_t)r0 * P;
    size_t row_len = P;
    if (path == LL_TILED) {
      for (int r = 0; r < rc; ++r) {
        const double* p = src + (size_t)r * P;
        fill_hyper_row(rows.data() + (size_t)r * (3 + d), p[0], fit_amp ? d * exp(p[1]) : 1.0, white_noise,
                       p + 1 + (fit_amp ? 1 : 0), d);
      }
      src = rows.data();
      row_len = 3 + d;
    }
    const bool pin_ok = (size_t)rc * row_len <= apgp_handle::PIN_DOUBLES / 2 && (size_t)rc <= apgp_handle::PIN_DOUBLES / 2;
    if (pin_ok) { memcpy(h->pin, src, (size_t)rc * row_len * 8); src = h->pin; }
    CU(cudaMemcpyAsync(h->bhyper.p, src, (size_t)rc * row_len * 8, cudaMemcpyHostToDevice, h->stream));
    int nl = 0;
    if (path == LL_SMALL) {
      // one restart per CTA, everything in shared memory: a single launch per optimiser round
      CUI(launch_loglik_small(h->X.as<double>(), h->y.as<double>(), N, d, h->bhyper.as<double>(), fit_amp, noise, rc,
                              h->bll.as<double>(), grad_host ? h->bgrad.as<double>() : nullptr, h->stream)); ++nl;
      if (grad_host)
        CU(cudaMemcpyAsync(gtmp.data(), h->bgrad.p, (size_t)rc * (2 + d) * 8, cudaMemcpyDeviceToHost, h->stream));
    } else if (path == LL_GROUP) {
      CUI(launch_loglik_group(h->X.as<double>(), h->y.as<double>(), N, d, Np, h->bhyper.as<double>(), fit_amp, noise, rc,
                              h->num_sms, h->gws.p, h->bll.as<double>(), h->stream)); ++nl;
    } else if (path == LL_GROUP_GRAD) {
      // one cluster per restart: factorisation, inverse and trace products in a single launch
      CUI(launch_loglik_grad_group(h->X.as<double>(), h->y.as<double>(), N, d, Np, h->bhyper.as<double>(), fit_amp, noise,
                                   rc, h->num_sms, h->gws.p, h->bll.as<double>(), h->bgrad.as<double>(), h->stream)); ++nl;
      CU(cudaMemcpyAsync(gtmp.data(), h->bgrad.p, (size_t)rc * (2 + d) * 8, cudaMemcpyDeviceToHost, h->stream));
    } else {
      FactorBatch fb{rc, N, Np, h->bK.as<double>(), h->bDinv.as<double>(), h->br.as<double>(), h->bscal.as<double>(),
                     h->binfo.as<int>()};
      CUI(launch_build_K(h->X.as<double>(), h->y.as<double>(), N, d, h->bhyper.as<double>(), fb, h->stream)); ++nl;
      CUI(launch_cholesky(fb, h->num_sms, h->stream, &nl));
      CUI(launch_loglik_finish(fb, h->bll.as<double>(), h->stream)); ++nl;
    }
    double* lldst = pin_ok ? h->pin + apgp_handle::PIN_DOUBLES / 2 : ll_host + r0;
    CU(cudaMemcpyAsync(lldst, h->bll.p, (size_t)rc * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (pin_ok) memcpy(ll_host + r0, lldst, (size_t)rc * 8);
    h->launches += nl;
    for (int r = 0; r < rc; ++r) {
      const double* p = P_host + (size_t)(r0 + r) * P;
      bool fin = true;
      for (int i = 0; i < P; ++i) fin = fin && isfinite(p[i]);
      double& ll = ll_host[r0 + r];
      if (!fin || !isfinite(ll)) ll = -INFINITY;
      if (grad_host) {                       // [sum alpha, d/dlog_c, d/dlogM..] -> george order, amplitude slot optional
        const double* gr = gtmp.data() + (size_t)r * (2 + d);
        double* o = grad_host + (size_t)(r0 + r) * P;
        int k = 0;
        o[k++] = gr[0];
        if (fit_amp) o[k++] = gr[1];
        for (int i = 0; i < d; ++i) o[k++] = gr[2 + i];
        if (ll == -INFINITY) for (int i = 0; i < P; ++i) o[i] = 0.0;
      }
    }
  }
  return APGP_OK;
}

int apgp_sampler_run(apgp_handle* h, const apgp_sampler_opts* o, const double* p0, double* chain, double* logp,
                     double* blob, int* naccept, int on_host) {
  if (!h || !o || !p0 || !chain || !logp || !blob || !naccept) return fail(APGP_ERR_ARG, "apgp_sampler_run: null argument");
  if (!h->factored) return fail(APGP_NOT_COMPUTED, "apgp_sampler_run: GP not computed");
  if (o->nens < 1 || o->nwalkers < 2 || (o->nwalkers & 1) || o->nwalkers > 1024 || o->nsteps < 1 || o->thin < 1)
    return fail(APGP_ERR_ARG, "apgp_sampler_run: need nens>=1, even 2<=nwalkers<=1024, nsteps>=1, thin>=1");
  if ((size_t)o->nwalkers * (24 * h->d + 72) + 64 > 200 * 1024)
    return fail(APGP_ERR_ARG, "apgp_sampler_run: nwalkers x ndim too large for one CTA's shared memory "
                              "(need nwalkers * (24 ndim + 72) bytes <= 200 KB); use more ensembles of fewer walkers");
  Guard g(h->device);
  const int d = h->d;
  const size_t W = (size_t)o->nens * o->nwalkers;
  const size_t nst = (size_t)(o->nsteps / o->thin);
  const size_t Ns = o->nwalkers / 2;
  const bool replay = o->replay_zz != nullptr;
  if (replay && (!o->replay_inds || !o->replay_rint || !o->replay_logu))
    return fail(APGP_ERR_ARG, "apgp_sampler_run: replay needs all four buffers");
  SamplerParams p;
  memset(&p, 0, sizeof(p));
  p.nens = o->nens; p.nwalk = o->nwalkers; p.d = d; p.nsteps = o->nsteps; p.N = h->N; p.Npad = h->Npad;
  p.Xs = h->Xs.as<double>(); p.alphaA = h->alphaA.as<double>();
  for (int i = 0; i < d; ++i) { p.qscale[i] = sqrt(0.5 * exp(-h->log_metric[i])); p.lo[i] = o->lo[i]; p.hi[i] = o->hi[i]; }
  p.mean = h->mean; p.lnprior_const = o->lnprior_const; p.a = o->a; p.seed = o->seed; p.thin = o->thin;
  if (on_host) {
    CUI(h->s_p0.reserve(W * d * 8)); CUI(h->s_chain.reserve(nst * W * d * 8));
    CUI(h->s_logp.reserve(nst * W * 8)); CUI(h->s_blob.reserve(nst * W * 8)); CUI(h->s_nacc.reserve(W * 4));
    CU(cudaMemcpyAsync(h->s_p0.p, p0, W * d * 8, cudaMemcpyHostToDevice, h->stream));
    p.p0 = h->s_p0.as<double>(); p.chain = h->s_chain.as<double>(); p.logp = h->s_logp.as<double>();
    p.blob = h->s_blob.as<double>(); p.naccept = h->s_nacc.as<int>();
    if (replay) {
      const size_t ns = (size_t)o->nens * o->nsteps;
      CUI(h->s_ri.reserve(ns * o->nwalkers * 4)); CUI(h->s_rz.reserve(ns * 2 * Ns * 8));
      CUI(h->s_rr.reserve(ns * 2 * Ns * 4)); CUI(h->s_rl.reserve(ns * 2 * Ns * 8));
      CU(cudaMemcpyAsync(h->s_ri.p, o->replay_inds, ns * o->nwalkers * 4, cudaMemcpyHostToDevice, h->stream));
      CU(cudaMemcpyAsync(h->s_rz.p, o->replay_zz, ns * 2 * Ns * 8, cudaMemcpyHostToDevice, h->stream));
      CU(cudaMemcpyAsync(h->s_rr.p, o->replay_rint, ns * 2 * Ns * 4, cudaMemcpyHostToDevice, h->stream));
      CU(cudaMemcpyAsync(h->s_rl.p, o->replay_logu, ns * 2 * Ns * 8, cudaMemcpyHostToDevice, h->stream));
      p.r_inds = h->s_ri.as<int>(); p.r_zz = h->s_rz.as<double>(); p.r_rint = h->s_rr.as<int>(); p.r_logu = h->s_rl.as<double>();
    }
  } else {
    p.p0 = p0; p.chain = chain; p.logp = logp; p.blob = blob; p.naccept = naccept;
    p.r_inds = o->replay_inds; p.r_zz = o->replay_zz; p.r_rint = o->replay_rint; p.r_logu = o->replay_logu;
  }
  // Host results of more than a few MB: the chain runs as up to 8 launches (whole stored rows each; the kernel resumes
  // from the previous piece's last stored row with the draws indexed by the global step, so the chain is the same bit
  // for bit) and piece k's rows cross PCIe on the copy stream while piece k+1 samples.  APGP_SAMPLER_PIECES overrides.
  int pieces = 1;
  if (on_host && !replay && nst >= 2) {
    const size_t out_bytes = nst * W * (size_t)(d + 2) * 8;
    if (out_bytes >= ((size_t)4 << 20)) pieces = nst < 8 ? (int)nst : 8;
    if (const char* pv = getenv("APGP_SAMPLER_PIECES")) { const int v = atoi(pv); if (v >= 1) pieces = v > (int)nst ? (int)nst : v; }
  }
  if (pieces <= 1) {
    int nl = 0;
    CUI(launch_sampler(p, h->stream, &nl));
    h->launches += nl;
    if (on_host) {
      CU(cudaMemcpyAsync(chain, p.chain, nst * W * d * 8, cudaMemcpyDeviceToHost, h->stream));
      CU(cudaMemcpyAsync(logp, p.logp, nst * W * 8, cudaMemcpyDeviceToHost, h->stream));
      CU(cudaMemcpyAsync(blob, p.blob, nst * W * 8, cudaMemcpyDeviceToHost, h->stream));
      CU(cudaMemcpyAsync(naccept, p.naccept, W * 4, cudaMemcpyDeviceToHost, h->stream));
      CU(cudaStreamSynchronize(h->stream));
    }
    return APGP_OK;
  }
  { int st_ = ensure_pipeline(h); if (st_ != APGP_OK) return st_; }
  double* const dchain = h->s_chain.as<double>();
  double* const dlogp = h->s_logp.as<double>();
  double* const dblob = h->s_blob.as<double>();
  std::vector<cudaEvent_t> ev((size_t)pieces, nullptr);
  std::vector<size_t> row0((size_t)pieces + 1, 0);
  for (int k = 0; k <= pieces; ++k) row0[k] = nst * (size_t)k / pieces;
  int rc = APGP_OK;
  auto cleanup = [&]() { for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e); };
  p.nsteps_total = o->nsteps;
  for (int k = 0; k < pieces && rc == APGP_OK; ++k) {            // every piece is queued before the host blocks in a copy
    const size_t r0 = row0[k], r1 = row0[k + 1];
    p.step_base = (int)(r0 * o->thin);
    p.nsteps = (k == pieces - 1) ? o->nsteps - p.step_base : (int)((r1 - r0) * o->thin);
    p.p0 = k == 0 ? h->s_p0.as<double>() : dchain + (r0 - 1) * W * d;
    p.chain = dchain + r0 * W * d; p.logp = dlogp + r0 * W; p.blob = dblob + r0 * W;
    int nl = 0;
    if (launch_sampler(p, h->stream, &nl)) { rc = fail(APGP_ERR_CUDA, "apgp_sampler_run: launch failed"); break; }
    h->launches += nl;
    if (cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(ev[k], h->stream) != cudaSuccess)
      rc = fail(APGP_ERR_CUDA, "apgp_sampler_run: event");
  }
  for (int k = 0; k < pieces && rc == APGP_OK; ++k) {
    const size_t r0 = row0[k], nr = row0[k + 1] - r0;
    if (cudaStreamWaitEvent(h->copy_out, ev[k], 0) != cudaSuccess ||
        cudaMemcpyAsync(chain + r0 * W * d, dchain + r0 * W * d, nr * W * d * 8, cudaMemcpyDeviceToHost, h->copy_out) != cudaSuccess ||
        cudaMemcpyAsync(logp + r0 * W, dlogp + r0 * W, nr * W * 8, cudaMemcpyDeviceToHost, h->copy_out) != cudaSuccess ||
        cudaMemcpyAsync(blob + r0 * W, dblob + r0 * W, nr * W * 8, cudaMemcpyDeviceToHost, h->copy_out) != cudaSuccess)
      rc = fail(APGP_ERR_CUDA, "apgp_sampler_run: copy");
  }
  if (rc == APGP_OK && cudaMemcpyAsync(naccept, p.naccept, W * 4, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess)
    rc = fail(APGP_ERR_CUDA, "apgp_sampler_run: copy");
  cudaStreamSynchronize(h->stream);
  cudaStreamSynchronize(h->copy_out);
  cleanup();
  if (rc == APGP_OK && cudaGetLastError() != cudaSuccess) rc = fail(APGP_ERR_CUDA, "apgp_sampler_run: device error");
  return rc;
}

// ---- multi-GPU: one handle per GPU, NCCL over NVLink (comm.cu) ------------------------------------------------------
int apgp_comm_unique_id(char id_out[128]) {
  if (!id_out) return fail(APGP_ERR_ARG, "apgp_comm_unique_id: null argument");
  if (comm_unique_id(id_out)) return fail(APGP_ERR_COMM, comm_last_error());
  return APGP_OK;
}
int apgp_comm_group_start(void) { if (comm_group_start()) return fail(APGP_ERR_COMM, comm_last_error()); return APGP_OK; }
int apgp_comm_group_end(void) { if (comm_group_end()) return fail(APGP_ERR_COMM, comm_last_error()); return APGP_OK; }

int apgp_comm_init(apgp_handle* h, const char id[128], int rank, int world) {
  if (!h || !id || world < 1 || rank < 0 || rank >= world) return fail(APGP_ERR_ARG, "apgp_comm_init: bad argument");
  Guard g(h->device);
  if (h->comm) { comm_destroy(h->comm); h->comm = nullptr; }
  if (comm_init(&h->comm, id, rank, world)) return fail(APGP_ERR_COMM, comm_last_error());
  h->comm_rank = rank; h->comm_world = world;
  return APGP_OK;
}
int apgp_comm_destroy(apgp_handle* h) {
  if (!h) return APGP_OK;
  Guard g(h->device);
  if (h->comm) { cudaStreamSynchronize(h->stream); comm_destroy(h->comm); h->comm = nullptr; }
  h->comm_rank = 0; h->comm_world = 1;
  return APGP_OK;
}

// header of a broadcast factorisation: everything host-side that apgp_factorize leaves in the handle
struct FactorHeader {
  int N, d, Np, Npad, factored;
  double mean, amp, white_noise, logdet, loglik;
  double log_metric[APGP_MAX_DIM];
};

int apgp_comm_broadcast_factor(apgp_handle* h, int root) {
  if (!h || !h->comm) return fail(APGP_ERR_ARG, "apgp_comm_broadcast_factor: apgp_comm_init first");
  if (root < 0 || root >= h->comm_world) return fail(APGP_ERR_ARG, "apgp_comm_broadcast_factor: bad root");
  Guard g(h->device);
  const bool is_root = h->comm_rank == root;
  if (is_root && !h->factored) return fail(APGP_NOT_COMPUTED, "apgp_comm_broadcast_factor: the root's GP is not computed");
  FactorHeader hd;
  memset(&hd, 0, sizeof(hd));
  if (is_root) {
    hd.N = h->N; hd.d = h->d; hd.Np = h->Np; hd.Npad = h->Npad; hd.factored = 1;
    hd.mean = h->mean; hd.amp = h->amp; hd.white_noise = h->white_noise; hd.logdet = h->logdet; hd.loglik = h->loglik;
    for (int i = 0; i < h->d; ++i) hd.log_metric[i] = h->log_metric[i];
  }
  CUI(h->c_hdr.reserve(sizeof(hd)));
  if (is_root) CU(cudaMemcpyAsync(h->c_hdr.p, &hd, sizeof(hd), cudaMemcpyHostToDevice, h->stream));
  if (comm_broadcast_bytes(h->comm, h->c_hdr.p, sizeof(hd), root, h->stream)) return fail(APGP_ERR_COMM, comm_last_error());
  CU(cudaMemcpyAsync(&hd, h->c_hdr.p, sizeof(hd), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (!hd.factored || hd.N < 1 || hd.d < 1 || hd.d > APGP_MAX_DIM) return fail(APGP_ERR_COMM, "apgp_comm_broadcast_factor: bad header");
  const int N = hd.N, d = hd.d, Np = hd.Np;
  if (!is_root) {
    h->N = N; h->d = d; h->Np = Np; h->Npad = hd.Npad;
    h->mean = hd.mean; h->amp = hd.amp; h->white_noise = hd.white_noise; h->logdet = hd.logdet; h->loglik = hd.loglik;
    for (int i = 0; i < d; ++i) h->log_metric[i] = hd.log_metric[i];
    h->has_training = true; h->has_hyper = true; h->factored = false;
    CUI(h->X.reserve((size_t)N * d * 8)); CUI(h->y.reserve((size_t)N * 8));
    CUI(h->K.reserve((size_t)Np * Np * 8)); CUI(h->Dinv.reserve((size_t)Np * 64 * 8)); CUI(h->r.reserve((size_t)Np * 8));
    CUI(h->Linv.reserve((size_t)Np * Np * 8)); CUI(h->work.reserve((size_t)Np * Np * 8));
    CUI(h->alpha.reserve((size_t)Np * 8)); CUI(h->alphaA.reserve((size_t)h->Npad * 8)); CUI(h->Xs.reserve((size_t)d * h->Npad * 8));
    CUI(h->scal.reserve(4 * 8)); CUI(h->info.reserve(4)); CUI(h->hyper.reserve((3 + APGP_MAX_DIM) * 8)); CUI(h->qscale.reserve(APGP_MAX_DIM * 8));
    const int BN = predict_tile_bn(d);
    CUI(h->LinvF.reserve((size_t)linvf_total_tiles(h->Npad, BN) * BN * 16 * 8));
  }
  struct { DevBuf* b; size_t bytes; } parts[] = {
      {&h->X, (size_t)N * d * 8}, {&h->y, (size_t)N * 8}, {&h->K, (size_t)Np * Np * 8}, {&h->Dinv, (size_t)Np * 64 * 8},
      {&h->r, (size_t)Np * 8}, {&h->Linv, (size_t)Np * Np * 8}, {&h->alpha, (size_t)Np * 8}, {&h->hyper, (size_t)(3 + d) * 8},
      {&h->scal, 16}};
  for (auto& pt : parts)
    if (comm_broadcast_bytes(h->comm, pt.b->p, pt.bytes, root, h->stream)) return fail(APGP_ERR_COMM, comm_last_error());
  if (!is_root) {
    int nl = 0;
    { int st_ = pack_predict_operands(h, &nl); if (st_ != APGP_OK) return st_; }
    h->launches += nl;
  }
  CU(cudaStreamSynchronize(h->stream));
  h->factored = true;
  return APGP_OK;
}

int apgp_comm_allgather(apgp_handle* h, const double* send, double* recv, long long count, int on_host) {
  if (!h || !h->comm || !send || !recv || count < 0) return fail(APGP_ERR_ARG, "apgp_comm_allgather: bad argument");
  if (count == 0) return APGP_OK;
  Guard g(h->device);
  const double* s = send; double* r = recv;
  if (on_host) {
    CUI(h->c_send.reserve((size_t)count * 8)); CUI(h->c_recv.reserve((size_t)count * 8 * h->comm_world));
    CU(cudaMemcpyAsync(h->c_send.p, send, (size_t)count * 8, cudaMemcpyHostToDevice, h->stream));
    s = h->c_send.as<double>(); r = h->c_recv.as<double>();
  }
  if (comm_allgather_doubles(h->comm, s, r, (size_t)count, h->stream)) return fail(APGP_ERR_COMM, comm_last_error());
  if (on_host) {
    CU(cudaMemcpyAsync(recv, r, (size_t)count * 8 * h->comm_world, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  return APGP_OK;
}

// ---- integrated autocorrelation time (emcee's estimator) of a chain, on the device -----------------------------
int apgp_integrated_time(apgp_handle* h, const double* chain, long long n_total, int W, int d, long long discard, int thin,
                         double c, int on_host, double* tau_out, int* window_out) {
  if (!h || !chain || !tau_out) return fail(APGP_ERR_ARG, "apgp_integrated_time: null argument");
  if (n_total < 1 || W < 1 || d < 1 || thin < 1 || discard < 0) return fail(APGP_ERR_ARG, "apgp_integrated_time: bad shape");
  const long long off = discard + thin - 1;                 // emcee: chain[discard + thin - 1 :: thin]
  if (off >= n_total) return fail(APGP_ERR_ARG, "apgp_integrated_time: nothing left after discard/thin");
  const long long nll = (n_total - off + thin - 1) / thin;
  if (nll > (1ll << 30)) return fail(APGP_ERR_ARG, "apgp_integrated_time: chain too long");
  const int n = (int)nll;
  Guard g(h->device);
  if (!autocorr_fits(n, 1)) return APGP_NEEDS_HOST;          // series does not fit one CTA's shared memory
  const double* src = chain;
  if (on_host) {
    const size_t bytes = (size_t)n_total * W * d * 8;
    CUI(h->ac_stage.reserve(bytes));
    CU(cudaMemcpyAsync(h->ac_stage.p, chain, bytes, cudaMemcpyHostToDevice, h->stream));
    src = h->ac_stage.as<double>();
  }
  std::vector<double> f;
  int T = 256;
  for (int k = 0; k < d; ++k) { tau_out[k] = NAN; if (window_out) window_out[k] = -1; }
  std::vector<char> found(d, 0);
  for (;;) {
    if (T > n) T = n;
    if (!autocorr_fits(n, T)) return APGP_NEEDS_HOST;
    int G, nchunk;
    const size_t pb = autocorr_partial_bytes(W, d, T, h->num_sms, &G, &nchunk);
    CUI(h->ac_part.reserve(pb));
    CUI(h->ac_f.reserve((size_t)d * T * 8));
    int nl = 0;
    CUI(launch_autocorr(src, off, thin, n, W, d, T, h->num_sms, h->ac_part.as<double>(), h->ac_f.as<double>(), h->stream, &nl));
    h->launches += nl;
    f.resize((size_t)d * T);
    CU(cudaMemcpyAsync(f.data(), h->ac_f.p, (size_t)d * T * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    bool all = true;
    for (int k = 0; k < d; ++k) {
      if (found[k]) continue;
      // emcee.autocorr.auto_window: m = arange(n) < c * taus; window = argmin(m) if any(m) else n - 1.
      // argmin(m) is the FIRST M where the condition fails -- and 0 when it never fails (argmin of an all-True
      // array), in which case emcee reports tau(0) = 2 f(0) - 1 = 1; kept.  (All-False needs taus[0] <= 0 or NaN:
      // the first failure is then M = 0 and the reported value is the same NaN.)
      double cum = 0.0, tau0 = NAN;
      int win = -1;
      double tw = NAN;
      for (int M = 0; M < T; ++M) {
        cum += f[(size_t)k * T + M];
        const double taus = 2.0 * cum - 1.0;
        if (M == 0) tau0 = taus;
        if (!((double)M < c * taus)) { win = M; tw = taus; break; }
      }
      if (win < 0 && T == n) { win = 0; tw = tau0; }
      if (win >= 0) { found[k] = 1; tau_out[k] = tw; if (window_out) window_out[k] = win; }
      else all = false;
    }
    if (all) return APGP_OK;
    if (T == n) return APGP_OK;
    if (T >= 4096) return APGP_NEEDS_HOST;                    // window beyond 4096 lags: let the caller use its FFT path
    T *= 4;
  }
}

// ---- device-resident optimisers ---------------------------------------------------------------------
static int resolve_opt(const apgp_opt_opts* o, int n, OptimizeParams& q) {
  if (o->method != APGP_OPT_NELDER_MEAD && o->method != APGP_OPT_POWELL) return -1;
  const long long INF = 1LL << 62;
  long long mi = o->maxiter, mf = o->maxfev;
  const long long def = (long long)n * (o->method == APGP_OPT_NELDER_MEAD ? 200 : 1000);   // SciPy's defaults
  if (mi < 0 && mf < 0) { mi = def; mf = def; }
  else if (mi < 0) mi = (mf >= INF) ? def : INF;
  else if (mf < 0) mf = (mi >= INF) ? def : INF;
  q.method = o->method; q.adaptive = o->adaptive; q.xtol = o->xtol; q.ftol = o->ftol; q.maxiter = mi; q.maxfun = mf;
  return 0;
}

static int opt_stage(apgp_handle* h, const double* in, size_t nin, size_t nx, int R) {
  CUI(h->o_in.reserve(nin * 8)); CUI(h->o_x.reserve(nx * 8)); CUI(h->o_f.reserve((size_t)R * 8));
  CUI(h->o_stats.reserve((size_t)R * 24));
  const double* src = in;
  if (nin <= apgp_handle::PIN_DOUBLES / 2) { memcpy(h->pin, in, nin * 8); src = h->pin; }
  CU(cudaMemcpyAsync(h->o_in.p, src, nin * 8, cudaMemcpyHostToDevice, h->stream));
  return APGP_OK;
}

static int opt_fetch(apgp_handle* h, size_t nx, int R, double* x_out, double* f_out, long long* stats) {
  CU(cudaMemcpyAsync(x_out, h->o_x.p, nx * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(f_out, h->o_f.p, (size_t)R * 8, cudaMemcpyDeviceToHost, h->stream));
  if (stats) CU(cudaMemcpyAsync(stats, h->o_stats.p, (size_t)R * 24, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return APGP_OK;
}

int apgp_minimize_utility(apgp_handle* h, const apgp_predict_opts* obj, const apgp_opt_opts* opt, const double* x0,
                          int R, double* x_out, double* f_out, long long* stats, int evaluate_only) {
  if (!h || !obj || !opt || !x0 || !x_out || !f_out) return fail(APGP_ERR_ARG, "apgp_minimize_utility: null argument");
  if (!h->factored) return fail(APGP_NOT_COMPUTED, "apgp_minimize_utility: GP not computed");
  if (obj->utility < APGP_UTIL_AGP || obj->utility > APGP_UTIL_NEGMEAN)
    return fail(APGP_ERR_ARG, "apgp_minimize_utility: objective must be AGP, BAPE, Jones or NEGMEAN");
  if (R < 1) return APGP_OK;
  Guard g(h->device);
  const int d = h->d;
  OptimizeParams q;
  if (resolve_opt(opt, d, q)) return fail(APGP_ERR_ARG, "apgp_minimize_utility: bad method");
  UtilityPointParams u;
  memset(&u, 0, sizeof(u));
  u.N = h->N; u.d = d; u.Npad = h->Npad; u.ldL = h->Np;
  u.Xs = h->Xs.as<double>(); u.alphaA = h->alphaA.as<double>(); u.Linv = h->Linv.as<double>();
  u.amp = h->amp; u.mean = h->mean; u.ybest = obj->ybest; u.zeta = obj->zeta; u.kind = obj->utility; u.has_box = obj->has_box;
  for (int i = 0; i < d; ++i) { u.lo[i] = obj->lo[i]; u.hi[i] = obj->hi[i]; u.qscale[i] = sqrt(0.5 * exp(-h->log_metric[i])); }
  { int st_ = opt_stage(h, x0, (size_t)R * d, (size_t)R * d, R); if (st_ != APGP_OK) return st_; }
  CUI(launch_minimize_utility(u, q, R, h->o_in.as<double>(), h->o_x.as<double>(), h->o_f.as<double>(),
                              h->o_stats.as<long long>(), evaluate_only ? 0 : 1, h->stream));
  h->launches += 1;
  return opt_fetch(h, (size_t)R * d, R, x_out, f_out, stats);
}

// largest training set the cluster-per-restart optimiser takes: beyond it one objective evaluation is so long that a
// host-driven optimiser over apgp_loglik_batch loses nothing, and R x Np^2 workspaces get large
static const int GROUP_OPT_MAX_N = 4096;
int apgp_minimize_nll_fits(const apgp_handle* h, int P) {
  if (!h || !h->has_training) return 0;
  if (minimize_nll_fits(h->N, h->d, P) && !getenv("APGP_NLL_GROUP")) return 1;
  return (minimize_nll_group_fits(P) && h->N <= GROUP_OPT_MAX_N) ? 2 : 0;
}

int apgp_minimize_nll(apgp_handle* h, const apgp_opt_opts* opt, const double* p0, int R, int P, int fit_amp,
                      double white_noise, int default_prior, double* p_out, double* f_out, long long* stats,
                      int evaluate_only) {
  if (!h || !opt || !p0 || !p_out || !f_out) return fail(APGP_ERR_ARG, "apgp_minimize_nll: null argument");
  if (!h->has_training) return fail(APGP_ERR_ARG, "apgp_minimize_nll: no training set");
  const int d = h->d, N = h->N;
  if (P != 1 + (fit_amp ? 1 : 0) + d) return fail(APGP_ERR_ARG, "apgp_minimize_nll: P != 1 + fit_amp + d");
  const int path = apgp_minimize_nll_fits(h, P);
  if (!path)
    return fail(APGP_ERR_ARG, "apgp_minimize_nll: training set too large for the device optimisers (N <= 4096); "
                              "drive apgp_loglik_batch from the host optimiser instead");
  if (R < 1) return APGP_OK;
  Guard g(h->device);
  OptimizeParams q;
  if (resolve_opt(opt, P, q)) return fail(APGP_ERR_ARG, "apgp_minimize_nll: bad method");
  if (path == 1) {
    { int st_ = opt_stage(h, p0, (size_t)R * P, (size_t)R * P, R); if (st_ != APGP_OK) return st_; }
    CUI(launch_minimize_nll(h->X.as<double>(), h->y.as<double>(), N, d, P, fit_amp ? 1 : 0, default_prior ? 1 : 0,
                            exp(white_noise) + TINY2, q, R, h->o_in.as<double>(), h->o_x.as<double>(), h->o_f.as<double>(),
                            h->o_stats.as<long long>(), evaluate_only ? 0 : 1, h->stream));
    h->launches += 1;
    return opt_fetch(h, (size_t)R * P, R, p_out, f_out, stats);
  }
  // one cluster per restart, matrices in L2-resident global workspace; the restart axis is chunked to ~4 GiB of it
  const int Np = h->Np;
  int Rc = (int)((4ull << 30) / ((size_t)Np * Np * 8)); if (Rc < 1) Rc = 1; if (Rc > R) Rc = R;
  CUI(h->gws.reserve(chol_group_ws_bytes(Np, Rc)));
  for (int r0 = 0; r0 < R; r0 += Rc) {
    const int rc = (R - r0 < Rc) ? (R - r0) : Rc;
    { int st_ = opt_stage(h, p0 + (size_t)r0 * P, (size_t)rc * P, (size_t)rc * P, rc); if (st_ != APGP_OK) return st_; }
    CUI(launch_minimize_nll_group(h->X.as<double>(), h->y.as<double>(), N, d, Np, P, fit_amp ? 1 : 0, default_prior ? 1 : 0,
                                  exp(white_noise) + TINY2, q, rc, h->num_sms, h->gws.p, h->o_in.as<double>(),
                                  h->o_x.as<double>(), h->o_f.as<double>(), h->o_stats.as<long long>(),
                                  evaluate_only ? 0 : 1, h->stream));
    h->launches += 1;
    { int st_ = opt_fetch(h, (size_t)rc * P, rc, p_out + (size_t)r0 * P, f_out + r0, stats ? stats + 3 * (size_t)r0 : nullptr);
      if (st_ != APGP_OK) return st_; }
  }
  return APGP_OK;
}

int apgp_get_alpha(apgp_handle* h, double* alpha) {
  if (!h || !alpha) return fail(APGP_ERR_ARG, "null argument");
  if (!h->factored) return fail(APGP_NOT_COMPUTED, "GP not computed");
  Guard g(h->device);
  CU(cudaMemcpyAsync(alpha, h->alpha.p, (size_t)h->N * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return APGP_OK;
}

static int get_square(apgp_handle* h, const DevBuf& b, double* out) {
  if (!h || !out) return fail(APGP_ERR_ARG, "null argument");
  if (!h->factored) return fail(APGP_NOT_COMPUTED, "GP not computed");
  Guard g(h->device);
  CU(cudaMemcpy2DAsync(out, (size_t)h->N * 8, b.p, (size_t)h->Np * 8, (size_t)h->N * 8, h->N, cudaMemcpyDeviceToHost,
                       h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < h->N; ++i)
    for (int j = i + 1; j < h->N; ++j) out[(size_t)i * h->N + j] = 0.0;
  return APGP_OK;
}
static int debug_exp(apgp_handle* h, const double* s, int n, double* out, int variant);
int apgp_debug_exp_neg(apgp_handle* h, const double* s, int n, double* out) { return debug_exp(h, s, n, out, 0); }
int apgp_debug_exp_neg256(apgp_handle* h, const double* s, int n, double* out) { return debug_exp(h, s, n, out, 1); }
}  // extern "C"
static int debug_exp(apgp_handle* h, const double* s, int n, double* out, int variant) {
  if (!h || !s || !out || n < 1) return fail(APGP_ERR_ARG, "apgp_debug_exp_neg");
  Guard g(h->device);
  CUI(h->stage_in.reserve((size_t)n * 8)); CUI(h->stage_out.reserve((size_t)n * 8));
  CU(cudaMemcpyAsync(h->stage_in.p, s, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
  CUI(launch_exp_neg_test(h->stage_in.as<double>(), n, h->stage_out.as<double>(), h->stream, variant));
  CU(cudaMemcpyAsync(out, h->stage_out.p, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return APGP_OK;
}
extern "C" {
int apgp_debug_group_plan(int N, int num_sms, int d, long long Q, int requested, int* G_out, int* tab512) {
  // host-only: the work split the grouped variance kernel would use (no device needed; exercised by the CPU tests)
  if (!G_out || N < 1 || num_sms < 1 || d < 1) return fail(APGP_ERR_ARG, "apgp_debug_group_plan");
  const int Npad = (N + 63) / 64 * 64;
  const int G = predict_group_size(Npad, num_sms, requested, d, Q, DMMA_GROUP_TILE);
  *G_out = G;
  if (tab512 && G > 1) predict_group_plan(Npad, num_sms, G, d, tab512, DMMA_GROUP_TILE);
  return APGP_OK;
}
int apgp_debug_read_prof(long long* out16) { return out16 ? read_prof(out16) : APGP_ERR_ARG; }
int apgp_get_linv(apgp_handle* h, double* linv) { return get_square(h, h->Linv, linv); }
int apgp_get_chol(apgp_handle* h, double* L) { return get_square(h, h->K, L); }

int apgp_debug_last_var_path(const apgp_handle* h, int* path) {
  if (!h || !path) return fail(APGP_ERR_ARG, "apgp_debug_last_var_path");
  *path = h->last_var_path;
  return APGP_OK;
}

int apgp_debug_last_loglik_path(const apgp_handle* h, int* path) {
  if (!h || !path) return fail(APGP_ERR_ARG, "apgp_debug_last_loglik_path");
  *path = h->last_loglik_path;
  return APGP_OK;
}

int apgp_debug_i8_operands(apgp_handle* h, unsigned char* linv_i8, double* rowscale, unsigned char* panel, int* npad) {
  if (!h || !h->factored || !h->i8_packed) return fail(APGP_ERR_ARG, "apgp_debug_i8_operands: int8 operands not packed");
  if (panel && h->last_var_path != 4) return fail(APGP_ERR_ARG, "apgp_debug_i8_operands: last variance call was not int8");
  Guard g(h->device);
  if (npad) *npad = h->Npad;
  if (linv_i8) CU(cudaMemcpyAsync(linv_i8, h->LinvI8.p, linv_i8_bytes(h->Npad), cudaMemcpyDeviceToHost, h->stream));
  if (rowscale) CU(cudaMemcpyAsync(rowscale, h->i8scale.p, (size_t)h->Npad * 8, cudaMemcpyDeviceToHost, h->stream));
  // group 0, buffer 0 of the grouped kernel's scratch: the first 128-query tile of the last call
  if (panel)
    CU(cudaMemcpyAsync(panel, h->scratch.p, (size_t)I8_GROUP_TILE.bm * I8_GROUP_TILE.panel_bytes * h->Npad,
                       cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return APGP_OK;
}

int apgp_debug_pack_linv_i8(apgp_handle* h, const double* M, int n, double amp, unsigned char* out, double* rowscale) {
  if (!h || !M || !out || !rowscale || n < 1 || n > 8192) return fail(APGP_ERR_ARG, "apgp_debug_pack_linv_i8");
  Guard g(h->device);
  const int Npad = (n + 63) / 64 * 64;
  const size_t nb = linv_i8_bytes(Npad);
  void *dm = nullptr, *dout = nullptr, *dsc = nullptr;
  cudaError_t e = cudaMalloc(&dm, (size_t)n * n * 8);
  if (e == cudaSuccess) e = cudaMalloc(&dout, nb);
  if (e == cudaSuccess) e = cudaMalloc(&dsc, (size_t)Npad * 8);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dm, M, (size_t)n * n * 8, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess)
    e = (cudaError_t)launch_pack_linv_i8((const double*)dm, n, n, Npad, amp, (unsigned char*)dout, (double*)dsc, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, nb, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(rowscale, dsc, (size_t)Npad * 8, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(dm); cudaFree(dout); cudaFree(dsc);
  if (e != cudaSuccess) return fail(APGP_ERR_CUDA, "apgp_debug_pack_linv_i8", e);
  h->launches += 1;
  return APGP_OK;
}

}  // extern "C"
