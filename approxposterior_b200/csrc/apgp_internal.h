// Internal (C++) interface between the libapgp translation units.  Not part of the C-ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace apgp {

// cudaFuncSetAttribute applies to the CURRENT device only, and a process may hold handles on several GPUs
// (apgp_create(device)): remember the opt-in per device ordinal, not per process.
struct PerDeviceOnce {
  unsigned long long done[2] = {0ull, 0ull};
  int dev = -1;
  // true when the attribute still has to be set on the current device; call mark() after it was set
  bool needed() {
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 128) { dev = -1; return true; }
    return !((done[dev >> 6] >> (dev & 63)) & 1ull);
  }
  void mark() { if (dev >= 0) done[dev >> 6] |= 1ull << (dev & 63); }
};

// ---- predict ---------------------------------------------------------------------
struct PredictParams {
  const double* Xq;        // [Q][d] queries, row-major (device)
  long long Q;
  int d;
  int N;                   // true number of training points
  int Npad;                // padded to a multiple of the variance kernel's BN
  const double* Xs;        // [d][Npad] training inputs, SoA, pre-scaled by sqrt(0.5/M_i), zero padded
  const double* alphaA;    // [Npad]  A * K^{-1}(y-m), zero padded
  const double* LinvF;     // fragment-tiled A * L^{-1} (see common.cuh)
  double* scratch;         // [grid][BM*Npad] per-CTA K* panels (L2-resident working set)
  double qscale[APGP_MAXD];
  double lo[APGP_MAXD];
  double hi[APGP_MAXD];
  int has_box;             // apply box prior gate lo <= q <= hi (utility -> +inf outside)
  double mean;             // constant mean m
  double amp;              // k** = A
  double* mu;              // [Q] out (may be null)
  double* var;             // [Q] out (may be null)
  double* util;            // [Q] out (may be null)
  int utility_kind;        // 0 none, 1 AGP, 2 BAPE, 3 Jones
  double ybest, zeta;
  int* grp_arrive;         // grouped kernel: [ngroups] arrival counters (zeroed per launch)
  double* grp_part;        // grouped kernel: [ngroups][2 (mu, ss)][2 buffers][Npad/64][256] per-block partial sums
  int* grp_plan;           // grouped kernel: work-split tables (plan_group_split), 4 x GROUP_MAX_BLOCKS ints
  const unsigned char* LinvI8;   // int8 engine: digit planes of A * L^{-1} (predict_i8.cu)
  const double* i8scale;   // int8 engine: [Npad] per-row scale of those digits
};

// grouped variance kernels: at most GROUP_MAX_BLOCKS 64-column blocks, Npad <= 8192
constexpr int GROUP_MAX_BLOCKS = 128;

// one-tile-per-CTA variance kernel: block-row height BN of its LinvF tiling (and the padding of Npad), from d
int predict_tile_bn(int d);

// returns cudaError_t as int; *launches incremented by the number of kernel launches issued
int launch_predict_var(const PredictParams& p, int num_sms, cudaStream_t st, int* launches);
// at most PREDICT_FEW_MAX queries: one CTA per query against the explicit row-major inverse (pure latency path)
constexpr long long PREDICT_FEW_MAX = 16;
size_t predict_few_ws_bytes();
int launch_predict_few(const PredictParams& p, const double* Linv, int ld, void* ws, cudaStream_t st, int* launches);
int launch_exp_neg_test(const double* s, int n, double* out, cudaStream_t st, int variant = 0);
int launch_predict_mean(const PredictParams& p, int num_sms, cudaStream_t st, int* launches);
size_t predict_scratch_bytes(int Npad, int num_sms, int d);
// What the group planner needs to know about a grouped kernel's tile
struct GroupTile {
  int bm;                  // queries per tile
  int panel_bytes;         // panel bytes per (query, training point)
  double phase1_scale;     // cost of building a 64-column panel block, relative to the DMMA tile's (plan_group_split)
  int max_d;               // largest input dimension the kernel takes
};
extern const GroupTile DMMA_GROUP_TILE;   // predict_var_group_kernel, 256 x 64 (predict.cu)
extern const GroupTile I8_GROUP_TILE;     // predict_var_i8_kernel, 128 x 64 (predict_i8.cu)
// grouped kernels: G CTAs share one query tile so the K* panels in flight stay in L2 (predict.cu).
// requested < 0: automatic choice; returns 1 when grouping is off / not applicable
int predict_group_size(int Npad, int num_sms, int requested, int d, long long Q, const GroupTile& tile);
void predict_group_plan(int Npad, int num_sms, int G, int d, int* tab /*[4 * GROUP_MAX_BLOCKS]*/, const GroupTile& tile);
size_t predict_group_scratch_bytes(int Npad, int num_sms, int G, const GroupTile& tile);
size_t predict_group_part_bytes(int Npad, int num_sms, int G);
int launch_predict_var_grouped(const PredictParams& p, int num_sms, int G, cudaStream_t st, int* launches);
// int8 tensor-core variance engine (grouped launch only): exact-integer split of the triangular product
bool predict_i8_fits(int Npad, int d);
size_t linv_i8_bytes(int Npad);
int launch_pack_linv_i8(const double* Linv, int ld, int N, int Npad, double amp, unsigned char* out, double* rowscale,
                        cudaStream_t st);
int launch_predict_var_i8(const PredictParams& p, int num_sms, int G, cudaStream_t st, int* launches);
int launch_pack_linv(const double* Linv, int ld, int N, int Npad, int BN, double amp, double* LinvF, cudaStream_t st);
int launch_pack_xs(const double* X, int N, int d, int Npad, const double* qscale_dev, double* Xs, cudaStream_t st);

// ---- factor (batched blocked Cholesky on 64x64 tiles) ------------------------------
struct FactorBatch {
  int R;                   // batch size (restarts); 1 for the single predict GP
  int N;                   // true size
  int Np;                  // padded to multiple of 64
  double* K;               // [R][Np][Np] row-major; lower triangle in/out (L on exit)
  double* Dinv;            // [R][Np/64][64][64] inverses of the diagonal blocks of L
  double* r;               // [R][Np] rhs (y - mean) in, z = L^{-1} r out
  double* logdet;          // [R] out: 2*sum(log L_ii)
  int* info;               // [R] out: 0 ok, k+1 = not positive definite at pivot k
};
// hyper[R][3 + d]: mean, amp, noise_var, invM_0..invM_{d-1}
int launch_build_K(const double* X, const double* y, int N, int d, const double* hyper, const FactorBatch& fb, cudaStream_t st);
int launch_cholesky(const FactorBatch& fb, int num_sms, cudaStream_t st, int* launches);
// explicit inverse of the lower-triangular factor (single matrix): Linv[Np][Np]
int launch_tri_inverse(const double* L, const double* Dinv, int Np, double* Linv, double* work, cudaStream_t st, int* launches);
// alpha = L^{-T} z  using the explicit inverse
int launch_linvT_matvec(const double* Linv, int Np, const double* z, double* alpha, cudaStream_t st);
int launch_loglik_finish(const FactorBatch& fb, double* ll, cudaStream_t st);
// one refinement step alpha += K^{-1}((y - m) - K alpha) through the explicit inverse, residual in double-double;
// w1, w2: [Np] work vectors
int launch_refine_alpha(const double* X, const double* y, int N, int d, int Np, const double* hyper_dev,
                        const double* Linv, double* alpha, double* w1, double* w2, cudaStream_t st, int* launches);
// bordered append of one training point to an existing factorisation (needs N + 1 <= Np)
int launch_append_point(const double* X, int N, int d, int Np, const double* xnew_dev, const double* hyper_dev, double kappa,
                        double rnew, double* L, double* Linv, double* z, double* alpha, double* kvec, double* lvec,
                        double* uvec, double* scal, int* status, cudaStream_t st, int* launches);
// batched log-likelihood of P [R][1 + fit_amp + d] (george order; noise = e^{white_noise} + TINY^2) by the evaluators of
// loglik.cuh, the same bits as the device optimisers' objective.  Small: one restart per CTA, everything in shared memory,
// usable when loglik_small_smem(N, d) <= 220 KB
size_t loglik_small_smem(int N, int d);
int launch_loglik_small(const double* X, const double* y, int N, int d, const double* P, int fit_amp, double noise, int R,
                        double* ll, double* grad /*[R][2+d] or null*/, cudaStream_t st);
// group: one CLUSTER per restart for larger N (chol_group.cuh), the matrix in L2-resident global workspace
int chol_group_cluster(int Np, int R, int num_sms);
size_t chol_group_ws_bytes(int Np, int R);
int launch_loglik_group(const double* X, const double* y, int N, int d, int Np, const double* P, int fit_amp, double noise,
                        int R, int num_sms, void* ws_bytes, double* ll, cudaStream_t st);
// the same with gradients (loglik_grad_group_kernel): grad [R][2 + d] = [sum alpha, d/dlog_constant, d/dlog M_0 ..], zeros
// where ll is -inf; the workspace adds the transposed inverse of L, alpha and the per-tile partials to the factorisation's
size_t loglik_grad_group_ws_bytes(int Np, int d, int R);
int launch_loglik_grad_group(const double* X, const double* y, int N, int d, int Np, const double* P, int fit_amp,
                             double noise, int R, int num_sms, void* ws_bytes, double* ll, double* grad, cudaStream_t st);
// gradient pieces: Kinv = Linv^T Linv (lower), then tr-products; grad_dev needs grad_loglik_doubles(Np, d) doubles
size_t grad_loglik_doubles(int Np, int d);
int launch_grad_loglik(const double* X, int N, int d, int Np, const double* Linv, const double* alpha,
                       const double* hyper_dev, int fit_amp, double* work /*[Np*Np]*/, double* grad_dev, cudaStream_t st,
                       int* launches);


// ---- device-resident optimisers (optimize.cu) ------------------------------------
struct OptimizeParams {
  int method;              // 0 Nelder-Mead, 1 Powell
  int adaptive;            // Nelder-Mead {"adaptive": True}
  double xtol, ftol;       // Nelder-Mead xatol/fatol, Powell xtol/ftol
  long long maxiter, maxfun;   // resolved by the caller with SciPy's default rules
};
struct UtilityPointParams {  // single-query predict + utility, read straight from the handle's factorisation
  int N, d, Npad, ldL;
  const double* Xs;        // [d][Npad] scaled SoA
  const double* alphaA;    // [Npad]
  const double* Linv;      // [ldL][ldL] row-major explicit L^{-1}
  double amp, mean, ybest, zeta;
  int kind;                // 1 AGP, 2 BAPE, 3 Jones, 4 -(mean)
  int has_box;
  double lo[APGP_MAXD], hi[APGP_MAXD], qscale[APGP_MAXD];
};
// mode 0: evaluate the objective at the R points; mode 1: minimise from the R starts (one CTA each).
// stats_dev [R][3] = (function evaluations, iterations, SM clock cycles) or null.
int launch_minimize_utility(const UtilityPointParams& u, const OptimizeParams& q, int R, const double* x0_dev,
                            double* x_out_dev, double* f_out_dev, long long* stats_dev, int mode, cudaStream_t st);
bool minimize_nll_fits(int N, int d, int P);
int read_prof(long long* out16);   // -DAPGP_PROF builds: per-phase cycle counters of the nll objective (zeros otherwise)
bool minimize_nll_group_fits(int P);
int launch_minimize_nll_group(const double* X_dev, const double* y_dev, int N, int d, int Np, int P, int fit_amp,
                              int default_prior, double noise, const OptimizeParams& q, int R, int num_sms, void* ws_bytes,
                              const double* p0_dev, double* p_out_dev, double* f_out_dev, long long* stats_dev, int mode,
                              cudaStream_t st);
int launch_minimize_nll(const double* X_dev, const double* y_dev, int N, int d, int P, int fit_amp, int default_prior,
                        double noise, const OptimizeParams& q, int R, const double* p0_dev, double* p_out_dev,
                        double* f_out_dev, long long* stats_dev, int mode, cudaStream_t st);

// ---- sampler ---------------------------------------------------------------------
struct SamplerParams {
  int nens, nwalk, d, nsteps, N, Npad;
  const double* Xs;        // [d][Npad] scaled SoA
  const double* alphaA;    // [Npad]
  double qscale[APGP_MAXD];
  double lo[APGP_MAXD], hi[APGP_MAXD];
  double mean;
  double lnprior_const;
  double a;                // stretch scale
  unsigned long long seed;
  const double* p0;        // [nens*nwalk][d]
  double* chain;           // [nsteps][nens*nwalk][d]
  double* logp;            // [nsteps][nens*nwalk]
  double* blob;            // [nsteps][nens*nwalk]
  int* naccept;            // [nens*nwalk]
  double* final_state;     // [nens*nwalk][d] (may be null)
  // replay buffers (all null => Philox); layout per ensemble e:
  const int* r_inds;       // [nens][nsteps][nwalk] colour 0/1
  const double* r_zz;      // [nens][nsteps][2][nwalk/2]
  const int* r_rint;       // [nens][nsteps][2][nwalk/2]
  const double* r_logu;    // [nens][nsteps][2][nwalk/2]
  int thin;                // store every `thin` steps (>=1)
  // a chain run as several launches (apgp_sampler_run pipelines the D2H of one piece under the next piece's kernel):
  // this launch covers steps [step_base, step_base + nsteps) of a chain of nsteps_total steps (0: nsteps) -- the
  // counter-based draws and the replay rows are indexed by the GLOBAL step, chain / logp / blob point at this piece's
  // first row, p0 is the previous piece's last stored row, naccept keeps counting (zeroed when step_base == 0)
  int step_base, nsteps_total;
};
int launch_sampler(const SamplerParams& p, cudaStream_t st, int* launches);

// ---- integrated autocorrelation time of a device-resident chain (autocorr.cu) -------
bool autocorr_fits(int n, int T);
size_t autocorr_partial_bytes(int W, int d, int T, int num_sms, int* G_out, int* nchunk_out);
int launch_autocorr(const double* chain, long long off, int thin, int n, int W, int d, int T, int num_sms, double* partial,
                    double* f_dev, cudaStream_t st, int* launches);

// ---- NCCL plumbing (comm.cu; NCCL bound at run time with dlopen) ---------------------
int comm_unique_id(char out[128]);
int comm_init(void** comm_out, const char id_bytes[128], int rank, int world);
int comm_destroy(void* comm);
int comm_broadcast_bytes(void* comm, void* buf_dev, size_t bytes, int root, cudaStream_t st);
int comm_allgather_doubles(void* comm, const double* send_dev, double* recv_dev, size_t count, cudaStream_t st);
int comm_group_start();
int comm_group_end();
const char* comm_last_error();

}  // namespace apgp
