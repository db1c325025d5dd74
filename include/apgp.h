/* libapgp -- C-ABI of the B200-native GP-surrogate engine behind approxposterior's hot path.
 *
 * Every entry point replaces one call the reference (dflemin3/approxposterior v0.4) makes into
 * george / emcee; the reference call site is cited on each declaration (paths relative to the
 * reference repo).  The reference has no FFI of its own (pure Python over george's pybind11
 * module), so this header *is* the boundary a maintainer would bind with ctypes -- see
 * INTEGRATION.md for the stub.
 *
 * Conventions
 *   - plain C: opaque handle, raw pointers + sizes, int status returns; no C++ types cross.
 *   - status 0 = ok; > 0 = data condition (APGP_NOT_POSDEF, ...); < 0 = CUDA/argument error, text
 *     via apgp_last_error().
 *   - all arrays are fp64, C-contiguous.  Arguments named *_dev are device pointers on the
 *     handle's device; `on_host` flags say whether bulk buffers are host (the library stages the
 *     H2D/D2H copies on the handle's stream) or device pointers.  Small parameter vectors
 *     (hyper-parameters, bounds) are always host pointers.
 *   - a handle is bound to one device and one stream; it is not thread-safe.
 *   - there is no CPU fallback: every function fails (status < 0) without a CUDA device.
 */
#ifndef APGP_H_
#define APGP_H_

#ifdef __cplusplus
extern "C" {
#endif

#define APGP_OK 0
#define APGP_NOT_POSDEF 1        /* covariance not positive definite (george: LinAlgError) */
#define APGP_NOT_COMPUTED 2      /* predict/log-likelihood before a successful factorisation */
#define APGP_NEEDS_REFACTOR 3    /* apgp_append_point: padded buffers are full, call set_training + factorize */
#define APGP_NEEDS_HOST 4        /* apgp_integrated_time: chain longer than one CTA's shared memory / window beyond 4096 lags;
                                    apgp_loglik_batch: gradients requested under a forced value-only kernel
                                    (APGP_LOGLIK_PATH = group | tiled) */
#define APGP_ERR_ARG (-1)
#define APGP_ERR_CUDA (-2)
#define APGP_ERR_NOMEM (-3)
#define APGP_ERR_COMM (-4)       /* NCCL could not be loaded / a collective failed */

#define APGP_MAX_DIM 32

#define APGP_UTIL_NONE 0
#define APGP_UTIL_AGP 1          /* utility.py:99-142  */
#define APGP_UTIL_BAPE 2         /* utility.py:145-189 */
#define APGP_UTIL_JONES 3        /* utility.py:192-250 */
#define APGP_UTIL_NEGMEAN 4      /* -(GP mean): findMAP's objective, approx.py:909-914 (apgp_minimize_utility only) */

typedef struct apgp_handle apgp_handle;

const char* apgp_last_error(void);
int apgp_version(void);

/* lifecycle -- george.GP(...) construction at gpUtils.py:176-177 and approx.py:712-715 */
int apgp_create(apgp_handle** out, int device);
int apgp_destroy(apgp_handle* h);
int apgp_set_stream(apgp_handle* h, void* cuda_stream);           /* cudaStream_t; NULL = library-owned stream */
/* Forget the training set, hyper-parameters and factorisation but keep every device buffer, the stream and the pinned
 * staging area: lets a caller that builds a fresh george.GP per design point (approx.py:712-717) recycle handles
 * instead of paying stream creation, cudaHostAlloc and a dozen cudaMallocs each time. */
int apgp_reset(apgp_handle* h);
int apgp_synchronize(apgp_handle* h);
long long apgp_launch_count(const apgp_handle* h);                /* kernels launched so far by this handle */

/* training set -- george.GP.compute(x) at gpUtils.py:178, approx.py:717 (x part) and the `y`
 * argument of predict/log_likelihood.  X is [N][d] row-major, y is [N]. */
int apgp_set_training(apgp_handle* h, const double* X, const double* y, int N, int d, int on_host);

/* hyper-parameters -- george.GP.set_parameter_vector(p) at gpUtils.py:74,243,253; approx.py:716.
 *   mean        constant mean (p[0])
 *   amp         effective kernel amplitude A = ndim*exp(log_constant), 1.0 without `a*kernel`
 *   log_metric  [d] log M_i, M_i the squared length scale of ExpSquaredKernel (gpUtils.py:160)
 *   white_noise frozen log-variance added to diag(K) (gpUtils.py:176-177; default -12) */
int apgp_set_hyper(apgp_handle* h, double mean, double amp, const double* log_metric, double white_noise);

/* factorise -- george.GP.compute/recompute (gpUtils.py:178,244,254; approx.py:717):
 * K = A exp(-1/2 r^2_M) + (e^{wn} + TINY^2) I ; blocked Cholesky; alpha; explicit L^{-1}.
 * Returns APGP_NOT_POSDEF (and *info = 1-based failing pivot) when K is not positive definite.
 * *logdet = log|K|, *loglik = log-likelihood of the stored y (george.GP.log_likelihood,
 * gpUtils.py:78,247); either may be NULL. */
int apgp_factorize(apgp_handle* h, double* logdet, double* loglik, int* info);

/* Append ONE training point (x_new [d], y_new; host) to the current factorisation with a bordered O(N^2)
 * update of L, L^-1, alpha, log|K| and the log-likelihood -- instead of the from-scratch refactorisation the
 * reference performs for every new design point (approx.py:693-717).  Hyper-parameters are unchanged.
 * Returns APGP_NEEDS_REFACTOR when the 64-padded buffers are full (caller re-uploads and factorises),
 * APGP_NOT_POSDEF when the bordered pivot is not positive. */
int apgp_append_point(apgp_handle* h, const double* x_new, double y_new, double* logdet, double* loglik);

typedef struct apgp_predict_opts {
  int want_var;                  /* 0: mean only (approx.py:178-180); 1: mean+variance (utility.py:131,178,224) */
  int utility;                   /* APGP_UTIL_*; needs want_var=1 */
  int has_box;                   /* 1: utility = +inf outside [lo,hi] (the priorFn gate, utility.py:126,173,219) */
  double lo[APGP_MAX_DIM];
  double hi[APGP_MAX_DIM];
  double ybest;                  /* Jones: max(y) (utility.py:232) */
  double zeta;                   /* Jones: exploration parameter (utility.py:192, default 0.01) */
} apgp_predict_opts;

/* batched george.GP.predict(y, Xq, return_cov=False, return_var=want_var) + utility epilogue.
 * Xq [Q][d]; mu/var/util [Q], each may be NULL.  on_host: Xq and outputs are host buffers. */
int apgp_predict(apgp_handle* h, const double* Xq, long long Q, double* mu, double* var, double* util,
                 const apgp_predict_opts* opts, int on_host);

/* george.GP.grad_log_likelihood(y, quiet=True) at gpUtils.py:110.  grad (host) has 1+fit_amp+d
 * entries ordered [mean, (log_constant), log M_0..]; zeros when the GP is not computed. */
int apgp_grad_log_likelihood(apgp_handle* h, int fit_amp, double* grad);

/* Batched log-likelihood for R hyper-parameter vectors at once -- what gpUtils._nll (gpUtils.py:46-80)
 * evaluates one at a time inside optimizeGP's restarts (gpUtils.py:223-247).
 * P_host [R][P], rows in george order [mean, (log_constant), log M_0 .. log M_{d-1}], P = 1+fit_amp+d.
 * ll_host [R]: log-likelihood, -inf when not positive definite / non-finite (quiet=True semantics).
 * grad_host [R][P] or NULL: gradient of the log-likelihood in the same parameter order (what gpUtils._grad_nll,
 * gpUtils.py:83-111, evaluates one vector at a time); zeros where ll is -inf.
 * Kernels (apgp_debug_last_loglik_path): one restart per CTA with everything in shared memory while
 * N(N+1)/2 + N(d+3) + d + 12 doubles fit 220 KB (N <= ~224); beyond, ONE launch of the fused cluster-per-vector kernel
 * (covariance build, look-ahead blocked Cholesky, reductions; csrc/chol_group.cuh), or for at most 8 vectors of
 * N > 1984 the multi-launch tiled sequence.  The first two return exactly -f of apgp_minimize_nll(default_prior=0).
 * With grad_host: the one-restart-per-CTA kernel while it fits, else ONE launch of the cluster-per-vector kernel with
 * gradients (the same factorisation, then L^-1, alpha and the trace products; its ll is the value kernel's bit for bit)
 * for every larger N, few large matrices included.
 * APGP_LOGLIK_PATH = small | group | tiled overrides the choice of value kernel; group_grad forces the cluster kernel with
 * gradients at any N (group for value-only calls).  Gradients under a forced group or tiled kernel return
 * APGP_NEEDS_HOST (use apgp_grad_log_likelihood per vector).
 * Does not disturb the handle's current factorisation. */
int apgp_loglik_batch(apgp_handle* h, const double* P_host, int R, int P, int fit_amp, double white_noise,
                      double* ll_host, double* grad_host);

typedef struct apgp_sampler_opts {
  int nens;                      /* independent ensembles */
  int nwalkers;                  /* walkers per ensemble (even, >= 2) */
  int nsteps;
  int thin;                      /* store every thin-th step (>= 1) */
  double a;                      /* stretch scale (emcee default 2.0) */
  unsigned long long seed;       /* Philox key */
  double lo[APGP_MAX_DIM];       /* box prior (approx.py:171-173 with a uniform lnprior) */
  double hi[APGP_MAX_DIM];
  double lnprior_const;          /* value stored in the "lnprior" blob for accepted points */
  /* optional replay of recorded draws (all NULL => Philox); host or device like the bulk buffers:
   * inds [nens][nsteps][nwalkers] int32, zz/logu [nens][nsteps][2][nwalkers/2] fp64, rint same shape int32 */
  const int* replay_inds;
  const double* replay_zz;
  const int* replay_rint;
  const double* replay_logu;
} apgp_sampler_opts;

/* emcee.EnsembleSampler(nwalkers, ndim, log_prob_fn=_gpll).sample(initial_state, iterations)
 * as driven from approx.py:839-847.  p0 [nens*nwalkers][d];
 * chain [nsteps/thin][nens*nwalkers][d], logp/blob [nsteps/thin][nens*nwalkers], naccept [nens*nwalkers] int32.
 * One CTA per ensemble, or -- few ensembles with enough work per half-step -- a thread-block cluster of 2/4/8 CTAs
 * per ensemble (same chains bit for bit).  nwalkers * (24 ndim + 72) bytes must fit one CTA's shared memory.
 * on_host=1 with more than 4 MB of results: the chain runs as up to 8 launches (whole stored rows each; the kernel
 * resumes from the previous piece's last stored row, draws indexed by the global step: the same chain bit for bit) and
 * the rows of one piece cross PCIe while the next piece samples.  APGP_SAMPLER_PIECES=k overrides (1: one launch). */
int apgp_sampler_run(apgp_handle* h, const apgp_sampler_opts* opts, const double* p0, double* chain, double* logp,
                     double* blob, int* naccept, int on_host);

/* ---- multi-GPU: one handle per GPU, NCCL over NVLink / NVSwitch (bound at run time: dlopen libnccl.so.2) ----------
 * The path shards by independent units (queries / ensembles / restarts: SURVEY 8e), so the only exchanges are the
 * replication of a factorised GP and the concatenation of per-rank results -- what a multi-process driver around
 * approx.py:664-672 (candidate scores), :839-847 (chains) and gpUtils.py:223-254 (restart results) needs.
 *   apgp_comm_unique_id      rank 0 creates the 128-byte NCCL id; the caller distributes it (file, MPI, TCP store)
 *   apgp_comm_init           ncclCommInitRank on the handle's device (collective over all `world` handles; several
 *                            handles of ONE process must be initialised between apgp_comm_group_start/_end)
 *   apgp_comm_broadcast_factor  replicate the root's factorisation (training set, hyper-parameters, L, L^-1, alpha,
 *                            log-likelihood) into every other handle, which then predicts / samples without having
 *                            factorised: <= 2 Np^2 doubles over NVLink instead of an O(N^3) refactorisation per GPU
 *   apgp_comm_allgather      recv[world][count] <- every rank's send[count] (rank order); host or device buffers */
int apgp_comm_unique_id(char id_out[128]);
int apgp_comm_init(apgp_handle* h, const char id[128], int rank, int world);
int apgp_comm_destroy(apgp_handle* h);
int apgp_comm_group_start(void);
int apgp_comm_group_end(void);
int apgp_comm_broadcast_factor(apgp_handle* h, int root);
int apgp_comm_allgather(apgp_handle* h, const double* send, double* recv, long long count, int on_host);

/* emcee.EnsembleSampler.get_autocorr_time(discard, thin, c, tol=0) / thin, as mcmcUtils.estimateBurnin calls it
 * (mcmcUtils.py:198; approx.py:853): integrated autocorrelation time per dimension of chain [n_total][W][d] restricted to
 * chain[discard + thin - 1 :: thin] -- walker-averaged normalised autocorrelation, Sokal window with constant c
 * (emcee: 5).  The chain may stay where apgp_sampler_run(on_host=0) left it: nothing but d x T doubles crosses PCIe.
 * tau_out [d] (host), window_out [d] (host, may be NULL).  Returns APGP_NEEDS_HOST when the series does not fit one
 * CTA's shared memory (n > ~27 000 samples) or the window lies beyond 4096 lags. */
int apgp_integrated_time(apgp_handle* h, const double* chain, long long n_total, int W, int d, long long discard, int thin,
                         double c, int on_host, double* tau_out, int* window_out);

/* ---- device-resident local optimisers: one CTA per start, the whole multistart in ONE launch ----------------- */
#define APGP_OPT_NELDER_MEAD 0
#define APGP_OPT_POWELL 1
typedef struct apgp_opt_opts {
  int method;                    /* APGP_OPT_* : scipy.optimize.minimize(method="nelder-mead" | "powell") */
  int adaptive;                  /* Nelder-Mead options={"adaptive": True} (utility.py:307-308) */
  double xtol, ftol;             /* Nelder-Mead xatol/fatol, Powell xtol/ftol (SciPy default 1e-4 each) */
  long long maxiter, maxfev;     /* < 0: None (SciPy's default rule: N*200 / N*1000); >= 2^62: inf */
} apgp_opt_opts;

/* utility.minimizeObjective's inner loop (utility.py:332-371): scipy.optimize.minimize(fn, x0[r], method=...)["x"]
 * for R starts at once on the current factorisation.  fn = obj->utility in {AGP, BAPE, JONES} evaluated as
 * utility.py:99-250 does (single-query predict with variance + epilogue; +inf outside obj's box when has_box,
 * the priorFn gate), or NEGMEAN = -(GP mean) with the same gate (findMAP, approx.py:909-914).
 * x0, x_out [R][d], f_out [R] = fn(x_out[r]); stats [R][3] or NULL = (function evaluations, optimiser iterations,
 * SM clock cycles spent by that start's CTA); all host buffers.  evaluate_only=1 returns
 * fn(x0[r]) without optimising (x_out = x0): the exact function the optimiser minimises, for tests. */
int apgp_minimize_utility(apgp_handle* h, const apgp_predict_opts* obj, const apgp_opt_opts* opt, const double* x0,
                          int R, double* x_out, double* f_out, long long* stats, int evaluate_only);

/* gpUtils.optimizeGP's inner loop (gpUtils.py:223-247): scipy.optimize.minimize(_nll, p0[r], method=...)["x"] for
 * R restarts at once; _nll as gpUtils.py:46-80 (+inf when default_prior and any |p[1:]| > 20 -- gpUtils.py:22-43 --,
 * when the covariance is not positive definite or the likelihood is not finite).  Rows in george order
 * [mean, (log_constant), log M_0..], P = 1 + fit_amp + d.  apgp_minimize_nll_fits() says which kernel runs: 1 = one
 * restart per CTA with everything in shared memory (N <= ~220), 2 = one thread-block CLUSTER per restart with the
 * matrix in L2-resident global memory (N <= 4096; optimiser state replicated in every CTA of the cluster), 0 = too
 * large: drive apgp_loglik_batch from a host optimiser.  Does not disturb the handle's current factorisation. */
int apgp_minimize_nll(apgp_handle* h, const apgp_opt_opts* opt, const double* p0, int R, int P, int fit_amp,
                      double white_noise, int default_prior, double* p_out, double* f_out, long long* stats,
                      int evaluate_only);
int apgp_minimize_nll_fits(const apgp_handle* h, int P);

/* test/diagnostic accessors (host outputs): alpha [N], Linv [N][N] row-major (lower), L likewise */
int apgp_get_alpha(apgp_handle* h, double* alpha);
int apgp_get_linv(apgp_handle* h, double* linv);
int apgp_get_chol(apgp_handle* h, double* L);
/* exp(-s), s >= 0, as evaluated inside the fused predict kernel (table + degree-5 polynomial); host buffers */
int apgp_debug_exp_neg(apgp_handle* h, const double* s, int n, double* out);
/* the 256-entry-table / degree-4 form used by the sampler and the mean-only predict kernel */
int apgp_debug_exp_neg256(apgp_handle* h, const double* s, int n, double* out);
/* host-only planning of the grouped variance kernel for a training set of N points on a GPU with num_sms SMs and a
 * call of Q queries: *G_out = CTAs per query tile (requested: -1 automatic, else as apgp_set_group); tab512 (may be NULL)
 * receives [full group | last group] x [owner of block-row ib | owner of panel column block cb] x 128 ints. */
int apgp_debug_group_plan(int N, int num_sms, int d, long long Q, int requested, int* G_out, int* tab512);
/* kernel of the handle's last predict call with variances: 0 none yet, 1 few-query kernel, 2 one-tile DMMA kernel (also
 * the fallback when the cooperative grouped launch does not fit), 3 grouped DMMA kernel, 4 grouped int8 kernel */
int apgp_debug_last_var_path(const apgp_handle* h, int* path);
/* kernel of the handle's last apgp_loglik_batch call: 0 none yet, 1 one restart per CTA (with or without gradients),
 * 2 one cluster per restart, 3 multi-launch tiled sequence, 4 one cluster per restart with gradients (every batched
 * gradient call above the one-CTA class; a call that returned APGP_NEEDS_HOST leaves the previous value) */
int apgp_debug_last_loglik_path(const apgp_handle* h, int* path);
/* the int8 engine's operands as the kernel reads them (host outputs, each may be NULL): linv_i8 the digit planes of
 * amp * L^-1 (nblk (nblk + 1) / 2 * 28672 bytes, nblk = Npad / 64), rowscale the Npad row scales 2^(ex_i - 38) (0 for
 * padding rows), panel the digit panel of the first 128-query tile of the last call (128 * 7 * Npad bytes; only when
 * that call ran on the int8 kernel), *npad the padded training-set size.  APGP_ERR_ARG when the operands are not
 * packed, or a panel is asked for and the last variance call did not run on the int8 kernel. */
int apgp_debug_i8_operands(apgp_handle* h, unsigned char* linv_i8, double* rowscale, unsigned char* panel, int* npad);
/* run the int8 engine's operand pack on the lower triangle of the host n x n matrix M (n <= 8192, padded to a multiple
 * of 64 as Npad): out and rowscale receive what apgp_debug_i8_operands returns for a factorisation with L^-1 = M */
int apgp_debug_pack_linv_i8(apgp_handle* h, const double* M, int n, double amp, unsigned char* out, double* rowscale);
/* profiling builds (-DAPGP_PROF): read and reset 16 per-phase SM-cycle counters of the log-likelihood objective */
int apgp_debug_read_prof(long long* out16);
/* CTAs that share one query tile in the 256x64 variance kernel (their K* panels then stay in L2 instead of streaming
 * through HBM): 0 = one tile per CTA, -1 = automatic (by training-set size, and by the number of query tiles of the
 * call: a few-tile call is spread over more CTAs for latency), 2..64 = fixed group size.  Default -1. */
int apgp_set_group(apgp_handle* h, int group);
/* engine of the variance product in grouped predict calls: APGP_VAR_ENGINE_I8 (default) runs it on the int8 tensor
 * cores as an exact-integer split of the FP64 operands, at N >= 1024 where that is faster; APGP_VAR_ENGINE_DMMA keeps
 * the FP64 tensor-core kernel everywhere.  The mean is bit-identical between the two.  Environment:
 * APGP_PREDICT_VAR_ENGINE=i8|dmma, read by apgp_create / apgp_reset. */
#define APGP_VAR_ENGINE_DMMA 0
#define APGP_VAR_ENGINE_I8 1
int apgp_set_var_engine(apgp_handle* h, int engine);
/* predict calls of at most 16 queries (the reference asks for ONE point per call: utility.py:131,178,224) run a few-query
 * kernel -- several CTAs per query against the explicit inverse -- instead of a 256-query tile of the DMMA kernels:
 * enable != 0 (default) / 0 = always the tiled kernels.  Environment: APGP_PREDICT_FEW, read by apgp_create / apgp_reset. */
int apgp_set_predict_few(apgp_handle* h, int enable);

#ifdef __cplusplus
}
#endif
#endif /* APGP_H_ */
