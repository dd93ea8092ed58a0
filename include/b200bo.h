/*
 * b200bo.h - C ABI of the B200-native GP-surrogate + acquisition engine.
 *
 * This is the drop-in boundary for ONE hot path of bayesian-optimization/BayesianOptimization
 * (v3.3.0): GP fit at given hyper-parameters -> batched posterior predict -> acquisition ->
 * argmin/top-k.  The reference has no FFI; its plugin surface is Python duck-typing on
 * sklearn's GaussianProcessRegressor and bayes_opt.acquisition.AcquisitionFunction
 * (SURVEY.md section 8b).  Every entry point below names the reference code it replaces
 * (R/ = /root/reference/, SK/ = site-packages/sklearn/).  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *  - plain pointers and sizes only; all matrices are row-major (C order) IEEE fp64, exactly
 *    the numpy arrays the reference passes around.
 *  - "host" entry points take HOST buffers and do their own H2D/D2H copies (synchronous).
 *    "_dev" entry points take DEVICE pointers and a cudaStream_t (as void*) and are
 *    asynchronous w.r.t. the host unless stated.
 *  - every function returns B200BO_OK (0) or a negative error code; b200bo_last_error()
 *    returns a thread-local message.  There is NO CPU fallback anywhere behind this ABI:
 *    without a CUDA device every compute entry point returns B200BO_ERR_CUDA.
 */
#ifndef B200BO_H
#define B200BO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200BO_VERSION 200 /* 0.2.0 */

/* error codes */
#define B200BO_OK 0
#define B200BO_ERR_CUDA (-1)       /* CUDA runtime failure / no device */
#define B200BO_ERR_ARG (-2)        /* invalid argument */
#define B200BO_ERR_NOT_PD (-3)     /* kernel matrix not positive definite (np.linalg.LinAlgError) */
#define B200BO_ERR_UNSUPPORTED (-4)/* kernel / option outside the supported set (NotImplementedError) */
#define B200BO_ERR_STATE (-5)      /* handle not fitted */

/* kernel families: SK/gaussian_process/kernels.py Matern (:1685-1786), RBF (:1530-1587) */
#define B200BO_KERNEL_MATERN 0
#define B200BO_KERNEL_RBF 1
/* Matern smoothness codes */
#define B200BO_NU_05 0
#define B200BO_NU_15 1
#define B200BO_NU_25 2
#define B200BO_NU_INF 3

/* acquisition kinds: R/bayes_opt/acquisition.py:485 (UCB), :847-849 (EI), :660-661 (PoI) */
#define B200BO_ACQ_UCB 0
#define B200BO_ACQ_EI 1
#define B200BO_ACQ_POI 2
#define B200BO_ACQ_NONE 3 /* predict only: no acquisition epilogue */

#define B200BO_MAX_GPS 8   /* 1 target GP + up to 7 constraint GPs per call */
#define B200BO_MAX_DIM 64  /* max input dimension d */
#define B200BO_MAX_TOPK 64 /* max n_smart seeds returned by argmin_topk */

/* per-dimension input transforms of bayes_opt.parameter.wrap_kernel
 * (R/bayes_opt/parameter.py:484-487): identity for floats (:222-234), np.round for ints (:308-320) */
#define B200BO_XFORM_IDENTITY 0
#define B200BO_XFORM_ROUND 1

typedef struct b200bo_gp b200bo_gp; /* opaque: one GP's device-resident factorisation */

/* kernel hyper-parameters: const_value * k(x/length_scale, x'/length_scale) [+ noise_level * delta(x, x')]
 * (ConstantKernel * {Matern,RBF} [+ WhiteKernel]; const_value = 1 for a bare kernel, noise_level = 0 without a
 * WhiteKernel term, SK/gaussian_process/kernels.py:1205-1330: the term adds noise_level to the diagonal of K(X,X)
 * and to the prior variance kernel_.diag(X*), and nothing to K(X*,X)). */
typedef struct {
    int32_t family;            /* B200BO_KERNEL_* */
    int32_t nu;                /* B200BO_NU_* (ignored for RBF) */
    int32_t n_length_scale;    /* 1 (isotropic) or d (anisotropic) */
    int32_t reserved;
    double const_value;        /* ConstantKernel factor; 1.0 when absent */
    const double* length_scale;/* host pointer, n_length_scale entries */
    double noise_level;        /* WhiteKernel term; 0.0 when absent */
} b200bo_kernel;

/* One acquisition evaluation: the closure built by AcquisitionFunction._get_acq
 * (R/bayes_opt/acquisition.py:171-219):  -base_acq(mu, sigma) [* prod_j p_j(x)]. */
/* Which kernels evaluate a batch.  AUTO: the tiled persistent kernel or the small-batch kernels, chosen
 * from the batch size m.  STABLE: chosen from the model size only - an optimiser's objective f(x) and its
 * finite-difference stencil f(x + h e_i) arrive as batches of different sizes and must be summed in the same
 * order (SP/optimize/_numdiff.py forms (f(x+h) - f(x)) / 1.5e-8). */
#define B200BO_PATH_AUTO 0
#define B200BO_PATH_STABLE 1

typedef struct {
    int32_t kind;              /* B200BO_ACQ_* */
    int32_t n_gps;             /* 1 + number of constraint GPs */
    int32_t path;              /* B200BO_PATH_* */
    int32_t reserved;
    double kappa;              /* UCB */
    double xi;                 /* EI / PoI */
    double y_max;              /* EI / PoI */
    b200bo_gp* gps[B200BO_MAX_GPS]; /* gps[0] = target GP; gps[1..] = ConstraintModel GPs */
    double lb[B200BO_MAX_GPS]; /* lb[j], ub[j] for gps[j] (j >= 1); +-inf allowed */
    double ub[B200BO_MAX_GPS]; /* (R/bayes_opt/constraint.py:200-221) */
} b200bo_acq;

/* ---- library / device ---------------------------------------------------------------- */
int b200bo_version(void);
const char* b200bo_last_error(void);
int b200bo_device_count(void);
/* number of kernel launches issued by this library in this process so far (bench.py's
 * gpu_launches claim is the difference across the timed region). */
int64_t b200bo_launch_count(void);

/* ---- GP handle ------------------------------------------------------------------------ */
int b200bo_gp_create(b200bo_gp** out, int device);
void b200bo_gp_destroy(b200bo_gp* gp);

/* Arithmetic of the N^2 term (V = L^-1 K*^T and sum V^2) in the fused predict/acquisition kernel:
 *   B200BO_PRECISION_FP64  exact fp64 (mma.sync f64 / DFMA); parity bar 1e-5 (default)
 *   B200BO_PRECISION_FP32  "fp32 mode": 3xTF32 on tcgen05 tensor cores, fp32 accumulate in TMEM;
 *                          K*, the mean and the acquisition epilogue stay fp64; tolerance 1e-3.
 * A call uses the precision of gps[0].  (BASELINE configs[2]: fp32 vs fp64 tolerance.) */
#define B200BO_PRECISION_FP64 0
#define B200BO_PRECISION_FP32 1
int b200bo_gp_set_precision(b200bo_gp* gp, int precision);

/* enable != 0: the handle's fit-side work (set_data / fit / lml) is issued on a CUDA stream of its own
 * instead of the legacy default stream, so that several handles driven from different host threads
 * factorise concurrently - the independent L-BFGS-B restarts of the hyper-parameter search
 * (SK/gaussian_process/_gpr.py:321-340 runs them one after the other).  Every entry point still returns
 * with its results complete; handles are not thread-safe individually (one thread per handle). */
int b200bo_gp_set_private_stream(b200bo_gp* gp, int enable);

/* Optional per-dimension input transform (wrap_kernel); xform has d entries or NULL. Must be
 * set before fit.  Replaces R/bayes_opt/parameter.py:484-487 for float/int parameters. */
int b200bo_gp_set_transform(b200bo_gp* gp, const int32_t* xform, int d);

/* Replaces the tail of GaussianProcessRegressor.fit (SK/gaussian_process/_gpr.py:275-285,
 * :349-367): y normalisation, K = k(X,X), K_ii += alpha, L = chol(K), alpha_ = K^-1 y, plus
 * the triangular inverse L^-1 the predict kernel streams.  X: (n,d) host, y: (n,) host.
 * Returns B200BO_ERR_NOT_PD when the factorisation meets a non-positive pivot; *info (nullable)
 * then receives the 1-based pivot index (LAPACK dpotrf convention). */
int b200bo_gp_fit(b200bo_gp* gp, const double* X, const double* y, int64_t n, int d,
                  const b200bo_kernel* kern, double alpha, int normalize_y, int64_t* info);

/* Incremental factor update (no counterpart in the reference, which always re-factorises:
 * R/bayes_opt/acquisition.py:84, :1130-1135): append ONE training point at the hyper-parameters of
 * the last b200bo_gp_fit in O(N^2) - new row of K, L (pivot checked) and L^-1, new y statistics and
 * alpha_.  Results equal a from-scratch fit on the extended data to round-off.  Returns
 * B200BO_ERR_STATE when the padded capacity is exhausted (caller refits), B200BO_ERR_NOT_PD as fit. */
int b200bo_gp_append(b200bo_gp* gp, const double* x_new, double y_new, int64_t* info);

/* Replaces GaussianProcessRegressor.log_marginal_likelihood(theta, eval_gradient)
 * (SK/gaussian_process/_gpr.py:541-656) on the training set of the last b200bo_gp_set_data /
 * b200bo_gp_fit call.  grad (nullable) receives d LML / d log(theta): [log const_value if
 * has_const & 1], then log length_scale (1 or d entries), then [log noise_level if has_const & 2].
 * Non-PD -> *lml = -inf, grad = 0 (as :590-593) and the call still returns B200BO_OK. */
int b200bo_gp_set_data(b200bo_gp* gp, const double* X, const double* y, int64_t n, int d,
                       int normalize_y);
int b200bo_gp_lml(b200bo_gp* gp, const b200bo_kernel* kern, double alpha, int has_const,
                  double* lml, double* grad);

/* Read back fitted state (tests / sklearn attribute parity: L_, alpha_, _y_train_mean/_std). */
#define B200BO_GET_L 0        /* (n,n) lower Cholesky factor, upper triangle zero */
#define B200BO_GET_ALPHA 1    /* (n,) alpha_ */
#define B200BO_GET_YSTATS 2   /* (2,) y_mean, y_std */
#define B200BO_GET_K 3        /* (n,n) K + alpha*I */
#define B200BO_GET_LINV 4     /* (n,n) L^-1 (lower) */
int b200bo_gp_get(b200bo_gp* gp, int what, double* out, int64_t len);
int64_t b200bo_gp_n(const b200bo_gp* gp);
int b200bo_gp_dim(const b200bo_gp* gp);

/* ---- predict / acquisition: HOST buffers --------------------------------------------- */
/* Replaces GaussianProcessRegressor.predict(X, return_std) (SK/gaussian_process/_gpr.py:446-500).
 * Xc: (m,d) host; mu: (m,) host; sd: (m,) host or NULL (mean only); n_clamped (nullable)
 * receives the number of negative variances set to 0 (the reference warns, :485-491). */
int b200bo_gp_predict(b200bo_gp* gp, const double* Xc, int64_t m, double* mu, double* sd,
                      int64_t* n_clamped);

/* Replaces GaussianProcessRegressor.predict(X, return_cov=True) (SK/gaussian_process/_gpr.py:464-475):
 * cov = (K(X*,X*) - V^T V) * y_std^2 with V = L^-1 K*^T.  mu: (m,), cov: (m,m) host.  1 <= m <= 16384.
 * The only caller in the reference is BayesianOptimization.predict (R/bayes_opt/bayesian_optimization.py:238). */
int b200bo_gp_predict_cov(b200bo_gp* gp, const double* Xc, int64_t m, double* mu, double* cov);

/* Replaces the closure returned by AcquisitionFunction._get_acq (R/bayes_opt/acquisition.py:
 * 171-219) incl. ConstraintModel.predict (R/bayes_opt/constraint.py:153-221):
 * acq_neg[i] = -base_acq(mu_i, sigma_i) * prod_j p_j(x_i).  Xc: (m,d) host, acq_neg: (m,) host. */
int b200bo_acq_eval(const b200bo_acq* spec, const double* Xc, int64_t m, double* acq_neg);

/* Replaces AcquisitionFunction._random_sample_minimize's evaluation + selection
 * (R/bayes_opt/acquisition.py:311-317): evaluates the closure on Xc and returns
 *   best_idx/best_val = np.argmin semantics (first NaN wins; ties -> lowest index),
 *   topk_idx/topk_val = the k smallest in (value, index) order, NaN last (np.argsort order).
 * acq_neg (nullable) additionally receives all m values.  The values are NOT materialised otherwise: every CTA of the
 * fused kernel keeps its k best (key, index) pairs and a small kernel merges the lists.  Batches of >= 2 chunks
 * (8 x 128 x #SM rows) are uploaded chunk by chunk on a copy stream behind the kernel.  A NaN / inf candidate coordinate
 * is detected where the kernels read it and reported as B200BO_ERR_ARG ("Input X contains NaN or infinity.", what
 * sklearn's validate_data raises on the reference path); the same holds for b200bo_acq_eval / b200bo_gp_predict. */
int b200bo_acq_argmin_topk(const b200bo_acq* spec, const double* Xc, int64_t m, int k,
                           double* best_val, int64_t* best_idx, double* topk_val,
                           int64_t* topk_idx, double* acq_neg);

/* ---- predict / acquisition: DEVICE buffers (candidates resident in HBM) --------------- */
/* d_Xc: (m,d) device fp64.  d_acq_neg, d_mu, d_sd: (m,) device or NULL.
 * If k > 0: d_sel receives (k+1) records {double value; int64 index}: record 0 = argmin,
 * records 1..k = top-k (device memory, 16*(k+1) bytes).  index_base is added to every index
 * (global index of this shard's first candidate).  stream: cudaStream_t. */
int b200bo_acq_eval_dev(const b200bo_acq* spec, const double* d_Xc, int64_t m,
                        double* d_acq_neg, double* d_mu, double* d_sd, int k, void* d_sel,
                        int64_t index_base, void* stream);

/* ---- throughput mode: device-side candidate source ------------------------------------ */
/* The reference draws the M candidates on the host (TargetSpace.random_sample, R/bayes_opt/target_space.py:
 * 565-603: column j = rng.uniform(lo_j, hi_j, M) from MT19937) - ~10^8 doubles/s, slower than the fp32-mode
 * kernel consumes them.  In throughput mode candidate i, column j is  lo_j + (hi_j - lo_j) * u,  u the 53-bit
 * uniform from Philox4x32-10 with counter (i + index_base, j/2) and key `seed`, generated INSIDE the fused
 * kernel: the candidate matrix never exists in host memory or HBM.  Rows depend only on (seed, global index),
 * so results are identical for any tiling and any number of GPUs.  This is an opt-in mode: it does not
 * reproduce the reference's RNG stream (parity mode = the host entry points above).
 * lo, hi: (d,) host.  best_x: (d,), topk_x: (k,d) host - the winners' coordinates, regenerated on the device. */
int b200bo_acq_argmin_topk_philox(const b200bo_acq* spec, uint64_t seed, const double* lo, const double* hi,
                                  int64_t m, int64_t index_base, int k, double* best_val, int64_t* best_idx,
                                  double* best_x, double* topk_val, int64_t* topk_idx, double* topk_x);
/* Device-resident flavour: only the (k+1) selection records are produced (d_sel as in b200bo_acq_eval_dev). */
int b200bo_acq_select_philox_dev(const b200bo_acq* spec, uint64_t seed, const double* lo, const double* hi,
                                 int64_t m, int64_t index_base, int k, void* d_sel, void* stream);
/* Rows of the Philox candidate matrix for given global indices (idx < 0 -> NaN row).  out: (n_idx, d) host. */
int b200bo_philox_rows(int device, uint64_t seed, const double* lo, const double* hi, int d,
                       const int64_t* idx, int64_t n_idx, double* out);

/* ---- multi-GPU (one process, several devices of one box) -------------------------------- */
/* SURVEY.md 8e: candidates are independent given the model, so a batch shards by rows over G devices, the
 * O(N^2) model state is replicated, and ONE exchange merges the per-device (argmin, top-k) records:
 * an ncclAllGather of (k+1) 16-byte records per device over NVLink (communicators from ncclCommInitAll,
 * created on first use for a device list and cached), then a merge kernel on device 0.  The reference has no
 * counterpart (single process, single thread: R/bayes_opt/acquisition.py:274-320).
 *
 * b200bo_gp_replicate: copy the fitted state of `src` (what predict needs: scaled X, L^-1, alpha_, statistics)
 * to a new handle on `device` with peer copies - no re-factorisation.  The replica is predict-only. */
int b200bo_gp_replicate(const b200bo_gp* src, int device, b200bo_gp** out);
/* specs[g] is the acquisition on device g (its gps[] are handles living on ONE device; all specs describe the
 * same model).  Rows [m*g/G, m*(g+1)/G) go to device g (remainder to the low devices); results as
 * b200bo_acq_argmin_topk with GLOBAL row indices - bit-identical to the single-device call. */
int b200bo_multi_gpu_acq_argmin_topk(const b200bo_acq* specs, int n_dev, const double* Xc, int64_t m, int k,
                                     double* best_val, int64_t* best_idx, double* topk_val,
                                     int64_t* topk_idx);
int b200bo_multi_gpu_acq_argmin_topk_philox(const b200bo_acq* specs, int n_dev, uint64_t seed, const double* lo,
                                            const double* hi, int64_t m, int64_t index_base, int k,
                                            double* best_val, int64_t* best_idx, double* best_x,
                                            double* topk_val, int64_t* topk_idx, double* topk_x);
/* Closure values for a batch split over the devices: rows [offsets[g], offsets[g+1]) on device g
 * (offsets: (n_dev+1,) host, or NULL for an even split).  Used by the lockstep L-BFGS-B driver to run seed r's
 * requests on device r mod G (R/bayes_opt/acquisition.py:364-374).  No collective. */
int b200bo_multi_gpu_acq_eval(const b200bo_acq* specs, int n_dev, const double* Xc, int64_t m,
                              const int64_t* offsets, double* acq_neg);

/* Duration (ms) of the most recent fused predict+acquisition kernel launched through a
 * device or host entry point on this thread, measured with CUDA events on its stream.
 * Synchronises on the stop event. */
int b200bo_last_kernel_ms(float* ms);
/* Work of the most recent fused predict+acquisition call on this thread (all chunks of a streamed host batch):
 * *screened = candidates that went through the screen of the pruned selection (0 when the call was not
 * pruned), *evaluated = candidates that went through the full L^-1 K*^T product (pilot + survivors when pruned,
 * else all of them).  Synchronises on the call's stop event. */
int b200bo_last_select_stats(int64_t* screened, int64_t* evaluated);

#ifdef __cplusplus
}
#endif
#endif /* B200BO_H */
