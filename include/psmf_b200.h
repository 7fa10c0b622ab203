/*
 * psmf_b200.h -- C ABI of the B200-native PSMF / rPSMF per-timestep filter.
 *
 * This is the drop-in boundary for the reference's filter hot path.  The
 * reference (alan-turing-institute/rPSMF) has no FFI of its own: its boundary
 * is two Python surfaces, which the package rpsmf_b200/ re-creates on top of
 * this library through ctypes (see INTEGRATION.md):
 *
 *   flat model functions   ExperimentImpute/rPSMF.py:39-148  robust_PSMF(...)
 *                          ExperimentImpute/PSMF.py:39-95    ProbabilisticSequentialMatrixFactorizer(...)
 *   class surface          pypsmf/psmf/psmf.py:14-248,275-331   PSMFIter, PSMFRecursive
 *                          pypsmf/psmf/rpsmf.py:11-184,187-334  rPSMFIter, rPSMFIterMissing, rPSMFRecursive
 *
 * Conventions
 *   - every buffer is a CALLER-OWNED DEVICE pointer (e.g. torch tensor
 *     data_ptr()); the library never frees it.  The library owns only its
 *     workspace (tiled copy of C, reduction scratch, NVLink mailboxes).
 *   - all functions return 0 on success, <0 on error (PSMF_E_*); the text of the
 *     last error of a handle is available from psmf_last_error().  Nothing
 *     throws or exits across the ABI.
 *   - one host thread per handle.  Kernels are enqueued on the caller's stream
 *     (a cudaStream_t passed as void*); psmf_run does not synchronise.
 *   - small state (x, P, V, Q, theta, rho, lambda) is always float64.  `dtype`
 *     selects the storage type of C, Y and Yrec (f64 or f32); all reductions
 *     and the r x r solves are float64 in both modes.
 */
#ifndef PSMF_B200_H
#define PSMF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct psmf_engine* psmf_handle;

#define PSMF_MAX_RANK 16
#define PSMF_MAX_PEERS 8
#define PSMF_MAILBOX_BLOB_BYTES 128   /* psmf_mailbox_export: 64-byte CUDA IPC handle + 64-byte plan record */

/* storage dtype of C / Y / Yrec */
#define PSMF_F64 0
#define PSMF_F32 1

/* flags */
#define PSMF_ROBUST        1   /* rPSMF: Student-t scales omega/phi, Q,R,lambda evolve (rPSMF.py:105,112-115,133-135) */
#define PSMF_SIMPLIFIED    2   /* ExperimentSynthetic overrides: P_bar=P, eta=tr(R)/d, x_t=x_bar (synthetic_psmf.py:78-100) */
#define PSMF_CUPDATE_VT    4   /* C += e (V x)'/N  (rPSMF.py:111, psmf.py:132); unset: C += e (V' x)'/N (PSMF.py:80) */
#define PSMF_FIXED_LAMBDA  16  /* rpsmf.py:36-40 */
#define PSMF_LL_STUDENT    32  /* theta gradient of the Student-t incremental likelihood (rpsmf.py:62-71); unset: Gaussian
                               * form (psmf.py:57-64; with a mask: rpsmf.py:196-200)                                   */
#define PSMF_NAN_MASK      64  /* missing entries of Y are NaN (the raw data form, rPSMF.py:160-164) and io->M must be NULL:
                               * m = !isnan(y), y := 0 where missing (== rPSMF.py:198-202 done on the fly; no mask stream) */

#define PSMF_RHO_VECTOR   128  /* R is diagonal but NOT uniform (psmf.py:144-152 takes the Woodbury branch for any diagonal R; the
                               * flat functions accept any (d, d) R): `rho` of psmf_set_state / psmf_get_state is then
                               * (n_series, d) = diag(R).  One GPU, direct-load kernel.
                               * Not with PSMF_XCHG_EXTERNAL (psmf_create refuses it): that exchange shards by rows. */
#define PSMF_GRAD_LINEAR  256  /* PSMF_DYN_LINEAR only: grad_out is the gradient of the summed incremental log-likelihood with
                               * respect to A and c (x_bar = A x + c, N, eta and V held fixed, as for the cos gradient):
                               * [G_A = sum_k gf_k x_{k-1}' (r x r row-major) | G_c = sum_k gf_k (r)] per series, gf_k =
                               * d ell_k / d x_bar_k.  d ell / d theta = <dA/dtheta, G_A>_F + <dc/dtheta, G_c> for any A(theta),
                               * c(theta): the caller closes the chain rule.  All kernels; row-sharded ranks agree bit for bit */
#define PSMF_LOGLIK       512  /* scal_out is PSMF_NSCAL_LL wide and carries the value of the learning objective and the one-step
                               * predictive log-density of every step (PSMF_SCAL_NLL, PSMF_SCAL_LOGPRED below); nothing is
                               * computed when scal_out is NULL.  Any flags, dynamics, mask encoding, kernel and sharding;
                               * row-sharded ranks write bit-identical records.  A non-finite value does not mark the step bad. */

/* dynamics f_theta(x, k) of the predict half (psmf.py:104-115) */
#define PSMF_DYN_IDENTITY 0    /* RandomWalk, nonlinearities.py:42-56; Impute scripts */
#define PSMF_DYN_COS      1    /* cos(2 pi theta k + x), synthetic_psmf.py:105-106 */
#define PSMF_DYN_LINEAR   2    /* x_bar = A x + c, F = A (psmf.py:104-115 with a linear f; ExperimentChange/PSMF.m:29-30):
                                * A, c from psmf_set_linear_dynamics                                          */
#define PSMF_DYN_EXTERNAL 3    /* x_bar and F = df/dx supplied by the caller, one step per psmf_run */

/* kernels (psmf_config.kernel; psmf_launch_info2 reports the one that ran) */
#define PSMF_KERNEL_AUTO   0
#define PSMF_KERNEL_DIRECT 1   /* direct-load kernel: any shape */
#define PSMF_KERNEL_STREAM 2   /* TMA-staged, software-pipelined kernel: one large series */
#define PSMF_KERNEL_BATCH  3   /* resident batch kernel: one CTA per series, C in shared memory for the whole launch */

/* statistics exchange between the GPUs that share one series by rows (psmf_config.exchange) */
#define PSMF_XCHG_NVLINK   0   /* inside the kernel: peer stores into NVLink mailboxes (psmf_mailbox_*) */
#define PSMF_XCHG_EXTERNAL 1   /* by the caller: psmf_run (one step) leaves the statistics of this GPU's rows in the
                                * buffer of psmf_stats_buffer; the caller all-reduces (sum) it in place on the same
                                * stream -- ncclAllReduce, MPI, anything -- and calls psmf_run_finish.  The NCCL
                                * baseline of bench.py, and the way to shard a series across nodes.              */

/* fused evaluation record written to eval_out: (n_series, PSMF_NEVAL) float64 (common.py:79-94) */
#define PSMF_NEVAL 4
#define PSMF_EVAL_SSE    0   /* sum over E of (y_hat - y_orig)^2   -> Epred = sqrt(SSE / COUNT), rPSMF.py:139 */
#define PSMF_EVAL_INSIDE 1   /* entries of E with y_orig inside y_hat -+ sig sqrt(U)  (rPSMF.py:121-123, common.py:87-94) */
#define PSMF_EVAL_COUNT  2   /* entries of E */

/* error codes */
#define PSMF_OK          0
#define PSMF_E_INVALID  -1
#define PSMF_E_CUDA     -2
#define PSMF_E_NOMEM    -3
#define PSMF_E_STATE    -4

/* per-step scalar record written to scal_out: (n_series, n_steps, PSMF_NSCAL) float64 */
#define PSMF_NSCAL 8
#define PSMF_SCAL_A      0   /* a = x_bar' V x_bar          rPSMF.py:93  */
#define PSMF_SCAL_ETA    1   /* eta_k                        rPSMF.py:108 */
#define PSMF_SCAL_N      2   /* N_k = a + eta                rPSMF.py:109 */
#define PSMF_SCAL_OMEGA  3   /* omega_k                      rPSMF.py:105 */
#define PSMF_SCAL_PHI    4   /* phi_k                        rPSMF.py:114 */
#define PSMF_SCAL_SSE    5   /* e' S^-1 e                    rPSMF.py:105 */
#define PSMF_SCAL_LAMBDA 6   /* lambda entering the step */
#define PSMF_SCAL_RHO    7   /* rho (R = rho I) entering the step */
/* PSMF_LOGLIK: (n_series, n_steps, PSMF_NSCAL_LL), entries 0..7 as above.  Per step, over the n = n_obs observed rows, with
 * q1 = sum_obs e_i^2, N = a + eta and lambda entering the step; both are exactly 0 for a step with every row missing.
 *   PSMF_SCAL_NLL     nll_k, the incremental negative log-likelihood that grad_out differentiates (the d ell_k / d f of
 *                     PSMF_DYN_COS / PSMF_DYN_EXTERNAL / PSMF_GRAD_LINEAR, with N, eta and V held fixed):
 *                       Gaussian:               (n/2) log(2 pi N) + q1 / (2 N)
 *                       PSMF_LL_STUDENT:        lgamma(lambda/2) - lgamma((lambda+n)/2) + (n/2) log(lambda pi N)
 *                                               + ((lambda+n)/2) log(1 + q1 / (lambda N))
 *                     i.e. -log of N(y_obs; C_o x_bar, N I) or of the t_lambda density with that scale.  The normalising
 *                     constants are included; they do not change the gradient.
 *   PSMF_SCAL_LOGPRED log p(y_obs,k | y_<k) under the filter's own predictive covariance S_obs = C_o Pbar C_o' + diag(rho_i + a):
 *                       log det S_obs = sum_obs log(rho_i + a) + log det(I + Pbar G)   (matrix-determinant lemma; the second
 *                                       term from the pivots of the elimination that solves for K, 0 with PSMF_SIMPLIFIED)
 *                       Delta^2       = diff_obs' S_obs^-1 diff_obs = w1 q1 - b'K b  (PSMF_RHO_VECTOR: sum_obs w_i e_i^2 - b'K b;
 *                                       PSMF_SIMPLIFIED: S_obs^-1 = diag(w_i), no b'K b)
 *                       Gaussian:     -(n log(2 pi) + log det S_obs + Delta^2) / 2
 *                       PSMF_ROBUST:  multivariate t with lambda degrees of freedom: lgamma((lambda+n)/2) - lgamma(lambda/2)
 *                                     - (n/2) log(lambda pi) - log det S_obs / 2 - ((lambda+n)/2) log(1 + Delta^2 / lambda) */
#define PSMF_NSCAL_LL     10
#define PSMF_SCAL_NLL     8
#define PSMF_SCAL_LOGPRED 9

typedef struct psmf_config {
    int64_t d;          /* rows of C held by this engine (the local shard)                         */
    int64_t d_global;   /* rows of the whole series: denominators of eta/omega/phi (== d if 1 GPU)  */
    int32_t r;          /* latent rank, 1..PSMF_MAX_RANK                                            */
    int32_t n_series;   /* independent series batched in this engine (>=1); no communication       */
    int32_t dtype;      /* PSMF_F64 | PSMF_F32                                                      */
    int32_t flags;      /* PSMF_ROBUST | ...                                                        */
    int32_t dynamics;   /* PSMF_DYN_*                                                               */
    int32_t device;     /* CUDA device ordinal                                                      */
    int32_t world_size; /* GPUs sharing ONE series by rows (1 = no exchange)                       */
    int32_t rank;
    int32_t ctas;       /* CTAs per series, 0 = auto                                                */
    int32_t kernel;     /* PSMF_KERNEL_* (error if the forced kernel is not eligible for the shape)         */
    double  alpha;      /* V scale (rpsmf.py:45-51), 1.0 unless use_scaling                        */
    double  beta;       /* P scale                                                                  */
    int32_t exchange;   /* PSMF_XCHG_* (world_size > 1)                                             */
    int32_t reserved;   /* 0                                                                        */
} psmf_config;

typedef struct psmf_io {
    const void*    Y;          /* (n_series, n_steps, ldy) time-major observations, zero-filled where missing */
    int64_t        ldy;        /* elements between consecutive time steps (>= d)                      */
    int64_t        y_series_stride;
    const uint8_t* M;          /* (n_series, n_steps, ldm) 1 = observed, 0 = missing; NULL = all observed */
    int64_t        ldm;
    int64_t        m_series_stride;
    double*        X_out;      /* (n_series, n_steps, r) filtered x_t, or NULL   (X[:, t], rPSMF.py:104) */
    void*          Yrec_out;   /* (n_series, n_steps, ldrec) C x_bar (unmasked), or NULL (Yrec, rPSMF.py:89) */
    int64_t        ldrec;
    int64_t        rec_series_stride;
    double*        scal_out;   /* (n_series, n_steps, PSMF_NSCAL), PSMF_LOGLIK: PSMF_NSCAL_LL; or NULL  */
    const double*  xbar_ext;   /* PSMF_DYN_EXTERNAL: (n_series, r)                                    */
    const double*  F_ext;      /* PSMF_DYN_EXTERNAL: (n_series, r, r) row-major                       */
    double*        grad_out;   /* (n_series, r) sum over the run of d ell_k / d theta (PSMF_DYN_COS), or NULL
                                * (_store_gradient, psmf.py:167-177); PSMF_DYN_EXTERNAL: d ell_k / d f of the one step;
                                * PSMF_GRAD_LINEAR: (n_series, r*r + r) [G_A row-major | G_c] summed over this run       */
    /* fused evaluation (all NULL / 0 = off): RMSE of the one-step predictions over the entries marked in E and the
     * number of original values inside the sig-sigma interval, accumulated in the row pass -- no (n, d) Yrec /
     * YrecL / YrecH arrays (rPSMF.py:67-69,121-123,139; common.py:79-94).  Direct-load and batch kernels only. */
    const void*    Yorig;      /* (n_series, n_steps, ldy) original values, same strides as Y (YorigInt)   */
    const uint8_t* E;          /* (n_series, n_steps, lde) 1 = evaluate here (Mmiss)                      */
    int64_t        lde;
    int64_t        e_series_stride;
    double         sig;        /* interval half-width in sigmas                                          */
    double*        eval_out;   /* (n_series, PSMF_NEVAL) sums over THIS run                              */
} psmf_io;

/* lifecycle ------------------------------------------------------------------------------------ */
int  psmf_create(psmf_handle* out, const psmf_config* cfg);
int  psmf_destroy(psmf_handle h);
const char* psmf_last_error(psmf_handle h);   /* h may be NULL: error of the last failed psmf_create */
int  psmf_version(void);

/* state round trip (sweep carry-over: psmf.py:75-83, rPSMF.py:75-79).  Any pointer may be NULL = leave /
 * skip.  C is (n_series, d, r) row-major in the engine dtype; V, P, Q are (n_series, r, r) row-major
 * float64; x, theta (n_series, r); rho, lambda (n_series) float64 (PSMF_RHO_VECTOR: rho is (n_series, d)). */
int  psmf_set_state(psmf_handle h, const void* C, const double* V, const double* P, const double* x,
                    const double* Q, const double* rho, const double* lambda, const double* theta, void* stream);
int  psmf_get_state(psmf_handle h, void* C, double* V, double* P, double* x,
                    double* Q, double* rho, double* lambda, double* theta, void* stream);

/* the hot path: n_steps filter steps starting at absolute time index k0 (the `t` argument handed to the
 * nonlinearity for the first step; pypsmf counts from 1).                                           */
int  psmf_run(psmf_handle h, const psmf_io* io, int64_t n_steps, int64_t k0, void* stream);

/* PSMF_XCHG_EXTERNAL: the statistics vector of one step (device pointer owned by the library, `count` doubles) and
 * the second half of a step (see PSMF_XCHG_EXTERNAL).  `io` and `k0` are those of the preceding psmf_run.       */
int  psmf_stats_buffer(psmf_handle h, double** dev_ptr, int32_t* count);
int  psmf_run_finish(psmf_handle h, const psmf_io* io, int64_t k0, void* stream);

/* PSMF_DYN_LINEAR: A (r, r) row-major and c (r) or NULL, device pointers, copied. One A per engine (all series). */
int  psmf_set_linear_dynamics(psmf_handle h, const double* A, const double* c, void* stream);

/* forecast (PSMFIter.predict, psmf.py:182-188): roll x through the dynamics for n_pred steps from the engine's
 * current state (absolute index of the first forecast step = k0) and emit C x.  Xpred_in (n_series, n_pred, r)
 * replaces the roll-out (PSMF_DYN_EXTERNAL: the caller owns f); Xpred_out (n_series, n_pred, r) and Ypred_out
 * (n_series, n_pred, ldp) in the engine dtype may be NULL.                                                 */
int  psmf_predict(psmf_handle h, int64_t n_pred, int64_t k0, const double* Xpred_in, double* Xpred_out, void* Ypred_out,
                  int64_t ldp, int64_t pred_series_stride, void* stream);

/* Efull of the imputation experiment (rPSMF.py:137-140): over the entries marked in E, the sum of
 * (C X - Yorig)^2 with the engine's CURRENT C and the filtered X (n_series, n_steps, r) of the sweep, and their
 * number -> out (n_series, 2).  No (d, n) product is materialised.                                         */
int  psmf_eval_full(psmf_handle h, const double* X, int64_t n_steps, const void* Yorig, int64_t ldy, int64_t y_series_stride,
                    const uint8_t* E, int64_t lde, int64_t e_series_stride, double* out, void* stream);

/* ingest (rPSMF.py:160-164,198-202): src (d, n) row-major float64 on the device with NaN = missing -> time-major
 * Y_out (n, ldy) of `dtype` (NaN kept if keep_nan, else zero-filled) and / or M_out (n, ldm) with 1 = observed.  */
int  psmf_ingest(int32_t device, const double* src, int64_t d, int64_t n, int32_t dtype, int32_t keep_nan, void* Y_out, int64_t ldy,
                 uint8_t* M_out, int64_t ldm, void* stream);
/* (d, n) row-major bytes -> time-major (n, ld) bytes, 1 where non-zero (M, Mmiss narrowed to one byte by the host) */
int  psmf_transpose_mask(int32_t device, const uint8_t* src, int64_t d, int64_t n, uint8_t* dst, int64_t ld, void* stream);
/* one sweep of prepare_missing (common.py:66-75) on time-major NaN-encoded Y (n, ldy): row i loses the `seg` entries
 * from starts[i] on that are not NaN yet (Y <- NaN, E <- 1); *count_dev += entries removed.  psmf_count_nan gives
 * NumMissDefault (common.py:65).  starts: d int64 on the device, drawn by the caller's generator.                */
int  psmf_missing_segments(int32_t device, int32_t dtype, void* Y, int64_t ldy, uint8_t* E, int64_t lde, int64_t d, int64_t n,
                           const int64_t* starts, int32_t seg, uint64_t* count_dev, void* stream);
int  psmf_count_nan(int32_t device, int32_t dtype, const void* Y, int64_t ldy, int64_t d, int64_t n, uint64_t* count_dev, void* stream);

/* synchronise the stream of the last run and report the device status word:
 * *first_bad_step = -1 if every step produced finite N/omega/phi, else the first offending step.
 * Returns PSMF_E_STATE (text in psmf_last_error) if a wait inside the kernel expired -- a peer GPU or CTA stopped
 * answering for PSMF_SPIN_TIMEOUT_MS (environment, default 10000) -- or if a peer GPU turned out to run a
 * different kernel; the launch has then drained with invalid results instead of hanging.              */
int  psmf_status(psmf_handle h, int64_t* first_bad_step);

/* introspection used by bench.py / tests, describing the last psmf_run: CTAs per series, threads per CTA,
 * dynamic smem bytes, kernels launched, which kernel ran (PSMF_KERNEL_*) and, for the TMA-staged kernel, its
 * shared-memory chunk slots and whether C stayed resident in shared memory.                          */
int  psmf_launch_info(psmf_handle h, int32_t* ctas, int32_t* threads, int32_t* smem_bytes, int32_t* launches);
int  psmf_launch_info2(psmf_handle h, int32_t* kernel, int32_t* nslot, int32_t* resident);

/* debug: record globaltimer stamps for the first `steps` filter steps of every following psmf_run into dev_buf
 * (steps * (16 + 2 * 160) uint64: 16 slots per step for the control CTA and the first pass warp of data CTA 0, then
 * per-CTA pass end / start times; scratch/trace.py decodes them).  dev_buf == NULL disables.           */
int  psmf_set_trace(psmf_handle h, uint64_t* dev_buf, int32_t steps);

/* multi-GPU row sharding (world_size > 1): NVLink mailbox for the per-step statistics exchange.
 * Each rank exports a blob of PSMF_MAILBOX_BLOB_BYTES (the CUDA IPC handle of its mailbox + a plan record: rank,
 * shape, flags, which kernels its shard is eligible for), gathers all ranks' blobs in rank order through the
 * host-side process group, and connects.  psmf_mailbox_connect checks that all ranks were created with the same
 * configuration and makes the kernel choice COLLECTIVELY (every rank derives it from the same n records): the
 * TMA-staged kernel only if every shard is eligible, else the direct-load kernel everywhere.           */
int  psmf_mailbox_export(psmf_handle h, void* blob);
int  psmf_mailbox_connect(psmf_handle h, const void* all_blobs, int32_t n);

#ifdef __cplusplus
}
#endif
#endif /* PSMF_B200_H */
