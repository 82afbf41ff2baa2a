/*
 * tame_b200.h -- C ABI of libtame_b200.so: the B200-native (sm_100a, FP64) variational update loop of
 * Temporal AME (naive mean-field, "good" and "bad" structured mean-field).
 *
 * The reference (Alfieriek/Python-Temporal-AME-SVI) is pure Python and has no FFI/plugin registry; its
 * boundary for this path is the Python class contract of src/inference/ (SURVEY.md section 8b).  Every entry
 * point below names the reference routine (file:line under /root/reference) that it replaces; the Python
 * classes in python-temporal-ame-svi_b200/tame_b200/inference.py bind them with ctypes and keep the reference's
 * class names, keyword arguments and error behaviour.  INTEGRATION.md shows the binding a maintainer would
 * add to the reference itself.
 *
 * Conventions
 *   - plain C types, no torch types.  All matrices row-major, FP64.
 *   - "dev" pointers are CUDA device pointers on the handle's device, "host" pointers are host memory.
 *   - every function returns 0 on success, a negative TAME_E* code otherwise; tame_last_error() returns a
 *     human-readable message for the calling thread's most recent failure.
 *   - one host thread per handle; work is ordered on the handle's stream (tame_set_stream).
 *   - state layout: x = [a, b, U(r), V(r)], d = 2 + 2r.
 *       Y      (n_rows_local, n, T, 2)   Y[i,j,t,:] = (y_ij, y_ji)       src/models/temporal_ame.py:176,209-216
 *       X_mean (n, T, d)                                                  src/inference/structured_mf.py:77
 *       X_cov  (n, T, d, d)                                               src/inference/structured_mf.py:80
 *   - single GPU: n_rows_local == n.  Multi GPU (world > 1): rows are dealt to ranks in panels of `panel`
 *     consecutive nodes, panel b belongs to rank b % world; a rank stores its panels' rows of Y back to back
 *     in increasing node order.  X_mean is replicated, X_cov rows of foreign nodes are only valid after
 *     tame_gather_state().
 */
#ifndef TAME_B200_H
#define TAME_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TAME_MODE_NAIVE 0 /* TemporalAMENaiveMFVI                     src/inference/naive_mf.py:29        */
#define TAME_MODE_GOOD 1  /* TemporalAMEStructuredMFVI("good")        src/inference/structured_mf.py:28   */
#define TAME_MODE_BAD 2   /* TemporalAMEStructuredMFVI("bad")         src/inference/structured_mf.py:270  */

#define TAME_OK 0
#define TAME_EINVAL (-1)   /* bad argument / unsupported shape (r must be 1..8)                           */
#define TAME_ECUDA (-2)    /* CUDA runtime error                                                           */
#define TAME_ESTATE (-3)   /* call order violated (e.g. sweep before bind)                                 */
#define TAME_EHANG (-4)    /* the in-kernel watchdog of the Gauss-Seidel chain fired                       */
#define TAME_ENCCL (-5)    /* NCCL error                                                                   */
#define TAME_ENOMEM (-6)

#define TAME_MAX_R 8

typedef struct tame_handle tame_handle;

/* Hyper-parameters of one fit: what the reference reads from `model` inside the loop
 * (model.R_inv, model.R, model.Phi, model.Q, model.Sigma, model.Psi; structured_mf.py:127-128,154-158,177-180,229-237). */
typedef struct tame_config {
    int32_t n;           /* nodes                                                                          */
    int32_t T;           /* time steps                                                                     */
    int32_t r;           /* latent_dim, 1..TAME_MAX_R                                                      */
    int32_t mode;        /* TAME_MODE_*                                                                    */
    double lr;           /* learning_rate (damping), structured_mf.py:282-287                              */
    double Rinv[4];      /* model.R_inv                                                                    */
    double logdet_R;     /* torch.logdet(model.R)                                                          */
    double logdet_Q;     /* torch.logdet(model.Q)                                                          */
    double logdet_S0;    /* torch.logdet(blockdiag(Sigma, Psi))                                            */
    const double* Phi;   /* host, d*d : model.Phi                                                          */
    const double* Qinv;  /* host, d*d : inv(model.Q)                                                       */
    const double* S0inv; /* host, d*d : inv(blockdiag(Sigma, Psi))                                         */
    int32_t device;      /* CUDA device ordinal                                                            */
    int32_t world;       /* number of ranks sharing this fit (1 = single GPU)                              */
    int32_t rank;        /* this rank                                                                      */
    int32_t panel;       /* rows per panel (multiple of 32); 0 = library default                           */
} tame_config;

/* ---- library ------------------------------------------------------------------------------------------ */
const char* tame_version(void);
const char* tame_last_error(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
int64_t tame_launch_count(void);

/* ---- handle life cycle --------------------------------------------------------------------------------- */
/* replaces the constructor chain base.py:60-82 / base.py:301-312 as far as device state is concerned */
int tame_create(const tame_config* cfg, tame_handle** out);
int tame_destroy(tame_handle* h);
int tame_set_stream(tame_handle* h, void* cuda_stream);
/* rows of Y held by this rank (== n when world == 1) */
int tame_local_rows(const tame_handle* h, int32_t* n_rows_local);

/* Bind the observations (device, read-only during the fit; self.Y = model.Y, base.py:71).  Runs the one-off
 * pass that builds the sweep-invariant sums  h_a[i,t] = sum_{j!=i} (p*y0 + q*y1),  h_b[i,t] = sum (q*y0 + p*y1)
 * -- the [a,b] rows of sum_j J'R^-1 y_ij in structured_mf.py:324.                                            */
int tame_bind_Y(tame_handle* h, const double* Y_dev);
/* The same for float observations (the reference's default dtype): Y stays float in HBM, half the bytes of the
 * double layout, and every dyad is widened to double when a kernel loads it -- the arithmetic, the state and the
 * results are those of tame_bind_Y on the widened Y, bit for bit.  The handle remembers the element type until the
 * next bind; rebinding with the other type is allowed. */
int tame_bind_Y_f32(tame_handle* h, const float* Y_dev);
/* Bind the variational state; it is updated IN PLACE like the reference's self.X_mean / self.X_cov
 * (structured_mf.py:282-287). */
int tame_bind_state(tame_handle* h, double* X_mean_dev, double* X_cov_dev);

/* ---- the hot path --------------------------------------------------------------------------------------- */
/* One Gauss-Seidel sweep: _update_step, structured_mf.py:211-287 / naive_mf.py:193-282 (+ _compute_observation_terms
 * structured_mf.py:289-326).  Nodes 0..n-1 in order, times 0..T-1 in order inside a node; each block is written
 * back before the next one reads it.  Asynchronous on the handle's stream.                                    */
int tame_sweep(tame_handle* h);
/* _compute_elbo (structured_mf.py:115-209 / naive_mf.py:89-191) fused with _compute_reconstruction_error
 * (base.py:314-326 -> temporal_ame.py:255-291).  out6 (host) = {ELBO, LL, LP0, LPT, H, MSE}.  Synchronises. */
int tame_elbo_mse(tame_handle* h, double* out6_host);
/* sweep + elbo_mse: one iteration of the body of fit(), base.py:170-180. */
int tame_iterate(tame_handle* h, double* out6_host);
/* BaseVariationalInference.fit, base.py:127-208, including the early stop of :183-203.  Traces are host
 * arrays of max_iter doubles; *n_done receives the number of iterations performed.  The patience counter
 * and previous ELBO live in the call, exactly as in the reference (a second fit() starts them afresh). */
int tame_fit(tame_handle* h, int32_t max_iter, double tolerance, double* elbo_trace_host, double* mse_trace_host,
             int32_t* n_done);

/* The whole loop of fit() on the DEVICE in one cooperative launch (k_fit: per iteration totals -> sweep -> covariance
 * blend -> ELBO/MSE -> the stop rule of base.py:183-203, grid-wide barriers in between), asynchronous on the handle's
 * stream: nothing returns to the host per iteration.  Traces / iteration count are written to DEVICE buffers
 * (max_iter doubles each, one int32).  Single GPU, small problems (what tame_fit_batch queues for every fit). */
int tame_fit_device(tame_handle* h, int32_t max_iter, double tolerance, double* elbo_trace_dev, double* mse_trace_dev,
                    int32_t* n_done_dev);
/* The same fit through HOST buffers: copies Y, X_mean, X_cov to the device, runs tame_fit, copies the state
 * back.  This is the end-to-end entry bench.py times (`e2e`).  Single GPU only. */
int tame_fit_host(const tame_config* cfg, const double* Y_host, double* X_mean_host, double* X_cov_host,
                  int32_t max_iter, double tolerance, double* elbo_trace_host, double* mse_trace_host,
                  int32_t* n_done);
/* tame_fit_host with float Y (tame_bind_Y_f32): stages half the bytes of Y; the state stays double. */
int tame_fit_host_f32(const tame_config* cfg, const float* Y_host, double* X_mean_host, double* X_cov_host,
                      int32_t max_iter, double tolerance, double* elbo_trace_host, double* mse_trace_host,
                      int32_t* n_done);

/* BASELINE config 5 (experiments/sensitivity_analysis.py:117-183: many independent small fits, one per grid point
 * and method): n_fits independent problems, each with its own tame_config and device buffers (Y_dev[f] is (n,n,T,2),
 * X_mean_dev[f] (n,T,d), X_cov_dev[f] (n,T,d,d), updated in place).  Traces are host arrays of n_fits * max_iter
 * doubles (row f = fit f); n_done[f] = iterations performed by fit f (early stop per fit, base.py:183-203).
 * Fits are independent Gauss-Seidel chains.  Default path (single-GPU fits with n <= 1024 on one device): every fit is ONE
 * cooperative launch of the whole-fit kernel (tame_fit_device: all iterations and the stop rule on the device), queued
 * largest fit first, round-robin on `n_streams` CUDA streams (0 = default 16, or TAME_BATCH_STREAMS) from the calling
 * thread; every stream re-points ONE handle per latent dimension, sized for the largest n and T of the batch, at its fits
 * (no allocation or device-wide synchronisation per fit); the host only waits at the end.  Otherwise (or with TAME_BATCH=host): one host thread per stream runs the host-driven loop of tame_fit.
 * The call returns when all fits are done. */
int tame_fit_batch(int32_t n_fits, const tame_config* cfgs, const double* const* Y_dev, double* const* X_mean_dev,
                   double* const* X_cov_dev, int32_t max_iter, double tolerance, double* elbo_traces_host,
                   double* mse_traces_host, int32_t* n_done, int32_t n_streams);
/* tame_fit_batch with float Y for every fit (tame_bind_Y_f32); everything else as above. */
int tame_fit_batch_f32(int32_t n_fits, const tame_config* cfgs, const float* const* Y_dev, double* const* X_mean_dev,
                       double* const* X_cov_dev, int32_t max_iter, double tolerance, double* elbo_traces_host,
                       double* mse_traces_host, int32_t* n_done, int32_t n_streams);

/* ---- data generation (the step before the path: TemporalAMEModel.generate_data, temporal_ame.py:200-216) - */
/* Y[i,j,t,:] = (mu0[i,j] + e0, mu0[j,i] + e1), (e0,e1) ~ N(0, R) per unordered dyad and time, mirrored for
 * j < i, zero diagonal; mu0[i,j] = a_i + b_j + U_i.V_j from X_true (n,T,d) on the device.  Counter-based
 * Philox keyed by (dyad, t), so every rank generates exactly its own rows of the same global Y.  Same
 * distribution as the reference, not the same stream.  Writes rows [row_begin,row_end) of global Y to Y_dev
 * (row-major, row_end-row_begin rows). */
int tame_generate_Y(int32_t n, int32_t T, int32_t r, const double R[4], const double* X_true_dev, uint64_t seed,
                    int32_t row_begin, int32_t row_end, double* Y_dev, void* cuda_stream);
/* The same Y stored as float: computed in double exactly as above and rounded once per value, so it equals
 * tame_generate_Y's output cast to float and stays mirror-consistent. */
int tame_generate_Y_f32(int32_t n, int32_t T, int32_t r, const double R[4], const double* X_true_dev, uint64_t seed,
                        int32_t row_begin, int32_t row_end, float* Y_dev, void* cuda_stream);

/* ---- alignment (the step after the fit in every driver: src/utils/alignment.py; demo.py:135-137) ------------ */
/* align_temporal_states (alignment.py:224-313) fused with the error of compute_alignment_error (:316-385).
 * X_est, X_true, X_aligned: (n, T, d) device arrays, d = 2 + 2r.
 *   align_each_time != 0: per time step, (a,b) rows get a sign flip when the flipped row is closer; U and V are each
 *     rotated by R = U Vt of svd(X_true' X_est) (last singular direction negated if det R < 0, :76-90) and then sign-
 *     flipped row by row (:204-214).
 *   align_each_time == 0: one 2r x 2r rotation from the temporal means of the multiplicative block (:286-311).
 * rot_dev (optional, device): the rotations, (T, 2, r, r) or (2r, 2r).  mse_host (optional, host): mean((X_aligned -
 * X_true)^2); passing it synchronises the stream.  The same call with T = 1 is the static (n, d) case of
 * compute_alignment_error (:362-369). */
int tame_align_states(int32_t n, int32_t T, int32_t r, const double* X_est_dev, const double* X_true_dev,
                      int32_t align_each_time, double* X_aligned_dev, double* rot_dev, double* mse_host, void* cuda_stream);
/* align_signs (alignment.py:106-166) on `rows` vectors of `width` entries: a vector is negated when that brings it
 * strictly closer to its target.  mse_host optional as above. */
int tame_align_signs(int64_t rows, int32_t width, const double* X_est_dev, const double* X_true_dev, double* X_aligned_dev,
                     double* mse_host, void* cuda_stream);
/* procrustes_alignment (alignment.py:31-103) of two (n, k) matrices, k <= 16: X_aligned = X_est R (times the optimal
 * scale when scaling != 0, :95-101); rot_dev (optional) receives R (k, k). */
int tame_procrustes(int32_t n, int32_t k, const double* X_est_dev, const double* X_true_dev, int32_t scaling,
                    double* X_aligned_dev, double* rot_dev, void* cuda_stream);

/* ---- diagnostics (src/utils/diagnostics.py; experiments/multiplicative_strength_comparison.py:46-89) ------------- */
/* compute_temporal_contributions (diagnostics.py:170-217): per time step the mean over node pairs of (a_i + b_j)^2
 * (compute_additive_contribution :82-122) and of (U_i . V_j)^2 (compute_multiplicative_contribution :125-167), with or
 * without the diagonal pairs.  X (n, T, d) device; additive_dev / multiplicative_dev: T doubles, device. */
int tame_contributions(int32_t n, int32_t T, int32_t r, const double* X_dev, int32_t exclude_diagonal, double* additive_dev,
                       double* multiplicative_dev, void* cuda_stream);
/* compute_uv_correlation_over_time (multiplicative_strength_comparison.py:46-89) / compute_uv_product_correlation
 * (diagnostics.py:528-561, T = 1): Pearson correlation of the flattened n x n products U V' of the estimate and of the
 * truth, per time step.  corr_dev: T doubles, device. */
int tame_uv_correlation(int32_t n, int32_t T, int32_t r, const double* X_est_dev, const double* X_true_dev, double* corr_dev,
                        void* cuda_stream);
/* compute_state_prediction_error (diagnostics.py:254-273): mean((A - B)^2) over `count` doubles.  Synchronises. */
int tame_state_mse(int64_t count, const double* A_dev, const double* B_dev, double* mse_host, void* cuda_stream);

/* ---- multi GPU ------------------------------------------------------------------------------------------ */
/* 128-byte NCCL unique id: rank 0 creates it, the caller ships it to the other ranks (torch.distributed),
 * every rank calls tame_comm_init.  After that tame_sweep broadcasts each finished panel's means from its
 * owner and tame_elbo_mse all-reduces the partial sums. */
int tame_comm_unique_id(void* id128_host);
int tame_comm_init(tame_handle* h, const void* id128_host);
/* Fused multi-GPU sweep: every rank exports the CUDA IPC handle (64 bytes) of its hand-over buffer, the caller
 * all-gathers the handles (torch.distributed) and every rank imports the world*64-byte table.  After that tame_sweep runs
 * the persistent kernel on every rank: the owner of a node writes its {new mean, tag} slots straight into the peers'
 * buffers over NVLink and the peers' time-step warps follow.  Without it the stream-ordered panel scheduler (NCCL
 * broadcast per 64-node block) is used. */
int tame_ipc_export(tame_handle* h, void* handle64_host);
int tame_ipc_import(tame_handle* h, const void* handles_host);
/* Same, for ranks that live in ONE process (one handle per device): every rank's handle is passed directly, peer access
 * is enabled between the devices and the hand-over buffers are used through their plain device pointers. */
int tame_peer_attach(tame_handle* h, tame_handle* const* all_handles);
/* all-gather the X_cov rows (X_mean is already replicated) so every rank holds the full state */
int tame_gather_state(tame_handle* h);

/* 1 when tame_bind_Y verified Y[j,i,t,:] == swap(Y[i,j,t,:]) bit for bit (the ELBO pass then streams the i<j half), else 0 */
int tame_y_symmetric(const tame_handle* h);

/* ---- diagnostics ----------------------------------------------------------------------------------------- */
/* device time of the last tame_sweep / tame_elbo_mse in milliseconds, measured with CUDA events on the
 * handle's stream; *_kernel_ms of the dominant kernel(s) inside it. */
int tame_last_timing(tame_handle* h, double* sweep_ms, double* elbo_ms, double* contract_ms, double* chain_ms,
                     double* llmse_ms);
int tame_set_timing(tame_handle* h, int32_t enabled);
/* timing probes of the last fused sweep (k_sweep): [0..7] the warp pair of time step 0, [8..15] of time step T-1:
 * {start ns, chain-warp cycles waiting for the NEXT node's inputs, end ns, helper cycles waiting for streaming units, for the hand-over of (i,t-1), for
 *  the chain warp, cells done, chain-warp cycles waiting for its inputs} */
int tame_debug_probes(tame_handle* h, uint64_t* out16_host);
/* with TAME_TRACE=1 in the environment at tame_create: per 32-node sub-block, the globaltimer stamps (ns) at which the
 * helper of time step 0 started / stopped waiting for the sub-block's streaming unit (2 entries per sub-block) */
int tame_debug_trace(tame_handle* h, uint64_t* out_host, int32_t n_entries);

#ifdef __cplusplus
}
#endif
#endif /* TAME_B200_H */
