/*
 * pcs_b200.h -- C ABI of the B200-native bundle-adjustment inner loop (libpcs_b200.so).
 *
 * Drop-in boundary for pyCamSet's residual / Jacobian callbacks and the solver step that consumes them.
 * Plain pointers and sizes only; no torch / numpy types.  Every entry point cites the reference interface
 * it replaces (paths relative to the pyCamSet repository, v1.1.2).
 *
 * Conventions
 *   - All floating point is IEEE FP64.  Index arrays are int32 unless stated.
 *   - Observation table = the reference's `dd` (target_detections.py:51-55) split into structure-of-arrays:
 *     cam[N], pose[N] (image number), key[N] (flattened key), uv[N][2].
 *   - Parameter string (abstract_function_blocks.py:777-820, :669-681):
 *       [ intr C x 9 | extr C x 6 | pose M x 6 | point K x 3 (self-calibration chain only) ]
 *     length L = 15 C + 6 M (+ 3 K).
 *   - free_map[L]: index of each parameter-string entry in the free vector x, or -1 when the entry is held
 *     fixed (the `conversion` renumbering of abstract_function_blocks.py:482-485).
 *   - Pointers are HOST pointers unless the function name ends in `_dev`; `_dev` functions take device
 *     pointers on the problem's device and enqueue on the problem's stream without synchronising.
 *   - Return value: 0 on success, negative pcs_status otherwise; pcs_last_error() gives the message
 *     (thread-local).  There is no CPU fallback: every call fails with PCS_ERR_CUDA when no device works.
 */
#ifndef PCS_B200_H
#define PCS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCS_API __attribute__((visibility("default")))

typedef struct pcs_problem pcs_problem;

typedef enum pcs_status {
    PCS_OK = 0,
    PCS_ERR_INVALID = -1,     /* bad argument (NULL pointer, size mismatch, index out of range) */
    PCS_ERR_CHAIN = -2,       /* unknown function-block chain: only the two shipped chains are accelerated */
    PCS_ERR_CUDA = -3,        /* CUDA runtime error (message in pcs_last_error) */
    PCS_ERR_UNSUPPORTED = -4, /* operation not defined for this chain / configuration */
    PCS_ERR_NUMERIC = -5      /* solver breakdown (non positive-definite system) */
} pcs_status;

/* Chain ids.  The key is the tuple of function-block class names, exactly what the reference uses to name
 * its generated kernels (abstract_function_blocks.py:297, :504). */
typedef enum pcs_chain {
    PCS_CHAIN_TEMPLATE = 0, /* projection + extrinsic3D + template_points           (template_handler.py:152)        */
    PCS_CHAIN_SELFCAL = 1   /* projection + extrinsic3D + rigidTform3d + free_point (standard_bundle_handler.py:182) */
} pcs_chain;

/* Maps "projection_extrinsic3D_template_points" etc. to a chain id; PCS_ERR_CHAIN for anything else. */
PCS_API int pcs_chain_from_name(const char* block_names_joined_by_underscore);

typedef struct pcs_problem_desc {
    int32_t chain;          /* pcs_chain */
    int32_t device;         /* CUDA device ordinal */
    int64_t n_obs;          /* N */
    int32_t n_cams;         /* C */
    int32_t n_poses;        /* M */
    int32_t n_keys;         /* K */
    int32_t inputs_on_device; /* non-zero: cam/pose/key/uv below are device pointers (template/free_map stay host) */
    const int32_t* cam;     /* [N] */
    const int32_t* pose;    /* [N] */
    const int32_t* key;     /* [N] */
    const double* uv;       /* [N][2] */
    const double* template_xyz; /* [K][3], chain 0; ignored (may be NULL) for chain 1 */
    const int32_t* free_map;    /* [L] or NULL (= every parameter free) */
    void* stream;           /* cudaStream_t to run on, or NULL for a stream owned by the problem */
} pcs_problem_desc;

typedef struct pcs_problem_info {
    int32_t chain, n_cams, n_poses, n_keys;
    int32_t cols_per_row;   /* P: 21 or 24 */
    int32_t device;
    int64_t n_obs;
    int64_t n_params;       /* L */
    int64_t n_free;
    int64_t nnz;            /* CSR non-zeros of the (2N x n_free) Jacobian */
    int64_t n_segments;     /* distinct (camera, pose) pairs with at least one observation */
} pcs_problem_info;

/* Build the static problem state on the device: observation SoA, gather structure, CSR row offsets and the
 * (camera, pose)-sorted layout used by the normal-equation kernel.
 * Replaces optimisation_function.make_full_loss_fn / make_jacobean set-up (abstract_function_blocks.py:656-667),
 * get_block_param_inds (:192-233) and make_jac_CSR_columns_row_pointers (:465-489). */
PCS_API int pcs_problem_create(const pcs_problem_desc* desc, pcs_problem** out);
PCS_API int pcs_problem_destroy(pcs_problem* p);
PCS_API int pcs_problem_get_info(const pcs_problem* p, pcs_problem_info* info);
PCS_API const char* pcs_last_error(void);

/* Parameters.  set_param_string loads the full dense string (fixed values included) -- the output of
 * optimisation_function.build_param_list (abstract_function_blocks.py:669-681).  set_free scatters the free
 * vector x into it -- TemplateBundlePrimitive.return_bundle_primitives + fill_flat
 * (template_handler.py:63-78, compiled_helpers.py:155-177).  get_param_string reads the dense string back. */
PCS_API int pcs_set_param_string(pcs_problem* p, const double* params /*[L]*/);
PCS_API int pcs_set_free(pcs_problem* p, const double* x /*[n_free]*/);
PCS_API int pcs_get_param_string(pcs_problem* p, double* params /*[L]*/);

/* loss_fun(x) -> float64[2N], interleaved (x, y) per observation in dd row order
 * (template_handler.py:157-170; generated full_loss, abstract_function_blocks.py:351-387).
 * x == NULL evaluates at the current parameters. */
PCS_API int pcs_residual(pcs_problem* p, const double* x, double* r_out /*[2N]*/);
PCS_API int pcs_residual_dev(pcs_problem* p, const double* x_dev, double* r_dev);

/* jac_fn(x) -> csr_array (2N x n_free): structure once, values per call
 * (template_handler.py:172-193; generated full_jac + matflow, abstract_function_blocks.py:552-652,
 *  matmul_map.py:147-243).  Column order within a row = chain parameter order, fixed columns absent. */
PCS_API int pcs_csr_structure(pcs_problem* p, int64_t* col_idx /*[nnz]*/, int64_t* row_ptr /*[2N+1]*/);
PCS_API int pcs_jacobian_values(pcs_problem* p, const double* x, double* vals_out /*[nnz]*/);
PCS_API int pcs_jacobian_values_dev(pcs_problem* p, const double* x_dev, double* vals_dev);

/* Segment table of the normal equations: one entry per (camera, pose) pair with observations, sorted by
 * (camera, pose).  W[s] couples seg_cam[s] with seg_pose[s]. */
PCS_API int pcs_segments(pcs_problem* p, int32_t* seg_cam /*[S]*/, int32_t* seg_pose /*[S]*/, int64_t* seg_len /*[S]*/);

/* Fused residual + Jacobian + J^T J / J^T r (both chains).  No reference counterpart: scipy's LSMR consumes the
 * CSR Jacobian instead (optimisation_handling.py:88-98); defined as the blocks of J.T @ J and J.T @ r of the
 * reference Jacobian with no parameter fixed:
 *   U[C][15][15], gc[C][15]  camera blocks (9 intrinsic + 6 extrinsic columns)
 *   V[M][6][6],  gp[M][6]    pose blocks
 *   W[S][15][6]              camera x pose coupling per segment
 *   cost = r . r
 * Any output pointer may be NULL to skip its copy-out (results stay on the device for pcs_lm_*). */
PCS_API int pcs_normal_equations(pcs_problem* p, const double* x, double* U, double* gc, double* V, double* gp,
                                 double* W, double* cost);
/* Device-resident variant: evaluates into the problem's own buffers; pointers to them via pcs_device_buffers. */
PCS_API int pcs_normal_equations_dev(pcs_problem* p, const double* x_dev);

/* Self-calibration chain (projection + extrinsic3D + rigidTform3d + free_point, standard_bundle_handler.py:129-226;
 * free_point: function_block_implementations.py:216-240): the blocks of J.T @ J / J.T @ r that involve the target points,
 * as of the last pcs_normal_equations* call (U, V, W, gc, gp of this chain are the blocks above):
 *   Pk[K][3][3], gk[K][3]     point blocks
 *   Xck[C][K][15][3]          camera x point coupling (zero for pairs without observations)
 *   Ymk[M][K][6][3]           pose x point coupling
 * Any pointer may be NULL.  PCS_ERR_UNSUPPORTED when (45 C + 18 M) K > 2^27 (the dense tables are not allocated). */
PCS_API int pcs_point_blocks(pcs_problem* p, double* Pk, double* gk, double* Xck, double* Ymk);

/* Arithmetic of the fused normal-equation kernel (pcs_normal_equations*, and every evaluation inside pcs_lm_solve).
 *   PCS_PRECISION_FP64  (default) everything FP64: blocks agree with J.T @ J of the reference Jacobian to 1e-9.
 *   PCS_PRECISION_MIXED residual, cost and the gradients gc / gp stay FP64 (bit-for-bit the same evaluation; the LM fixed
 *                       point g = 0 is unchanged); the J^T J blocks U, V, W -- which only precondition the step -- are
 *                       accumulated on the BF16 tensor path (two-term split, FP32 accumulation per (camera, pose) segment,
 *                       FP64 across segments): entries within ~1e-4 sqrt(d_a d_b) of the FP64 blocks.
 * No reference counterpart (the reference never forms J^T J). */
typedef enum pcs_precision { PCS_PRECISION_FP64 = 0, PCS_PRECISION_MIXED = 1 } pcs_precision;
PCS_API int pcs_set_normal_precision(pcs_problem* p, int precision);

/* Dense normal equations over the free parameters (both chains; small problems: n_free^2 doubles of HBM):
 * JtJ[n_free][n_free] (full symmetric), Jtr[n_free], cost. */
PCS_API int pcs_normal_dense(pcs_problem* p, const double* x, double* JtJ, double* Jtr, double* cost);

typedef struct pcs_device_buffers {
    double* params;  /* [L] */
    double* U;       /* [C][15][15] */
    double* gc;      /* [C][15] */
    double* V;       /* [M][6][6] */
    double* gp;      /* [M][6] */
    double* W;       /* [S][15][6] */
    double* cost;    /* [1] */
    double* residual;/* [2N] scratch used by pcs_residual */
    void* stream;    /* cudaStream_t */
} pcs_device_buffers;
PCS_API int pcs_device_buffers_get(pcs_problem* p, pcs_device_buffers* out);

/* Multi-GPU hook.  Observations are sharded by target pose: every rank owns the pose blocks of its poses and a
 * PARTIAL sum of the camera blocks.  pcs_lm_solve calls this callback (work enqueued on `stream`) to combine n
 * doubles in place across ranks: the Schur-reduced camera system [S | rhs | gc | cost] once per linear solve and
 * one vector of 5 + world_size step scalars once per iteration (both op 0 = sum; op 1 = max is part of the contract
 * but currently unused).  The Python host installs a torch.distributed (NCCL) all-reduce here; it must return 0 on
 * success. */
typedef int (*pcs_allreduce_fn)(void* user, double* buf_dev, int64_t n, int op, void* stream);
PCS_API int pcs_set_allreduce(pcs_problem* p, pcs_allreduce_fn fn, void* user, int rank, int world_size);

/* Initialiser cost evaluation: bundle_adjustment_costfn (compiled_helpers.py:517-549, distortion :438-460) as
 * estimate_camera_relative_poses drives it (template_handler.py:510-593) -- all `n_tables` candidate pose tables in
 * one call over the problem's resident observations.
 *   im_points  [n_tables][M][K][3]  target points transformed by each image's candidate pose
 *   proj [C][3][4] = K_c [R_c | t_c],  intrinsics [C][3][3],  dists [C][5] = (k1, k2, p1, p2, k3)
 *   errors     [n_tables][2N] projected-minus-measured pixels, dd row order (or NULL to skip: 16 B/obs/table of PCIe)
 *   per_image  [n_tables][M]  sum over the observations of image m of |error| (template_handler.py:550-560), or NULL */
PCS_API int pcs_costfn(pcs_problem* p, int n_tables, const double* im_points, const double* proj, const double* intrinsics,
                       const double* dists, double* errors, double* per_image);

/* Scale estimate of the self-calibration gauge transform: SelfBundleHandler.apply_gauge_transform
 * (standard_bundle_handler.py:339-410, the cdist tables of :360-366).  Over all pairs i < j of visible points whose
 * reference distance is np.isclose(., square_size, rtol, atol): *sum_ratio = sum d_ref / d_estimate, *n_pairs = their
 * number (the reference's s is the mean).  Host buffers; estimate / reference [n_points][3], visible [n_points] bytes. */
PCS_API int pcs_gauge_scale(int device, int64_t n_points, const double* estimate, const double* reference, const uint8_t* visible,
                            double square_size, double rtol, double atol, double* sum_ratio, int64_t* n_pairs);

/* Multi-GPU, raw evaluation: one-shot all-reduce (sum, rank order) of the camera blocks [U | gc | cost] over NVLink
 * peer memory -- the only exchange step of a pose-sharded normal-equation evaluation (C * 240 + 1 doubles, latency
 * bound).  Every rank allocates a zero-initialised buffer of pcs_p2p_buffer_bytes(p, world) that all peers have mapped
 * (e.g. torch.distributed._symmetric_memory) and passes the world's pointers, own buffer at index `rank`.
 * pcs_p2p_allreduce_setup marks the slots of the rank's own buffer as empty (a sentinel NaN; the call synchronises the
 * problem's stream) -- the caller must put a barrier across the ranks between the setup call and the first exchange.
 * pcs_p2p_allreduce_camera_blocks enqueues one kernel (one CTA per peer) on the problem's stream: the rank's block is
 * pushed into its slot at every peer without fence or flag, the arrival of the data is the signal (csrc/pcs_p2p.cu);
 * all ranks must call it the same number of times.
 * pcs_p2p_status: *timed_out = 1 if a poll ever gave up waiting for a peer (the sums of that exchange are then
 * invalid); synchronises the stream.  No reference counterpart (the reference is single-process). */
PCS_API int64_t pcs_p2p_buffer_bytes(const pcs_problem* p, int world_size);
PCS_API int pcs_p2p_allreduce_setup(pcs_problem* p, int rank, int world_size, void* const* peer_buffers, int64_t buffer_bytes);
PCS_API int pcs_p2p_allreduce_camera_blocks(pcs_problem* p);
PCS_API int pcs_p2p_status(pcs_problem* p, int* timed_out);

/* Levenberg-Marquardt on the device (replaces scipy.optimize.least_squares TRF + LSMR as driven by
 * run_bundle_adjustment, optimisation_handling.py:52-117). */
/* Termination, tested in this order in every iteration, after the damped step dx has been solved at the current
 * linearisation point x (x, dx and g = J^T r range over the FREE parameters only; fixed entries of the parameter string
 * do not enter any norm):
 *   gtol  |g|_inf < gtol                          status 1, x is returned (the step is not taken);
 *   xtol  |dx|_2 < xtol (xtol + |x|_2)            status 3, x is returned (the step is not taken);
 *   ftol  after an ACCEPTED step, (c - c') / c < ftol with c, c' = r.r before / after the step: status 2, x + dx returned.
 * A step is accepted when rho = (c - c') / pred > 0, pred = dx . (lambda D dx - g), D = diag(J^T J); then
 * lambda <- max(lambda_min, lambda max(1/3, 1 - (2 rho - 1)^3)), nu = 2; otherwise lambda <- min(lambda_max, lambda nu),
 * nu <- 2 nu, and reaching lambda_max ends the solve with status -1.  max_iter counts accepted and rejected steps. */
typedef struct pcs_lm_options {
    int32_t max_iter;      /* default 100 (the reference's max_nfev, template_handler.py:24-31) */
    int32_t verbose;
    double lambda0;        /* initial damping, default 1e-3 */
    double ftol, xtol, gtol; /* default 1e-8 (scipy least_squares defaults) */
    double lambda_min, lambda_max;
} pcs_lm_options;

typedef struct pcs_lm_stats {
    int32_t iterations;    /* accepted + rejected steps */
    int32_t n_eval_normal; /* fused normal-equation evaluations */
    int32_t n_eval_cost;   /* residual-only evaluations */
    int32_t status;        /* 0 max_iter, 1 gtol, 2 ftol, 3 xtol, <0 failure */
    double cost_initial, cost_final; /* 0.5 * r.r, scipy's convention */
    double grad_norm_inf;
    double lambda_final;
    double seconds;        /* device time of the whole solve, CUDA events */
} pcs_lm_stats;

PCS_API void pcs_lm_default_options(pcs_lm_options* o);
PCS_API int pcs_lm_solve(pcs_problem* p, const double* x0 /*[n_free]*/, const pcs_lm_options* opts,
                         double* x_out /*[n_free]*/, pcs_lm_stats* stats);

/* Parameter covariance at x (host buffers; x == NULL: the current parameters).  With H = J^T J over the free parameters,
 * r the residual and N the number of observations, the unit-weight covariance Sigma = H^-1 is returned in parts:
 *   cam   [15 C][15 C]  the full camera block, camera-major, 15 entries per camera (9 intrinsics, then 6 extrinsics: the
 *                       layout of U);
 *   pose  [M][6][6]     the marginal block of every pose;
 *   point [K][3][3]     the marginal block of every target point (self-calibration chain only; ignored otherwise);
 *   s2                  r.r / dof, dof = 2 N - (number of observed free parameters); NaN when dof <= 0;
 *   dof.
 * The covariance of the estimate is s2 * Sigma.  Any output may be NULL.  Camera x pose and camera x point
 * cross-covariances are not returned (O(C M) numbers).
 * An entry is exactly 0 when either of its parameters is fixed; otherwise NaN when either is unobserved (a free parameter
 * whose diagonal of J^T J is zero).  Unobserved parameters are decoupled from all others: no other entry depends on them.
 * Sigma comes from the factors of the LM solver's reduced system at lambda = 0 (S = A - Z Z^T = L L^T, Z = W L_b^-T):
 *   reduced set    S^-1 = X^T X,                     X = L^-1;
 *   eliminated set L_b^-T (I + X_b^T X_b) L_b^-1,    X_b = L^-1 Z_b
 * (csrc/pcs_cov.cu).  The eliminated set is the poses, or on the self-calibration chain the points when 3 K > 6 M.
 * The normal equations are always FP64, whatever pcs_set_normal_precision selects (the setting is kept).
 * Side effects: those of pcs_normal_equations(p, x, NULL, ...): the parameters become x and the device block buffers hold
 * the evaluation at x; a later pcs_lm_solve behaves as it would without this call.
 * Errors: PCS_ERR_NUMERIC when the undamped reduced system or an eliminated block is not positive definite (typically: the
 * gauge is not fixed); PCS_ERR_UNSUPPORTED with an all-reduce hook of world size > 1, and on the dense self-calibration
 * fallback (no point tables, or PCS_LM_SELFCAL=dense).
 * No reference counterpart: with scipy's solver the covariance comes from result.jac (optimisation_handling.py:52-117). */
PCS_API int pcs_covariance(pcs_problem* p, const double* x /*[n_free] or NULL*/, double* cam, double* pose, double* point,
                           double* s2, int64_t* dof);

/* Dense symmetric positive definite solve S x = b with the persistent tiled Cholesky kernel, the kernel every
 * factorisation of the library uses (in pcs_lm_solve the counterpart of the LSMR solve inside scipy's TRF,
 * optimisation_handling.py:88-98).  Host buffers; A is column-major [n][n], only the lower triangle is read.
 * *info: 0 ok, 1 not positive definite (PCS_ERR_NUMERIC), -2 the kernel's grid barrier timed out (PCS_ERR_CUDA).
 * Exposed so that the solver kernel can be tested on its own. */
PCS_API int pcs_spd_solve(int device, int64_t n, const double* A, const double* b, double* x /*[n]*/, int* info);

/* S -= Z Z^T on the lower triangle, the pose-elimination update of the reduced camera system as pcs_lm_solve runs it
 * (stream-K tiled FP64 tensor-path kernel, csrc/pcs_schur.cu).  Host buffers; Z is column-major [k][n] (n rows
 * contiguous), S column-major [n][n], only its lower triangle is updated.  Exposed so that the kernel can be tested
 * on its own. */
PCS_API int pcs_syrk_sub(int device, int64_t n, int64_t k, const double* Z, double* S);

/* Block sparsity of the pose elimination inside pcs_lm_solve.  A camera that does not see a pose leaves a zero 15 x 6
 * block in Z; the pattern is static, so the solver orders the pose columns by visibility pattern and visits only the
 * (96-row tile pair, 16-column slab) units of S -= Z Z^T whose operands are both non-zero (csrc/pcs_schur.cu).
 * *fraction = visited units / all units; 1.0 means the dense iteration space is used (pattern too dense to pay, or
 * PCS_LM_SCHUR=dense).  Builds the solver workspace if it does not exist yet.  Diagnostic; no reference counterpart
 * (scipy's LSMR never forms the reduced system, optimisation_handling.py:88-98). */
PCS_API int pcs_lm_schur_fraction(pcs_problem* p, double* fraction);

/* Optional kernel timing: when enabled, every launch of the fused normal-equation kernel is bracketed by a pair of
 * CUDA events on the problem's stream (a ring of 1024 pairs, so a timed loop needs no synchronisation inside).
 * pcs_timing_get returns the duration (ms) of the most recent launch, pcs_timing_get_all the durations of the last
 * launches since timing was enabled, oldest first (both synchronise on the events they read). */
PCS_API int pcs_timing_enable(pcs_problem* p, int on);
PCS_API int pcs_timing_get(pcs_problem* p, double* normal_kernel_ms);
PCS_API int pcs_timing_get_all(pcs_problem* p, double* ms, int64_t capacity, int64_t* n_out);

/* Number of kernels of this library launched so far for the residual / Jacobian / normal-equation evaluations of
 * this problem.  bench.py reports the difference
 * over its timed region as `gpu_launches`. */
PCS_API int pcs_launch_count(const pcs_problem* p, int64_t* n_kernels);

/* Library / device probe: returns the device's SM count, or a negative pcs_status. */
PCS_API int pcs_device_sm_count(int device);
PCS_API const char* pcs_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PCS_B200_H */
