// pcs_solver.cu -- Levenberg-Marquardt on the device.
//
// Replaces scipy.optimize.least_squares (TRF + LSMR, x_scale='jac') as driven by run_bundle_adjustment
// (optimisation_handling.py:52-117).  The reference never forms J^T J; here the fused kernel delivers the
// block normal equations and each LM step (solve_step) eliminates one set of B x B diagonal blocks (BlockSet: the poses,
// B = 6, or the target points, B = 3; lm_path decides which):
//   factor the damped blocks (k_lm_block_factor<B>), form the reduced system over the cameras (+ the second block set of
//   the self-calibration chain) S = A + lambda D - Z Z^T with Z = (coupling) L_b^-T (k_lm_init_reduced<B>, the Z kernels,
//   k_schur_syrk in pcs_schur.cu), [all-reduce S | rhs across ranks], dense SPD solve (k_chol_solve, pcs_chol.cu),
//   back-substitute the eliminated blocks (k_lm_block_back<B>), move to the trial point and evaluate it with the full
//   normal-equation kernel into the second output set -- one host synchronisation per iteration.
//   template chain:  the poses are eliminated, the reduced system is over the cameras (15 C).
//   self-calibration: poses AND target points are block diagonal but coupled to each other, so one of the two sets is
//                    eliminated -- the larger one.  Points eliminated (3 K > 6 M, single rank): reduced system over
//                    cameras + poses [[U, .], [W^T, V]] - Z Z^T with Z = [Xck; Ymk] L_k^-T.  Poses eliminated
//                    (otherwise): the points join the cameras in the reduced system (15 C + 3 K unknowns: point blocks
//                    Pk, camera x point blocks Xck on the A side, pose x point blocks Ymk next to W on the coupling side).
//                    Problems whose dense (camera, key) / (pose, key) tables would not fit fall back to the dense
//                    (n_free x n_free) normal matrix, factored by the same k_chol_solve, with a residual-only trial pass.
//   The pose elimination skips the structurally zero blocks of Z (static unit list, pcs_schur.cu).
// Marquardt scaling (lambda * diag(J^T J)) plays the role of x_scale='jac'; Nielsen's gain-ratio update
// drives lambda.  Fixed parameters are rows / columns replaced by the identity.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "pcs_internal.cuh"
#include "pcs_math.cuh"

namespace pcs {

// A set of B x B diagonal blocks of the normal equations: the poses (B = 6) or the target points (B = 3).  block_set()
// builds it from the problem whenever it is used, because the normal-equation outputs alternate between two buffers
// (swap_normal_buffers).
struct BlockSet {
    int B = 0;                       // 6: poses, 3: target points, 0: no set
    int n = 0;                       // number of blocks
    int64_t off = 0;                 // first parameter of the set in the parameter string
    const double* blk = nullptr;     // [n][B][B] V / Pk
    const double* g = nullptr;       // [n][B]    gp / gk
    const uint8_t* mask = nullptr;   // [n] free bits
    const int32_t* slot = nullptr;   // [n] column slot of block b in Z (pose elimination with a Schur plan), nullptr = b
};

// The LM path, fixed when the workspace is built (lm_path): the eliminated block set (elim_B = 6: poses, 3: target
// points, 0: none -- the dense self-calibration fallback) and the second block set that joins the cameras in the reduced
// system (red_B = 3: the points, 6: the poses, 0: none -- template chain).
struct LmPath {
    int elim_B = 0, red_B = 0;
};

struct LmWorkspace {
    LmPath path;
    int64_t nc = 0;          // order of the reduced system nl, rounded up to a multiple of 32 (identity rows) so that every
                             // tile of the Cholesky kernel is full and moves with 16-byte copies, whatever C, M and K are
    int64_t nl = 0;          // logical order: 15 C + the second set's unknowns (3 K, 6 M or none)
    int64_t np = 0;          // eliminated unknowns: 6 M or 3 K
    double* L = nullptr;     // [n_elim][B * B] lower Cholesky factors of the damped eliminated blocks
    double* y = nullptr;     // [n_elim][B]     L_b^-1 (-g_b)
    double* Z = nullptr;     // [np][nc] column-major (nc rows): coupling L_b^-T
    SchurPlan plan;          // static block sparsity of Z: pose column order + non-zero (tile, slab) units (pcs_schur.cu)
    int32_t* seg_of = nullptr;   // poses in the reduced system: [C][M] segment of (camera, pose) or -1 (placement of W)
    double* red = nullptr;   // [S nc*nc | rhs nc | gc nc | cost 1]  (all-reduce unit)
    int64_t red_doubles = 0;
    double* delta = nullptr; // [Lparams]
    double* backup = nullptr;// [Lparams]
    double* scal = nullptr;  // [8] device scalars: pred, |dx|^2, |x|^2, ginf, cost_trial, flag
    int* info = nullptr;
    // dense SPD solve (k_chol_solve) of order nc, or n_free on the dense path: diagonal-block factors, grid barrier counter
    double* Ldiag = nullptr;   // [ceil(n / 32)][32 * 32] row-major lower factors of the diagonal tiles
    unsigned long long* bar = nullptr;
    unsigned long long bar_base = 0;
    int chol_grid = 0;         // co-resident CTAs of k_chol_solve
    // second set of normal-equation outputs: the trial point is evaluated speculatively with the full kernel
    double* ne_alt = nullptr;
    double* ne_orig = nullptr;
    // one pinned read-back per iteration: scal[8] | info | cost of the linearisation point (gathered on the device)
    double* h_read = nullptr;   // pinned [10]
    double* d_read = nullptr;   // [10]
    double* comb = nullptr;     // [5 + world] multi-rank: the step scalars of all ranks in ONE sum all-reduce (see k_lm_pack_scalars)
    // dense path
    double* H = nullptr;     // [n_free^2 + n_free + 1] = JtJ | Jtr | cost  (aliases p->dense)
    double* Hd = nullptr;    // damped copy [n_free^2]
    double* rhs = nullptr;   // [n_free]
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // device time of a solve (owned by the workspace: no leak on error returns)
    // pcs_covariance: X_I = L^-1 [nc][nc]
    double* cov_Xi = nullptr;
};

static inline int grid_for(int64_t n, int block) { return (int)((n + block - 1) / block); }

// per block (one thread each): Cholesky of the damped, masked B x B block, y = L^-1 (-g); fixed / unobserved coordinates
// are identity rows
template <int B>
__global__ void k_lm_block_factor(int n, double lambda, const double* __restrict__ blk, const double* __restrict__ g,
                                  const uint8_t* __restrict__ blk_mask, double* __restrict__ Lout, double* __restrict__ yout,
                                  double* __restrict__ scal)
{
    int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    const unsigned mask = blk_mask[m];
    double A[B][B], b[B];
#pragma unroll
    for (int i = 0; i < B; ++i) {
        const bool fi = mask & (1u << i);
        b[i] = fi ? -g[(int64_t)m * B + i] : 0.0;
#pragma unroll
        for (int j = 0; j < B; ++j) {
            const bool fj = mask & (1u << j);
            double v = (fi && fj) ? blk[(int64_t)m * (B * B) + i * B + j] : 0.0;
            if (i == j) v = (fi && v > 0.0) ? v + lambda * v : 1.0;  // fixed or unobserved: identity row
            A[i][j] = v;
        }
    }
    bool ok = true;
#pragma unroll
    for (int j = 0; j < B; ++j) {
        double d = A[j][j];
#pragma unroll
        for (int k = 0; k < j; ++k) d -= A[j][k] * A[j][k];
        if (!(d > 0.0)) { ok = false; d = 1.0; }
        d = sqrt(d);
        A[j][j] = d;
        const double inv = 1.0 / d;
#pragma unroll
        for (int i = j + 1; i < B; ++i) {
            double s = A[i][j];
#pragma unroll
            for (int k = 0; k < j; ++k) s -= A[i][k] * A[j][k];
            A[i][j] = s * inv;
        }
    }
    if (!ok) scal[5] = 1.0;
    // y = L^-1 b
#pragma unroll
    for (int i = 0; i < B; ++i) {
        double s = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s -= A[i][k] * b[k];
        b[i] = s / A[i][i];
    }
#pragma unroll
    for (int i = 0; i < B; ++i) {
        yout[(int64_t)m * B + i] = b[i];
#pragma unroll
        for (int j = 0; j < B; ++j) Lout[(int64_t)m * (B * B) + i * B + j] = (j <= i) ? A[i][j] : 0.0;
    }
}

// One row of a coupling block times L_b^-T: z = x L_b^-T (forward substitution L_b z^T = x^T; x reads as zero unless
// row_free, and so does every entry whose bit is clear in `live`), and dot += z . y_b -- a row of Z and its share of the
// reduced right-hand side.  Lb = the factor of block b, y = [n][B] (all blocks)
template <int B>
__device__ __forceinline__ void tri_row(const double* x, bool row_free, unsigned live, const double* Lb, const double* y, int b,
                                        double (&z)[B], double& dot)
{
#pragma unroll
    for (int i = 0; i < B; ++i) {
        double v = (row_free && (live & (1u << i))) ? x[i] : 0.0;
#pragma unroll
        for (int k = 0; k < i; ++k) v -= Lb[i * B + k] * z[k];
        z[i] = v / Lb[i * B + i];
        dot = fma(z[i], y[(int64_t)b * B + i], dot);
    }
}

// Z rows of one segment: z = w L^-T  (solve L z^T = w^T), scattered into the dense column-major Z.  The same threads
// also form the pose part of the reduced right-hand side, rhs_c -= Z_{c,m} y_m: segments are sorted by camera, so a
// block's contributions fall on at most a few cameras and are combined in shared memory before they reach global
// memory (one FP64 reduction per block, camera and row instead of one per segment and row).
constexpr int Z_CAM_WIN = 4;
__global__ void __launch_bounds__(256)
k_lm_segment_Z(int64_t S, int64_t nc, const int32_t* __restrict__ seg_cam, const int32_t* __restrict__ seg_pose,
               const double* __restrict__ W, const double* __restrict__ L, const double* __restrict__ y,
               const uint16_t* __restrict__ cam_mask, const uint8_t* __restrict__ pose_mask, const int32_t* __restrict__ pose_slot,
               double* __restrict__ Z, double* __restrict__ rhs)
{
    __shared__ double s_acc[Z_CAM_WIN * 15];
    __shared__ int s_c0;
    const int64_t t0 = blockIdx.x * (int64_t)blockDim.x;
    if (threadIdx.x < Z_CAM_WIN * 15) s_acc[threadIdx.x] = 0.0;
    if (threadIdx.x == 0) s_c0 = seg_cam[min(t0 / 15, S - 1)];
    __syncthreads();
    const int64_t t = t0 + threadIdx.x;
    if (t < S * 15) {
        const int64_t s = t / 15;
        const int a = (int)(t % 15);
        const int c = seg_cam[s], m = seg_pose[s];
        const bool row_free = cam_mask[c] & (1u << a);
        const unsigned pm = pose_mask[m];
        double z[6], dot = 0.0;
        tri_row<6>(W + s * 90 + a * 6, row_free, pm, L + (int64_t)m * 36, y, m, z, dot);
        const int64_t col0 = 6 * (int64_t)(pose_slot ? pose_slot[m] : m);
#pragma unroll
        for (int i = 0; i < 6; ++i) Z[(col0 + i) * nc + (int64_t)c * 15 + a] = z[i];
        const int cw = c - s_c0;
        if (dot != 0.0) {
            if (cw >= 0 && cw < Z_CAM_WIN) atomicAdd(&s_acc[cw * 15 + a], -dot);
            else atomicAdd(rhs + (int64_t)c * 15 + a, -dot);
        }
    }
    __syncthreads();
    if (threadIdx.x < Z_CAM_WIN * 15) {
        const double v = s_acc[threadIdx.x];
        if (v != 0.0) atomicAdd(rhs + (int64_t)(s_c0 + threadIdx.x / 15) * 15 + threadIdx.x % 15, v);
    }
}

// S = [[U + lambda D, .], [X^T, P + lambda D]] (lower triangle; cameras first, then -- self-calibration chain -- the
// second block set P of n B x B blocks: the target points (B = 3, coupling X = Xck) or the poses (B = 6, coupling X = the
// W blocks placed through seg_of)), masked, every other entry zero (each entry of S is written exactly once: no memset);
// rhs = -g masked, g copy (for the convergence test); also clears the step scalars and the factorisation status.
// Template chain: no second set (nl = 15 C), either instantiation.
template <int B>
__global__ void k_lm_init_reduced(int C, int n, int64_t nc, int64_t nl, double lambda, const double* __restrict__ U,
                                  const double* __restrict__ gc, const double* __restrict__ cost, const uint16_t* __restrict__ cam_mask,
                                  const double* __restrict__ P, const double* __restrict__ gP, const uint8_t* __restrict__ P_mask,
                                  const double* __restrict__ Xck, const double* __restrict__ W, const int32_t* __restrict__ seg_of,
                                  double* __restrict__ Smat, double* __restrict__ rhs, double* __restrict__ gcopy,
                                  double* __restrict__ cost_out, double* __restrict__ scal, int* __restrict__ info)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < 8) scal[t] = 0.0;
    if (t == 8) { *info = 0; *cost_out = *cost; }
    if (t >= nc * nc) return;
    const int64_t col = t / nc, row = t % nc;      // column-major S
    const int64_t n_cam = 15 * (int64_t)C;
    double v = 0.0;
    if (row >= nl || col >= nl) {       // padding rows: zero here, identity after the all-reduce (k_lm_fix_diag)
        if (row == col) { rhs[row] = 0.0; gcopy[row] = 0.0; }
    } else if (row < n_cam && col < n_cam) {
        const int c = (int)(row / 15), a = (int)(row % 15), cb = (int)(col / 15), b = (int)(col % 15);
        if (c == cb) {
            const unsigned mask = cam_mask[c];
            const bool fa = mask & (1u << a), fb = mask & (1u << b);
            v = (fa && fb) ? U[(int64_t)c * 225 + a * 15 + b] : 0.0;
            if (a == b) {
                // fixed rows: zero here, set to the identity after the all-reduce (k_lm_fix_diag)
                v = fa ? v + lambda * v : 0.0;
                rhs[row] = fa ? -gc[row] : 0.0;
                gcopy[row] = fa ? gc[row] : 0.0;
            }
        }
    } else if (row >= n_cam && col >= n_cam) {
        const int64_t jr = row - n_cam, jc = col - n_cam;
        const int k = (int)(jr / B), a = (int)(jr % B), kb = (int)(jc / B), b = (int)(jc % B);
        if (k == kb) {
            const unsigned mask = P_mask[k];
            const bool fa = mask & (1u << a), fb = mask & (1u << b);
            v = (fa && fb) ? P[(int64_t)k * (B * B) + a * B + b] : 0.0;
            if (a == b) {
                v = fa ? v + lambda * v : 0.0;
                rhs[row] = fa ? -gP[jr] : 0.0;
                gcopy[row] = fa ? gP[jr] : 0.0;
            }
        }
    } else if (row >= n_cam) {   // second-set row (block k, coordinate a), camera column (camera c, coordinate i)
        const int64_t jr = row - n_cam;
        const int k = (int)(jr / B), a = (int)(jr % B), c = (int)(col / 15), i = (int)(col % 15);
        if (B == 3) {            // points: Xck[c][k][i][a]
            if ((P_mask[k] & (1u << a)) && (cam_mask[c] & (1u << i))) v = Xck[(((int64_t)c * n + k) * 15 + i) * 3 + a];
        } else {                 // poses: W_s[i][a] of the segment s of (camera c, pose k)
            const int32_t s = seg_of[(int64_t)c * n + k];
            if (s >= 0 && (P_mask[k] & (1u << a)) && (cam_mask[c] & (1u << i))) v = W[(int64_t)s * 90 + i * 6 + a];
        }
    }
    Smat[t] = v;
}

// Point rows of Z (self-calibration chain): for every (pose, key) pair and point coordinate a, z = Ymk[m][k][:, a]^T L_m^-T,
// scattered into the dense column-major Z next to the camera rows, and rhs[point row] -= z . y_m.  Pairs without
// observations are all-zero blocks and are skipped (Z is cleared once: its sparsity pattern is static).
__global__ void __launch_bounds__(256)
k_lm_point_Z(int M, int K, int64_t nc, int64_t row0, const double* __restrict__ Ymk, const double* __restrict__ L,
             const double* __restrict__ y, const uint8_t* __restrict__ pose_mask, const uint8_t* __restrict__ key_mask,
             const int32_t* __restrict__ pose_slot, double* __restrict__ Z, double* __restrict__ rhs)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= (int64_t)M * K * 3) return;
    const int a = (int)(t % 3);
    const int64_t mk = t / 3;
    const int k = (int)(mk % K), m = (int)(mk / K);
    const double* Y = Ymk + mk * 18;
    double w[6];
    bool any = false;
#pragma unroll
    for (int i = 0; i < 6; ++i) { w[i] = Y[3 * i + a]; any = any || (w[i] != 0.0); }
    if (!any) return;
    const bool row_free = key_mask[k] & (1u << a);
    const unsigned pm = pose_mask[m];
    double z[6], dot = 0.0;
    tri_row<6>(w, row_free, pm, L + (int64_t)m * 36, y, m, z, dot);
    const int64_t row = row0 + 3 * (int64_t)k + a;
    const int64_t col0 = 6 * (int64_t)(pose_slot ? pose_slot[m] : m);
#pragma unroll
    for (int i = 0; i < 6; ++i) Z[(col0 + i) * nc + row] = z[i];
    if (dot != 0.0) atomicAdd(rhs + row, -dot);
}

// ---- point elimination (self-calibration chain, 3 K > 6 M) ------------------------------------------------------------
__global__ void k_seg_of(int64_t S, int M, const int32_t* __restrict__ seg_cam, const int32_t* __restrict__ seg_pose, int32_t* __restrict__ seg_of)
{
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s < S) seg_of[(int64_t)seg_cam[s] * M + seg_pose[s]] = (int32_t)s;
}

// Z rows of the point elimination: for reduced row r (camera or pose unknown) and point k, z = x L_k^-T with x the 1 x 3
// coupling block row (Xck / Ymk), written to the dense column-major Z [3 K][nc]; rhs[r] -= z . y_k.  A thread handles one
// row and PT_CHUNK consecutive points (one reduction per thread, consecutive rows in consecutive lanes).
constexpr int PT_CHUNK = 4;
__global__ void __launch_bounds__(128)
k_lm_point_elim_Z(int C, int M, int K, int64_t nc, int64_t nl, const double* __restrict__ Xck, const double* __restrict__ Ymk,
                  const double* __restrict__ L, const double* __restrict__ y, const uint16_t* __restrict__ cam_mask,
                  const uint8_t* __restrict__ pose_mask, const uint8_t* __restrict__ key_mask, double* __restrict__ Z,
                  double* __restrict__ rhs)
{
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int k0 = blockIdx.y * PT_CHUNK;
    if (r >= nc) return;
    const int64_t n_cam = 15 * (int64_t)C;
    const bool is_cam = r < n_cam, live = r < nl;
    int blk = 0, a = 0;
    bool row_free = false;
    if (live) {
        if (is_cam) { blk = (int)(r / 15); a = (int)(r % 15); row_free = cam_mask[blk] & (1u << a); }
        else { blk = (int)((r - n_cam) / 6); a = (int)((r - n_cam) % 6); row_free = pose_mask[blk] & (1u << a); }
    }
    double dot = 0.0;
    for (int k = k0; k < min(K, k0 + PT_CHUNK); ++k) {
        double z[3] = {0.0, 0.0, 0.0};
        if (row_free) {
            const double* x = is_cam ? Xck + (((int64_t)blk * K + k) * 15 + a) * 3 : Ymk + (((int64_t)blk * K + k) * 6 + a) * 3;
            tri_row<3>(x, true, key_mask[k], L + (int64_t)k * 9, y, k, z, dot);
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) Z[(3 * (int64_t)k + i) * nc + r] = z[i];   // every entry is written: no memset
    }
    if (dot != 0.0) atomicAdd(rhs + r, -dot);
}

// rows whose diagonal is exactly zero after the reduction (fixed, or unobserved by every rank) -> identity
__global__ void k_lm_fix_diag(int64_t nc, double* __restrict__ Smat)
{
    int64_t a = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (a < nc && Smat[a * nc + a] == 0.0) Smat[a * nc + a] = 1.0;
}

// delta_b = L_b^-T (y_b - Z_b^T delta_r), one warp per eliminated block: the B dot products t_i = Z[:, B slot(b) + i] .
// delta_r (Z is column-major with nc contiguous rows per column, so the lanes stride over one column: coalesced) are
// formed here instead of by a library GEMV over the whole of Z, then lane 0 runs the B x B back substitution.  delta_r is
// the solution of the reduced system (all nc rows); delta_b the set's part of the parameter-string step.
template <int B>
__global__ void __launch_bounds__(128)
k_lm_block_back(int n, int64_t nc, const double* __restrict__ L, const double* __restrict__ y, const double* __restrict__ Z,
                const int32_t* __restrict__ slot, const double* __restrict__ delta_r, double* __restrict__ delta_b)
{
    const int m = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (m >= n) return;
    double t[B];
#pragma unroll
    for (int i = 0; i < B; ++i) t[i] = 0.0;
    const double* Zm = Z + (int64_t)(slot ? slot[m] : m) * B * nc;
    for (int64_t a = lane; a < nc; a += 32) {
        const double d = delta_r[a];
#pragma unroll
        for (int i = 0; i < B; ++i) t[i] = fma(Zm[i * nc + a], d, t[i]);
    }
#pragma unroll
    for (int i = 0; i < B; ++i)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t[i] += __shfl_xor_sync(0xffffffffu, t[i], o);
    if (lane != 0) return;
    const double* Lm = L + (int64_t)m * (B * B);
    double v[B];
#pragma unroll
    for (int i = 0; i < B; ++i) v[i] = y[(int64_t)m * B + i] - t[i];
#pragma unroll
    for (int i = B - 1; i >= 0; --i) {
        double s = v[i];
#pragma unroll
        for (int k = i + 1; k < B; ++k) s -= Lm[k * B + i] * v[k];
        v[i] = s / Lm[i * B + i];
    }
#pragma unroll
    for (int i = 0; i < B; ++i) delta_b[(int64_t)m * B + i] = v[i];
}

// delta (parameter-string layout): [intr | extr | pose (| point)] from the camera (15 per camera), pose and point parts of
// the step, each read from the reduced solution or, for the eliminated set, from delta itself (written by
// k_lm_block_back).  Also accumulates pred = sum delta (lambda D delta + b), |delta|^2, |x|^2 and |g|_inf of the LOCAL
// pose part plus (rank 0 only for the replicated camera / point norms) the replicated part; D and b are this rank's
// partial sums.
__global__ void k_lm_assemble_delta(int C, int M, int K3, double lambda, const double* __restrict__ dc, const double* __restrict__ dp,
                                    const double* __restrict__ dk, const double* __restrict__ U, const double* __restrict__ gc, const double* __restrict__ V,
                                    const double* __restrict__ gp, const double* __restrict__ Pk, const double* __restrict__ gk,
                                    const uint16_t* __restrict__ cam_mask, const uint8_t* __restrict__ pose_mask,
                                    const uint8_t* __restrict__ key_mask, const double* __restrict__ params,
                                    double* __restrict__ delta, double* __restrict__ scal, int rank0, int pts_ginf)
{
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t n_cam = 15 * (int64_t)C, n_pose = 6 * (int64_t)M;
    const int64_t total = n_cam + n_pose + K3;
    double pred = 0.0, dx2 = 0.0, x2 = 0.0, ginf = 0.0;
    if (t < total) {
        double d, D, g;
        bool replicated, f;
        if (t < n_cam) {
            int c, a;
            if (t < 9 * (int64_t)C) { c = (int)(t / 9); a = (int)(t % 9); }
            else { c = (int)((t - 9 * (int64_t)C) / 6); a = 9 + (int)((t - 9 * (int64_t)C) % 6); }
            f = cam_mask[c] & (1u << a);
            d = f ? dc[c * 15 + a] : 0.0;
            D = f ? U[c * 225 + a * 16] : 0.0;
            g = f ? gc[c * 15 + a] : 0.0;
            replicated = true;
        } else if (t < n_cam + n_pose) {
            const int64_t r = t - n_cam;
            const int m = (int)(r / 6), a = (int)(r % 6);
            f = pose_mask[m] & (1u << a);
            d = f ? dp[r] : 0.0;
            D = f ? V[(int64_t)m * 36 + a * 7] : 0.0;
            g = f ? gp[r] : 0.0;
            replicated = false;
        } else {
            const int64_t j = t - n_cam - n_pose;
            const int k = (int)(j / 3), a = (int)(j % 3);
            f = key_mask[k] & (1u << a);
            d = f ? dk[j] : 0.0;
            D = f ? Pk[(int64_t)k * 9 + a * 4] : 0.0;
            g = f ? gk[j] : 0.0;
            replicated = true;
            if (pts_ginf) ginf = fabs(g);   // point elimination: the point gradient is not part of the reduced copy
        }
        delta[t] = d;
        pred = d * (lambda * D * d - g);
        if (!replicated || rank0) {
            dx2 = d * d;
            x2 = f ? params[t] * params[t] : 0.0;   // |x| of the xtol test is the norm of the FREE vector
        }
        if (!replicated) ginf = fabs(g);  // the replicated gradient norm is taken from the all-reduced copy (k_lm_take_step)
    }
    // block reduction
    __shared__ double sh[4][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        pred += __shfl_xor_sync(0xffffffffu, pred, o);
        dx2 += __shfl_xor_sync(0xffffffffu, dx2, o);
        x2 += __shfl_xor_sync(0xffffffffu, x2, o);
        ginf = fmax(ginf, __shfl_xor_sync(0xffffffffu, ginf, o));
    }
    if (lane == 0) { sh[0][warp] = pred; sh[1][warp] = dx2; sh[2][warp] = x2; sh[3][warp] = ginf; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, b = 0, c2 = 0, g2 = 0;
        for (int w = 0; w < (blockDim.x >> 5); ++w) { a += sh[0][w]; b += sh[1][w]; c2 += sh[2][w]; g2 = fmax(g2, sh[3][w]); }
        atomicAdd(scal + 0, a);
        atomicAdd(scal + 1, b);
        atomicAdd(scal + 2, c2);
        // non-negative doubles order like their bit patterns
        atomicMax((unsigned long long*)(scal + 3), (unsigned long long)__double_as_longlong(g2));
    }
}

// backup <- params, params += delta (the move to the trial point), and scal[4] = |g_cam|_inf in the same launch
// (nc = 0, the dense fallback: the move alone)
__global__ void k_lm_take_step(int64_t L, int64_t nc, const double* __restrict__ delta, double* __restrict__ params,
                               double* __restrict__ backup, const double* __restrict__ gcopy, double* __restrict__ scal)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < L) {
        const double v = params[i];
        backup[i] = v;
        params[i] = v + delta[i];
    }
    double m = i < nc ? fabs(gcopy[i]) : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.0) atomicMax((unsigned long long*)(scal + 4), (unsigned long long)__double_as_longlong(m));
}

// Multi-rank: everything that has to be combined across ranks after the trial evaluation goes into ONE sum all-reduce:
// comb = [pred | |dx|^2 | |x|^2 | trial cost | pose-factorisation failure flag | per-rank slots of the pose gradient
// inf-norm (own slot set, others 0)]; after the sum every rank holds all the norms and takes their maximum, and a
// failure on any rank is seen by all of them, so the ranks take the same branch (k_lm_gather_readback).
__global__ void k_lm_pack_scalars(const double* __restrict__ scal, const double* __restrict__ cost_trial, int rank, int world,
                                  double* __restrict__ comb)
{
    const int t = threadIdx.x + blockIdx.x * blockDim.x;
    if (t < 3) comb[t] = scal[t];
    else if (t == 3) comb[3] = *cost_trial;
    else if (t == 4) comb[4] = scal[5];
    else if (t < 5 + world) comb[t] = (t - 5 == rank) ? scal[3] : 0.0;
}

// everything the host reads after an iteration, gathered into one buffer: scal[0..7] | info | cost of the linearisation.
// comb != nullptr: the all-reduced scalars of k_lm_pack_scalars replace the rank-local ones.
__global__ void k_lm_gather_readback(const double* __restrict__ scal, const int* __restrict__ info, const double* __restrict__ cost_lin,
                                     const double* __restrict__ cost_trial, const double* __restrict__ comb, int world,
                                     double* __restrict__ out)
{
    const int t = threadIdx.x;
    if (t < 8) {
        double v = scal[t];
        if (comb) {
            if (t < 3) v = comb[t];
            else if (t == 3) { v = 0.0; for (int r = 0; r < world; ++r) v = fmax(v, comb[5 + r]); }
            else if (t == 5) v = comb[4];
            else if (t == 6) v = comb[3];
        } else if (t == 6 && cost_trial) v = *cost_trial;
        out[t] = v;
    }
    if (t == 8) out[8] = (double)*info;
    if (t == 9) out[9] = *cost_lin;
}

// dense path: Hd = H + lambda diag(H), rhs = -g, clears the factorisation status; pred / norms after the solve
__global__ void k_dense_damp(int64_t n, double lambda, const double* __restrict__ H, const double* __restrict__ g,
                             double* __restrict__ Hd, double* __restrict__ rhs, int* __restrict__ info)
{
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t == 0) *info = 0;
    if (t >= n * n) return;
    const int64_t i = t / n, j = t % n;
    double v = H[t];
    if (i == j) {
        v += lambda * fmax(v, 1e-12);
        rhs[i] = -g[i];
    }
    Hd[t] = v;
}

__global__ void k_dense_delta(int64_t n, double lambda, const double* __restrict__ d, const double* __restrict__ H,
                              const double* __restrict__ g, const int32_t* __restrict__ free_idx, const double* __restrict__ params,
                              double* __restrict__ delta_full, double* __restrict__ scal)
{
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double pred = 0, dx2 = 0, x2 = 0, ginf = 0;
    if (j < n) {
        const double dj = d[j];
        const int32_t pi = free_idx[j];
        delta_full[pi] = dj;
        pred = dj * (lambda * fmax(H[j * n + j], 1e-12) * dj - g[j]);
        dx2 = dj * dj;
        x2 = params[pi] * params[pi];
        ginf = fabs(g[j]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        pred += __shfl_xor_sync(0xffffffffu, pred, o);
        dx2 += __shfl_xor_sync(0xffffffffu, dx2, o);
        x2 += __shfl_xor_sync(0xffffffffu, x2, o);
        ginf = fmax(ginf, __shfl_xor_sync(0xffffffffu, ginf, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(scal + 0, pred);
        atomicAdd(scal + 1, dx2);
        atomicAdd(scal + 2, x2);
        atomicMax((unsigned long long*)(scal + 3), (unsigned long long)__double_as_longlong(ginf));
    }
}

__global__ void k_gather_free(int64_t n, const int32_t* __restrict__ free_idx, const double* __restrict__ params, double* __restrict__ x)
{
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < n) x[j] = params[free_idx[j]];
}

// the two sets of normal-equation outputs [U | gc | cost | pad | V | gp | W] trade places
static void swap_normal_buffers(pcs_problem* p, LmWorkspace* w)
{
    double* other = (p->ne == w->ne_orig) ? w->ne_alt : w->ne_orig;
    const int64_t o_gc = p->gc - p->ne, o_cost = p->cost - p->ne, o_V = p->V - p->ne, o_gp = p->gp - p->ne, o_W = p->W - p->ne;
    const int64_t o_P = p->Pk ? p->Pk - p->ne : 0, o_gk = p->Pk ? p->gk - p->ne : 0, o_X = p->Pk ? p->Xck - p->ne : 0,
                  o_Y = p->Pk ? p->Ymk - p->ne : 0;
    const bool pts = p->Pk != nullptr;
    p->ne = other; p->U = other; p->gc = other + o_gc; p->cost = other + o_cost; p->V = other + o_V; p->gp = other + o_gp;
    p->W = other + o_W;
    if (pts) { p->Pk = other + o_P; p->gk = other + o_gk; p->Xck = other + o_X; p->Ymk = other + o_Y; }
}

void lm_free(pcs_problem* p)
{
    LmWorkspace* w = (LmWorkspace*)p->lm_ws;
    if (!w) return;
    // a solve that returned early on an error may have left the problem on the second output set
    if (w->ne_alt && w->ne_orig && p->ne == w->ne_alt) swap_normal_buffers(p, w);
    schur_plan_free(&w->plan);
    if (w->seg_of) cudaFree(w->seg_of);
    double* ptrs[] = {w->L, w->y, w->Z, w->red, w->delta, w->backup, w->scal, w->Hd, w->rhs, w->Ldiag, w->ne_alt, w->cov_Xi};
    for (double* q : ptrs) if (q) cudaFree(q);
    if (w->info) cudaFree(w->info);
    if (w->bar) cudaFree(w->bar);
    if (w->h_read) cudaFreeHost(w->h_read);
    if (w->d_read) cudaFree(w->d_read);
    if (w->comb) cudaFree(w->comb);
    if (w->ev0) cudaEventDestroy(w->ev0);
    if (w->ev1) cudaEventDestroy(w->ev1);
    delete w;
    p->lm_ws = nullptr;
}

// The LM path of the problem: the one its workspace was built for, else the one a workspace built now takes.  Template
// chain: the poses are eliminated.  Self-calibration chain: poses AND points are block diagonal but coupled to each other,
// so only one of them can go; the larger one does (3 K point unknowns against 6 M pose unknowns -- on the reference's
// ccube fixture a reduced system of 162 instead of 1503 unknowns).  The point elimination is single-rank: its reduced
// system contains the (rank-local) poses.  Without the (camera, key) / (pose, key) tables (p->Pk) the self-calibration
// chain takes the dense fallback.  Switch for A/B runs and tests, read whenever a workspace is built:
// PCS_LM_SELFCAL=dense forces the dense fallback of the self-calibration chain, PCS_LM_SELFCAL=poses its pose elimination.
static LmPath lm_path(const pcs_problem* p)
{
    if (p->lm_ws) return ((const LmWorkspace*)p->lm_ws)->path;
    if (p->chain == PCS_CHAIN_TEMPLATE) return {6, 0};
    const char* env = std::getenv("PCS_LM_SELFCAL");
    if (!p->Pk || (env && env[0] == 'd')) return {0, 0};
    const bool points = p->world == 1 && 3 * (int64_t)p->K > 6 * (int64_t)p->M && !(env && env[0] == 'p');
    return points ? LmPath{3, 6} : LmPath{6, 3};
}

// the block set B of the problem's current normal-equation outputs (B = 0: the empty set)
static BlockSet block_set(const pcs_problem* p, const LmWorkspace* w, int B)
{
    BlockSet s;
    s.B = B;
    if (B == 6) {
        s.n = p->M; s.off = 15 * (int64_t)p->C; s.blk = p->V; s.g = p->gp; s.mask = p->pose_mask; s.slot = w->plan.pose_slot;
    } else if (B == 3) {
        s.n = p->K; s.off = 15 * (int64_t)p->C + 6 * (int64_t)p->M; s.blk = p->Pk; s.g = p->gk; s.mask = p->key_mask;
    }
    return s;
}

static int lm_prepare_impl(pcs_problem* p, LmWorkspace* w);

// The workspace is published on the problem only after every allocation succeeded; a failure half-way (out of memory
// for Z, n_free over the dense limit, ...) frees what was built, so that the next call starts from scratch instead of
// launching on NULL buffers.  It is laid out for the world size of the moment (the path, the all-reduce buffers):
// pcs_set_allreduce frees it when the world size changes.
static int lm_prepare(pcs_problem* p)
{
    if (p->lm_ws) return PCS_OK;
    LmWorkspace* w = new LmWorkspace();
    w->path = lm_path(p);
    p->lm_ws = w;
    const int rc = lm_prepare_impl(p, w);
    if (rc != PCS_OK) lm_free(p);
    return rc;
}

static int lm_prepare_impl(pcs_problem* p, LmWorkspace* w)
{
    // PCS_LM_SCHUR=dense (A/B runs and tests, read whenever a workspace is built): the full iteration space (identity
    // column order) of the pose elimination
    const char* env_schur = std::getenv("PCS_LM_SCHUR");
    const bool dense_schur = env_schur && env_schur[0] == 'd';
    PCS_CUDA(cudaMalloc((void**)&w->delta, (size_t)p->L * 8));
    PCS_CUDA(cudaMalloc((void**)&w->backup, (size_t)p->L * 8));
    PCS_CUDA(cudaMalloc((void**)&w->scal, 8 * 8));
    PCS_CUDA(cudaMalloc((void**)&w->info, sizeof(int)));
    PCS_CUDA(cudaMalloc((void**)&w->d_read, 10 * 8));
    PCS_CUDA(cudaMallocHost((void**)&w->h_read, 10 * 8));
    PCS_CUDA(cudaMemsetAsync(w->delta, 0, (size_t)p->L * 8, p->stream));
    PCS_CUDA(cudaEventCreate(&w->ev0));
    PCS_CUDA(cudaEventCreate(&w->ev1));
    if (w->path.elim_B) {
        const BlockSet e = block_set(p, w, w->path.elim_B), r = block_set(p, w, w->path.red_B);
        w->nl = 15 * (int64_t)p->C + (int64_t)r.B * r.n;   // cameras (+ the second set)
        w->np = (int64_t)e.B * e.n;                        // eliminated unknowns
        w->nc = (w->nl + 31) / 32 * 32;
        PCS_CUDA(cudaMalloc((void**)&w->L, (size_t)(w->np * e.B) * 8));
        PCS_CUDA(cudaMalloc((void**)&w->y, (size_t)w->np * 8));
        PCS_CUDA(cudaMalloc((void**)&w->Z, (size_t)(w->nc * w->np) * 8));
        PCS_CUDA(cudaMemsetAsync(w->Z, 0, (size_t)(w->nc * w->np) * 8, p->stream));  // sparsity pattern is static
        if (r.B == 6) {
            PCS_CUDA(cudaMalloc((void**)&w->seg_of, (size_t)p->C * p->M * sizeof(int32_t)));
            PCS_CUDA(cudaMemsetAsync(w->seg_of, 0xff, (size_t)p->C * p->M * sizeof(int32_t), p->stream));
            if (p->n_seg) k_seg_of<<<grid_for(p->n_seg, 256), 256, 0, p->stream>>>(p->n_seg, p->M, p->seg_cam, p->seg_pose, w->seg_of);
            PCS_CUDA(cudaGetLastError());
        }
        // block-sparse pose elimination
        if (e.B == 6 && !dense_schur) PCS_TRY(schur_plan_build(p, w->nc, w->nl, &w->plan));
        w->red_doubles = w->nc * w->nc + 2 * w->nc + 1;
        PCS_CUDA(cudaMalloc((void**)&w->red, (size_t)w->red_doubles * 8));
        PCS_TRY(chol_prepare(p->device, w->nc, &w->Ldiag, &w->bar, &w->chol_grid));
        PCS_CUDA(cudaMalloc((void**)&w->ne_alt, (size_t)p->ne_doubles * 8));
        w->ne_orig = p->ne;
        PCS_CUDA(cudaMalloc((void**)&w->comb, (size_t)(5 + p->world) * 8));
    } else {
        const int64_t n = p->n_free;
        PCS_REQUIRE(n > 0 && n <= 32768, "dense LM path needs 0 < n_free <= 32768");
        if (!p->dense) PCS_CUDA(cudaMalloc((void**)&p->dense, (size_t)(n * n + n + 1) * 8));
        w->H = p->dense;
        PCS_CUDA(cudaMalloc((void**)&w->Hd, (size_t)(n * n) * 8));
        PCS_CUDA(cudaMalloc((void**)&w->rhs, (size_t)n * 8));
        PCS_TRY(chol_prepare(p->device, n, &w->Ldiag, &w->bar, &w->chol_grid));
    }
    return PCS_OK;
}

// evaluate the block normal equations at the current p->params (tables refreshed, reduction targets cleared in the same launch)
static int eval_normal(pcs_problem* p)
{
    PCS_TRY(launch_prepare(p, false, nullptr, p->ne, ne_zero_doubles(p)));
    PCS_TRY(launch_normal_blocks(p, true));
    if (p->chain == PCS_CHAIN_SELFCAL) PCS_TRY(launch_point_blocks(p));
    return PCS_OK;
}

// The reduced system at damping lambda, built in w->red and ready for the factorisation: S (lower triangle; fixed and
// unobserved unknowns are identity rows), rhs = -g_red - Z y, the gradient copy and the cost; w->L / w->y hold the
// eliminated blocks' Cholesky factors and L_b^-1 (-g_b), w->Z the coupling L_b^-T.  Multi-rank: S | rhs | g | cost are
// all-reduced here.  The first half of every LM step, and what pcs_covariance factors at lambda = 0.
static int build_reduced(pcs_problem* p, LmWorkspace* w, double lambda)
{
    cudaStream_t st = p->stream;
    const int64_t nc = w->nc, np = w->np;
    const BlockSet e = block_set(p, w, w->path.elim_B), r = block_set(p, w, w->path.red_B);
    double* Smat = w->red;
    double* rhs = w->red + nc * nc;
    double* gcopy = rhs + nc;
    double* cost_r = gcopy + nc;
    const auto init = r.B == 6 ? k_lm_init_reduced<6> : k_lm_init_reduced<3>;
    init<<<grid_for(std::max<int64_t>(nc * nc, 9), 256), 256, 0, st>>>(p->C, r.n, nc, w->nl, lambda, p->U, p->gc, p->cost, p->cam_mask,
                                                                      r.blk, r.g, r.mask, p->Xck, p->W, w->seg_of, Smat, rhs, gcopy,
                                                                      cost_r, w->scal, w->info);
    const auto factor = e.B == 6 ? k_lm_block_factor<6> : k_lm_block_factor<3>;
    factor<<<grid_for(e.n, 128), 128, 0, st>>>(e.n, lambda, e.blk, e.g, e.mask, w->L, w->y, w->scal);
    if (e.B == 3) {
        k_lm_point_elim_Z<<<dim3(grid_for(nc, 128), (p->K + PT_CHUNK - 1) / PT_CHUNK), 128, 0, st>>>(p->C, p->M, p->K, nc, w->nl, p->Xck, p->Ymk, w->L,
                                                                                                  w->y, p->cam_mask, p->pose_mask, p->key_mask, w->Z, rhs);
    } else {
        if (p->n_seg)
            k_lm_segment_Z<<<grid_for(p->n_seg * 15, 256), 256, 0, st>>>(p->n_seg, nc, p->seg_cam, p->seg_pose, p->W, w->L, w->y,
                                                                         p->cam_mask, p->pose_mask, e.slot, w->Z, rhs);
        if (r.B == 3)
            k_lm_point_Z<<<grid_for((int64_t)p->M * p->K * 3, 256), 256, 0, st>>>(p->M, p->K, nc, 15 * (int64_t)p->C, p->Ymk, w->L, w->y,
                                                                                 p->pose_mask, p->key_mask, e.slot, w->Z, rhs);
    }
    PCS_CUDA(cudaGetLastError());
    PCS_TRY(launch_schur_syrk(st, p->sm_count, nc, np, w->Z, Smat, &w->plan));
    if (p->allreduce) {
        int rc = p->allreduce(p->allreduce_user, w->red, w->red_doubles, 0, (void*)st);
        if (rc != 0) { set_error("all-reduce callback failed"); return PCS_ERR_CUDA; }
    }
    k_lm_fix_diag<<<grid_for(nc, 256), 256, 0, st>>>(nc, Smat);
    return PCS_OK;
}

// A = L L^T and rhs <- A^-1 rhs for A of order n (leading dimension ld, lower triangle read), with the workspace's
// Cholesky-kernel state: the kernel leaves the off-diagonal tiles of L in A, the diagonal ones in Ldiag, and only ever
// raises w->info, which must be zero on entry
static int chol_solve(pcs_problem* p, LmWorkspace* w, int64_t n, double* A, int64_t ld, double* rhs)
{
    return launch_chol_solve(p->stream, w->chol_grid, n, A, ld, rhs, w->Ldiag, w->bar, &w->bar_base, w->info);
}

// One damped solve of the block path at the current linearisation, enqueued without synchronising.  Afterwards w->delta
// holds the step (parameter-string layout), w->scal = {pred, |dx|^2, |x|^2, |g_pose|_inf, |g_cam|_inf, flag, trial cost, -},
// w->info the factorisation status and cost_r (inside w->red) the all-reduced r.r of the linearisation point.
static int solve_step(pcs_problem* p, LmWorkspace* w, double lambda)
{
    cudaStream_t st = p->stream;
    const int64_t nc = w->nc, n_cam = 15 * (int64_t)p->C;
    double* rhs = w->red + nc * nc;
    PCS_TRY(build_reduced(p, w, lambda));
    PCS_TRY(chol_solve(p, w, nc, w->red, nc, rhs));
    const BlockSet e = block_set(p, w, w->path.elim_B);
    p->n_launches += e.B == 6 ? 8 : 7;
    // rhs now holds the reduced part of the step (cameras, then the second set); the eliminated set's part is written in
    // place into the parameter-string delta
    double* de = w->delta + e.off;
    const auto back = e.B == 6 ? k_lm_block_back<6> : k_lm_block_back<3>;
    back<<<grid_for((int64_t)e.n * 32, 128), 128, 0, st>>>(e.n, nc, w->L, w->y, w->Z, e.slot, rhs, de);
    const double* dp = e.B == 6 ? de : rhs + n_cam;
    const double* dk = e.B == 3 ? de : rhs + n_cam;
    const int K3 = p->chain == PCS_CHAIN_SELFCAL ? 3 * p->K : 0;
    k_lm_assemble_delta<<<grid_for(n_cam + 6 * (int64_t)p->M + K3, 128), 128, 0, st>>>(
        p->C, p->M, K3, lambda, rhs, dp, dk, p->U, p->gc, p->V, p->gp, p->Pk, p->gk, p->cam_mask, p->pose_mask, p->key_mask,
        p->params, w->delta, w->scal, p->rank == 0, e.B == 3);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;   // multi-rank: pred, |dx|^2, |x|^2 and the pose gradient norm are still rank-local here (k_lm_pack_scalars)
}

}  // namespace pcs

using namespace pcs;

extern "C" {

void pcs_lm_default_options(pcs_lm_options* o)
{
    if (!o) return;
    o->max_iter = 100;
    o->verbose = 0;
    o->lambda0 = 1e-3;
    o->ftol = o->xtol = o->gtol = 1e-8;
    o->lambda_min = 1e-12;
    o->lambda_max = 1e12;
}

// dense normal equations at the current parameters, device-resident (pcs_core.cu)
int pcs_normal_dense_dev_internal(pcs_problem* p);

static int lm_solve_impl(pcs_problem* p, const double* x0, const pcs_lm_options* opts_in, double* x_out, pcs_lm_stats* stats)
{
    PCS_REQUIRE(p && x_out, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    pcs_lm_options o;
    if (opts_in) o = *opts_in; else pcs_lm_default_options(&o);
    if (p->world > 1 && lm_path(p).elim_B == 0) {
        // the dense self-calibration fallback is not combined across ranks: refuse instead of letting the replicated
        // camera / point parameters diverge silently
        set_error("pcs_lm_solve: the dense self-calibration fallback is single-rank");
        return PCS_ERR_UNSUPPORTED;
    }
    PCS_TRY(lm_prepare(p));
    LmWorkspace* w = (LmWorkspace*)p->lm_ws;
    cudaStream_t st = p->stream;
    cudaEvent_t ev0 = w->ev0, ev1 = w->ev1;
    PCS_CUDA(cudaEventRecord(ev0, st));
    if (x0) {
        PCS_TRY(ensure_pinned(p, std::max<int64_t>(p->n_free, 1)));
        std::memcpy(p->h_pin, x0, (size_t)p->n_free * 8);
        PCS_CUDA(cudaMemcpyAsync(p->x, p->h_pin, (size_t)p->n_free * 8, cudaMemcpyHostToDevice, st));
        PCS_TRY(launch_scatter_x(p, p->x));
    }
    const bool block = w->path.elim_B != 0;   // block path (both chains); false: dense self-calibration fallback
    const int64_t n = p->n_free;
    int n_normal = 0, n_cost = 0, status = 0, it = 0;
    double lambda = o.lambda0, nu = 2.0;
    double cost = 0.0, cost0 = 0.0, ginf = 0.0;
    double h_scal[8] = {0};

    auto eval_lin = [&]() -> int {  // normal equations at p->params; returns r.r in `cost`
        ++n_normal;
        if (block) return eval_normal(p);
        return pcs_normal_dense_dev_internal(p);
    };
    int rc = eval_lin();
    bool have_cost = false;
    while (rc == PCS_OK && it < o.max_iter) {
        ++it;
        double ginf_cam = 0.0, cost_lin = 0.0, cost_new = 0.0;
        int h_info = 0;
        if (block) {
            // Block path: the damped solve, the step and the evaluation of the TRIAL point with the full
            // normal-equation kernel (into the second output set) are enqueued back to back and read with ONE
            // synchronisation per iteration.  An accepted step already has its linearisation; a rejected one only
            // costs the difference between the full kernel and a residual-only pass.
            rc = solve_step(p, w, lambda);
            if (rc != PCS_OK) break;
            double* gcopy = w->red + w->nc * w->nc + w->nc;
            k_lm_take_step<<<grid_for(std::max<int64_t>(p->L, w->nc), 256), 256, 0, st>>>(p->L, w->nc, w->delta, p->params, w->backup,
                                                                                       gcopy, w->scal);
            swap_normal_buffers(p, w);
            rc = eval_lin();
            if (rc != PCS_OK) break;
            const double* comb = nullptr;
            if (p->allreduce) {   // one combined all-reduce of the step scalars and the trial cost
                k_lm_pack_scalars<<<grid_for(5 + p->world, 64), 64, 0, st>>>(w->scal, p->cost, p->rank, p->world, w->comb);
                if (p->allreduce(p->allreduce_user, w->comb, 5 + p->world, 0, (void*)st) != 0) {
                    set_error("all-reduce callback failed");
                    rc = PCS_ERR_CUDA;
                    break;
                }
                comb = w->comb;
            }
            k_lm_gather_readback<<<1, 32, 0, st>>>(w->scal, w->info, gcopy + w->nc, p->cost, comb, p->world, w->d_read);
            PCS_CUDA(cudaMemcpyAsync(w->h_read, w->d_read, 10 * 8, cudaMemcpyDeviceToHost, st));
            PCS_CUDA(cudaStreamSynchronize(st));
            std::memcpy(h_scal, w->h_read, 8 * 8);
            h_info = (int)w->h_read[8];
            cost_lin = w->h_read[9];
            ginf_cam = h_scal[4];
            cost_new = h_scal[6];
            rc = chol_status(h_info);
            if (rc == PCS_OK && h_scal[5] != 0.0) rc = PCS_ERR_NUMERIC;
        } else {
            double *H = w->H, *g = w->H + n * n, *c = g + n;
            PCS_CUDA(cudaMemsetAsync(w->scal, 0, 8 * 8, st));
            k_dense_damp<<<grid_for(n * n, 256), 256, 0, st>>>(n, lambda, H, g, w->Hd, w->rhs, w->info);
            PCS_TRY(chol_solve(p, w, n, w->Hd, n, w->rhs));
            k_dense_delta<<<grid_for(n, 128), 128, 0, st>>>(n, lambda, w->rhs, H, g, p->free_idx, p->params, w->delta, w->scal);
            PCS_CUDA(cudaMemcpyAsync(h_scal, w->scal, 8 * 8, cudaMemcpyDeviceToHost, st));
            PCS_CUDA(cudaMemcpyAsync(&h_info, w->info, sizeof(int), cudaMemcpyDeviceToHost, st));
            PCS_CUDA(cudaMemcpyAsync(&cost_lin, c, 8, cudaMemcpyDeviceToHost, st));
            PCS_CUDA(cudaStreamSynchronize(st));
            rc = chol_status(h_info);
        }
        // the block path has already moved to the trial point: undo = old parameters + old output set
        auto undo_trial = [&]() -> int {
            if (!block) return PCS_OK;
            PCS_CUDA(cudaMemcpyAsync(p->params, w->backup, (size_t)p->L * 8, cudaMemcpyDeviceToDevice, st));
            swap_normal_buffers(p, w);
            --n_normal;   // the speculative evaluation is not a linearisation that was used
            ++n_cost;
            return PCS_OK;
        };
        if (rc == PCS_ERR_NUMERIC) {  // not positive definite at this damping: raise lambda and retry
            rc = undo_trial();
            lambda = std::min(lambda * 10.0, o.lambda_max);
            if (lambda >= o.lambda_max) { status = -1; break; }
            continue;
        }
        if (rc != PCS_OK) break;
        if (!have_cost) { cost = cost0 = cost_lin; have_cost = true; }
        ginf = std::max(ginf_cam, h_scal[3]);
        if (ginf < o.gtol) { status = 1; rc = undo_trial(); break; }
        const double pred = h_scal[0], dx = std::sqrt(h_scal[1]), xn = std::sqrt(h_scal[2]);
        if (dx < o.xtol * (o.xtol + xn)) { status = 3; rc = undo_trial(); break; }
        if (!block) {
            // trial point, residual-only pass
            k_lm_take_step<<<grid_for(p->L, 256), 256, 0, st>>>(p->L, 0, w->delta, p->params, w->backup, nullptr, w->scal);
            PCS_TRY(launch_prepare(p));
            PCS_TRY(launch_cost_only(p, w->scal + 6));
            ++n_cost;
            if (p->allreduce && p->allreduce(p->allreduce_user, w->scal + 6, 1, 0, (void*)st) != 0) {
                set_error("all-reduce callback failed");
                rc = PCS_ERR_CUDA;
                break;
            }
            PCS_CUDA(cudaMemcpyAsync(&cost_new, w->scal + 6, 8, cudaMemcpyDeviceToHost, st));
            PCS_CUDA(cudaStreamSynchronize(st));
        }
        const double actual = cost - cost_new;          // in units of r.r
        const double rho = (pred > 0.0 && std::isfinite(cost_new)) ? actual / pred : -1.0;
        if (o.verbose)
            std::fprintf(stderr, "[pcs lm] it %3d  cost %.9e  trial %.9e  rho %8.3g  lambda %.2e  |g| %.2e  |dx| %.2e\n", it,
                         0.5 * cost, 0.5 * cost_new, rho, lambda, ginf, dx);
        if (rho > 0.0) {
            const double rel = actual / std::max(cost, 1e-300);
            cost = cost_new;
            const double f = 1.0 - std::pow(2.0 * rho - 1.0, 3.0);
            lambda = std::max(o.lambda_min, lambda * std::max(1.0 / 3.0, f));
            nu = 2.0;
            if (!block) {
                rc = eval_lin();
                if (rc != PCS_OK) break;
            }
            if (rel < o.ftol) { status = 2; break; }
        } else {
            if (block) rc = undo_trial();
            else PCS_CUDA(cudaMemcpyAsync(p->params, w->backup, (size_t)p->L * 8, cudaMemcpyDeviceToDevice, st));
            lambda = std::min(o.lambda_max, lambda * nu);
            nu *= 2.0;
            if (lambda >= o.lambda_max) { status = -1; break; }
        }
    }
    if (block && p->ne != w->ne_orig) {   // callers hold pointers into the original output set (pcs_device_pointers)
        PCS_CUDA(cudaMemcpyAsync(w->ne_orig, p->ne, (size_t)p->ne_doubles * 8, cudaMemcpyDeviceToDevice, st));
        swap_normal_buffers(p, w);
    }
    if (rc == PCS_OK) {
        PCS_TRY(launch_prepare(p));
        if (n) {
            k_gather_free<<<grid_for(n, 256), 256, 0, st>>>(n, p->free_idx, p->params, p->x);
            PCS_CUDA(cudaMemcpyAsync(x_out, p->x, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        }
    }
    PCS_CUDA(cudaEventRecord(ev1, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ev0, ev1);
    if (stats) {
        stats->iterations = it; stats->n_eval_normal = n_normal; stats->n_eval_cost = n_cost; stats->status = status;
        stats->cost_initial = 0.5 * cost0; stats->cost_final = 0.5 * cost; stats->grad_norm_inf = ginf;
        stats->lambda_final = lambda; stats->seconds = ms * 1e-3;
    }
    return rc;
}

int pcs_lm_schur_fraction(pcs_problem* p, double* fraction)
{
    PCS_REQUIRE(p && fraction, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    PCS_TRY(lm_prepare(p));
    const LmWorkspace* w = (const LmWorkspace*)p->lm_ws;
    *fraction = w->plan.units ? w->plan.fraction : 1.0;
    return PCS_OK;
}

static int covariance_impl(pcs_problem* p, const double* x, double* cam, double* pose, double* point, double* s2, int64_t* dof)
{
    PCS_CUDA(cudaSetDevice(p->device));
    if (p->world > 1) {
        set_error("pcs_covariance: the covariance is single-rank (an all-reduce hook is installed)");
        return PCS_ERR_UNSUPPORTED;
    }
    if (lm_path(p).elim_B == 0) {
        set_error("pcs_covariance: the dense self-calibration fallback has no block path to factor");
        return PCS_ERR_UNSUPPORTED;
    }
    PCS_TRY(lm_prepare(p));
    LmWorkspace* w = (LmWorkspace*)p->lm_ws;
    cudaStream_t st = p->stream;
    const int64_t nc = w->nc, np = w->np, n_cam = 15 * (int64_t)p->C;
    if (!w->cov_Xi) PCS_CUDA(cudaMalloc((void**)&w->cov_Xi, (size_t)(nc * nc) * 8));
    if (x && p->n_free > 0) {
        PCS_TRY(ensure_pinned(p, p->n_free));
        std::memcpy(p->h_pin, x, (size_t)p->n_free * 8);
        PCS_CUDA(cudaMemcpyAsync(p->x, p->h_pin, (size_t)p->n_free * 8, cudaMemcpyHostToDevice, st));
        PCS_TRY(launch_scatter_x(p, p->x));
    }
    // FP64 normal equations whatever precision the LM iterations use
    const int precision = p->normal_precision;
    p->normal_precision = PCS_PRECISION_FP64;
    const int rc_eval = eval_normal(p);
    p->normal_precision = precision;
    PCS_TRY(rc_eval);
    double* Smat = w->red;
    PCS_TRY(build_reduced(p, w, 0.0));
    // the factor: off-diagonal tiles of L in S, diagonal tiles in Ldiag
    PCS_TRY(chol_solve(p, w, nc, Smat, nc, w->red + nc * nc));
    // X = L^-1 [I | Z] in place (Z's columns become X_b), then Sigma_red = X_I^T X_I into S (negated), Sigma_bb over L_b
    PCS_TRY(cov_forward_substitution(st, nc, Smat, w->Ldiag, w->cov_Xi, w->Z, np));
    PCS_TRY(cov_reduced_inverse(st, p->sm_count, nc, w->cov_Xi, Smat));
    const BlockSet e = block_set(p, w, w->path.elim_B);
    PCS_TRY(cov_block_marginals(st, e.n, e.B, nc, w->Z, e.slot, w->L));
    // copy-out layout in the (now free) X_I buffer: cam [15 C][15 C], then the reduced set's pose or point blocks
    double* out_cam = w->cov_Xi;
    double* out_red = w->cov_Xi + n_cam * n_cam;
    double* n_obs = w->scal + 7;   // cleared by the reduced-system build
    PCS_TRY(cov_assemble(st, p, nc, w->path.red_B, e.B, Smat, w->L, out_cam, out_red, n_obs));
    // the LM path clears Z once and relies on its static zero pattern
    PCS_CUDA(cudaMemsetAsync(w->Z, 0, (size_t)(nc * np) * 8, st));
    double* h = w->h_read;
    PCS_CUDA(cudaMemcpyAsync(h, w->scal, 8 * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaMemcpyAsync(h + 8, w->info, sizeof(int), cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaMemcpyAsync(h + 9, p->cost, 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    int info = 0;
    std::memcpy(&info, h + 8, sizeof(int));
    int rc = chol_status(info);
    if (rc == PCS_OK && h[5] != 0.0) rc = PCS_ERR_NUMERIC;
    if (rc == PCS_ERR_NUMERIC)
        set_error("pcs_covariance: the undamped normal equations are not positive definite (is the gauge fixed?)");
    PCS_TRY(rc);
    const int64_t d = 2 * p->N - (int64_t)h[7];
    if (dof) *dof = d;
    if (s2) *s2 = d > 0 ? h[9] / (double)d : std::nan("");
    if (cam) PCS_CUDA(cudaMemcpyAsync(cam, out_cam, (size_t)(n_cam * n_cam) * 8, cudaMemcpyDeviceToHost, st));
    double* pose_src = e.B == 6 ? w->L : out_red;
    double* point_src = e.B == 3 ? w->L : out_red;
    if (pose && p->M) PCS_CUDA(cudaMemcpyAsync(pose, pose_src, (size_t)p->M * 36 * 8, cudaMemcpyDeviceToHost, st));
    if (point && p->chain == PCS_CHAIN_SELFCAL && p->K)
        PCS_CUDA(cudaMemcpyAsync(point, point_src, (size_t)p->K * 9 * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_covariance(pcs_problem* p, const double* x, double* cam, double* pose, double* point, double* s2, int64_t* dof)
{
    PCS_REQUIRE(p, "NULL argument");
    return covariance_impl(p, x, cam, pose, point, s2, dof);
}

int pcs_lm_solve(pcs_problem* p, const double* x0, const pcs_lm_options* opts_in, double* x_out, pcs_lm_stats* stats)
{
    const int rc = lm_solve_impl(p, x0, opts_in, x_out, stats);
    // an error return in the middle of an iteration can leave the problem on the second output set: callers hold
    // pointers into the original one (pcs_device_buffers_get), so the problem always leaves on it
    LmWorkspace* w = p ? (LmWorkspace*)p->lm_ws : nullptr;
    if (w && w->ne_alt && w->ne_orig && p->ne == w->ne_alt) swap_normal_buffers(p, w);
    return rc;
}

}  // extern "C"
