// pcs_cov.cu -- covariance of the bundle-adjustment solution from the factored reduced system (pcs_covariance).
//
// The LM workspace eliminates one block-diagonal set (poses, or the target points) and factors the reduced system
// S = A - Z Z^T = L L^T (k_chol_solve, pcs_chol.cu), Z = W L_b^-T scattered per eliminated block b.  At lambda = 0:
//   reduced set     Sigma_red = S^-1 = X_I^T X_I,                    X_I = L^-1
//   eliminated set  Sigma_bb  = L_b^-T (I + X_b^T X_b) L_b^-1,       X_b = L^-1 Z_b
// The kernels here:
//   * k_cov_tile_inverse   the 32 x 32 diagonal factors of L (Ldiag, row-major) -> their inverses, in place;
//   * k_cov_forward        L X = B in place for all right-hand sides at once, B = [identity | Z]: one CTA per panel of
//                          128 columns walks the 32-row steps of L top-down, X_k = L_kk^-1 (B_k - L_{k,<k} X_{<k}).  The
//                          update is a GEMM on the FP64 tensor path (DMMA m8n8k4, operands streamed global -> shared
//                          memory through a 3-stage ring of 16-deep slabs, as k_schur_syrk does); the off-diagonal tiles
//                          of L are read from S, where k_chol_solve leaves them.  Identity panels start at their own
//                          diagonal (the rows above it stay zero);
//   * k_cov_transpose      X_I -> X_I^T in place, so that k_schur_syrk (which forms Z Z^T of a column-major [k][n] Z)
//                          forms X_I^T X_I;
//   * k_cov_block_marginals one warp per eliminated block: Gram X_b^T X_b, then L_b^-T (I + G) L_b^-1;
//   * k_cov_assemble       masking (fixed -> 0, unobserved -> NaN), the count of observed free parameters, copy-out layout.
#include <algorithm>

#include "pcs_internal.cuh"

namespace pcs {

namespace {

constexpr int FT = 32;            // row step = tile edge of the Cholesky factor
constexpr int FW = 128;           // right-hand sides per CTA
constexpr int FK = 16;            // slab depth
constexpr int F_THREADS = 256;    // 8 warps, warp w owns columns [16 w, 16 w + 16) of the panel, all 32 rows
constexpr int F_STAGES = 3;
constexpr int ALD = FT + 8;       // A slab [FK][ALD]: element (row r, k) at k * ALD + r
constexpr int BLD = FK + 4;       // B slab [FW][BLD]: element (k, column c) at c * BLD + k
constexpr int A_DOUBLES = FK * ALD;
constexpr int B_DOUBLES = FW * BLD;
constexpr int STAGE_DOUBLES = A_DOUBLES + B_DOUBLES;
constexpr int DLD = FT + 8;       // epilogue: L_kk^-1 [FT][DLD], element (r, k) at k * DLD + r
constexpr int TLD = FT + 4;       // epilogue: B_k - update [FW][TLD], element (r, c) at c * TLD + r
static_assert(FT * DLD + FW * TLD <= F_STAGES * STAGE_DOUBLES, "the epilogue reuses the stage ring");

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Ldiag[k] (row-major lower 32 x 32) -> its inverse, column-major (element (r, c) at c * 32 + r); thread c solves L x = e_c
__global__ void __launch_bounds__(FT) k_cov_tile_inverse(double* __restrict__ Ldiag)
{
    __shared__ double Ls[FT][FT + 1];
    double* D = Ldiag + (int64_t)blockIdx.x * FT * FT;
    const int c = threadIdx.x;
    for (int r = 0; r < FT; ++r) Ls[r][c] = D[r * FT + c];
    __syncthreads();
    double x[FT];
#pragma unroll
    for (int r = 0; r < FT; ++r) {
        double s = r == c ? 1.0 : 0.0;
#pragma unroll
        for (int q = 0; q < r; ++q) s = fma(-Ls[r][q], x[q], s);
        x[r] = r < c ? 0.0 : s / Ls[r][r];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < FT; ++r) D[c * FT + r] = x[r];
}

__global__ void k_cov_identity(int64_t n, double* __restrict__ X)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < n * n) X[t] = (t / n == t % n) ? 1.0 : 0.0;
}

// L X = B in place.  Panels [0, n_id): columns of X_I (B = identity, already in Xi); the rest: columns of Z.
__global__ void __launch_bounds__(F_THREADS, 2)
k_cov_forward(int64_t nc, const double* __restrict__ S, const double* __restrict__ Dinv, double* __restrict__ Xi, int n_id,
              double* __restrict__ Z, int64_t np)
{
    extern __shared__ __align__(16) double fs[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t4 = lane & 3;
    const bool id = (int)blockIdx.x < n_id;
    double* const B = id ? Xi : Z;
    const int64_t ncols = id ? nc : np;
    const int64_t c0 = (int64_t)FW * (id ? blockIdx.x : blockIdx.x - n_id);
    const int nb = (int)(nc / FT);
    const int k_first = id ? (int)(c0 / FT) : 0;     // identity panel: rows above its first column are zero
    const int64_t r_lo = (int64_t)FT * k_first;

    for (int k = k_first; k < nb; ++k) {
        double acc[4][2][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        const int n_slabs = (int)(((int64_t)FT * k - r_lo) / FK);
        auto fetch = [&](int s) {
            if (s < n_slabs) {
                double* As = fs + (s % F_STAGES) * STAGE_DOUBLES;
                double* Bs = As + A_DOUBLES;
                const int64_t kk0 = r_lo + (int64_t)s * FK;
                {   // L rows [32 k, 32 k + 32) x columns [kk0, kk0 + 16): 256 copies of 16 bytes
                    const int kk = threadIdx.x >> 4, r = (threadIdx.x & 15) * 2;
                    cp_async16(As + kk * ALD + r, S + (kk0 + kk) * nc + (int64_t)FT * k + r);
                }
#pragma unroll
                for (int q = 0; q < (FW * FK / 2) / F_THREADS; ++q) {   // X rows [kk0, kk0 + 16) of the panel's columns
                    const int e = threadIdx.x + q * F_THREADS, c = e >> 3, r = (e & 7) * 2;
                    if (c0 + c < ncols) cp_async16(Bs + c * BLD + r, B + (c0 + c) * nc + kk0 + r);
                    else { Bs[c * BLD + r] = 0.0; Bs[c * BLD + r + 1] = 0.0; }
                }
            }
            cp_async_commit();
        };
        fetch(0);
        fetch(1);
        for (int s = 0; s < n_slabs; ++s) {
            cp_async_wait<F_STAGES - 2>();
            __syncthreads();
            fetch(s + 2);
            const double* A = fs + (s % F_STAGES) * STAGE_DOUBLES + g;
            const double* Bw = fs + (s % F_STAGES) * STAGE_DOUBLES + A_DOUBLES + (16 * warp + g) * BLD + t4;
#pragma unroll
            for (int ks = 0; ks < FK / 4; ++ks) {
                double a[4], b[2];
#pragma unroll
                for (int i = 0; i < 4; ++i) a[i] = A[(4 * ks + t4) * ALD + 8 * i];
#pragma unroll
                for (int j = 0; j < 2; ++j) b[j] = Bw[8 * j * BLD + 4 * ks];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 2; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
        }
        cp_async_wait<0>();
        __syncthreads();   // the ring is free: epilogue
        double* Dt = fs;
        double* T = fs + FT * DLD;
#pragma unroll
        for (int q = 0; q < (FT * FT / 2) / F_THREADS; ++q) {
            const int e = threadIdx.x + q * F_THREADS, kk = e >> 4, r = (e & 15) * 2;
            cp_async16(Dt + kk * DLD + r, Dinv + (int64_t)k * FT * FT + kk * FT + r);
        }
        cp_async_commit();
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int c = 16 * warp + 8 * j + 2 * t4 + h, r = 8 * i + g;
                    const double b = c0 + c < ncols ? B[(c0 + c) * nc + (int64_t)FT * k + r] : 0.0;
                    T[c * TLD + r] = b - acc[i][j][h];
                    acc[i][j][h] = 0.0;
                }
        cp_async_wait<0>();
        __syncthreads();
        // X_k = L_kk^-1 (B_k - update)
        const double* Tw = T + (16 * warp + g) * TLD + t4;
#pragma unroll
        for (int ks = 0; ks < FT / 4; ++ks) {
            double a[4], b[2];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = Dt[(4 * ks + t4) * DLD + 8 * i + g];
#pragma unroll
            for (int j = 0; j < 2; ++j) b[j] = Tw[8 * j * TLD + 4 * ks];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int c = 16 * warp + 8 * j + 2 * t4 + h;
                    if (c0 + c < ncols) B[(c0 + c) * nc + (int64_t)FT * k + 8 * i + g] = acc[i][j][h];
                }
        // X_k is read back through L2 (cp.async.cg) by the next steps of this CTA; the epilogue buffers become the ring again
        __threadfence();
        __syncthreads();
    }
}

// in-place transpose of the n x n matrix X (n a multiple of 32): tile pairs (bi, bj), bi >= bj, swap through shared memory
__global__ void __launch_bounds__(256) k_cov_transpose(int64_t n, double* __restrict__ X)
{
    __shared__ double a[32][33], b[32][33];
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    double* P = X + (int64_t)32 * bj * n + 32 * bi;   // tile (bi, bj): element (r, c) at P[c * n + r]
    double* Q = X + (int64_t)32 * bi * n + 32 * bj;   // tile (bj, bi)
    for (int c = ty; c < 32; c += 8) { a[c][tx] = P[c * n + tx]; b[c][tx] = Q[c * n + tx]; }
    __syncthreads();
    for (int c = ty; c < 32; c += 8) { P[c * n + tx] = b[tx][c]; Q[c * n + tx] = a[tx][c]; }
}

// one warp per eliminated block b: G = X_b^T X_b (X_b = the B columns of the substituted Z at B slot[b]), then
// Sigma_bb = L_b^-T (I + G) L_b^-1, written over the block's factor L_b ([B][B] row-major lower)
template <int B>
__global__ void __launch_bounds__(128)
k_cov_block_marginals(int n_blocks, int64_t nc, const double* __restrict__ X, const int32_t* __restrict__ slot, double* __restrict__ L)
{
    constexpr int NG = B * (B + 1) / 2;
    const int b = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (b >= n_blocks) return;
    const double* Xb = X + (int64_t)B * (slot ? slot[b] : b) * nc;
    double G[NG];
#pragma unroll
    for (int q = 0; q < NG; ++q) G[q] = 0.0;
    for (int64_t r = lane; r < nc; r += 32) {
        double z[B];
#pragma unroll
        for (int i = 0; i < B; ++i) z[i] = Xb[i * nc + r];
        int q = 0;
#pragma unroll
        for (int i = 0; i < B; ++i)
#pragma unroll
            for (int j = 0; j <= i; ++j) { G[q] = fma(z[i], z[j], G[q]); ++q; }
    }
#pragma unroll
    for (int q = 0; q < NG; ++q)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) G[q] += __shfl_xor_sync(0xffffffffu, G[q], o);
    if (lane != 0) return;
    double* Lb = L + (int64_t)b * B * B;
    double l[B][B], m[B][B];
#pragma unroll
    for (int i = 0; i < B; ++i)
#pragma unroll
        for (int j = 0; j < B; ++j) l[i][j] = Lb[i * B + j];
    int q = 0;
#pragma unroll
    for (int i = 0; i < B; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) { m[i][j] = m[j][i] = G[q] + (i == j ? 1.0 : 0.0); ++q; }
    // T = L^-T M (columns of M by back substitution with L^T), then Sigma = L^-T T^T
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
        double t[B][B];
#pragma unroll
        for (int c = 0; c < B; ++c)
#pragma unroll
            for (int i = B - 1; i >= 0; --i) {
                double s = pass == 0 ? m[i][c] : m[c][i];
#pragma unroll
                for (int k = i + 1; k < B; ++k) s -= l[k][i] * t[k][c];
                t[i][c] = s / l[i][i];
            }
#pragma unroll
        for (int i = 0; i < B; ++i)
#pragma unroll
            for (int j = 0; j < B; ++j) m[i][j] = t[i][j];
    }
#pragma unroll
    for (int i = 0; i < B; ++i)
#pragma unroll
        for (int j = 0; j < B; ++j) Lb[i * B + j] = 0.5 * (m[i][j] + m[j][i]);
}

struct CovAssemble {
    int C, M, K;
    int64_t nc;
    int red_B, elim_B;                 // reduced-set blocks after the cameras (6: poses, 3: points, 0: none); eliminated (6 / 3)
    const double* S;                   // -Sigma_red, lower triangle
    double* elim;                      // Sigma_bb [n_elim][elim_B^2], masked in place
    double* out_cam;                   // [15 C][15 C]
    double* out_red;                   // [n_red][red_B^2]
    const double *U, *V, *Pk;
    const uint16_t* cam_mask;
    const uint8_t *pose_mask, *key_mask;
    double* n_observed;                // observed free parameters (diagonal entries counted once)
};

// parameter r of a block set: 15 per camera, 6 per pose, 3 per point
__device__ __forceinline__ void param_state(const CovAssemble& A, int B, int64_t r, bool& fixed, bool& unobserved)
{
    double d;
    bool f;
    if (B == 15) { const int c = (int)(r / 15), a = (int)(r % 15); f = A.cam_mask[c] & (1u << a); d = A.U[(int64_t)c * 225 + a * 16]; }
    else if (B == 6) { const int m = (int)(r / 6), a = (int)(r % 6); f = A.pose_mask[m] & (1u << a); d = A.V[(int64_t)m * 36 + a * 7]; }
    else { const int k = (int)(r / 3), a = (int)(r % 3); f = A.key_mask[k] & (1u << a); d = A.Pk[(int64_t)k * 9 + a * 4]; }
    fixed = !f;
    unobserved = f && d == 0.0;
}

__global__ void k_cov_assemble(CovAssemble A, int64_t n_cam_entries, int64_t n_red_entries, int64_t n_elim_entries)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    bool count = false;
    if (t < n_cam_entries + n_red_entries + n_elim_entries) {
        int B;
        int64_t ra, rb, row0;     // parameters a, b inside their set; row0: offset of the set in the reduced system
        double* out;
        const double* src = nullptr;
        if (t < n_cam_entries) {
            const int64_t n = 15 * (int64_t)A.C;
            B = 15; ra = t / n; rb = t % n; row0 = 0; out = A.out_cam + t; src = A.S;
        } else {
            const int64_t u = t < n_cam_entries + n_red_entries ? t - n_cam_entries : t - n_cam_entries - n_red_entries;
            const bool red = t < n_cam_entries + n_red_entries;
            B = red ? A.red_B : A.elim_B;
            const int64_t blk = u / (B * B);
            const int i = (int)(u % (B * B)) / B, j = (int)(u % B);
            ra = blk * B + i; rb = blk * B + j; row0 = 15 * (int64_t)A.C;
            if (red) { out = A.out_red + u; src = A.S; }
            else out = A.elim + u;
        }
        double v;
        if (src) {
            const int64_t hi = row0 + max(ra, rb), lo = row0 + min(ra, rb);
            v = -src[lo * A.nc + hi];
        } else {
            v = *out;
        }
        bool fa, ua, fb, ub;
        param_state(A, B, ra, fa, ua);
        param_state(A, B, rb, fb, ub);
        if (fa || fb) v = 0.0;
        else if (ua || ub) v = __longlong_as_double(0x7ff8000000000000ll);
        *out = v;
        count = ra == rb && !fa && !ua;
    }
    const unsigned n = __popc(__ballot_sync(0xffffffffu, count));
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(A.n_observed, (double)n);
}

size_t forward_smem_bytes() { return (size_t)F_STAGES * STAGE_DOUBLES * sizeof(double); }

}  // namespace

int cov_forward_substitution(cudaStream_t st, int64_t nc, const double* S, double* Ldiag, double* Xi, double* Z, int64_t np)
{
    const int nb = (int)(nc / FT);
    k_cov_tile_inverse<<<nb, FT, 0, st>>>(Ldiag);
    k_cov_identity<<<(int)((nc * nc + 255) / 256), 256, 0, st>>>(nc, Xi);
    PCS_CUDA(cudaGetLastError());
    const int n_id = (int)((nc + FW - 1) / FW), n_z = (int)((np + FW - 1) / FW);
    PCS_CUDA(ensure_dynamic_smem(k_cov_forward, forward_smem_bytes()));
    k_cov_forward<<<n_id + n_z, F_THREADS, forward_smem_bytes(), st>>>(nc, S, Ldiag, Xi, n_id, Z, np);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

int cov_reduced_inverse(cudaStream_t st, int sm_count, int64_t nc, double* Xi, double* S)
{
    PCS_CUDA(cudaMemsetAsync(S, 0, (size_t)(nc * nc) * 8, st));
    const int nb = (int)(nc / 32);
    k_cov_transpose<<<dim3(nb, nb), 256, 0, st>>>(nc, Xi);
    PCS_CUDA(cudaGetLastError());
    return launch_schur_syrk(st, sm_count, nc, nc, Xi, S, nullptr);   // S = -X_I^T X_I (lower triangle)
}

int cov_block_marginals(cudaStream_t st, int n_blocks, int B, int64_t nc, const double* X, const int32_t* slot, double* L)
{
    if (n_blocks <= 0) return PCS_OK;
    const int grid = (int)(((int64_t)n_blocks * 32 + 127) / 128);
    if (B == 6) k_cov_block_marginals<6><<<grid, 128, 0, st>>>(n_blocks, nc, X, slot, L);
    else k_cov_block_marginals<3><<<grid, 128, 0, st>>>(n_blocks, nc, X, slot, L);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

int cov_assemble(cudaStream_t st, const pcs_problem* p, int64_t nc, int red_B, int elim_B, const double* S, double* elim,
                 double* out_cam, double* out_red, double* n_observed)
{
    CovAssemble A;
    A.C = p->C; A.M = p->M; A.K = p->K; A.nc = nc; A.red_B = red_B; A.elim_B = elim_B;
    A.S = S; A.elim = elim; A.out_cam = out_cam; A.out_red = out_red;
    A.U = p->U; A.V = p->V; A.Pk = p->Pk; A.cam_mask = p->cam_mask; A.pose_mask = p->pose_mask; A.key_mask = p->key_mask;
    A.n_observed = n_observed;
    auto n_blocks = [&](int B) -> int64_t { return B == 6 ? p->M : (B == 3 ? p->K : 0); };
    const int64_t n_cam = 225 * (int64_t)p->C * p->C;
    const int64_t n_red = n_blocks(red_B) * red_B * red_B, n_elim = n_blocks(elim_B) * elim_B * elim_B;
    const int64_t total = n_cam + n_red + n_elim;
    if (total == 0) return PCS_OK;
    k_cov_assemble<<<(int)((total + 255) / 256), 256, 0, st>>>(A, n_cam, n_red, n_elim);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

}  // namespace pcs
