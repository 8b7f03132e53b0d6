// pcs_chol.cu -- dense SPD solve  S x = b, one persistent kernel: every factorisation of the library.
//
// Factors the reduced camera system of the LM step (the counterpart of the LSMR solve inside scipy's TRF,
// optimisation_handling.py:88-98), the dense self-calibration fallback and the covariance.  n = 15 C is small (480 at 32
// cameras, 1920 at 128): the factorisation is a chain of n dependent pivots, so what matters is the latency of one block
// step, not throughput.  A vendor potrf + potrs took ~240 + ~90 us at n = 480; this kernel needs one grid barrier per
// 32-column block step:
//
//   * 32 x 32 tiles of the lower triangle, in place in global memory (L2-resident); b rides along as one more block
//     row, so the forward substitution is part of the factorisation.
//   * Phase k (k = 0 .. nb-1), separated by one grid barrier: every CTA that owns a tile of block column k rebuilds the
//     diagonal tile itself -- A_kk minus the (lagged) rank-32 update with panel k-1 -- and factors it in one warp
//     (row per lane, pivots broadcast by shuffles), so nobody waits for a "diagonal done" message; it then applies the
//     lagged update to its own tile and solves it against L_kk^T.  Tiles right of the panel only get the lagged update.
//   * The tiles right of the panel are visited in 2 x 2 groups that share their four operand tiles of panel k-1 and have
//     all (up to) eight tile fetches in flight together: a visit is bound by the latency of its fetches from L2.
//   * The back substitution  x = L^-T y  is a dataflow over the whole grid without barriers: block column k belongs to CTA
//     (nb - 1 - k) mod grid, which streams the tiles of its column through a ring of shared-memory buffers, subtracts
//     L_ik^T x_i as the x_i arrive in a sentinel-initialised mailbox (the data is the signal: no fence, no flag), solves
//     its triangle in one warp and publishes x_k.  n is bounded by the device memory, not by the SM.
// Work is assigned round-robin per phase, panel tiles first (one per CTA while the grid is wide enough), then the groups.
// The kernel is launched cooperatively (co-residency is required by the barrier); loads of data written by other
// CTAs bypass L1 (ld.global.cg).
#include <algorithm>

#include "pcs_internal.cuh"

namespace pcs {

namespace {

constexpr int TB = 32;               // tile edge
constexpr int TP = 34;               // padded row length of a tile in shared memory (even: 16-byte aligned rows)
constexpr int TILE_DOUBLES = TB * TP;
constexpr int CHOL_THREADS = 128;
constexpr int CH_WARPS = CHOL_THREADS / 32;
constexpr unsigned FULL = 0xffffffffu;
constexpr unsigned long long XSENTINEL = 0x7ff8deadbeefcafeull;   // a NaN payload no computation produces: "x not published yet"

struct CholProblem {
    double* A;        // [n][ld] column-major, lower triangle
    double* rhs;      // [n]
    double* Ldiag;    // [nb][32 * 32] row-major
    unsigned long long* bar;   // monotonic arrival counter, never reset: the launch passes the value it starts from
    unsigned long long bar_base;
    int* info;
    int64_t n, ld;
    int nb;
    double* xbuf;                // [nb * 32] back substitution mailbox: x as it is published (XSENTINEL = not yet)
    long long* trace;   // optional [nb + 1][8] globaltimer stamps of CTA 0 (tools/chol_trace.cu), else nullptr
};

__device__ __forceinline__ void trace_stamp(const CholProblem& P, int k, int slot)
{
    if (P.trace && blockIdx.x == 0 && threadIdx.x == 0) {
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        P.trace[k * 8 + slot] = t;
    }
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Shared-memory tiles are COLUMN-major, S[c * TP + r] = element (r, c): that is the layout of the matrix in global
// memory, so a full tile moves with 16-byte asynchronous copies (two rows of one column per copy) and a factored
// diagonal tile is at the same time L^T in row-major form (row j = column j of L, contiguous for tile_trsm).

// element (r, c) of tile (bi, bj); bi == nb is the right-hand-side row.  Rows / columns past n are padded with the identity.
__device__ __forceinline__ double tile_load(const CholProblem& P, int bi, int bj, int r, int c)
{
    const int64_t gc = (int64_t)TB * bj + c, gr = (int64_t)TB * bi + r;
    const bool rhs_row = bi == P.nb;
    const bool in = gc < P.n && (rhs_row ? r == 0 : gr < P.n);
    const double* src = rhs_row ? P.rhs + gc : P.A + gc * P.ld + gr;
    double v = (gc >= P.n && bi == bj && r == c) ? 1.0 : 0.0;
    if (in) v = __ldcg(src);
    return v;
}

__device__ __forceinline__ bool tile_is_full(const CholProblem& P, int bi, int bj)
{
    return bi < P.nb && (int64_t)TB * (bi + 1) <= P.n && (int64_t)TB * (bj + 1) <= P.n && (P.ld & 1) == 0;
}

// start fetching tile (bi, bj) into S; complete after cp_async_wait_all() + __syncthreads()
__device__ __forceinline__ void tile_fetch(const CholProblem& P, int bi, int bj, double* __restrict__ S)
{
    if (tile_is_full(P, bi, bj)) {
        const double* src = P.A + (int64_t)TB * bj * P.ld + (int64_t)TB * bi;
#pragma unroll
        for (int q = 0; q < (TB * TB / 2) / CHOL_THREADS; ++q) {
            const int e = threadIdx.x + q * CHOL_THREADS, c = e >> 4, r = (e & 15) * 2;
            cp_async16(S + c * TP + r, src + (int64_t)c * P.ld + r);
        }
    } else {
        // ragged tiles and the right-hand-side row: all guarded loads first (one round trip), then the stores
        const int r = threadIdx.x & 31, c0 = threadIdx.x >> 5;
        double v[TB / CH_WARPS];
#pragma unroll
        for (int q = 0; q < TB / CH_WARPS; ++q) v[q] = tile_load(P, bi, bj, r, c0 + q * CH_WARPS);
#pragma unroll
        for (int q = 0; q < TB / CH_WARPS; ++q) S[(c0 + q * CH_WARPS) * TP + r] = v[q];
    }
}

__device__ __forceinline__ void tile_store(const CholProblem& P, int bi, int bj, const double* __restrict__ S)
{
    if (tile_is_full(P, bi, bj)) {
        double* dst = P.A + (int64_t)TB * bj * P.ld + (int64_t)TB * bi;
#pragma unroll
        for (int q = 0; q < (TB * TB / 2) / CHOL_THREADS; ++q) {
            const int e = threadIdx.x + q * CHOL_THREADS, c = e >> 4, r = (e & 15) * 2;
            *reinterpret_cast<double2*>(dst + (int64_t)c * P.ld + r) = *reinterpret_cast<const double2*>(S + c * TP + r);
        }
        return;
    }
    const int r = threadIdx.x & 31;
    for (int c = threadIdx.x >> 5; c < TB; c += CHOL_THREADS / 32) {
        const int64_t gc = (int64_t)TB * bj + c;
        if (gc >= P.n) continue;
        if (bi == P.nb) { if (r == 0) P.rhs[gc] = S[c * TP]; continue; }
        const int64_t gr = (int64_t)TB * bi + r;
        if (gr < P.n) P.A[gc * P.ld + gr] = S[c * TP + r];
    }
}

// T -= X Y^T (32 x 32 tiles in shared memory) by warps [W0, W0 + NW) of the CTA, NW = 4 or 3.  A thread owns row r and
// a contiguous, even-aligned block of columns (8 each for four warps; 12 / 10 / 10 for three), so the Y operand
// arrives with 16-byte broadcast loads; one accumulation chain per column keeps the FP64 pipe fed.
template <int W0, int NW>
__device__ __forceinline__ void tile_update(double* __restrict__ T, const double* __restrict__ X, const double* __restrict__ Y)
{
    static_assert(NW == 4 || NW == 3, "column blocks are laid out for 3 or 4 warps");
    const int r = threadIdx.x & 31, w = (int)(threadIdx.x >> 5) - W0;
    if (w < 0 || w >= NW) return;
    constexpr int NP = NW == 4 ? 4 : 6;                       // column pairs per thread (upper bound)
    const int c_lo = NW == 4 ? 8 * w : (w == 0 ? 0 : 2 + 10 * w);
    const int np = NW == 4 ? 4 : (w == 0 ? 6 : 5);
    double acc[2 * NP];
#pragma unroll
    for (int q = 0; q < NP; ++q) {
        acc[2 * q] = q < np ? T[(c_lo + 2 * q) * TP + r] : 0.0;
        acc[2 * q + 1] = q < np ? T[(c_lo + 2 * q + 1) * TP + r] : 0.0;
    }
#pragma unroll 4
    for (int t = 0; t < TB; ++t) {
        const double x = X[t * TP + r];
#pragma unroll
        for (int q = 0; q < NP; ++q) {
            if (q < np) {
                const double2 y = *reinterpret_cast<const double2*>(Y + t * TP + c_lo + 2 * q);
                acc[2 * q] = fma(-x, y.x, acc[2 * q]);
                acc[2 * q + 1] = fma(-x, y.y, acc[2 * q + 1]);
            }
        }
    }
#pragma unroll
    for (int q = 0; q < NP; ++q) {
        if (q < np) {
            T[(c_lo + 2 * q) * TP + r] = acc[2 * q];
            T[(c_lo + 2 * q + 1) * TP + r] = acc[2 * q + 1];
        }
    }
}

__device__ __forceinline__ double lds_f64(unsigned addr)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void lds_v2f64(unsigned addr, double& x, double& y)
{
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x), "=d"(y) : "r"(addr));
}

// branch-free reciprocal: MUFU.RCP64H seed (~20 bits) + two Newton steps (full double accuracy for normal arguments)
__device__ __forceinline__ double rcp_newton(double d)
{
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
    double e = fma(-d, y, 1.0);
    y = fma(y, e, y);
    e = fma(-d, y, 1.0);
    return fma(y, e, y);
}

// Cholesky of the 32 x 32 tile D (shared memory, column-major) by one warp, lane r = row r.
//   * The elimination runs in the square-root-free form (A = L' diag(d) L'^T); the 32 inverse square roots that turn
//     L' into the Cholesky factor are taken afterwards, off the dependent chain.
//   * Every lane tracks the pivot sequence itself: d_{j+1} = a'_{j+1,j+1} - u_{j+1,j}^2 / d_j, where a' (the diagonal
//     entry before step j) is fetched by a shuffle issued one step early and u comes from the column broadcast -- the
//     chain of a step is one reciprocal and one FMA, no shuffle, no compare.
//   * The column of step j reaches the other lanes through a double-buffered shared-memory vector.
// Results: D <- L (column-major, upper part zeroed), invd[j] = 1 / L_jj.  Returns false if a pivot is not positive.
__device__ __forceinline__ bool tile_factor(double* __restrict__ D, double* __restrict__ invd, double* __restrict__ colbuf /*[2][32]*/,
                                            int lane)
{
    double a[TB];
#pragma unroll
    for (int c = 0; c < TB; ++c) a[c] = D[c * TP + lane];
    bool ok = true;
    const unsigned cb_addr = (unsigned)__cvta_generic_to_shared(colbuf);
    double d = __shfl_sync(FULL, a[0], 0);        // pivot 0
    colbuf[lane] = a[0];
    __syncwarp();
#pragma unroll
    for (int j = 0; j < TB; ++j) {
        // column j, unscaled (cb[r] = a_rj), pulled into registers in one batch at the top of the step: issued through
        // volatile asm so that the loads stay ahead of the reciprocal chain instead of trickling in front of their uses
        const unsigned cb = cb_addr + (j & 1) * TB * 8;
        double cbv[TB];
        if ((j + 1) & 1) { if (j + 1 < TB) cbv[j + 1] = lds_f64(cb + (j + 1) * 8); }
#pragma unroll
        for (int c = (j + 2) & ~1; c < TB; c += 2) lds_v2f64(cb + c * 8, cbv[c], cbv[c + 1]);
        __syncwarp();                              // scheduling fence: keeps the batch of loads above the arithmetic
        ok = ok && (d > 0.0);
        if (lane == 0) invd[j] = d;                // pivots, turned into 1 / sqrt below
        const double inv = rcp_newton(d);
        if (j + 1 < TB) {
            // next pivot, on every lane: a'_{j+1,j+1} (before this step's update) - u^2 inv
            const double apd = __shfl_sync(FULL, a[j + 1], j + 1);
            const double u = cbv[j + 1];
            d = fma(-(u * u), inv, apd);
        }
        const double w = a[j] * inv;
#pragma unroll
        for (int c = j + 1; c < TB; ++c) a[c] = fma(-w, cbv[c], a[c]);
        if (j + 1 < TB) {
            colbuf[((j + 1) & 1) * TB + lane] = a[j + 1];
            __syncwarp();
        }
    }
    __syncwarp();
    const double rs = rsqrt(invd[lane]);           // lane j: 1 / sqrt(d_j)
    __syncwarp();
    invd[lane] = rs;
    __syncwarp();
#pragma unroll
    for (int c = 0; c < TB; ++c) D[c * TP + lane] = c <= lane ? a[c] * invd[c] : 0.0;
    return ok;
}

// X <- X L^-T for the 32 rows of tile T (shared memory), one row per lane; L (column-major: row j of the buffer is
// column j of L) and invd in shared memory
__device__ __forceinline__ void tile_trsm(double* __restrict__ T, const double* __restrict__ L, const double* __restrict__ invd, int lane)
{
    double x[TB];
#pragma unroll
    for (int c = 0; c < TB; ++c) x[c] = T[c * TP + lane];
#pragma unroll
    for (int j = 0; j < TB; ++j) {
        const double xj = x[j] * invd[j];
        x[j] = xj;
        const double* col = L + j * TP;      // col[c] = L[c][j]
        if (!(j & 1)) x[j + 1] = fma(-xj, col[j + 1], x[j + 1]);
#pragma unroll
        for (int c = (j + 2) & ~1; c < TB; c += 2) {
            const double2 l = *reinterpret_cast<const double2*>(col + c);
            x[c] = fma(-xj, l.x, x[c]);
            x[c + 1] = fma(-xj, l.y, x[c + 1]);
        }
    }
#pragma unroll
    for (int c = 0; c < TB; ++c) T[c * TP + lane] = x[c];
}

__device__ __forceinline__ void grid_barrier(unsigned long long* bar, unsigned long long target, int* info)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(bar, 1ull);
        unsigned long long v;
        int spins = 0;
        do {
            asm volatile("ld.acquire.gpu.u64 %0, [%1];" : "=l"(v) : "l"(bar) : "memory");
        } while (v < target && ++spins < (1 << 24));
        if (v < target) *info = -2;   // a CTA never arrived: give up instead of hanging the device
    }
    __syncthreads();
}

// tile t of phase k: panel tiles (i, k), i = k+1 .. nb first, then the trailing tiles (i, j), k < j <= i <= nb, (nb, nb) excluded
__device__ __forceinline__ void phase_tile(int k, int nb, int t, int& bi, int& bj)
{
    const int n_panel = nb - k;
    if (t < n_panel) { bi = k + 1 + t; bj = k; return; }
    t -= n_panel;
    // trailing: rows i = k+1 .. nb, columns j = k+1 .. min(i, nb-1)
    for (int i = k + 1; i <= nb; ++i) {
        const int w = ::min(i, nb - 1) - k;
        if (t < w) { bi = i; bj = k + 1 + t; return; }
        t -= w;
    }
    bi = -1; bj = -1;
}


__global__ void __launch_bounds__(CHOL_THREADS)
k_chol_solve(CholProblem P)
{
    extern __shared__ __align__(16) double ch_smem[];
    double* D = ch_smem;                       // diagonal tile / L_kk
    double* Pk = D + TILE_DOUBLES;             // L_{k,k-1}
    double* T = Pk + TILE_DOUBLES;             // the tile being processed
    double* X = T + TILE_DOUBLES;              // L_{i,k-1}
    double* Y = X + TILE_DOUBLES;              // L_{j,k-1}
    double* T2 = Y + TILE_DOUBLES;             // 2 x 2 groups of trailing tiles: three more tiles, a second row / column operand
    double* T3 = T2 + TILE_DOUBLES;
    double* T4 = T3 + TILE_DOUBLES;
    double* X2 = T4 + TILE_DOUBLES;
    double* Y2 = X2 + TILE_DOUBLES;
    double* invd = Y2 + TILE_DOUBLES;          // [32]
    double* colbuf = invd + TB;                // [2][32]
    double* yk = colbuf + 2 * TB;              // [32] back substitution: right-hand side of the block being solved
    __shared__ int s_bad;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nb = P.nb;
    if (threadIdx.x == 0) s_bad = 0;
    // the mailbox of the back substitution is emptied here; the grid barriers of the factorisation publish that
    for (int e = blockIdx.x * CHOL_THREADS + threadIdx.x; e < nb * TB; e += gridDim.x * CHOL_THREADS)
        reinterpret_cast<unsigned long long*>(P.xbuf)[e] = XSENTINEL;

    for (int k = 0; k < nb; ++k) {
        const int n_panel = nb - k;
        int n_tiles = n_panel;
        if (k > 0)   // phase 0 has no lagged update: only the panel is touched
            for (int i = k + 1; i <= nb; ++i) n_tiles += ::min(i, nb - 1) - k;
        const bool has_panel = (int)blockIdx.x < n_panel;     // then this CTA's first tile is the panel tile (k + 1 + blockIdx, k)
        trace_stamp(P, k, 0);
        int t_next = blockIdx.x;
        if (has_panel) {
            // all global loads of the critical path are issued together: diagonal tile, L_{k,k-1}, the panel tile and its L_{i,k-1}
            const int bi = k + 1 + (int)blockIdx.x;
            tile_fetch(P, k, k, D);
            if (k > 0) tile_fetch(P, k, k - 1, Pk);
            tile_fetch(P, bi, k, T);
            if (k > 0) tile_fetch(P, bi, k - 1, X);
            cp_async_wait_all();
            __syncthreads();
            trace_stamp(P, k, 5);
            if (k > 0) tile_update<0, CH_WARPS>(D, Pk, Pk);            // the diagonal tile, rebuilt locally (lagged update)
            __syncthreads();
            trace_stamp(P, k, 1);
            if (warp == 0) {                                           // warp 0 factors it ...
                const long long c0 = clock64();
                if (!tile_factor(D, invd, colbuf, lane) && lane == 0) s_bad = 1;
                if (P.trace && blockIdx.x == 0 && lane == 0) P.trace[k * 8 + 7] = clock64() - c0;   // cycles
            } else if (k > 0) {
                tile_update<1, CH_WARPS - 1>(T, X, Pk);                // ... while the others bring the panel tile up to date
            }
            __syncthreads();
            trace_stamp(P, k, 2);
            if (warp == 0) tile_trsm(T, D, invd, lane);
            else if (blockIdx.x == 0)                                  // L_kk for the back substitution, row-major
                for (int e = threadIdx.x - 32; e < TB * TB; e += CHOL_THREADS - 32) P.Ldiag[(int64_t)k * TB * TB + e] = D[(e & 31) * TP + (e >> 5)];
            __syncthreads();
            trace_stamp(P, k, 6);
            tile_store(P, bi, k, T);
            __syncthreads();
            t_next += gridDim.x;
        } else {
            trace_stamp(P, k, 5);
            trace_stamp(P, k, 1);
            trace_stamp(P, k, 2);
            trace_stamp(P, k, 6);
        }
        if (n_panel <= (int)gridDim.x) {
            // Trailing tiles (lagged update with panel k - 1) in 2 x 2 groups: rows I, I + 1 x columns J, J + 1 of the lower
            // triangle share their operands L_{I,k-1}, L_{I+1,k-1}, L_{J,k-1}, L_{J+1,k-1}, and all (up to) eight tiles of
            // a group are in flight together -- a visit is bound by the latency of its fetches from L2, not by the updates
            // (2.9 us per single-tile visit with three fetches; a group does four updates on eight fetches in one round
            // trip).  Groups are dealt round-robin, starting with the CTAs that have no panel tile in this phase.
            if (k > 0) {
                const int n_pairs = (nb - k + 1) / 2;                  // row pairs of rows k + 1 .. nb (the last one may be single)
                const int n_groups = n_pairs * (n_pairs + 1) / 2;
                int g0 = ((int)blockIdx.x - n_panel) % (int)gridDim.x;
                if (g0 < 0) g0 += gridDim.x;
                for (int g = g0; g < n_groups; g += gridDim.x) {
                    int a = 0, rem = g;
                    while (rem > a) { rem -= a + 1; ++a; }             // group (a, b), b <= a, row-major over the lower triangle
                    const int b = rem;
                    const int I = k + 1 + 2 * a, J = k + 1 + 2 * b;
                    const bool diag = a == b;
                    const bool r1 = I + 1 <= nb;                       // second row of the pair exists
                    // members: (I, J), (I + 1, J), (I + 1, J + 1) and, off the diagonal, (I, J + 1); columns stop at nb - 1
                    const bool m00 = J <= nb - 1, m10 = r1 && J <= nb - 1, m11 = r1 && J + 1 <= nb - 1 && J + 1 <= I + 1,
                               m01 = !diag && J + 1 <= nb - 1;
                    double* const Yj = diag ? X : Y;                   // on the diagonal the column operands are the row operands
                    double* const Yj1 = diag ? X2 : Y2;
                    if (m00) tile_fetch(P, I, J, T);
                    if (m10) tile_fetch(P, I + 1, J, T2);
                    if (m11) tile_fetch(P, I + 1, J + 1, T3);
                    if (m01) tile_fetch(P, I, J + 1, T4);
                    tile_fetch(P, I, k - 1, X);
                    if (r1) tile_fetch(P, I + 1, k - 1, X2);
                    if (!diag) {
                        tile_fetch(P, J, k - 1, Y);
                        if (m01 || m11) tile_fetch(P, J + 1, k - 1, Y2);
                    }
                    cp_async_wait_all();
                    __syncthreads();
                    if (m00) tile_update<0, CH_WARPS>(T, X, Yj);
                    if (m10) tile_update<0, CH_WARPS>(T2, X2, Yj);
                    if (m11) tile_update<0, CH_WARPS>(T3, X2, Yj1);
                    if (m01) tile_update<0, CH_WARPS>(T4, X, Yj1);
                    __syncthreads();
                    if (m00) tile_store(P, I, J, T);
                    if (m10) tile_store(P, I + 1, J, T2);
                    if (m11) tile_store(P, I + 1, J + 1, T3);
                    if (m01) tile_store(P, I, J + 1, T4);
                    __syncthreads();
                }
            }
        } else {
            // the grid is narrower than the panel (n > 32 x grid): one tile per visit, panel tiles included
            for (int t = t_next; t < n_tiles; t += gridDim.x) {
                int bi, bj;
                phase_tile(k, nb, t, bi, bj);
                const bool panel = bj == k;
                tile_fetch(P, bi, bj, T);
                if (k > 0) { tile_fetch(P, bi, k - 1, X); if (!panel) tile_fetch(P, bj, k - 1, Y); }
                cp_async_wait_all();
                __syncthreads();
                if (k > 0) tile_update<0, CH_WARPS>(T, X, panel ? Pk : Y);
                __syncthreads();
                if (panel) {
                    if (warp == 0) tile_trsm(T, D, invd, lane);
                    __syncthreads();
                }
                tile_store(P, bi, bj, T);
                __syncthreads();
            }
        }
        trace_stamp(P, k, 3);
        grid_barrier(P.bar, P.bar_base + (unsigned long long)(k + 1) * gridDim.x, P.info);
        trace_stamp(P, k, 4);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && s_bad) *P.info = 1;

    // Back substitution x = L^-T y, distributed over the grid as a dataflow (no grid barrier): block column k belongs to
    // CTA (nb - 1 - k) mod grid.  Its owner starts from y_k, subtracts L_ik^T x_i for i = nb - 1 .. k + 1 as the x_i are
    // published (tiles of the block column stream through a ring of shared-memory buffers ahead of the flags), solves the
    // 32 x 32 triangle L_kk^T x_k = y_k in one warp and publishes x_k: besides the result in `rhs` it is written into a
    // mailbox that was filled with a sentinel NaN at kernel start -- the consumers poll the values they need themselves, so
    // the arrival of the data IS the signal (no fence + flag + second load on the chain; 8-byte stores are atomic).
    // Every CTA walks its blocks in descending order and a block only waits for higher blocks, so the
    // highest unfinished block can always proceed (all CTAs are co-resident: cooperative launch).  The critical path is one
    // flag round trip + one tile product + one triangle per block; a single CTA streaming all of L (round 1) took 225 us at
    // n = 1504 and 350 us at n = 1920.
    trace_stamp(P, nb, 0);
    {
        double* const ring[8] = {T, X, Y, T2, T3, T4, X2, Y2};
        constexpr int RING = 8;
        const int c = threadIdx.x >> 2, q = threadIdx.x & 3;      // thread (c, q): column c of a tile, rows 8 q .. 8 q + 7
        for (int k = nb - 1 - (int)blockIdx.x; k >= 0; k -= gridDim.x) {
            // diagonal block (row-major lower factor) and y_k
            for (int e = threadIdx.x; e < TB * (TB / 2); e += CHOL_THREADS) {
                const int r = e >> 4, cc = (e & 15) * 2;
                cp_async16(D + r * TP + cc, P.Ldiag + (int64_t)k * TB * TB + r * TB + cc);
            }
            cp_async_commit();
            const int n_up = nb - 1 - k;                          // tiles (i, k), i = nb - 1 .. k + 1
            int issued = 0;
            for (int gq = 0; gq < RING - 1; ++gq) {               // always RING - 1 groups (empty ones past the last tile): tile u is group u + 1
                if (issued < n_up) { tile_fetch(P, nb - 1 - issued, k, ring[issued % RING]); ++issued; }
                cp_async_commit();
            }
            double acc = 0.0;                                     // threads with q == 0: (sum_i L_ik^T x_i)[c]
            for (int u = 0; u < n_up; ++u) {
                const int i = nb - 1 - u;
                if (issued < n_up) { tile_fetch(P, nb - 1 - issued, k, ring[issued % RING]); ++issued; }
                cp_async_commit();                                // (possibly empty: keeps the group count uniform)
                cp_async_wait_group<RING - 1>();                  // tile u (and the diagonal block) have landed
                __syncthreads();
                // x_i: every thread polls the eight values it needs until none of them is the sentinel
                const double* S = ring[u % RING] + c * TP + 8 * q;
                const unsigned long long* xb = reinterpret_cast<const unsigned long long*>(P.xbuf) + (int64_t)TB * i + 8 * q;
                unsigned long long xv[8];
                int spins = 0;
                bool ready;
                do {
                    ready = true;
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
                        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(xv[r]) : "l"(xb + r) : "memory");
                        ready = ready && xv[r] != XSENTINEL;
                    }
                } while (!ready && ++spins < (1 << 22));
                if (!ready) {                                     // a block was never published: give up instead of hanging
                    *P.info = -2;
#pragma unroll
                    for (int r = 0; r < 8; ++r) xv[r] = 0ull;
                }
                double part = 0.0;
#pragma unroll
                for (int r = 0; r < 8; r += 2) {
                    const double2 l = *reinterpret_cast<const double2*>(S + r);
                    part = fma(l.x, __longlong_as_double((long long)xv[r]), part);
                    part = fma(l.y, __longlong_as_double((long long)xv[r + 1]), part);
                }
                part += __shfl_xor_sync(FULL, part, 1);
                part += __shfl_xor_sync(FULL, part, 2);
                acc += part;
                __syncthreads();                                  // the buffer of tile u may be refilled
            }
            cp_async_wait_all();
            if (q == 0) {
                const int64_t gi = (int64_t)TB * k + c;
                yk[c] = (gi < P.n ? __ldcg(P.rhs + gi) : 0.0) - acc;
            }
            __syncthreads();
            if (warp == 0) {
                double yc = yk[lane];
                double lcol[TB];                    // column `lane` of L_kk: lcol[r] = L[r][lane]
#pragma unroll
                for (int r = 0; r < TB; ++r) lcol[r] = D[r * TP + lane];
                __syncwarp();                       // scheduling fence (see tile_factor)
                const double inv = rcp_newton(D[lane * TP + lane]);
#pragma unroll
                for (int r = TB - 1; r >= 0; --r) {
                    const double xr = __shfl_sync(FULL, yc * inv, r);
                    if (lane == r) yc = xr;
                    else if (lane < r) yc = fma(-lcol[r], xr, yc);
                }
                const int64_t gi = (int64_t)TB * k + lane;
                const double xo = gi < P.n ? yc : 0.0;            // padding rows publish a zero: nobody waits for them forever
                asm volatile("st.relaxed.gpu.global.f64 [%0], %1;" ::"l"(P.xbuf + (int64_t)TB * k + lane), "d"(xo) : "memory");
                if (gi < P.n) P.rhs[gi] = yc;
            }
            __syncthreads();                        // D / yk are reused by the next block of this CTA
        }
    }
    trace_stamp(P, nb, 1);
}

size_t chol_smem_bytes()
{
    return (size_t)(10 * TILE_DOUBLES + 4 * TB) * sizeof(double);
}

}  // namespace

// Workspace + launch geometry.  PCS_ERR_UNSUPPORTED when the kernel cannot be co-scheduled on the device.
int chol_prepare(int device, int64_t n, double** Ldiag, unsigned long long** bar, int* grid)
{
    const int nb = (int)((n + TB - 1) / TB);
    int max_optin = 0, sms = 0, coop = 0;
    PCS_CUDA(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    PCS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    PCS_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
    const size_t smem = chol_smem_bytes();
    int per_sm = 0;
    if (coop && smem <= (size_t)max_optin) {
        // monotone per (kernel, device): a later, smaller problem must not lower the opt-in of a live larger one
        PCS_CUDA(ensure_dynamic_smem(k_chol_solve, smem));
        PCS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_chol_solve, CHOL_THREADS, smem));
    }
    if (per_sm < 1) {
        set_error("the Cholesky kernel cannot be co-scheduled on this device: it needs a cooperative launch and one CTA with " +
                  std::to_string(smem) + " bytes of shared memory per SM");
        return PCS_ERR_UNSUPPORTED;
    }
    // work units of the widest phase: nb panel tiles + the 2 x 2 groups of the trailing tiles.  A grid wider than that only
    // makes the barrier slower (every CTA arrives on one counter)
    const int n_pairs0 = (nb + 1) / 2;
    const int n_tiles0 = nb + n_pairs0 * (n_pairs0 + 1) / 2;
    // diagonal-block factors, followed by the mailbox of the back substitution (nb x 32 doubles, reset by every launch)
    PCS_CUDA(cudaMalloc((void**)Ldiag, ((size_t)nb * TB * TB + (size_t)nb * TB) * sizeof(double)));
    PCS_CUDA(cudaMalloc((void**)bar, sizeof(unsigned long long)));
    PCS_CUDA(cudaMemset(*bar, 0, sizeof(unsigned long long)));
    *grid = std::max(1, std::min(sms, n_tiles0));
    return PCS_OK;
}

// *bar_base: the caller's running count of barrier arrivals on `bar` (starts at 0 with a zeroed counter); advanced here.
// `info` must be zero on entry (the kernel only ever raises it).
int launch_chol_solve(cudaStream_t st, int grid, int64_t n, double* A, int64_t ld, double* rhs, double* Ldiag,
                      unsigned long long* bar, unsigned long long* bar_base, int* info, long long* trace)
{
    CholProblem P;
    P.trace = trace;
    P.A = A; P.rhs = rhs; P.Ldiag = Ldiag; P.bar = bar; P.info = info; P.n = n; P.ld = ld;
    P.nb = (int)((n + TB - 1) / TB);
    P.xbuf = Ldiag + (size_t)P.nb * TB * TB;
    P.bar_base = *bar_base;
    *bar_base += (unsigned long long)P.nb * (unsigned long long)grid;
    void* args[] = {&P};
    PCS_CUDA(cudaLaunchCooperativeKernel((const void*)k_chol_solve, dim3(grid), dim3(CHOL_THREADS), args, chol_smem_bytes(), st));
    return PCS_OK;
}

// 1: a pivot was not positive; -2: a grid barrier or the back substitution's mailbox gave up waiting (the result is void)
int chol_status(int info)
{
    if (info == 0) return PCS_OK;
    if (info == -2) {
        set_error("the Cholesky kernel's grid barrier timed out");
        return PCS_ERR_CUDA;
    }
    return PCS_ERR_NUMERIC;
}

}  // namespace pcs

extern "C" int pcs_spd_solve(int device, int64_t n, const double* A, const double* b, double* x, int* info)
{
    using namespace pcs;
    PCS_REQUIRE(n > 0 && A && b && x, "NULL argument or n <= 0");
    PCS_CUDA(cudaSetDevice(device));
    double *dA = nullptr, *db = nullptr, *Ldiag = nullptr;
    unsigned long long* bar = nullptr;
    unsigned long long bar_base = 0;
    int* dinfo = nullptr;
    int grid = 0;
    int rc = chol_prepare(device, n, &Ldiag, &bar, &grid);
    auto cleanup = [&]() { cudaFree(dA); cudaFree(db); cudaFree(Ldiag); cudaFree(bar); cudaFree(dinfo); };
    if (rc != PCS_OK) { cleanup(); return rc; }
    cudaError_t e = cudaMalloc((void**)&dA, (size_t)(n * n) * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&db, (size_t)n * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&dinfo, sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpy(dA, A, (size_t)(n * n) * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, b, (size_t)n * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(dinfo, 0, sizeof(int));
    if (e != cudaSuccess) { set_error(std::string("pcs_spd_solve: ") + cudaGetErrorString(e)); cleanup(); return PCS_ERR_CUDA; }
    rc = launch_chol_solve(nullptr, grid, n, dA, n, db, Ldiag, bar, &bar_base, dinfo, nullptr);
    int h_info = 0;
    if (rc == PCS_OK) {
        e = cudaDeviceSynchronize();
        if (e == cudaSuccess) e = cudaMemcpy(x, db, (size_t)n * 8, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(&h_info, dinfo, sizeof(int), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { set_error(std::string("pcs_spd_solve: ") + cudaGetErrorString(e)); rc = PCS_ERR_CUDA; }
    }
    if (info) *info = h_info;
    cleanup();
    if (rc == PCS_OK) rc = chol_status(h_info);
    if (rc == PCS_ERR_NUMERIC) set_error("pcs_spd_solve: matrix is not positive definite");
    return rc;
}
