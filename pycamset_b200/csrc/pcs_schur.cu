// pcs_schur.cu -- reduced camera system: S -= Z Z^T (lower triangle), the rank-6M update that eliminates the poses.
//
// Part of the LM step that stands in for scipy's TRF / LSMR solve (optimisation_handling.py:88-98): with
// Z = W L^-T (15 C x 6 M, dense when every camera sees every pose) the Schur complement of the pose blocks is
// S = U + lambda D - Z Z^T.  A vendor DSYRK reaches a third of the FP64 pipe on this shape (n = 480, k = 12000: few
// output tiles, long k); this kernel is shaped for it:
//   * 96 x 96 output tiles of the lower triangle; the (tile, k) iteration space is linearised and cut into one
//     contiguous range per SM ("stream-K"), so all SMs finish together whatever the tile count; a CTA flushes its
//     accumulators with FP64 reductions whenever its range leaves a tile (at most twice).
//   * Operands stream global -> shared memory with 16-byte asynchronous copies through a 3-stage ring of 16-column
//     slabs; Z is column-major, so a slab row (96 consecutive matrix rows of one column) is contiguous.
//   * 8 warps, warp tile 48 x 24 = 6 x 3 DMMA m8n8k4 accumulators; A and B fragments of a k-step are plain 8-byte
//     loads from the slab (row stride 104 doubles: the minimum two wavefronts per load).
//   * Block sparsity (LIST variant): a camera that does not see a pose leaves a zero 15 x 6 block in Z.  The sparsity
//     pattern is static, so schur_plan_build() orders the pose columns by their visibility pattern (poses seen by the same
//     row blocks become neighbours) and lists the (tile, slab) units whose two operand slabs are both non-zero; the kernel
//     then streams that list instead of the full iteration space.  On the 32-camera ring (every pose seen by half of the
//     cameras) 57 % of the units remain; on the dome (95 % fill) the list is not used.
#include <algorithm>
#include <numeric>
#include <vector>

#include "pcs_internal.cuh"

namespace pcs {

namespace {

constexpr int ST = 96;            // tile edge
constexpr int SK = 16;            // slab depth (columns of Z per stage)
constexpr int SLD = ST + 8;       // slab row stride in doubles
constexpr int S_STAGES = 3;
constexpr int S_THREADS = 256;
constexpr int SLAB_DOUBLES = SK * SLD;              // one operand slab
constexpr int STAGE_DOUBLES = 2 * SLAB_DOUBLES;     // A rows + B rows

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ void cp_async_zfill(void* smem, const void* gmem, int bytes, int src_bytes)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    if (bytes == 16)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sa), "l"(gmem), "r"(src_bytes) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sa), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// lower-triangle tile t -> (ti, tj), ti >= tj, row-major enumeration
__device__ __forceinline__ void tile_of(int t, int& ti, int& tj)
{
    ti = 0;
    while (t > ti) { t -= ti + 1; ++ti; }
    tj = t;
}

// Per-thread constants of the slab copies: a thread moves the same (column, row) positions of every slab, so the
// shared-memory offsets and the row / column offsets inside a slab are computed once.
template <bool ALIGNED>
struct FetchPlan {
    static constexpr int PER_SLAB = ALIGNED ? (SK * (ST / 2)) / S_THREADS : (SK * ST) / S_THREADS;   // copies per thread and slab
    int kk[PER_SLAB], row[PER_SLAB];   // column inside the slab, row inside the tile
    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int q = 0; q < PER_SLAB; ++q) {
            const int r = threadIdx.x + q * S_THREADS;
            if (ALIGNED) { kk[q] = r / (ST / 2); row[q] = 2 * (r % (ST / 2)); }
            else { kk[q] = r / ST; row[q] = r % ST; }
        }
    }
};

// fetch one stage: columns [k0, k0 + SK) of the rows of tiles ti (slab A) and tj (slab B)
template <bool ALIGNED>
__device__ __forceinline__ void fetch_stage(const FetchPlan<ALIGNED>& fp, double* __restrict__ stage, const double* __restrict__ Z,
                                            int64_t nc, int64_t np, int ti, int tj, int64_t k0)
{
#pragma unroll
    for (int slab = 0; slab < 2; ++slab) {
        const int64_t row0 = (int64_t)ST * (slab ? tj : ti);
#pragma unroll
        for (int q = 0; q < FetchPlan<ALIGNED>::PER_SLAB; ++q) {
            const int64_t row = row0 + fp.row[q], k = k0 + fp.kk[q];
            int src = 0;
            if (ALIGNED) { if (k < np) src = row + 1 < nc ? 16 : (row < nc ? 8 : 0); }
            else src = (k < np && row < nc) ? 8 : 0;
            const double* g = src ? Z + k * nc + row : Z;
            cp_async_zfill(stage + slab * SLAB_DOUBLES + fp.kk[q] * SLD + fp.row[q], g, ALIGNED ? 16 : 8, src);
        }
    }
}

constexpr int UL_CHUNK = 64;   // LIST: unit-list entries per shared-memory chunk (two chunks resident)

// LIST: the iteration space is the list `units` of non-zero (tile, slab) pairs -- entry = {ti << 16 | tj, slab}, sorted by
// tile -- instead of all n_lower x n_slabs pairs.
template <bool ALIGNED, bool LIST>
__global__ void __launch_bounds__(S_THREADS, 2)
k_schur_syrk(int64_t nc, int64_t np, const double* __restrict__ Z, double* __restrict__ S, int n_lower, int64_t n_slabs,
             const int2* __restrict__ unit_list, int64_t n_units)
{
    extern __shared__ __align__(16) double sy_smem[];
    __shared__ int2 ul[2][UL_CHUNK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t4 = lane & 3;
    const int wr = warp >> 2, wc = warp & 3;   // 2 x 4 warps: 48 rows x 24 columns each

    const int64_t units = LIST ? n_units : (int64_t)n_lower * n_slabs;
    const int64_t u0 = units * blockIdx.x / gridDim.x, u1 = units * (blockIdx.x + 1) / gridDim.x;
    if (u0 >= u1) return;
    // chunk j of this CTA's range sits in ul[j & 1]; chunk j + 1 is loaded when the computation enters chunk j (the fetches
    // run at most two units ahead of it)
    auto load_chunk = [&](int64_t j) {
        if (threadIdx.x < UL_CHUNK) {
            const int64_t u = u0 + UL_CHUNK * j + threadIdx.x;
            ul[j & 1][threadIdx.x] = u < u1 ? unit_list[u] : make_int2(-1, 0);
        }
    };
    auto entry = [&](int64_t u) -> int2 { const int64_t i = u - u0; return ul[(i / UL_CHUNK) & 1][i % UL_CHUNK]; };
    if (LIST) {
        load_chunk(0);
        load_chunk(1);
        __syncthreads();
    }
    FetchPlan<ALIGNED> fp;
    fp.init();

    double acc[6][3][2];
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    auto flush = [&](int ti, int tj) {
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int64_t row = (int64_t)ST * ti + wr * 48 + 8 * i + g;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int64_t col = (int64_t)ST * tj + wc * 24 + 8 * j + 2 * t4 + h;
                    if (row < nc && col <= row) atomicAdd(S + col * nc + row, -acc[i][j][h]);
                    acc[i][j][h] = 0.0;
                }
            }
    };

    // (tile, slab) of the unit being computed and of the unit being fetched, advanced incrementally (or read from the list)
    int c_tile = LIST ? 0 : (int)(u0 / n_slabs), cti = 0, ctj = 0;
    if (!LIST) tile_of(c_tile, cti, ctj);
    int f_tile = c_tile, fti = cti, ftj = ctj;
    int64_t f_slab = LIST ? 0 : u0 % n_slabs, f_u = u0;
    auto fetch_next = [&](int stage) {
        if (f_u < u1) {
            if (LIST) {
                const int2 e = entry(f_u);
                fetch_stage<ALIGNED>(fp, sy_smem + stage * STAGE_DOUBLES, Z, nc, np, e.x >> 16, e.x & 0xffff, (int64_t)e.y * SK);
                ++f_u;
            } else {
                fetch_stage<ALIGNED>(fp, sy_smem + stage * STAGE_DOUBLES, Z, nc, np, fti, ftj, f_slab * SK);
                ++f_u;
                if (++f_slab == n_slabs) { f_slab = 0; ++f_tile; tile_of(f_tile, fti, ftj); }
            }
        }
        cp_async_commit();
    };
    for (int s = 0; s < S_STAGES - 1; ++s) fetch_next(s);
    int c_stage = 0, f_stage = S_STAGES - 1;
    int64_t c_slab = LIST ? 0 : u0 % n_slabs;
    for (int64_t u = u0; u < u1; ++u) {
        cp_async_wait<S_STAGES - 2>();
        __syncthreads();   // stage u has landed for everybody; stage u - 1 has been consumed by everybody
        if (LIST) {
            const int64_t i = u - u0;
            if (i > 0 && i % UL_CHUNK == 0) load_chunk(i / UL_CHUNK + 1);   // replaces the chunk everybody has left
        }
        fetch_next(f_stage);
        f_stage = f_stage + 1 == S_STAGES ? 0 : f_stage + 1;
        const double* A = sy_smem + c_stage * STAGE_DOUBLES + wr * 48 + g;
        const double* B = sy_smem + c_stage * STAGE_DOUBLES + SLAB_DOUBLES + wc * 24 + g;
#pragma unroll
        for (int s = 0; s < SK / 4; ++s) {
            double a[6], b[3];
#pragma unroll
            for (int i = 0; i < 6; ++i) a[i] = A[(4 * s + t4) * SLD + 8 * i];
#pragma unroll
            for (int j = 0; j < 3; ++j) b[j] = B[(4 * s + t4) * SLD + 8 * j];
#pragma unroll
            for (int i = 0; i < 6; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        c_stage = c_stage + 1 == S_STAGES ? 0 : c_stage + 1;
        if (LIST) {
            const int2 e = entry(u);
            if (u + 1 == u1 || entry(u + 1).x != e.x) flush(e.x >> 16, e.x & 0xffff);   // the range leaves this tile
        } else if (++c_slab == n_slabs) {   // the range leaves this tile
            flush(cti, ctj);
            c_slab = 0;
            ++c_tile;
            tile_of(c_tile, cti, ctj);
        }
    }
    if (!LIST && c_slab != 0) flush(cti, ctj);
}

// segment s = (camera c, pose m): the row blocks (ST rows each) that camera c's 15 rows touch are non-zero for pose m
__global__ void k_pose_block_mask(int64_t S, const int32_t* __restrict__ seg_cam, const int32_t* __restrict__ seg_pose,
                                  unsigned long long* __restrict__ mask)
{
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int c = seg_cam[s];
    const int b0 = 15 * c / ST, b1 = (15 * c + 14) / ST;
    unsigned long long bits = 1ull << b0;
    if (b1 != b0) bits |= 1ull << b1;
    atomicOr(mask + seg_pose[s], bits);
}

}  // namespace

// S (n x n, column-major, lower triangle) -= Z Z^T with Z given column-major as [k][n]; plan (optional): the non-zero units
int launch_schur_syrk(cudaStream_t st, int sm_count, int64_t n, int64_t k, const double* Z, double* S, const SchurPlan* plan)
{
    if (n <= 0 || k <= 0) return PCS_OK;
    const int n_t = (int)((n + ST - 1) / ST);
    const int n_lower = n_t * (n_t + 1) / 2;
    const int64_t n_slabs = (k + SK - 1) / SK;
    const size_t smem = (size_t)S_STAGES * STAGE_DOUBLES * sizeof(double);
    const bool aligned = (n % 2 == 0) && ((reinterpret_cast<uintptr_t>(Z) & 15) == 0);
    const bool list = plan && plan->units;
    if (list && plan->n_units == 0) return PCS_OK;
    auto kern = list ? (aligned ? k_schur_syrk<true, true> : k_schur_syrk<false, true>) : (aligned ? k_schur_syrk<true, false> : k_schur_syrk<false, false>);
    PCS_CUDA(ensure_dynamic_smem(kern, smem));
    const int64_t units = list ? plan->n_units : (int64_t)n_lower * n_slabs;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(2 * (int64_t)sm_count, units));   // two CTAs per SM
    kern<<<grid, S_THREADS, smem, st>>>(n, k, Z, S, n_lower, n_slabs, list ? (const int2*)plan->units : nullptr, list ? plan->n_units : 0);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

void schur_plan_free(SchurPlan* plan)
{
    if (plan->pose_slot) cudaFree(plan->pose_slot);
    if (plan->units) cudaFree(plan->units);
    *plan = SchurPlan();
}

// Static block-sparsity plan of the pose elimination (see the header comment).  nl = logical order of the reduced system,
// rows [15 C, nl) are the target-point rows of the self-calibration chain (treated as dense).  Leaves the plan empty (dense
// SYRK, identity column order) when the reduced system has more than 64 row blocks or too few units would be skipped.
int schur_plan_build(pcs_problem* p, int64_t nc, int64_t nl, SchurPlan* plan)
{
    schur_plan_free(plan);
    const int n_t = (int)((nc + ST - 1) / ST);
    const int64_t M = p->M, n_slabs = (6 * M + SK - 1) / SK;
    // small systems: the whole update takes microseconds, the plan (allocations, a read-back, host-side sorting) milliseconds
    if (n_t > 64 || n_t < 3 || M < 256 || p->n_seg == 0) return PCS_OK;
    unsigned long long* d_mask = nullptr;
    PCS_CUDA(cudaMalloc((void**)&d_mask, (size_t)M * 8));
    std::vector<unsigned long long> mask((size_t)M);
    cudaError_t e = cudaMemsetAsync(d_mask, 0, (size_t)M * 8, p->stream);
    if (e == cudaSuccess) {
        k_pose_block_mask<<<(int)((p->n_seg + 255) / 256), 256, 0, p->stream>>>(p->n_seg, p->seg_cam, p->seg_pose, d_mask);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(mask.data(), d_mask, (size_t)M * 8, cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    cudaFree(d_mask);
    if (e != cudaSuccess) { set_error(std::string("schur_plan_build: ") + cudaGetErrorString(e)); return PCS_ERR_CUDA; }
    const int64_t n_cam_rows = 15 * (int64_t)p->C;
    if (nl > n_cam_rows) {   // point rows: every pose may touch them
        unsigned long long pts = 0;
        for (int b = (int)(n_cam_rows / ST); b <= (int)((nl - 1) / ST); ++b) pts |= 1ull << b;
        for (auto& m : mask) if (m) m |= pts;
    }
    // column order: poses with the same / similar visibility pattern next to each other
    std::vector<int32_t> order((size_t)M), slot((size_t)M);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return mask[a] < mask[b]; });
    for (int64_t i = 0; i < M; ++i) slot[order[i]] = (int32_t)i;
    // row blocks touched by the columns of every slab
    std::vector<unsigned long long> slab_any((size_t)n_slabs, 0ull);
    std::vector<int2> units;
    const int64_t total = (int64_t)n_t * (n_t + 1) / 2 * n_slabs;
    units.reserve((size_t)(total / 2 + 16));
    for (int ti = 0; ti < n_t; ++ti)
        for (int tj = 0; tj <= ti; ++tj) {
            const unsigned long long need = (1ull << ti) | (1ull << tj);
            for (int64_t s = 0; s < n_slabs; ++s) {
                const int64_t p0 = SK * s / 6, p1 = std::min<int64_t>(M - 1, (SK * s + SK - 1) / 6);
                bool nz = false;
                for (int64_t q = p0; q <= p1 && !nz; ++q) nz = (mask[order[q]] & need) == need;
                if (nz) units.push_back(make_int2((ti << 16) | tj, (int)s));
            }
        }
    plan->fraction = total ? (double)units.size() / (double)total : 1.0;
    if (plan->fraction > 0.85) return PCS_OK;   // nothing worth skipping: dense SYRK, identity column order
    PCS_CUDA(cudaMalloc((void**)&plan->pose_slot, (size_t)M * 4));
    PCS_CUDA(cudaMalloc((void**)&plan->units, std::max<size_t>(units.size(), 1) * sizeof(int2)));
    PCS_CUDA(cudaMemcpyAsync(plan->pose_slot, slot.data(), (size_t)M * 4, cudaMemcpyHostToDevice, p->stream));
    PCS_CUDA(cudaMemcpyAsync(plan->units, units.data(), units.size() * sizeof(int2), cudaMemcpyHostToDevice, p->stream));
    PCS_CUDA(cudaStreamSynchronize(p->stream));   // the host vectors go out of scope
    plan->n_units = (int64_t)units.size();
    return PCS_OK;
}

}  // namespace pcs

extern "C" int pcs_syrk_sub(int device, int64_t n, int64_t k, const double* Z, double* S)
{
    using namespace pcs;
    PCS_REQUIRE(n > 0 && k > 0 && Z && S, "NULL argument or empty shape");
    PCS_CUDA(cudaSetDevice(device));
    double *dZ = nullptr, *dS = nullptr;
    int sms = 0;
    PCS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    cudaError_t e = cudaMalloc((void**)&dZ, (size_t)(n * k) * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&dS, (size_t)(n * n) * 8);
    if (e == cudaSuccess) e = cudaMemcpy(dZ, Z, (size_t)(n * k) * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dS, S, (size_t)(n * n) * 8, cudaMemcpyHostToDevice);
    int rc = PCS_OK;
    if (e == cudaSuccess) rc = launch_schur_syrk(nullptr, sms, n, k, dZ, dS, nullptr);
    if (e == cudaSuccess && rc == PCS_OK) e = cudaDeviceSynchronize();
    if (e == cudaSuccess && rc == PCS_OK) e = cudaMemcpy(S, dS, (size_t)(n * n) * 8, cudaMemcpyDeviceToHost);
    cudaFree(dZ);
    cudaFree(dS);
    if (e != cudaSuccess) { set_error(std::string("pcs_syrk_sub: ") + cudaGetErrorString(e)); return PCS_ERR_CUDA; }
    return rc;
}
