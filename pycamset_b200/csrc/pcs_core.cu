// pcs_core.cu -- problem build, parameter handling, residual / Jacobian / normal-equation kernels and
// their C-ABI entry points (see include/pcs_b200.h for the reference interfaces each one replaces).
#include <cub/cub.cuh>

#include <algorithm>
#include <cstring>
#include <new>

#include "pcs_internal.cuh"
#include "pcs_math.cuh"

namespace pcs {

static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }

// ------------------------------------------------------------------------------------------------
// small utilities
// ------------------------------------------------------------------------------------------------
template <typename T>
static int dev_alloc(T** ptr, int64_t count)
{
    *ptr = nullptr;
    if (count <= 0) count = 1;
    PCS_CUDA(cudaMalloc((void**)ptr, (size_t)count * sizeof(T)));
    return PCS_OK;
}

template <typename T>
static void dev_free(T*& ptr)
{
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
}

int ensure_pinned(pcs_problem* p, int64_t doubles)
{
    if (p->h_pin_doubles >= doubles) return PCS_OK;
    if (p->h_pin) cudaFreeHost(p->h_pin);
    p->h_pin = nullptr;
    p->h_pin_doubles = 0;
    PCS_CUDA(cudaMallocHost((void**)&p->h_pin, (size_t)doubles * sizeof(double)));
    p->h_pin_doubles = doubles;
    return PCS_OK;
}

static inline int grid_for(int64_t n, int block) { return (int)((n + block - 1) / block); }

// ------------------------------------------------------------------------------------------------
// parameter kernels
// ------------------------------------------------------------------------------------------------
// x (free vector) -> parameter string; replaces fill_flat x3 (compiled_helpers.py:155-177)
__global__ void k_scatter_x(int64_t n_free, const int32_t* __restrict__ free_idx, const double* __restrict__ x,
                            double* __restrict__ params)
{
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < n_free) params[free_idx[j]] = x[j];
}

// Per-camera / per-pose tables: rotation matrices and their derivatives are computed ONCE per parameter
// update instead of once per observation (the reference calls Rodrigues inside the per-observation loop,
// function_block_implementations.py:150-182).
// Optionally fused into the same launch (the normal-equation evaluation runs it every step):
//   x != nullptr   : scatter the free vector into the parameter string first (fill_flat, compiled_helpers.py:155-177);
//                    threads [C + M, C + M + n_tail) handle the entries after the pose block (free points, chain 1)
//   zero != nullptr: clear `n_zero` doubles (the reduction targets of the normal-equation kernel)
__device__ __forceinline__ double param_value(double* __restrict__ params, const double* __restrict__ x,
                                              const int32_t* __restrict__ free_map, int64_t i)
{
    if (x) {
        const int32_t f = free_map[i];
        if (f >= 0) {
            const double v = x[f];
            params[i] = v;
            return v;
        }
    }
    return params[i];
}

__global__ void k_prepare_tables(int C, int M, int64_t n_tail, double* __restrict__ params, const double* __restrict__ x,
                                 const int32_t* __restrict__ free_map, double* __restrict__ camtab,
                                 double* __restrict__ posetab, double* __restrict__ dRtab, double* __restrict__ zero,
                                 int64_t n_zero, int64_t n_seg, const int32_t* __restrict__ seg_cam,
                                 const int32_t* __restrict__ seg_pose, double* __restrict__ segtab, double* __restrict__ pts4)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    pdl_launch_dependents();   // the evaluation kernel that follows may become resident now; it waits for this grid (pdl_wait)
    for (int64_t i = t; i < n_zero; i += (int64_t)gridDim.x * blockDim.x) zero[i] = 0.0;
    if (t < C) {
        const int64_t qi = 9 * t, ei = 9 * (int64_t)C + 6 * t;
        double* o = camtab + t * CAM_STRIDE;
        for (int k = 0; k < 9; ++k) o[CAM_Q + k] = param_value(params, x, free_map, qi + k);
        double e[6];
        for (int k = 0; k < 6; ++k) e[k] = param_value(params, x, free_map, ei + k);
        double r[3] = {e[0], e[1], e[2]}, R[9], Jl[9];
        rodrigues(r, R);
        rodrigues_left_jacobian(r, Jl);
        for (int k = 0; k < 9; ++k) o[CAM_R + k] = R[k];
        for (int k = 0; k < 3; ++k) o[CAM_T + k] = e[3 + k];
        for (int k = 0; k < 9; ++k) o[CAM_JL + k] = Jl[k];
        o[30] = o[31] = 0.0;
        if (dRtab) rodrigues_jac(r, dRtab + 27 * t);
    } else if (t < C + M) {
        const int64_t m = t - C;
        const int64_t ei = 15 * (int64_t)C + 6 * m;
        double* o = posetab + m * POSE_STRIDE;
        double e[6];
        for (int k = 0; k < 6; ++k) e[k] = param_value(params, x, free_map, ei + k);
        double r[3] = {e[0], e[1], e[2]}, R[9], Jl[9];
        rodrigues(r, R);
        rodrigues_left_jacobian(r, Jl);
        for (int k = 0; k < 9; ++k) o[POSE_R + k] = R[k];
        for (int k = 0; k < 3; ++k) o[POSE_T + k] = e[3 + k];
        for (int k = 0; k < 9; ++k) o[POSE_JL + k] = Jl[k];
        o[21] = o[22] = o[23] = 0.0;
        if (dRtab) rodrigues_jac(r, dRtab + 27 * t);
    } else if (t < (int64_t)C + M + n_tail) {
        // chain 1: the free points follow the pose block; they are also kept as 16-byte rows (pts4) for the kernels
        const int64_t j = t - C - M;
        const double v = param_value(params, x, free_map, 15 * (int64_t)C + 6 * (int64_t)M + j);
        pts4[4 * (j / 3) + j % 3] = v;
    } else if (segtab && t >= (int64_t)C + M + n_tail && t < (int64_t)C + M + n_tail + n_seg) {
        // residual kernel: one combined transform per (camera, pose) segment, X_c = (R_c R_m) X_t + (R_c t_m + t_c),
        // formed from the parameters themselves (not from the tables other threads of this launch are still writing)
        const int64_t s = t - C - M - n_tail;
        const int c = seg_cam[s], m = seg_pose[s];
        double ec[6], em[6], Rc[9], Rm[9];
        for (int k = 0; k < 6; ++k) {
            const int64_t ic = 9 * (int64_t)C + 6 * (int64_t)c + k, im = 15 * (int64_t)C + 6 * (int64_t)m + k;
            const int32_t fc = x ? free_map[ic] : -1, fm = x ? free_map[im] : -1;
            ec[k] = fc >= 0 ? x[fc] : params[ic];
            em[k] = fm >= 0 ? x[fm] : params[im];
        }
        rodrigues(ec, Rc);
        rodrigues(em, Rm);
        double* o = segtab + s * SEG_STRIDE;
        for (int a = 0; a < 3; ++a) {
            for (int b = 0; b < 3; ++b)
                o[SEG_R + 3 * a + b] = fma(Rc[3 * a], Rm[b], fma(Rc[3 * a + 1], Rm[3 + b], Rc[3 * a + 2] * Rm[6 + b]));
            o[SEG_T + a] = fma(Rc[3 * a], em[3], fma(Rc[3 * a + 1], em[4], fma(Rc[3 * a + 2], em[5], ec[3 + a])));
        }
        for (int k = 0; k < 9; ++k) {
            const int64_t iq = 9 * (int64_t)c + k;
            const int32_t fq = x ? free_map[iq] : -1;
            o[SEG_Q + k] = fq >= 0 ? x[fq] : params[iq];
        }
        o[SEG_Q + 9] = 0.0;
    }
}

int launch_scatter_x(pcs_problem* p, const double* x_dev)
{
    if (p->n_free > 0) {
        k_scatter_x<<<grid_for(p->n_free, 256), 256, 0, p->stream>>>(p->n_free, p->free_idx, x_dev, p->params);
        ++p->n_launches;
        PCS_CUDA(cudaGetLastError());
    }
    return PCS_OK;
}

// with_dR: also refresh the OpenCV dR/dr tables [C + M][27] the explicit-Jacobian / dense paths read.
// x_dev / zero: see k_prepare_tables (one launch instead of scatter + tables + memset).
int launch_prepare(pcs_problem* p, bool with_dR, const double* x_dev, double* zero, int64_t n_zero, bool with_seg)
{
    if (with_dR && !p->dRtab) PCS_TRY(dev_alloc(&p->dRtab, 27 * ((int64_t)p->C + p->M)));
    if (with_seg && !p->segtab) PCS_TRY(dev_alloc(&p->segtab, SEG_STRIDE * p->n_seg));
    const int64_t n_tail = p->L - 15 * (int64_t)p->C - 6 * (int64_t)p->M;   // chain 1: 3 K point coordinates, chain 0: none
    const int64_t threads = (int64_t)p->C + p->M + n_tail + (with_seg ? p->n_seg : 0);
    const int grid = (int)std::max<int64_t>(grid_for(threads, 128), std::min<int64_t>(grid_for(n_zero, 128), 2 * p->sm_count));
    k_prepare_tables<<<grid, 128, 0, p->stream>>>(p->C, p->M, n_tail, p->params, x_dev, p->free_map, p->camtab, p->posetab,
                                                  with_dR ? p->dRtab : nullptr, zero, zero ? n_zero : 0, p->n_seg, p->seg_cam,
                                                  p->seg_pose, with_seg ? p->segtab : nullptr, p->tmpl4);
    ++p->n_launches;
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

static inline const double* points_ptr(const pcs_problem* p)
{
    return p->chain == PCS_CHAIN_TEMPLATE ? p->tmpl : p->params + 15 * (int64_t)p->C + 6 * (int64_t)p->M;
}

// ------------------------------------------------------------------------------------------------
// K_res: residual, one thread per observation, dd row order.  44 algorithmic bytes / observation.
// ------------------------------------------------------------------------------------------------
// Rows of the per-segment table are fetched with 16-byte loads; the observation stream (segment id, key, (u, v)) is read
// once and bypasses L1 allocation.  Per lane: 22 + 4 doubles of table rows instead of the 34 + 3 of a separate pose and
// camera transform, in one dependent load level -- the kernel is bound by the bytes every lane has to RECEIVE through
// the L1 data pipe (128 B / clock / SM), not by HBM, so fewer row bytes per observation is what makes it faster.
__device__ __forceinline__ int ld_stream_i32(const int32_t* p)
{
    int v;
    asm("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double2 ld_stream_f64x2(const double2* p)
{
    double2 v;
    asm("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}

// One thread per observation.  Measured alternatives, none faster than this kernel's 32 us at 2.59 M observations
// (profiles/r2_kres_variants.txt): a persistent, software-pipelined variant (67 us: 60 registers, half the resident warps);
// a per-warp row cache in shared memory for (camera, pose)-sorted tables (33-34 us: L1 data-pipe wavefronts 65 -> 59 %,
// time unchanged -- a broadcast shared load still has to deliver 16 bytes to every lane); 2 / 4 observations per thread
// with all stream loads issued up front (33 / 35 us at 44 % / 34 % occupancy).  The time does not move with occupancy,
// memory-level parallelism or the wavefront count: what is constant across the variants is the number of bytes each lane
// receives through the load / store unit (232 B of rows and stream + 16 B stored per observation).
__global__ void __launch_bounds__(256)
k_residual(int64_t N, const int32_t* __restrict__ obs_seg, const int32_t* __restrict__ key, const double2* __restrict__ uv,
           const double* __restrict__ segtab, const double* __restrict__ pts4, double2* __restrict__ r_out)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    // the observation stream is static: it is requested before the wait for the table set-up launch
    const int s = ld_stream_i32(obs_seg + i), k = ld_stream_i32(key + i);
    const double2 o = ld_stream_f64x2(uv + i);
    pdl_wait();
    double T[SEG_STRIDE], Xt[4];
    {
        const double2* row = reinterpret_cast<const double2*>(segtab + (int64_t)s * SEG_STRIDE);
#pragma unroll
        for (int j = 0; j < SEG_STRIDE / 2; ++j) { const double2 v = row[j]; T[2 * j] = v.x; T[2 * j + 1] = v.y; }
        const double2* x2 = reinterpret_cast<const double2*>(pts4 + 4 * (int64_t)k);   // point rows are padded to 4 doubles
        const double2 a = x2[0], b = x2[1];
        Xt[0] = a.x; Xt[1] = a.y; Xt[2] = b.x;
    }
    double Xc[3];
    transform(T + SEG_R, T + SEG_T, Xt, Xc);
    const Proj p = project(T + SEG_Q, Xc);
    r_out[i] = make_double2(p.u - o.x, p.v - o.y);
}

int launch_residual(pcs_problem* p, double* r_dev)
{
    if (p->N == 0) return PCS_OK;
    PCS_CUDA(launch_pdl(k_residual, dim3(grid_for(p->N, 256)), dim3(256), 0, p->stream, p->N, (const int32_t*)p->obs_seg,
                        (const int32_t*)p->key, (const double2*)p->uv, (const double*)p->segtab, (const double*)p->tmpl4,
                        (double2*)r_dev));
    ++p->n_launches;
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

// cost-only evaluation (LM step acceptance): residual in registers, block reduction, one atomic per CTA
__global__ void __launch_bounds__(256)
k_cost(int64_t N, const int32_t* __restrict__ cam, const int32_t* __restrict__ pose, const int32_t* __restrict__ key,
       const double2* __restrict__ uv, const double* __restrict__ camtab, const double* __restrict__ posetab,
       const double* __restrict__ pts, double* __restrict__ cost)
{
    double acc = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = cam[i], m = pose[i], k = key[i];
        const double2 o = uv[i];
        const double* pt = pts + 3 * (int64_t)k;
        const double Xt[3] = {pt[0], pt[1], pt[2]};
        double res[2];
        eval_residual(camtab + (int64_t)c * CAM_STRIDE, posetab + (int64_t)m * POSE_STRIDE, Xt, o.x, o.y, res);
        acc = fma(res[0], res[0], fma(res[1], res[1], acc));
    }
    typedef cub::BlockReduce<double, 256> BR;
    __shared__ typename BR::TempStorage tmp;
    double s = BR(tmp).Sum(acc);
    if (threadIdx.x == 0) atomicAdd(cost, s);
}

int launch_cost_only(pcs_problem* p, double* cost_dev)
{
    PCS_CUDA(cudaMemsetAsync(cost_dev, 0, sizeof(double), p->stream));
    if (p->N == 0) return PCS_OK;
    int grid = std::min<int64_t>(grid_for(p->N, 256), (int64_t)p->sm_count * 8);
    k_cost<<<grid, 256, 0, p->stream>>>(p->N, p->cam, p->pose, p->key, (const double2*)p->uv, p->camtab, p->posetab,
                                        points_ptr(p), cost_dev);
    ++p->n_launches;
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

// ------------------------------------------------------------------------------------------------
// K_jac: explicit CSR values in the reference's order.  One thread per observation evaluates the 2 x P
// row pair in registers; a warp's rows are contiguous in the CSR value array, so they are compacted
// (fixed columns dropped) into shared memory and leave the SM as ONE bulk asynchronous copy
// (cp.async.bulk shared -> global, the TMA unit): the copy-out does not pass through the load / store
// unit, which is what bounds this kernel.  28 B in + 16 P B out per observation.
// ------------------------------------------------------------------------------------------------
template <int P>
__global__ void __launch_bounds__(128)
k_jacobian(int64_t N, const int32_t* __restrict__ cam, const int32_t* __restrict__ pose, const int32_t* __restrict__ key,
           const double2* __restrict__ uv, const double* __restrict__ camtab, const double* __restrict__ posetab,
           const double* __restrict__ dRtab, const double* __restrict__ pts, const uint16_t* __restrict__ cam_mask,
           const uint8_t* __restrict__ pose_mask, const uint8_t* __restrict__ key_mask, const int64_t* __restrict__ row_prefix,
           int C, double* __restrict__ vals)
{
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* ws = sm + warp * (64 * P);
    const int64_t w0 = (blockIdx.x * (int64_t)(blockDim.x >> 5) + warp) * 32;
    if (w0 >= N) return;
    const int64_t i = w0 + lane;
    const int64_t wend = min(N, w0 + 32);
    const int64_t base = row_prefix[w0];
    const int64_t total = 2 * (row_prefix[wend] - base);
    if (i < N) {
        const int c = cam[i], m = pose[i], k = key[i];
        const double2 o = uv[i];
        const double* pt = pts + 3 * (int64_t)k;
        const double Xt[3] = {pt[0], pt[1], pt[2]};
        const double* ct = camtab + (int64_t)c * CAM_STRIDE;
        const double* ptab = posetab + (int64_t)m * POSE_STRIDE;
        double res[2], Bc[6], Bm[6];
        ObsJac J;
        eval_obs(ct, ptab, Xt, o.x, o.y, res, J);
        reference_rotation_blocks(J, ptab, dRtab + 27 * (int64_t)c, dRtab + 27 * ((int64_t)C + m), Xt, Bc, Bm);
        double ju[P], jv[P];
        expand_rows<P>(J, Bc, Bm, ptab, ju, jv);
        uint32_t mask = (uint32_t)cam_mask[c] | ((uint32_t)pose_mask[m] << 15);
        if (P == 24) mask |= (uint32_t)key_mask[k] << 21;
        const int n = __popc(mask);
        int off = (int)(2 * (row_prefix[i] - base));
        double* du = ws + off;
        double* dv = du + n;
        int w = 0;
#pragma unroll
        for (int col = 0; col < P; ++col) {
            if (mask & (1u << col)) {
                du[w] = ju[col];
                dv[w] = jv[col];
                ++w;
            }
        }
    }
    double* out = vals + 2 * base;
    // 2 * base and `total` are even: source, destination and size are multiples of 16 bytes.  Every lane orders its own
    // (generic-proxy) shared-memory stores before the asynchronous proxy's read; lane 0 then issues the copy and holds the
    // CTA's shared memory until the unit has read it.
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0 && total > 0) {
        const unsigned src = (unsigned)__cvta_generic_to_shared(ws);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out), "r"(src), "r"((unsigned)(total * 8)) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

// CSR structure (make_jac_CSR_columns_row_pointers, abstract_function_blocks.py:465-489)
__global__ void k_csr_structure(int64_t N, int P, int C, int M, const int32_t* __restrict__ cam,
                                const int32_t* __restrict__ pose, const int32_t* __restrict__ key,
                                const int32_t* __restrict__ free_map, const int64_t* __restrict__ row_prefix,
                                int64_t* __restrict__ col_idx, int64_t* __restrict__ row_ptr)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i > N) return;
    if (i == N) {
        row_ptr[2 * N] = 2 * row_prefix[N];
        return;
    }
    const int64_t s = row_prefix[i], n = row_prefix[i + 1] - s;
    row_ptr[2 * i] = 2 * s;
    row_ptr[2 * i + 1] = 2 * s + n;
    const int64_t c = cam[i], m = pose[i], k = key[i];
    int64_t w = 2 * s;
    for (int col = 0; col < P; ++col) {
        int64_t g;
        if (col < 9) g = 9 * c + col;
        else if (col < 15) g = 9 * (int64_t)C + 6 * c + (col - 9);
        else if (col < 21) g = 15 * (int64_t)C + 6 * m + (col - 15);
        else g = 15 * (int64_t)C + 6 * (int64_t)M + 3 * k + (col - 21);
        const int32_t f = free_map[g];
        if (f >= 0) {
            col_idx[w] = f;
            col_idx[w + n] = f;
            ++w;
        }
    }
}

// mirror the upper triangles of U (15x15) and V (6x6) into the lower ones
__global__ void k_symmetrize_blocks(int64_t n_blocks, int dim, double* __restrict__ blocks)
{
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int per = dim * dim;
    if (t >= n_blocks * per) return;
    const int64_t blk = t / per;
    const int e = (int)(t % per), a = e / dim, b = e % dim;
    if (a > b) blocks[blk * per + e] = blocks[blk * per + b * dim + a];
}

// ------------------------------------------------------------------------------------------------
// Dense normal equations over the free parameters (both chains; small problems)
// ------------------------------------------------------------------------------------------------
template <int P>
__global__ void __launch_bounds__(128)
k_normal_dense(int64_t N, int C, int M, int64_t n_free, const int32_t* __restrict__ cam, const int32_t* __restrict__ pose,
               const int32_t* __restrict__ key, const double2* __restrict__ uv, const double* __restrict__ camtab,
               const double* __restrict__ posetab, const double* __restrict__ dRtab, const double* __restrict__ pts,
               const int32_t* __restrict__ free_map, double* JtJ, double* Jtr, double* cost)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int64_t c = cam[i], m = pose[i], k = key[i];
    const double2 o = uv[i];
    const double* pt = pts + 3 * k;
    const double Xt[3] = {pt[0], pt[1], pt[2]};
    const double* ptab = posetab + m * POSE_STRIDE;
    const double* ct = camtab + c * CAM_STRIDE;
    double res[2], Bc[6], Bm[6];
    ObsJac J;
    eval_obs(ct, ptab, Xt, o.x, o.y, res, J);
    reference_rotation_blocks(J, ptab, dRtab + 27 * c, dRtab + 27 * ((int64_t)C + m), Xt, Bc, Bm);
    double ju[P], jv[P];
    expand_rows<P>(J, Bc, Bm, ptab, ju, jv);
    int32_t f[P];
#pragma unroll
    for (int col = 0; col < P; ++col) {
        int64_t g;
        if (col < 9) g = 9 * c + col;
        else if (col < 15) g = 9 * (int64_t)C + 6 * c + (col - 9);
        else if (col < 21) g = 15 * (int64_t)C + 6 * m + (col - 15);
        else g = 15 * (int64_t)C + 6 * (int64_t)M + 3 * k + (col - 21);
        f[col] = free_map[g];
    }
    atomicAdd(cost, fma(res[0], res[0], res[1] * res[1]));
#pragma unroll
    for (int a = 0; a < P; ++a) {
        if (f[a] < 0) continue;
        atomicAdd(Jtr + f[a], fma(ju[a], res[0], jv[a] * res[1]));
#pragma unroll
        for (int b = a; b < P; ++b) {
            if (f[b] < 0) continue;
            const double v = fma(ju[a], ju[b], jv[a] * jv[b]);
            if (v == 0.0) continue;
            const int64_t lo = min(f[a], f[b]), hi = max(f[a], f[b]);
            atomicAdd(JtJ + lo * n_free + hi, v);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Self-calibration chain (projection + extrinsic3D + rigidTform3d + free_point, standard_bundle_handler.py:129-226):
// the blocks that involve the target points.  The camera / pose blocks U, V, W, g_c, g_m, r.r of this chain are the
// template chain's with X_t = point[k] and come from the fused kernel (pcs_normal.cu); this kernel adds, per observation
// (c, m, k) with B_k = Pm R_c R_m (2 x 3, function_block_implementations.py:226-240: d X_t / d point = I):
//     Pk[k]    += B_k^T B_k          (3 x 3)       gk[k] += B_k^T r
//     Xck[c,k] += [A | B_c]^T B_k    (15 x 3)      Ymk[m,k] += B_m^T B_k   (6 x 3)
// Rotation columns are in the reference's rvec parametrisation (tangent rows times the left Jacobian), like the blocks the
// fused kernel writes.  One lane per observation, FP64 reductions into the dense (camera, key) / (pose, key) tables:
// 75 reductions per observation -- this chain's problems are small (N = 4884 at the reference's fixture).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_normal_points(int64_t N, int K, const int32_t* __restrict__ cam, const int32_t* __restrict__ pose, const int32_t* __restrict__ key,
                const double2* __restrict__ uv, const double* __restrict__ camtab, const double* __restrict__ posetab,
                const double* __restrict__ pts4, double* __restrict__ Pk, double* __restrict__ gk, double* __restrict__ Xck,
                double* __restrict__ Ymk)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int64_t c = cam[i], m = pose[i], k = key[i];
    const double2 o = uv[i];
    const double* ct = camtab + c * CAM_STRIDE;
    const double* ptab = posetab + m * POSE_STRIDE;
    const double Xt[3] = {pts4[4 * k], pts4[4 * k + 1], pts4[4 * k + 2]};
    double res[2], Bc[6], Bm[6];
    ObsJac J;
    eval_obs(ct, ptab, Xt, o.x, o.y, res, J);
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            Bc[3 * r + a] = J.Wc[3 * r] * ct[CAM_JL + a] + J.Wc[3 * r + 1] * ct[CAM_JL + 3 + a] + J.Wc[3 * r + 2] * ct[CAM_JL + 6 + a];
            Bm[3 * r + a] = J.Wm[3 * r] * ptab[POSE_JL + a] + J.Wm[3 * r + 1] * ptab[POSE_JL + 3 + a] + J.Wm[3 * r + 2] * ptab[POSE_JL + 6 + a];
        }
    double ju[24], jv[24];
    expand_rows<24>(J, Bc, Bm, ptab, ju, jv);
    double* P = Pk + k * 9;
    double* X = Xck + (c * K + k) * 45;
    double* Y = Ymk + (m * K + k) * 18;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double bu = ju[21 + a], bv = jv[21 + a];
        atomicAdd(gk + 3 * k + a, fma(bu, res[0], bv * res[1]));
#pragma unroll
        for (int b = 0; b < 3; ++b) atomicAdd(P + 3 * a + b, fma(bu, ju[21 + b], bv * jv[21 + b]));
#pragma unroll
        for (int r = 0; r < 15; ++r) {
            const double v = fma(ju[r], bu, jv[r] * bv);
            if (v != 0.0) atomicAdd(X + 3 * r + a, v);
        }
#pragma unroll
        for (int r = 0; r < 6; ++r) atomicAdd(Y + 3 * r + a, fma(ju[15 + r], bu, jv[15 + r] * bv));
    }
}

int launch_point_blocks(pcs_problem* p)
{
    if (p->chain != PCS_CHAIN_SELFCAL || !p->Pk) {
        set_error("point blocks exist for the self-calibration chain (and need (45 C + 18 M) K <= 2^27)");
        return PCS_ERR_UNSUPPORTED;
    }
    if (p->N == 0) return PCS_OK;
    k_normal_points<<<grid_for(p->N, 128), 128, 0, p->stream>>>(p->N, p->K, p->cam, p->pose, p->key, (const double2*)p->uv, p->camtab,
                                                              p->posetab, p->tmpl4, p->Pk, p->gk, p->Xck, p->Ymk);
    ++p->n_launches;
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

// ------------------------------------------------------------------------------------------------
// problem build kernels
// ------------------------------------------------------------------------------------------------
__global__ void k_validate_and_count(int64_t N, int C, int M, int K, int P, const int32_t* __restrict__ cam,
                                     const int32_t* __restrict__ pose, const int32_t* __restrict__ key,
                                     const uint16_t* __restrict__ cam_mask, const uint8_t* __restrict__ pose_mask,
                                     const uint8_t* __restrict__ key_mask, int64_t* __restrict__ counts,
                                     uint64_t* __restrict__ sort_keys, uint32_t* __restrict__ sort_idx, int* __restrict__ bad)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i > N) return;
    if (i == N) {
        counts[N] = 0;
        return;
    }
    const int c = cam[i], m = pose[i], k = key[i];
    if (c < 0 || c >= C || m < 0 || m >= M || k < 0 || k >= K) {
        atomicExch(bad, 1);
        counts[i] = 0;
        sort_keys[i] = 0;
        sort_idx[i] = (uint32_t)i;
        return;
    }
    int n = __popc((unsigned)cam_mask[c]) + __popc((unsigned)pose_mask[m]);
    if (P == 24) n += __popc((unsigned)key_mask[k]);
    counts[i] = n;
    sort_keys[i] = (uint64_t)c * (uint64_t)M + (uint64_t)m;
    sort_idx[i] = (uint32_t)i;
}

__global__ void k_segment_flags(int64_t N, const uint64_t* __restrict__ keys, int32_t* __restrict__ flags)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < N) flags[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// seg_scan = inclusive scan of the segment-head flags (segment id + 1); writes the (camera, pose)-sorted SoA
__global__ void k_segment_fill(int64_t N, int M, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ perm,
                               const int32_t* __restrict__ key_in, const double2* __restrict__ uv_in,
                               const int32_t* __restrict__ seg_scan, int32_t* __restrict__ s_cam, int32_t* __restrict__ s_pose,
                               int32_t* __restrict__ s_key, double2* __restrict__ s_uv, int32_t* __restrict__ seg_cam,
                               int32_t* __restrict__ seg_pose, int64_t* __restrict__ seg_start, int32_t* __restrict__ obs_seg)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int32_t seg = seg_scan[i] - 1;
    const uint32_t src = perm[i];
    const int32_t c = (int32_t)(keys[i] / (uint64_t)M), m = (int32_t)(keys[i] % (uint64_t)M);
    s_cam[i] = c;
    s_pose[i] = m;
    s_key[i] = key_in[src];
    s_uv[i] = uv_in[src];
    obs_seg[src] = seg;
    if (i == 0 || keys[i] != keys[i - 1]) {
        seg_cam[seg] = c;
        seg_pose[seg] = m;
        seg_start[seg] = i;
    }
    if (i == N - 1) seg_start[seg + 1] = N;
}

}  // namespace pcs

using namespace pcs;

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* pcs_last_error(void) { return g_last_error.c_str(); }
const char* pcs_version(void) { return "pcs_b200 0.1 (sm_100a)"; }

int pcs_chain_from_name(const char* name)
{
    if (name && std::strcmp(name, "projection_extrinsic3D_template_points") == 0) return PCS_CHAIN_TEMPLATE;
    if (name && std::strcmp(name, "projection_extrinsic3D_rigidTform3d_free_point") == 0) return PCS_CHAIN_SELFCAL;
    set_error(std::string("unknown function-block chain '") + (name ? name : "(null)") +
              "': only projection_extrinsic3D_template_points and projection_extrinsic3D_rigidTform3d_free_point "
              "have CUDA kernels; there is no CPU fallback");
    return PCS_ERR_CHAIN;
}

int pcs_device_sm_count(int device)
{
    int n = 0;
    PCS_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device));
    return n;
}

int pcs_problem_destroy(pcs_problem* p)
{
    if (!p) return PCS_OK;
    cudaSetDevice(p->device);
    if (p->stream) cudaStreamSynchronize(p->stream);
    lm_free(p);
    p2p_free(p);
    dev_free(p->cam); dev_free(p->pose); dev_free(p->key); dev_free(p->uv); dev_free(p->tmpl); dev_free(p->tmpl4);
    dev_free(p->free_map); dev_free(p->free_idx); dev_free(p->cam_mask); dev_free(p->pose_mask); dev_free(p->key_mask);
    dev_free(p->row_prefix); dev_free(p->params); dev_free(p->x); dev_free(p->camtab); dev_free(p->posetab);
    dev_free(p->resid); dev_free(p->jvals); dev_free(p->seg_cam); dev_free(p->seg_pose); dev_free(p->seg_start);
    dev_free(p->s_key); dev_free(p->s_cam); dev_free(p->s_pose); dev_free(p->s_uv); dev_free(p->obs_seg); dev_free(p->segtab); dev_free(p->ne); dev_free(p->dense); dev_free(p->warp_seg[0]); dev_free(p->warp_seg[1]); dev_free(p->dRtab);
    if (p->h_pin) cudaFreeHost(p->h_pin);
    for (cudaEvent_t e : p->ev_a) cudaEventDestroy(e);
    for (cudaEvent_t e : p->ev_b) cudaEventDestroy(e);
    if (p->copy_stream) cudaStreamDestroy(p->copy_stream);
    for (cudaEvent_t e : p->part_done) if (e) cudaEventDestroy(e);
    if (p->copy_done) cudaEventDestroy(p->copy_done);
    if (p->own_stream && p->stream) cudaStreamDestroy(p->stream);
    delete p;
    return PCS_OK;
}

static int build_problem(pcs_problem* p, const pcs_problem_desc* d)
{
    const int64_t N = p->N;
    PCS_CUDA(cudaSetDevice(p->device));
    PCS_CUDA(cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, p->device));
    if (d->stream) {
        p->stream = (cudaStream_t)d->stream;
    } else {
        PCS_CUDA(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
        p->own_stream = true;
    }
    cudaStream_t st = p->stream;

    // --- observation SoA -------------------------------------------------------------------
    PCS_TRY(dev_alloc(&p->cam, N)); PCS_TRY(dev_alloc(&p->pose, N)); PCS_TRY(dev_alloc(&p->key, N));
    PCS_TRY(dev_alloc(&p->uv, 2 * N));
    const cudaMemcpyKind kind = d->inputs_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (N > 0) {
        PCS_CUDA(cudaMemcpyAsync(p->cam, d->cam, (size_t)N * 4, kind, st));
        PCS_CUDA(cudaMemcpyAsync(p->pose, d->pose, (size_t)N * 4, kind, st));
        PCS_CUDA(cudaMemcpyAsync(p->key, d->key, (size_t)N * 4, kind, st));
        PCS_CUDA(cudaMemcpyAsync(p->uv, d->uv, (size_t)N * 16, kind, st));
    }
    if (p->chain == PCS_CHAIN_TEMPLATE) {
        PCS_TRY(dev_alloc(&p->tmpl, 3 * (int64_t)p->K));
        PCS_CUDA(cudaMemcpyAsync(p->tmpl, d->template_xyz, (size_t)p->K * 24, cudaMemcpyHostToDevice, st));
        PCS_TRY(dev_alloc(&p->tmpl4, 4 * (int64_t)p->K));
        PCS_CUDA(cudaMemsetAsync(p->tmpl4, 0, (size_t)p->K * 32, st));
        PCS_CUDA(cudaMemcpy2DAsync(p->tmpl4, 32, d->template_xyz, 24, 24, (size_t)p->K, cudaMemcpyHostToDevice, st));
    } else {
        PCS_TRY(dev_alloc(&p->tmpl4, 4 * (int64_t)p->K));
        PCS_CUDA(cudaMemsetAsync(p->tmpl4, 0, (size_t)p->K * 32, st));
    }

    // --- free map, masks, free index list (host, O(L)) ---------------------------------------
    const int64_t L = p->L;
    std::vector<int32_t> fm(L);
    if (d->free_map) std::memcpy(fm.data(), d->free_map, (size_t)L * 4);
    else for (int64_t i = 0; i < L; ++i) fm[i] = (int32_t)i;
    int64_t n_free = 0;
    for (int64_t i = 0; i < L; ++i) if (fm[i] >= 0) ++n_free;
    std::vector<int32_t> fidx(std::max<int64_t>(n_free, 1), -1);
    for (int64_t i = 0; i < L; ++i) {
        if (fm[i] < 0) continue;
        PCS_REQUIRE(fm[i] < n_free && fidx[fm[i]] < 0, "free_map must be a bijection onto [0, n_free)");
        fidx[fm[i]] = (int32_t)i;
    }
    p->n_free = n_free;
    std::vector<uint16_t> cmask(std::max(p->C, 1));
    std::vector<uint8_t> pmask(std::max(p->M, 1)), kmask(std::max(p->K, 1), 0);
    for (int c = 0; c < p->C; ++c) {
        uint16_t mk = 0;
        for (int k = 0; k < 9; ++k) if (fm[9 * (int64_t)c + k] >= 0) mk |= (uint16_t)(1u << k);
        for (int k = 0; k < 6; ++k) if (fm[9 * (int64_t)p->C + 6 * (int64_t)c + k] >= 0) mk |= (uint16_t)(1u << (9 + k));
        cmask[c] = mk;
    }
    for (int m = 0; m < p->M; ++m) {
        uint8_t mk = 0;
        for (int k = 0; k < 6; ++k) if (fm[15 * (int64_t)p->C + 6 * (int64_t)m + k] >= 0) mk |= (uint8_t)(1u << k);
        pmask[m] = mk;
    }
    if (p->chain == PCS_CHAIN_SELFCAL)
        for (int k = 0; k < p->K; ++k) {
            uint8_t mk = 0;
            for (int j = 0; j < 3; ++j)
                if (fm[15 * (int64_t)p->C + 6 * (int64_t)p->M + 3 * (int64_t)k + j] >= 0) mk |= (uint8_t)(1u << j);
            kmask[k] = mk;
        }
    PCS_TRY(dev_alloc(&p->free_map, L)); PCS_TRY(dev_alloc(&p->free_idx, n_free));
    PCS_TRY(dev_alloc(&p->cam_mask, p->C)); PCS_TRY(dev_alloc(&p->pose_mask, p->M)); PCS_TRY(dev_alloc(&p->key_mask, p->K));
    PCS_CUDA(cudaMemcpyAsync(p->free_map, fm.data(), (size_t)L * 4, cudaMemcpyHostToDevice, st));
    if (n_free) PCS_CUDA(cudaMemcpyAsync(p->free_idx, fidx.data(), (size_t)n_free * 4, cudaMemcpyHostToDevice, st));
    PCS_CUDA(cudaMemcpyAsync(p->cam_mask, cmask.data(), (size_t)p->C * 2, cudaMemcpyHostToDevice, st));
    PCS_CUDA(cudaMemcpyAsync(p->pose_mask, pmask.data(), (size_t)p->M, cudaMemcpyHostToDevice, st));
    PCS_CUDA(cudaMemcpyAsync(p->key_mask, kmask.data(), (size_t)p->K, cudaMemcpyHostToDevice, st));

    // --- dynamic state ------------------------------------------------------------------------
    PCS_TRY(dev_alloc(&p->params, L)); PCS_TRY(dev_alloc(&p->x, n_free));
    PCS_TRY(dev_alloc(&p->camtab, (int64_t)p->C * CAM_STRIDE)); PCS_TRY(dev_alloc(&p->posetab, (int64_t)p->M * POSE_STRIDE));
    PCS_CUDA(cudaMemsetAsync(p->params, 0, (size_t)L * 8, st));

    // --- per-observation free-column counts, sort keys ------------------------------------------
    PCS_TRY(dev_alloc(&p->row_prefix, N + 1));
    uint64_t *keys_a = nullptr, *keys_b = nullptr;
    uint32_t *idx_a = nullptr, *idx_b = nullptr;
    int* bad = nullptr;
    int32_t *flags = nullptr, *seg_scan = nullptr;
    void* tmp = nullptr;
    int rc = PCS_OK;
    auto cleanup = [&]() {
        dev_free(keys_a); dev_free(keys_b); dev_free(idx_a); dev_free(idx_b); dev_free(bad); dev_free(flags); dev_free(seg_scan);
        if (tmp) cudaFree(tmp);
    };
#define BUILD_TRY(expr) do { rc = (expr); if (rc != PCS_OK) { cleanup(); return rc; } } while (0)
#define BUILD_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { set_error(std::string(#call) + " -> " + cudaGetErrorString(e__)); cleanup(); return PCS_ERR_CUDA; } } while (0)
    BUILD_TRY(dev_alloc(&keys_a, N)); BUILD_TRY(dev_alloc(&keys_b, N));
    BUILD_TRY(dev_alloc(&idx_a, N)); BUILD_TRY(dev_alloc(&idx_b, N));
    BUILD_TRY(dev_alloc(&bad, 1)); BUILD_TRY(dev_alloc(&flags, N));
    BUILD_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), st));
    k_validate_and_count<<<grid_for(N + 1, 256), 256, 0, st>>>(N, p->C, p->M, p->K, p->P, p->cam, p->pose, p->key,
                                                               p->cam_mask, p->pose_mask, p->key_mask, p->row_prefix,
                                                               keys_a, idx_a, bad);
    BUILD_CUDA(cudaGetLastError());
    int h_bad = 0;
    BUILD_CUDA(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BUILD_CUDA(cudaStreamSynchronize(st));
    if (h_bad) {
        set_error("observation table has a camera / pose / key index outside [0, n_cams) x [0, n_poses) x [0, n_keys)");
        cleanup();
        return PCS_ERR_INVALID;
    }
    size_t tmp_bytes = 0, need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, p->row_prefix, p->row_prefix, N + 1, st);
    tmp_bytes = std::max(tmp_bytes, need);
    int key_bits = 1;
    while (key_bits < 64 && ((uint64_t)1 << key_bits) < (uint64_t)std::max<int64_t>(1, (int64_t)p->C * p->M)) ++key_bits;
    cub::DeviceRadixSort::SortPairs(nullptr, need, keys_a, keys_b, idx_a, idx_b, N, 0, key_bits, st);
    tmp_bytes = std::max(tmp_bytes, need);
    cub::DeviceScan::InclusiveSum(nullptr, need, flags, flags, N, st);
    tmp_bytes = std::max(tmp_bytes, need);
    BUILD_CUDA(cudaMalloc(&tmp, std::max<size_t>(tmp_bytes, 16)));
    need = tmp_bytes;
    BUILD_CUDA(cub::DeviceScan::ExclusiveSum(tmp, need, p->row_prefix, p->row_prefix, N + 1, st));
    int64_t h_total = 0;
    BUILD_CUDA(cudaMemcpyAsync(&h_total, p->row_prefix + N, 8, cudaMemcpyDeviceToHost, st));

    // --- (camera, pose)-sorted layout -------------------------------------------------------------
    BUILD_TRY(dev_alloc(&p->s_key, N)); BUILD_TRY(dev_alloc(&p->s_cam, N)); BUILD_TRY(dev_alloc(&p->s_pose, N));
    BUILD_TRY(dev_alloc(&p->s_uv, 2 * N)); BUILD_TRY(dev_alloc(&seg_scan, N)); BUILD_TRY(dev_alloc(&p->obs_seg, N));
    int64_t n_seg = 0;
    if (N > 0) {
        need = tmp_bytes;
        BUILD_CUDA(cub::DeviceRadixSort::SortPairs(tmp, need, keys_a, keys_b, idx_a, idx_b, N, 0, key_bits, st));
        k_segment_flags<<<grid_for(N, 256), 256, 0, st>>>(N, keys_b, flags);
        need = tmp_bytes;
        BUILD_CUDA(cub::DeviceScan::InclusiveSum(tmp, need, flags, seg_scan, N, st));
        int32_t h_nseg = 0;
        BUILD_CUDA(cudaMemcpyAsync(&h_nseg, seg_scan + (N - 1), 4, cudaMemcpyDeviceToHost, st));
        BUILD_CUDA(cudaStreamSynchronize(st));
        n_seg = h_nseg;
    } else {
        BUILD_CUDA(cudaStreamSynchronize(st));
    }
    p->nnz = 2 * h_total;
    p->n_seg = n_seg;
    BUILD_TRY(dev_alloc(&p->seg_cam, n_seg)); BUILD_TRY(dev_alloc(&p->seg_pose, n_seg)); BUILD_TRY(dev_alloc(&p->seg_start, n_seg + 1));
    if (N > 0) {
        k_segment_fill<<<grid_for(N, 256), 256, 0, st>>>(N, p->M, keys_b, idx_b, p->key, (const double2*)p->uv, seg_scan, p->s_cam,
                                                         p->s_pose, p->s_key, (double2*)p->s_uv, p->seg_cam, p->seg_pose,
                                                         p->seg_start, p->obs_seg);
        BUILD_CUDA(cudaGetLastError());
    } else {
        BUILD_CUDA(cudaMemsetAsync(p->seg_start, 0, 8, st));
    }

    // --- normal-equation outputs: [U | gc | cost | pad | V | gp | W] -------------------------------------
    const int64_t nU = (int64_t)p->C * 225, ngc = (int64_t)p->C * 15, nV = (int64_t)p->M * 36, ngp = (int64_t)p->M * 6;
    const int64_t head = (nU + ngc + 1 + 1) / 2 * 2;
    // chain 1: point blocks and the dense camera x point / pose x point coupling tables sit between gp and W (all of
    // them are accumulated with reductions and cleared by the prepare launch); skipped when they would exceed 2^27 doubles
    int64_t nP = 0, ngk = 0, nX = 0, nY = 0;
    if (p->chain == PCS_CHAIN_SELFCAL && ((int64_t)p->C * 45 + (int64_t)p->M * 18) * p->K <= ((int64_t)1 << 27)) {
        nP = ((int64_t)p->K * 9 + 1) / 2 * 2; ngk = ((int64_t)p->K * 3 + 1) / 2 * 2; nX = (int64_t)p->C * p->K * 45 / 2 * 2 + 2; nY = (int64_t)p->M * p->K * 18;
    }
    p->ne_doubles = head + nV + ngp + nP + ngk + nX + nY + n_seg * 90;
    BUILD_TRY(dev_alloc(&p->ne, p->ne_doubles));
    p->U = p->ne; p->gc = p->U + nU; p->cost = p->gc + ngc; p->V = p->ne + head; p->gp = p->V + nV;
    double* q = p->gp + ngp;
    if (nP) { p->Pk = q; p->gk = p->Pk + nP; p->Xck = p->gk + ngk; p->Ymk = p->Xck + nX; q = p->Ymk + nY; }
    p->W = q;

    BUILD_CUDA(cudaStreamSynchronize(st));
    cleanup();
#undef BUILD_TRY
#undef BUILD_CUDA
    return PCS_OK;
}

int pcs_problem_create(const pcs_problem_desc* d, pcs_problem** out)
{
    PCS_REQUIRE(d && out, "desc / out is NULL");
    *out = nullptr;
    if (d->chain != PCS_CHAIN_TEMPLATE && d->chain != PCS_CHAIN_SELFCAL) {
        set_error("unknown chain id; only the two shipped function-block chains are accelerated (no CPU fallback)");
        return PCS_ERR_CHAIN;
    }
    PCS_REQUIRE(d->n_obs >= 0 && d->n_cams > 0 && d->n_poses > 0 && d->n_keys > 0, "sizes must be positive");
    PCS_REQUIRE(d->n_obs < ((int64_t)1 << 31), "n_obs must be below 2^31 per problem (shard by pose across GPUs)");
    PCS_REQUIRE(d->n_obs == 0 || (d->cam && d->pose && d->key && d->uv), "observation arrays are NULL");
    PCS_REQUIRE(d->chain != PCS_CHAIN_TEMPLATE || d->template_xyz, "template chain needs template_xyz");
    int n_dev = 0;
    PCS_CUDA(cudaGetDeviceCount(&n_dev));
    PCS_REQUIRE(d->device >= 0 && d->device < n_dev, "device ordinal out of range");
    pcs_problem* p = new (std::nothrow) pcs_problem();
    PCS_REQUIRE(p, "out of host memory");
    p->chain = d->chain; p->device = d->device; p->N = d->n_obs; p->C = d->n_cams; p->M = d->n_poses; p->K = d->n_keys;
    p->P = d->chain == PCS_CHAIN_TEMPLATE ? 21 : 24;
    p->L = 15 * (int64_t)p->C + 6 * (int64_t)p->M + (d->chain == PCS_CHAIN_SELFCAL ? 3 * (int64_t)p->K : 0);
    int rc = build_problem(p, d);
    if (rc != PCS_OK) {
        std::string keep = g_last_error;
        pcs_problem_destroy(p);
        set_error(keep);
        return rc;
    }
    *out = p;
    return PCS_OK;
}

int pcs_problem_get_info(const pcs_problem* p, pcs_problem_info* info)
{
    PCS_REQUIRE(p && info, "NULL argument");
    info->chain = p->chain; info->n_cams = p->C; info->n_poses = p->M; info->n_keys = p->K; info->cols_per_row = p->P;
    info->device = p->device; info->n_obs = p->N; info->n_params = p->L; info->n_free = p->n_free; info->nnz = p->nnz;
    info->n_segments = p->n_seg;
    return PCS_OK;
}

int pcs_set_param_string(pcs_problem* p, const double* params)
{
    PCS_REQUIRE(p && params, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    PCS_TRY(ensure_pinned(p, p->L));
    std::memcpy(p->h_pin, params, (size_t)p->L * 8);
    PCS_CUDA(cudaMemcpyAsync(p->params, p->h_pin, (size_t)p->L * 8, cudaMemcpyHostToDevice, p->stream));
    PCS_CUDA(cudaStreamSynchronize(p->stream));
    return PCS_OK;
}

int pcs_get_param_string(pcs_problem* p, double* params)
{
    PCS_REQUIRE(p && params, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    PCS_CUDA(cudaMemcpyAsync(params, p->params, (size_t)p->L * 8, cudaMemcpyDeviceToHost, p->stream));
    PCS_CUDA(cudaStreamSynchronize(p->stream));
    return PCS_OK;
}

// host x -> device x -> parameter string (x == NULL: keep current parameters)
static int upload_x(pcs_problem* p, const double* x)
{
    if (!x || p->n_free == 0) return PCS_OK;
    PCS_TRY(ensure_pinned(p, p->n_free));
    std::memcpy(p->h_pin, x, (size_t)p->n_free * 8);
    PCS_CUDA(cudaMemcpyAsync(p->x, p->h_pin, (size_t)p->n_free * 8, cudaMemcpyHostToDevice, p->stream));
    return launch_scatter_x(p, p->x);
}

int pcs_set_free(pcs_problem* p, const double* x)
{
    PCS_REQUIRE(p && x, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    PCS_TRY(upload_x(p, x));
    PCS_CUDA(cudaStreamSynchronize(p->stream));
    return PCS_OK;
}

int pcs_residual_dev(pcs_problem* p, const double* x_dev, double* r_dev)
{
    PCS_REQUIRE(p && r_dev, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    // two launches per call: [x scatter + camera / pose tables + per-segment transforms] and the residual kernel
    PCS_TRY(launch_prepare(p, false, x_dev, nullptr, 0, true));
    return launch_residual(p, r_dev);
}

int pcs_residual(pcs_problem* p, const double* x, double* r_out)
{
    PCS_REQUIRE(p && r_out, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    if (!p->resid) PCS_TRY(dev_alloc(&p->resid, 2 * p->N));
    const double* x_dev = nullptr;
    if (x && p->n_free > 0) {
        PCS_TRY(ensure_pinned(p, p->n_free));
        std::memcpy(p->h_pin, x, (size_t)p->n_free * 8);
        PCS_CUDA(cudaMemcpyAsync(p->x, p->h_pin, (size_t)p->n_free * 8, cudaMemcpyHostToDevice, p->stream));
        x_dev = p->x;
    }
    PCS_TRY(launch_prepare(p, false, x_dev, nullptr, 0, true));
    PCS_TRY(launch_residual(p, p->resid));
    if (p->N) PCS_CUDA(cudaMemcpyAsync(r_out, p->resid, (size_t)p->N * 16, cudaMemcpyDeviceToHost, p->stream));
    PCS_CUDA(cudaStreamSynchronize(p->stream));
    return PCS_OK;
}

int pcs_csr_structure(pcs_problem* p, int64_t* col_idx, int64_t* row_ptr)
{
    PCS_REQUIRE(p && col_idx && row_ptr, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    int64_t *d_col = nullptr, *d_rp = nullptr;
    PCS_TRY(dev_alloc(&d_col, p->nnz));
    int rc = dev_alloc(&d_rp, 2 * p->N + 1);
    if (rc != PCS_OK) { dev_free(d_col); return rc; }
    k_csr_structure<<<grid_for(p->N + 1, 256), 256, 0, p->stream>>>(p->N, p->P, p->C, p->M, p->cam, p->pose, p->key,
                                                                    p->free_map, p->row_prefix, d_col, d_rp);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && p->nnz) e = cudaMemcpyAsync(col_idx, d_col, (size_t)p->nnz * 8, cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(row_ptr, d_rp, (size_t)(2 * p->N + 1) * 8, cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    dev_free(d_col); dev_free(d_rp);
    if (e != cudaSuccess) { set_error(std::string("csr structure: ") + cudaGetErrorString(e)); return PCS_ERR_CUDA; }
    return PCS_OK;
}

int pcs_jacobian_values_dev(pcs_problem* p, const double* x_dev, double* vals_dev)
{
    PCS_REQUIRE(p && vals_dev, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    if (x_dev) PCS_TRY(launch_scatter_x(p, x_dev));
    PCS_TRY(launch_prepare(p, true));
    if (p->N == 0) return PCS_OK;
    const int grid = grid_for(p->N, 128);
    const size_t smem = (size_t)4 * 64 * p->P * sizeof(double);
    auto kern = p->P == 21 ? k_jacobian<21> : k_jacobian<24>;
    PCS_CUDA(ensure_dynamic_smem(kern, smem));
    kern<<<grid, 128, smem, p->stream>>>(p->N, p->cam, p->pose, p->key, (const double2*)p->uv, p->camtab, p->posetab, p->dRtab,
                                         points_ptr(p), p->cam_mask, p->pose_mask, p->key_mask, p->row_prefix, p->C, vals_dev);
    PCS_CUDA(cudaGetLastError());
    ++p->n_launches;
    return PCS_OK;
}

int pcs_jacobian_values(pcs_problem* p, const double* x, double* vals_out)
{
    PCS_REQUIRE(p && vals_out, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    if (!p->jvals) PCS_TRY(dev_alloc(&p->jvals, p->nnz));
    PCS_TRY(upload_x(p, x));
    PCS_TRY(pcs_jacobian_values_dev(p, nullptr, p->jvals));
    if (p->nnz) PCS_CUDA(cudaMemcpyAsync(vals_out, p->jvals, (size_t)p->nnz * 8, cudaMemcpyDeviceToHost, p->stream));
    PCS_CUDA(cudaStreamSynchronize(p->stream));
    return PCS_OK;
}

int pcs_segments(pcs_problem* p, int32_t* seg_cam, int32_t* seg_pose, int64_t* seg_len)
{
    PCS_REQUIRE(p, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    const int64_t S = p->n_seg;
    if (S == 0) return PCS_OK;
    if (seg_cam) PCS_CUDA(cudaMemcpyAsync(seg_cam, p->seg_cam, (size_t)S * 4, cudaMemcpyDeviceToHost, p->stream));
    if (seg_pose) PCS_CUDA(cudaMemcpyAsync(seg_pose, p->seg_pose, (size_t)S * 4, cudaMemcpyDeviceToHost, p->stream));
    std::vector<int64_t> start;
    if (seg_len) {
        start.resize(S + 1);
        PCS_CUDA(cudaMemcpyAsync(start.data(), p->seg_start, (size_t)(S + 1) * 8, cudaMemcpyDeviceToHost, p->stream));
    }
    PCS_CUDA(cudaStreamSynchronize(p->stream));
    if (seg_len) for (int64_t s = 0; s < S; ++s) seg_len[s] = start[s + 1] - start[s];
    return PCS_OK;
}

static int require_block_path(const pcs_problem* p)
{
    if (p->chain == PCS_CHAIN_SELFCAL && !p->Pk) {
        set_error("block normal equations of the self-calibration chain keep dense (camera, key) / (pose, key) tables and need "
                  "(45 C + 18 M) K <= 2^27; use pcs_normal_dense for this problem");
        return PCS_ERR_UNSUPPORTED;
    }
    return PCS_OK;
}

int pcs_normal_equations_dev(pcs_problem* p, const double* x_dev)
{
    PCS_REQUIRE(p, "NULL argument");
    PCS_TRY(require_block_path(p));
    PCS_CUDA(cudaSetDevice(p->device));
    // one launch: x -> parameter string, camera / pose tables, cleared reduction targets [U | gc | cost | pad | V | gp (| point blocks)]
    PCS_TRY(launch_prepare(p, false, x_dev, p->ne, ne_zero_doubles(p)));
    PCS_TRY(launch_normal_blocks(p, true));
    if (p->chain == PCS_CHAIN_SELFCAL) PCS_TRY(launch_point_blocks(p));
    return PCS_OK;
}

int pcs_point_blocks(pcs_problem* p, double* Pk, double* gk, double* Xck, double* Ymk)
{
    PCS_REQUIRE(p, "NULL argument");
    if (p->chain != PCS_CHAIN_SELFCAL) { set_error("point blocks exist for the self-calibration chain"); return PCS_ERR_UNSUPPORTED; }
    PCS_TRY(require_block_path(p));
    PCS_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = p->stream;
    if (Pk) PCS_CUDA(cudaMemcpyAsync(Pk, p->Pk, (size_t)p->K * 9 * 8, cudaMemcpyDeviceToHost, st));
    if (gk) PCS_CUDA(cudaMemcpyAsync(gk, p->gk, (size_t)p->K * 3 * 8, cudaMemcpyDeviceToHost, st));
    if (Xck) PCS_CUDA(cudaMemcpyAsync(Xck, p->Xck, (size_t)p->C * p->K * 45 * 8, cudaMemcpyDeviceToHost, st));
    if (Ymk) PCS_CUDA(cudaMemcpyAsync(Ymk, p->Ymk, (size_t)p->M * p->K * 18 * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_normal_equations(pcs_problem* p, const double* x, double* U, double* gc, double* V, double* gp, double* W,
                         double* cost)
{
    PCS_REQUIRE(p, "NULL argument");
    PCS_TRY(require_block_path(p));
    PCS_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = p->stream;
    // host x -> device (pinned staging), then one launch: scatter + tables + cleared reduction targets
    const double* x_dev = nullptr;
    if (x && p->n_free > 0) {
        PCS_TRY(ensure_pinned(p, p->n_free));
        std::memcpy(p->h_pin, x, (size_t)p->n_free * 8);
        PCS_CUDA(cudaMemcpyAsync(p->x, p->h_pin, (size_t)p->n_free * 8, cudaMemcpyHostToDevice, st));
        x_dev = p->x;
    }
    PCS_TRY(launch_prepare(p, false, x_dev, p->ne, ne_zero_doubles(p)));
    // W is by far the largest output (720 B per segment): the evaluation runs in parts and the copy-out of a finished
    // part's segments proceeds on a second stream while the next part is evaluated
    const int n_parts = (W && p->n_seg >= 4096) ? 4 : 1;
    if (n_parts > 1 && !p->copy_stream) {
        PCS_CUDA(cudaStreamCreateWithFlags(&p->copy_stream, cudaStreamNonBlocking));
        for (int k = 0; k < 8; ++k) PCS_CUDA(cudaEventCreateWithFlags(&p->part_done[k], cudaEventDisableTiming));
        PCS_CUDA(cudaEventCreateWithFlags(&p->copy_done, cudaEventDisableTiming));
    }
    for (int part = 0; part < n_parts; ++part) {
        PCS_TRY(launch_normal_blocks(p, true, part, n_parts));
        if (n_parts > 1) {
            const int64_t s0 = p->h_part_bounds[part], s1 = p->h_part_bounds[part + 1];
            PCS_CUDA(cudaEventRecord(p->part_done[part], st));
            if (s1 > s0) {
                PCS_CUDA(cudaStreamWaitEvent(p->copy_stream, p->part_done[part], 0));
                PCS_CUDA(cudaMemcpyAsync(W + s0 * 90, p->W + s0 * 90, (size_t)(s1 - s0) * 90 * 8, cudaMemcpyDeviceToHost, p->copy_stream));
            }
        }
    }
    if (p->chain == PCS_CHAIN_SELFCAL) PCS_TRY(launch_point_blocks(p));   // left on the device: pcs_point_blocks copies them out
    if (U) PCS_CUDA(cudaMemcpyAsync(U, p->U, (size_t)p->C * 225 * 8, cudaMemcpyDeviceToHost, st));
    if (gc) PCS_CUDA(cudaMemcpyAsync(gc, p->gc, (size_t)p->C * 15 * 8, cudaMemcpyDeviceToHost, st));
    if (V) PCS_CUDA(cudaMemcpyAsync(V, p->V, (size_t)p->M * 36 * 8, cudaMemcpyDeviceToHost, st));
    if (gp) PCS_CUDA(cudaMemcpyAsync(gp, p->gp, (size_t)p->M * 6 * 8, cudaMemcpyDeviceToHost, st));
    if (W && p->n_seg && n_parts == 1) PCS_CUDA(cudaMemcpyAsync(W, p->W, (size_t)p->n_seg * 90 * 8, cudaMemcpyDeviceToHost, st));
    if (cost) PCS_CUDA(cudaMemcpyAsync(cost, p->cost, 8, cudaMemcpyDeviceToHost, st));
    if (n_parts > 1) {
        PCS_CUDA(cudaEventRecord(p->copy_done, p->copy_stream));
        PCS_CUDA(cudaStreamWaitEvent(st, p->copy_done, 0));
    }
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

// dense normal equations at the current parameters, left on the device in p->dense = [JtJ | Jtr | cost]
int pcs_normal_dense_dev_internal(pcs_problem* p)
{
    const int64_t n = p->n_free;
    PCS_REQUIRE(n > 0 && n <= 32768, "dense normal equations need 0 < n_free <= 32768");
    if (!p->dense) PCS_TRY(dev_alloc(&p->dense, n * n + n + 1));
    PCS_TRY(launch_prepare(p, true));
    cudaStream_t st = p->stream;
    PCS_CUDA(cudaMemsetAsync(p->dense, 0, (size_t)(n * n + n + 1) * 8, st));
    double *dJ = p->dense, *dg = p->dense + n * n, *dc = dg + n;
    if (p->N) {
        if (p->P == 21)
            k_normal_dense<21><<<grid_for(p->N, 128), 128, 0, st>>>(p->N, p->C, p->M, n, p->cam, p->pose, p->key,
                                                                    (const double2*)p->uv, p->camtab, p->posetab, p->dRtab,
                                                                    points_ptr(p), p->free_map, dJ, dg, dc);
        else
            k_normal_dense<24><<<grid_for(p->N, 128), 128, 0, st>>>(p->N, p->C, p->M, n, p->cam, p->pose, p->key,
                                                                    (const double2*)p->uv, p->camtab, p->posetab, p->dRtab,
                                                                    points_ptr(p), p->free_map, dJ, dg, dc);
        PCS_CUDA(cudaGetLastError());
    }
    k_symmetrize_blocks<<<grid_for(n * n, 256), 256, 0, st>>>(1, (int)n, dJ);
    PCS_CUDA(cudaGetLastError());
    return PCS_OK;
}

int pcs_normal_dense(pcs_problem* p, const double* x, double* JtJ, double* Jtr, double* cost)
{
    PCS_REQUIRE(p && JtJ && Jtr && cost, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    PCS_TRY(upload_x(p, x));
    PCS_TRY(pcs_normal_dense_dev_internal(p));
    const int64_t n = p->n_free;
    cudaStream_t st = p->stream;
    double *dJ = p->dense, *dg = p->dense + n * n, *dc = dg + n;
    PCS_CUDA(cudaMemcpyAsync(JtJ, dJ, (size_t)(n * n) * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaMemcpyAsync(Jtr, dg, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaMemcpyAsync(cost, dc, 8, cudaMemcpyDeviceToHost, st));
    PCS_CUDA(cudaStreamSynchronize(st));
    return PCS_OK;
}

int pcs_device_buffers_get(pcs_problem* p, pcs_device_buffers* out)
{
    PCS_REQUIRE(p && out, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    if (!p->resid) PCS_TRY(dev_alloc(&p->resid, 2 * p->N));
    out->params = p->params; out->U = p->U; out->gc = p->gc; out->V = p->V; out->gp = p->gp; out->W = p->W;
    out->cost = p->cost; out->residual = p->resid; out->stream = (void*)p->stream;
    return PCS_OK;
}

int pcs_launch_count(const pcs_problem* p, int64_t* n_kernels)
{
    PCS_REQUIRE(p && n_kernels, "NULL argument");
    *n_kernels = p->n_launches;
    return PCS_OK;
}

constexpr int TIMING_RING = 1024;

int pcs_timing_enable(pcs_problem* p, int on)
{
    PCS_REQUIRE(p, "NULL argument");
    PCS_CUDA(cudaSetDevice(p->device));
    if (on && p->ev_a.empty()) {
        p->ev_a.resize(TIMING_RING);
        p->ev_b.resize(TIMING_RING);
        for (int i = 0; i < TIMING_RING; ++i) {
            PCS_CUDA(cudaEventCreate(&p->ev_a[i]));
            PCS_CUDA(cudaEventCreate(&p->ev_b[i]));
        }
    }
    if (on) p->timing_count = 0;
    p->timing = on != 0;
    return PCS_OK;
}

// most recent launch
int pcs_timing_get(pcs_problem* p, double* ms)
{
    PCS_REQUIRE(p && ms && !p->ev_a.empty() && p->timing_count > 0, "no timed launch recorded");
    PCS_CUDA(cudaSetDevice(p->device));
    const int i = (int)((p->timing_count - 1) % TIMING_RING);
    PCS_CUDA(cudaEventSynchronize(p->ev_b[i]));
    float f = 0.f;
    PCS_CUDA(cudaEventElapsedTime(&f, p->ev_a[i], p->ev_b[i]));
    *ms = f;
    return PCS_OK;
}

// durations (ms) of the last min(count, capacity, ring) launches since pcs_timing_enable(p, 1), oldest first
int pcs_timing_get_all(pcs_problem* p, double* ms, int64_t capacity, int64_t* n_out)
{
    PCS_REQUIRE(p && ms && n_out && !p->ev_a.empty(), "timing was never enabled");
    PCS_CUDA(cudaSetDevice(p->device));
    const int64_t n = std::min<int64_t>(std::min<int64_t>(p->timing_count, TIMING_RING), capacity);
    for (int64_t k = 0; k < n; ++k) {
        const int i = (int)((p->timing_count - n + k) % TIMING_RING);
        PCS_CUDA(cudaEventSynchronize(p->ev_b[i]));
        float f = 0.f;
        PCS_CUDA(cudaEventElapsedTime(&f, p->ev_a[i], p->ev_b[i]));
        ms[k] = f;
    }
    *n_out = n;
    return PCS_OK;
}

int pcs_set_normal_precision(pcs_problem* p, int precision)
{
    PCS_REQUIRE(p, "NULL argument");
    PCS_REQUIRE(precision == PCS_PRECISION_FP64 || precision == PCS_PRECISION_MIXED, "precision must be PCS_PRECISION_FP64 or PCS_PRECISION_MIXED");
    if (precision == PCS_PRECISION_MIXED && p->chain != PCS_CHAIN_TEMPLATE) {
        set_error("the mixed-precision normal-equation kernel exists for the template chain");
        return PCS_ERR_UNSUPPORTED;
    }
    p->normal_precision = precision;
    return PCS_OK;
}

int pcs_set_allreduce(pcs_problem* p, pcs_allreduce_fn fn, void* user, int rank, int world_size)
{
    PCS_REQUIRE(p, "NULL argument");
    PCS_REQUIRE(world_size >= 1 && rank >= 0 && rank < world_size, "rank / world_size out of range");
    if (world_size != p->world) {   // the LM workspace is laid out for one world size (its path, its all-reduce buffers)
        PCS_CUDA(cudaSetDevice(p->device));
        lm_free(p);
    }
    p->allreduce = world_size > 1 ? fn : nullptr;
    p->allreduce_user = user;
    p->rank = rank;
    p->world = world_size;
    return PCS_OK;
}

}  // extern "C"

