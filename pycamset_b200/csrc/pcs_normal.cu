// pcs_normal.cu -- K_ne: fused residual + analytic Jacobian + J^T J / J^T r (template chain), the north-star kernel.
//
// No reference counterpart computes J^T J (scipy's LSMR consumes the CSR Jacobian, optimisation_handling.py:88-98);
// the per-observation math is the reference chain projection + extrinsic3D + template_points
// (function_block_implementations.py:21-211, matmul_map.py:147-243) as restated in pcs_math.cuh.
//
// Design (B200, FP64):
//   * Observations are sorted by (camera, pose) at problem build; a "segment" is one (camera, pose) pair.
//   * A warp owns a contiguous range of WHOLE segments (balanced by observation count) and walks it in batches
//     of 32 observations (inputs of batch n+1 are prefetched while batch n runs), one lane per observation: the
//     lane evaluates residual and Jacobian in registers and parks its two augmented rows
//         J' = [cam(0..7) | cam(8..14) r]        (16 doubles each)
//     in shared memory -- 8 KB per warp, swizzled so that both the 16-byte row stores and the fragment loads below
//     are bank-conflict free.
//   * Only the CAMERA columns are accumulated per observation.  Inside one segment the six pose columns are the
//     six extrinsic columns times a constant adjoint,  [w_m | n] = [w_c | p] T,  T = [[R_c, 0], [[R_c t_m]x R_c, R_c]]
//     (rows in the tangent parametrisation, pcs_math.cuh), so V_m, g_m and W_{c,m} follow from the SEGMENT's camera
//     Gram matrix G_s at flush time:   W_s = G_s[:, 9:15] T,   V_m += T^T G_s[9:15, 9:15] T,   g_m += T^T g_s[9:15].
//     That halves the per-observation Gram work: 16 columns = exactly two 8-column tiles.
//   * The Gram update  G += J'^T J'  runs on the FP64 tensor path: per 2 observations (4 rows = one k-step) the warp
//     loads 2 fragment values per lane and issues 3 DMMA m8n8k4 (tile pairs AA, AB, BB).  A-fragment and B-fragment
//     of a tile are the same register.
//   * Two accumulator sets: the segment's (registers; flushed per segment on the tensor path: W by 16-byte plain
//     stores -- the warp owns the segment -- V/g_m by FP64 reductions) and the camera's running sums (U_c, g_c, r.r;
//     a 16 x 16 block in shared memory, flushed when the camera changes).
//   * Rotation rows are accumulated in the tangent parametrisation; the SO(3) left Jacobians are applied once per
//     block inside the flushes (Jl_m folded into the adjoint, Jl_c on three rows of W_s and on U_c / g_c).
//   HBM traffic per observation: (u,v) 16 B + camera, pose, key 12 B = 28 B read; outputs are O(segments).
#include <algorithm>

#include "pcs_internal.cuh"
#include "pcs_math.cuh"

namespace pcs {

constexpr int NE_WARPS = 4;                  // warps per CTA
constexpr int NE_TILE_DOUBLES = 64 * 8;      // one 8-column tile of the 64 staged rows
constexpr int NE_SCRATCH_DOUBLES = 64 + 192;           // Tbar (8 x 8, flush_segment) | running camera sums (tiles AA, AB, BB)
constexpr int NE_WARP_DOUBLES = 2 * NE_TILE_DOUBLES + NE_SCRATCH_DOUBLES;

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// Shared-memory position of staged row (observation slot o in 0..31, row r in {u, v}) and column c of one tile:
//   word(o, r, c) = 8 * rho(o, r) + (c ^ rot(o)),   rho = 2 o + (r ^ bit1(o)),   rot = 4 bit0(o) + 2 bit2(o)  (even).
// rho is a bijection onto 0..63.  With this swizzle
//   - the 16-byte stores of a quarter warp (8 consecutive o, fixed r and column pair) hit 8 distinct 16-byte banks;
//   - the 8-byte fragment loads of a half warp (4 rows of one k-step x 4 columns) hit 16 distinct 8-byte banks.
// For the fragment loads of k-step ks (rows o = 2 ks + jb, r = jr; column g8) this collapses to
//   word = 32 ks + (L ^ X(ks)),   L = 16 jb + 8 jr + (g8 ^ 4 jb),   X(ks) = 8 bit0(ks) + 2 bit1(ks).
__device__ __forceinline__ int stage_row(int o, int r) { return (2 * o + (r ^ ((o >> 1) & 1))) * 8; }
__device__ __forceinline__ int stage_rot(int o) { return 4 * (o & 1) + 2 * ((o >> 2) & 1); }

// Fragment (m8n8 accumulator) layout: lane holds rows lane >> 2, columns 2 (lane & 3) + {0, 1} of an 8 x 8 tile.
// Column order of the 16 accumulated columns: 0..14 = camera (9 intrinsic, 3 rotation (tangent), 3 translation), 15 = r.
struct NeAcc {
    double aa[2], ab[2], bb[2];
};

__device__ __forceinline__ void acc_zero(NeAcc& A) { A.aa[0] = A.aa[1] = A.ab[0] = A.ab[1] = A.bb[0] = A.bb[1] = 0.0; }

// Running camera sums: tiles AA = G[0:8,0:8], AB = G[0:8,8:16], BB = G[8:16,8:16] of the symmetric 16 x 16 matrix,
// 64 doubles each; element (row, col) of a tile sits at row * 8 + (col ^ bit1(row)), which makes the per-lane
// read-modify-write of flush_segment (rows lane >> 2, columns 2 (lane & 3) + i) bank-conflict free.
__device__ __forceinline__ int cam_tile_pos(int row, int col) { return row * 8 + (col ^ ((row >> 1) & 1)); }
__device__ __forceinline__ double cam_sum(const double* __restrict__ G, int a, int b)   // G(a, b), 0 <= a, b < 16
{
    if (a > b) { const int t = a; a = b; b = t; }
    if (b < 8) return G[cam_tile_pos(a, b)];
    if (a < 8) return G[64 + cam_tile_pos(a, b - 8)];
    return G[128 + cam_tile_pos(a - 8, b - 8)];
}

// double-precision shuffle of one of two registers: returns (sel ? x1 : x0) of lane `src`
__device__ __forceinline__ double shfl_pick(double x0, double x1, int src, bool sel)
{
    const double y0 = __shfl_sync(0xffffffffu, x0, src), y1 = __shfl_sync(0xffffffffu, x1, src);
    return sel ? y1 : y0;
}

// D (8 x 8, accumulator layout) = X (8 x 8, accumulator layout) * Tbar (8 x 8), as two DMMA k-steps; tb0 / tb1 are
// the lane's Tbar fragments for k = 0..3 / 4..7 (Tbar[4h + (lane & 3)][lane >> 2]).
__device__ __forceinline__ void tile_times_tbar(const double x[2], double tb0, double tb1, int lane, double d[2])
{
    d[0] = d[1] = 0.0;
    // A fragment element (row = lane >> 2, k = 4h + (lane & 3)) sits in lane (row * 4 + k / 2), register k & 1
    const int quad = lane & ~3, half = (lane & 3) >> 1;
    const bool odd = lane & 1;
    const double a0 = shfl_pick(x[0], x[1], quad + half, odd);
    const double a1 = shfl_pick(x[0], x[1], quad + 2 + half, odd);
    dmma884(d[0], d[1], a0, tb0);
    dmma884(d[0], d[1], a1, tb1);
}

// Segment flush.  S = this segment's camera Gram matrix G_s (fragments: aa = G[0:8,0:8], ab = G[0:8,8:16],
// bb = G[8:16,8:16]; column 8 + kk with kk = 0: k3, 1..3: camera rotation (tangent), 4..6: camera translation, 7: r).
// G = the running camera sums (shared memory).  With the adjoint folded with the pose's left Jacobian,
//     T' = [[R_c Jl_m, 0], [[s]x R_c Jl_m, R_c]],  s = R_c t_m,
// embedded as Tbar[1..6][0..5] = T', Tbar[7][6] = 1 (zero elsewhere), the pose blocks are three small products
// on the FP64 tensor path:
//     Wbar_A = ab Tbar, Wbar_B = bb Tbar   -> W_s[a][j] (a < 15, j < 6), final in the pose columns
//     Vbar   = Tbar^T Wbar_B               -> V_m += Vbar[0:6,0:6], g_m += Vbar[0:6,6]
// Rows 9..11 of W_s are then rotated from the camera's tangent frame with Jl_c (three shuffled rows).
__device__ __forceinline__ void flush_segment(NeAcc& S, int lane, int64_t seg, int c, int m,
                                              const double* __restrict__ camtab, const double* __restrict__ posetab,
                                              double* __restrict__ tbar, double* __restrict__ G, double* __restrict__ V,
                                              double* __restrict__ gp, double* __restrict__ W)
{
    if (lane < 9) {
        const double* Rc = camtab + (int64_t)c * CAM_STRIDE + CAM_R;
        const double* pm = posetab + (int64_t)m * POSE_STRIDE;
        const int i = lane / 3, j = lane - 3 * i;
        const int i1 = (i + 1) % 3, i2 = (i + 2) % 3;
        const double t0 = pm[POSE_T], t1 = pm[POSE_T + 1], t2 = pm[POSE_T + 2];
        const double j0 = pm[POSE_JL + j], j1 = pm[POSE_JL + 3 + j], j2 = pm[POSE_JL + 6 + j];
        const double s1 = Rc[3 * i1] * t0 + Rc[3 * i1 + 1] * t1 + Rc[3 * i1 + 2] * t2;
        const double s2 = Rc[3 * i2] * t0 + Rc[3 * i2 + 1] * t1 + Rc[3 * i2 + 2] * t2;
        const double q = Rc[3 * i] * j0 + Rc[3 * i + 1] * j1 + Rc[3 * i + 2] * j2;        // (R_c Jl_m)[i][j]
        const double q1 = Rc[3 * i1] * j0 + Rc[3 * i1 + 1] * j1 + Rc[3 * i1 + 2] * j2;
        const double q2 = Rc[3 * i2] * j0 + Rc[3 * i2 + 1] * j1 + Rc[3 * i2 + 2] * j2;
        tbar[(1 + i) * 8 + j] = q;
        tbar[(4 + i) * 8 + j] = s1 * q2 - s2 * q1;                                          // ([s]x R_c Jl_m)[i][j]
        tbar[(4 + i) * 8 + 3 + j] = Rc[3 * i + j];
    }
    {   // fold the segment into the running camera sums (three 8 x 8 tiles in shared memory, bank-conflict free)
        const int row = lane >> 2, cp = 2 * (lane & 3);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int e = cam_tile_pos(row, cp + i);
            G[e] += S.aa[i];
            G[64 + e] += S.ab[i];
            G[128 + e] += S.bb[i];
        }
    }
    __syncwarp();
    const double tb0 = tbar[(lane & 3) * 8 + (lane >> 2)], tb1 = tbar[(4 + (lane & 3)) * 8 + (lane >> 2)];
    double wa[2], wb[2];
    tile_times_tbar(S.ab, tb0, tb1, lane, wa);
    tile_times_tbar(S.bb, tb0, tb1, lane, wb);
    // Vbar = Tbar^T Wbar_B: the A fragment of Tbar^T is the same register as the B fragment of Tbar;
    // B fragment element (k = 4h + (lane & 3), n = lane >> 2) of Wbar_B sits in lane (k * 4 + n / 2), register n & 1
    double vb[2] = {0.0, 0.0};
    {
        const int n = lane >> 2;
        const bool odd = n & 1;
        const double b0 = shfl_pick(wb[0], wb[1], (lane & 3) * 4 + (n >> 1), odd);
        const double b1 = shfl_pick(wb[0], wb[1], (4 + (lane & 3)) * 4 + (n >> 1), odd);
        dmma884(vb[0], vb[1], tb0, b0);
        dmma884(vb[0], vb[1], tb1, b1);
    }
    const int row = lane >> 2, cp = 2 * (lane & 3);
    {   // rows 9..11 of W_s (rows 1..3 of Wbar_B) are in the camera's tangent frame: new row i = sum_i' Jl_c[i'][i] row i'
        const int q = lane & 3;
        const double x10 = __shfl_sync(0xffffffffu, wb[0], 4 + q), x11 = __shfl_sync(0xffffffffu, wb[1], 4 + q);
        const double x20 = __shfl_sync(0xffffffffu, wb[0], 8 + q), x21 = __shfl_sync(0xffffffffu, wb[1], 8 + q);
        const double x30 = __shfl_sync(0xffffffffu, wb[0], 12 + q), x31 = __shfl_sync(0xffffffffu, wb[1], 12 + q);
        if (row >= 1 && row <= 3) {
            const double* jl = camtab + (int64_t)c * CAM_STRIDE + CAM_JL + (row - 1);
            const double j0 = jl[0], j1 = jl[3], j2 = jl[6];
            wb[0] = x10 * j0 + x20 * j1 + x30 * j2;
            wb[1] = x11 * j0 + x21 * j1 + x31 * j2;
        }
    }
    if (cp < 6) {   // W_s[a][cp], W_s[a][cp + 1]: 16-byte stores
        double* Ws = W + seg * 90 + cp;
        *reinterpret_cast<double2*>(Ws + row * 6) = make_double2(wa[0], wa[1]);
        if (row < 7) *reinterpret_cast<double2*>(Ws + (8 + row) * 6) = make_double2(wb[0], wb[1]);
        if (row < 6) {
            atomicAdd(V + (int64_t)m * 36 + row * 6 + cp, vb[0]);
            atomicAdd(V + (int64_t)m * 36 + row * 6 + cp + 1, vb[1]);
        }
    } else if (row < 6) {
        atomicAdd(gp + (int64_t)m * 6 + row, vb[0]);   // column 6 of Vbar
    }
    acc_zero(S);
}

// Camera flush: the running camera sums (tangent parametrisation, shared memory) are mapped to the reference's
// rvec parametrisation, B = T^T B' T with T = diag(I9, Jl_c, I3, 1), and added to U_c (both triangles), g_c and r.r
// with FP64 reductions: every output entry is formed from at most 9 tile entries.  Runs once per (warp, camera).
__device__ __forceinline__ void flush_camera(int lane, int c, const double* __restrict__ camtab,
                                             double* __restrict__ G, double* __restrict__ U, double* __restrict__ gc,
                                             double* __restrict__ cost)
{
    const double* jl = camtab + (int64_t)c * CAM_STRIDE + CAM_JL;
    __syncwarp();
    double* Uc = U + (int64_t)c * 225;
    for (int e = lane; e < 256; e += 32) {
        const int a = e >> 4, b = e & 15;   // a, b = 15: the residual column
        const bool ra = a >= 9 && a < 12, rb = b >= 9 && b < 12;
        double v = 0.0;
        if (!ra && !rb) {
            v = cam_sum(G, a, b);
        } else if (ra && !rb) {
#pragma unroll
            for (int i = 0; i < 3; ++i) v += jl[3 * i + (a - 9)] * cam_sum(G, 9 + i, b);
        } else if (!ra && rb) {
#pragma unroll
            for (int i = 0; i < 3; ++i) v += cam_sum(G, a, 9 + i) * jl[3 * i + (b - 9)];
        } else {
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int k = 0; k < 3; ++k) v += jl[3 * i + (a - 9)] * cam_sum(G, 9 + i, 9 + k) * jl[3 * k + (b - 9)];
        }
        if (a < 15 && b < 15) atomicAdd(Uc + a * 15 + b, v);
        else if (a < 15) atomicAdd(gc + (int64_t)c * 15 + a, v);          // b == 15
        else if (b == 15) atomicAdd(cost, v);                              // a == b == 15
    }
    __syncwarp();
    for (int e = lane; e < 192; e += 32) G[e] = 0.0;   // the sums restart with the next camera
    __syncwarp();
}

// One k-step (2 observations = 4 staged rows) of the Gram update: fragment loads and the three DMMA.
__device__ __forceinline__ void gram_mma(NeAcc& S, double v0, double v1)
{
    dmma884(S.aa[0], S.aa[1], v0, v0);
    dmma884(S.ab[0], S.ab[1], v0, v1);
    dmma884(S.bb[0], S.bb[1], v1, v1);
}
__device__ __forceinline__ void gram_load(const double* __restrict__ f, double& v0, double& v1)
{
    v0 = f[0];
    v1 = f[NE_TILE_DOUBLES];
}

// Streamed observation loads: every observation is read exactly once per evaluation, so the loads bypass L1
// allocation and leave the (small) L1 that remains beside the staging buffers to the camera / pose / template rows.
__device__ __forceinline__ int ld_stream(const int32_t* p)
{
    int v;
    asm("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double2 ld_stream(const double2* p)
{
    double2 v;
    asm("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}

// One observation's inputs (sorted layout); c < 0 marks a lane past the end of the warp's range.
struct NeObs {
    int c, m, k;
    double2 uv;
};
__device__ __forceinline__ void load_obs(NeObs& o, int64_t i, int64_t end, const int32_t* __restrict__ s_cam,
                                         const int32_t* __restrict__ s_pose, const int32_t* __restrict__ s_key,
                                         const double2* __restrict__ s_uv)
{
    if (i < end) { o.c = ld_stream(s_cam + i); o.m = ld_stream(s_pose + i); o.k = ld_stream(s_key + i); o.uv = ld_stream(s_uv + i); }
    else { o.c = -1; o.m = -1; o.k = 0; o.uv = make_double2(0.0, 0.0); }
}

// Evaluated rows of one observation, as staged: tile 0 = [xD 1 0 0 Au0..3] / [0 0 yD 1 Av0..3],
// tile 1 = [Au4 Wc Pm r] per image row.
struct NeRows {
    double xD, yD, Au[5], Av[5], Pm[6], Wc[6], res[2];
};
__device__ __forceinline__ void eval_rows(const NeObs& o, const double* __restrict__ camtab, const double* __restrict__ posetab,
                                          const double* __restrict__ pts, NeRows& R)
{
    // lanes past the end evaluate row 0 of every table (never staged)
    const double* ct = camtab + (int64_t)max(o.c, 0) * CAM_STRIDE;
    const double* ptab = posetab + (int64_t)max(o.m, 0) * POSE_STRIDE;
    ObsJacCam J;
    eval_obs_cam(ct, ptab, pts + 4 * (int64_t)(o.c < 0 ? 0 : o.k), o.uv.x, o.uv.y, R.res, J);
    R.xD = J.xD; R.yD = J.yD;
#pragma unroll
    for (int i = 0; i < 5; ++i) { R.Au[i] = J.Au[i]; R.Av[i] = J.Av[i]; }
#pragma unroll
    for (int i = 0; i < 6; ++i) { R.Pm[i] = J.Pm[i]; R.Wc[i] = J.Wc[i]; }
}
// The first tile of a staged row pair is [xD 1 0 0 | Au0..3] / [0 0 yD 1 | Av0..3]: six of its sixteen entries are the
// constants 1 / 0.  Every lane always writes the same slot, so they are written once per kernel (stage_constants) and the
// per-observation staging is 12 sixteen-byte + 2 eight-byte stores instead of 16 sixteen-byte ones.
__device__ __forceinline__ void stage_constants(double* __restrict__ st_u, double* __restrict__ st_v, int st_rot)
{
    st_u[(0 ^ st_rot) + 1] = 1.0;
    *reinterpret_cast<double2*>(st_u + (2 ^ st_rot)) = make_double2(0.0, 0.0);
    *reinterpret_cast<double2*>(st_v + (0 ^ st_rot)) = make_double2(0.0, 0.0);
    st_v[(2 ^ st_rot) + 1] = 1.0;
}
__device__ __forceinline__ void stage_rows(const NeRows& R, double* __restrict__ st_u, double* __restrict__ st_v, int st_rot)
{
    st_u[0 ^ st_rot] = R.xD;
    st_v[2 ^ st_rot] = R.yD;
    *reinterpret_cast<double2*>(st_u + (4 ^ st_rot)) = make_double2(R.Au[0], R.Au[1]);
    *reinterpret_cast<double2*>(st_u + (6 ^ st_rot)) = make_double2(R.Au[2], R.Au[3]);
    *reinterpret_cast<double2*>(st_v + (4 ^ st_rot)) = make_double2(R.Av[0], R.Av[1]);
    *reinterpret_cast<double2*>(st_v + (6 ^ st_rot)) = make_double2(R.Av[2], R.Av[3]);
    {
        const double t1[8] = {R.Au[4], R.Wc[0], R.Wc[1], R.Wc[2], R.Pm[0], R.Pm[1], R.Pm[2], R.res[0]};
#pragma unroll
        for (int c = 0; c < 8; c += 2) *reinterpret_cast<double2*>(st_u + NE_TILE_DOUBLES + (c ^ st_rot)) = make_double2(t1[c], t1[c + 1]);
    }
    {
        const double t1[8] = {R.Av[4], R.Wc[3], R.Wc[4], R.Wc[5], R.Pm[3], R.Pm[4], R.Pm[5], R.res[1]};
#pragma unroll
        for (int c = 0; c < 8; c += 2) *reinterpret_cast<double2*>(st_v + NE_TILE_DOUBLES + (c ^ st_rot)) = make_double2(t1[c], t1[c + 1]);
    }
}

// (A variant with two observations per lane and loop trip -- two independent evaluation chains -- was measured at 0.177 ms
// against 0.135 ms: the second observation's rows spill.  Removed.)
template <int CTAS_PER_SM, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, CTAS_PER_SM)
k_normal(int n_warps, const int64_t* __restrict__ warp_seg, const int32_t* __restrict__ s_cam, const int32_t* __restrict__ s_pose,
         const int32_t* __restrict__ s_key, const double2* __restrict__ s_uv, const int64_t* __restrict__ seg_start,
         const double* __restrict__ camtab, const double* __restrict__ posetab, const double* __restrict__ pts,
         double* __restrict__ U, double* __restrict__ gc, double* __restrict__ cost, double* __restrict__ V,
         double* __restrict__ gp, double* __restrict__ W)
{
    extern __shared__ __align__(16) double ne_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* ws = ne_smem + warp * NE_WARP_DOUBLES;
    const int wg = blockIdx.x * WARPS + warp;
    pdl_launch_dependents();   // the exchange kernel of a pose-sharded evaluation may queue up behind this grid
    pdl_wait();                // tables, cleared targets (k_prepare_tables) and the warp ranges are complete from here on
    if (wg >= n_warps) return;

    // this warp's range of whole segments (k_warp_ranges)
    const int64_t sb = warp_seg[wg], se = warp_seg[wg + 1];
    if (sb >= se) return;
    const int64_t begin = seg_start[sb], end = seg_start[se];

    NeAcc S;   // the segment's accumulators; the camera's running sums live in shared memory
    acc_zero(S);
    double* const scratch = ws + 2 * NE_TILE_DOUBLES;   // Tbar: constant entries are written once
    scratch[lane] = 0.0;
    scratch[32 + lane] = lane == 30 ? 1.0 : 0.0;       // Tbar[7][6] = 1
    for (int e = lane; e < 192; e += 32) scratch[64 + e] = 0.0;
    int64_t cur_seg = sb - 1;   // segments are visited in order: a piece head advances this counter
    int cur_c = -1, cur_m = -1;
    int last_c = -1, last_m = -1;  // (camera, pose) of the last observation of the previous batch

    // lane constants of the staging layout
    double* const st_u = ws + stage_row(lane, 0);
    double* const st_v = ws + stage_row(lane, 1);
    const int st_rot = stage_rot(lane);
    stage_constants(st_u, st_v, st_rot);   // the 1 / 0 entries of the first tile never change: written once
    __syncwarp();
    const int g8 = lane >> 2, jb = (lane >> 1) & 1, jr = lane & 1;
    const int ld_L = 16 * jb + 8 * jr + (g8 ^ (4 * jb));
    // fragment address of k-step ks: ws + 32 ks + (ld_L ^ X(ks)), X(ks) = 8 bit0(ks) + 2 bit1(ks): four lane constants,
    // the rest of the address is a compile-time offset of the unrolled step
    const double* const fb0 = ws + ld_L;
    const double* const fb1 = ws + (ld_L ^ 8);
    const double* const fb2 = ws + (ld_L ^ 2);
    const double* const fb3 = ws + (ld_L ^ 10);

    // software prefetch: the inputs of the next trip are requested before the current trip is evaluated
    NeObs nxt;
    load_obs(nxt, begin + lane, end, s_cam, s_pose, s_key, s_uv);

    for (int64_t base = begin; base < end; base += 32) {
        const NeObs ob = nxt;
        NeRows rows;
        eval_rows(ob, camtab, posetab, pts, rows);
        // the next trip's stream loads are issued only now.  Issued at the top of the trip they shared a scoreboard with
        // this trip's table-row loads, so the first use of a row waited for the whole DRAM latency of the prefetch (17 % of
        // the warp samples sat on two such instructions); the Gram phase below is long enough to cover them: 131.1 -> 127.0
        // us at config 4 (a two-deep variant spills and gains nothing, nor does pulling the next trip's pose rows into L1
        // from pose indices loaded one trip further ahead).
        load_obs(nxt, base + 32 + lane, end, s_cam, s_pose, s_key, s_uv);
        const int cnt = (int)min((int64_t)32, end - base);
        const int c = ob.c, m = ob.m;
        // every lane stages its rows, also the lanes past the end of the range (they evaluated row 0 of every table: finite
        // values, masked out of the Gram steps below): without a predicate the stores are free to move up into the evaluation
        stage_rows(rows, st_u, st_v, st_rot);
        // piece heads: lanes whose (camera, pose) differs from the previous observation's
        int pc = __shfl_up_sync(0xffffffffu, c, 1), pm = __shfl_up_sync(0xffffffffu, m, 1);
        if (lane == 0) { pc = last_c; pm = last_m; }
        const unsigned heads = __ballot_sync(0xffffffffu, lane < cnt && (c != pc || m != pm));
        last_c = __shfl_sync(0xffffffffu, c, cnt - 1);
        last_m = __shfl_sync(0xffffffffu, m, cnt - 1);
        __syncwarp();
        unsigned pieces = heads | 1u;  // a batch may start in the middle of a segment
        while (pieces) {
            const int a = __ffs(pieces) - 1;
            pieces &= pieces - 1;
            const int b = pieces ? __ffs(pieces) - 1 : cnt;
            if ((heads >> a) & 1u) {
                if (cur_c >= 0) flush_segment(S, lane, cur_seg, cur_c, cur_m, camtab, posetab, scratch, scratch + 64, V, gp, W);
                const int nc = __shfl_sync(0xffffffffu, c, a);
                if (nc != cur_c && cur_c >= 0) flush_camera(lane, cur_c, camtab, scratch + 64, U, gc, cost);
                ++cur_seg; cur_c = nc; cur_m = __shfl_sync(0xffffffffu, m, a);
            }
            // k-steps (2 observations each) of the piece [a, b), fully unrolled: every fragment address is a lane constant
            // plus a compile-time offset.
            if (a == 0 && b == 32) {
                // the whole batch belongs to one segment (the common case): 16 unmasked steps, loads of four steps hoisted
#pragma unroll
                for (int k4 = 0; k4 < 16; k4 += 4) {
                    double v0[4], v1[4];
                    gram_load(fb0 + 32 * k4, v0[0], v1[0]);
                    gram_load(fb1 + 32 * (k4 + 1), v0[1], v1[1]);
                    gram_load(fb2 + 32 * (k4 + 2), v0[2], v1[2]);
                    gram_load(fb3 + 32 * (k4 + 3), v0[3], v1[3]);
#pragma unroll
                    for (int u = 0; u < 4; ++u) gram_mma(S, v0[u], v1[u]);
                }
            } else {
                // general piece: steps outside [a, b) are skipped (warp-uniform), steps shared with a neighbouring piece or
                // reaching past the end of the batch are masked per observation
#pragma unroll
                for (int ks = 0; ks < 16; ++ks) {
                    if (2 * ks + 2 <= a || 2 * ks >= b) continue;
                    const double* f = ((ks & 3) == 0 ? fb0 : (ks & 3) == 1 ? fb1 : (ks & 3) == 2 ? fb2 : fb3) + 32 * ks;
                    double v0, v1;
                    gram_load(f, v0, v1);
                    if (2 * ks < a || 2 * ks + 2 > b) {
                        const int o = 2 * ks + jb;
                        const bool ok = o >= a && o < b;
                        v0 = ok ? v0 : 0.0;
                        v1 = ok ? v1 : 0.0;
                    }
                    gram_mma(S, v0, v1);
                }
            }
        }
        __syncwarp();
    }
    if (cur_c >= 0) {
        flush_segment(S, lane, cur_seg, cur_c, cur_m, camtab, posetab, scratch, scratch + 64, V, gp, W);
        flush_camera(lane, cur_c, camtab, scratch + 64, U, gc, cost);
    }
}

// ================================================================================================================
// K_ne, mixed precision (opt-in, pcs_set_normal_precision): same mapping, same flushes, same outputs -- but the 16 x 16
// Gram update leaves the FP64 pipe.
//
// Measured on B200 (tools/mma_peak.cu, profiles/r2_mma_peak_b200.json): DFMA, DMMA and the legacy tensor path (HMMA) all
// issue through ONE pipe per sub-partition -- a DFMA costs 2.2 clocks, a DMMA m8n8k4 16, an HMMA (any shape / type) 8.6,
// and a DFMA + HMMA mix takes the SUM of the two.  The FP64 kernel spends 768 of ~1100 pipe clocks per batch of 32
// observations in its 48 DMMAs.  Here:
//   * residual, Jacobian rows, cost and the gradient g = J^T r stay FP64: every lane forms its 16 products
//     [J_u[a] r_u + J_v[a] r_v | r.r] in registers, parks them in an (swizzled) shared-memory table, and lane (a, half)
//     sums column a over the rows of the current piece -- 16 LDS + 16 DADD per lane and batch however the batch is cut
//     into pieces.  The fixed point of the LM iteration is defined by g = 0, so it is unchanged to FP64 accuracy.
//   * J^T J only preconditions the step.  Each Jacobian entry is split into two BF16 terms, x ~ hi + lo (16 mantissa bits,
//     truncation, relative error <= 2^-15), packed as (u-row, v-row) pairs -- exactly the k-pair a m16n8k16 fragment
//     register holds -- and the Gram is the full product (hi + lo)^T (hi + lo): 8 HMMA.16816.F32.BF16 per 8
//     observations, FP32 accumulators per SEGMENT (~40 observations), promoted to FP64 at the segment flush and summed
//     in FP64 across segments.  All four terms are kept: the result is then the exact Gram matrix of a Jacobian whose
//     entries are within 2^-15 of the true ones (a CONSISTENT perturbation, which Levenberg-Marquardt does not notice),
//     up to FP32 accumulation.  Measured effect on the solver: tests/test_gpu_mixed_precision.py (same iterates' cost to 1e-6, same
//     converged cost to 1e-9, iterations within 10 %).
//   * A-fragment and B-fragment of a column tile are the same registers (as in the FP64 kernel): per k-step a lane loads
//     4 x 8 bytes (hi / lo words of its two observations, columns g and g + 8 adjacent in the staged row).
// ================================================================================================================
constexpr int NEM_STAGE_DOUBLES = 512;   // 32 observations x 128 B: 16 hi words | 16 lo words (bf16 pairs (u, v))
constexpr int NEM_GSTRIDE = 18;          // row stride of the gradient-product table: 16-byte stores of 8 consecutive lanes and the
                                         // 8-byte column reads of a half warp are both bank-conflict free without any swizzle
constexpr int NEM_GBUF_DOUBLES = 32 * NEM_GSTRIDE;   // 32 x 16 FP64 gradient products (padded rows)
constexpr int NEM_WARP_DOUBLES = NEM_STAGE_DOUBLES + NEM_GBUF_DOUBLES + NE_SCRATCH_DOUBLES;

__device__ __forceinline__ void hmma_bf16(float d[4], unsigned a0, unsigned a1, unsigned a2, unsigned a3, unsigned b0, unsigned b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// Staged observation block (32 words): chunk c (4 words) sits at chunk c ^ swz(o); chunks 0..3 = hi words, 4..7 = lo
// words; inside the 16 words of a half, column col sits at 2 (col & 7) + (col >> 3): columns g and g + 8 are adjacent.
// swz is a bijection of o & 7 (conflict-free 16-byte stores of 8 consecutive lanes) whose bits 1, 2 are o & 3
// (conflict-free 8-byte fragment loads of a half warp: 4 observations x 4 column pairs).
__device__ __forceinline__ int nem_swz(int o) { return ((o & 3) << 1) | ((o >> 2) & 1); }

// split two FP64 values (the u-row and v-row entries of one column) into packed bf16 pairs: hi = truncated, lo = remainder
__device__ __forceinline__ void bf16_split_pair(double xu, double xv, unsigned& hi, unsigned& lo)
{
    const float fu = (float)xu, fv = (float)xv;
    const unsigned bu = __float_as_uint(fu), bv = __float_as_uint(fv);
    hi = __byte_perm(bu, bv, 0x7632);                                  // (bu >> 16) | (bv & 0xffff0000)
    const float lu = fu - __uint_as_float(bu & 0xffff0000u), lv = fv - __uint_as_float(bv & 0xffff0000u);   // exact
    lo = __byte_perm(__float_as_uint(lu), __float_as_uint(lv), 0x7632);
}

// Stage the two rows of one observation.  Column -> physical position pc = 2 (col & 7) + (col >> 3); chunk c holds
// positions 4c .. 4c + 3, i.e. columns (2c, 2c + 8, 2c + 1, 2c + 9):
//   c = 0: (xD | 0), (Au4 | Av4), (1 | 0), Wc0      c = 1: (0 | yD), Wc1, (0 | 1), Wc2
//   c = 2: Au0/Av0, Pm0, Au1/Av1, Pm1                c = 3: Au2/Av2, Pm2, Au3/Av3, 0
// Each chunk is split and stored as soon as it is formed (two 16-byte stores: hi words, lo words).
__device__ __forceinline__ void stage_chunk(unsigned* __restrict__ blk, int swz, int c, const unsigned hi[4], const unsigned lo[4])
{
    *reinterpret_cast<uint4*>(blk + ((c ^ swz) << 2)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(blk + (((4 + c) ^ swz) << 2)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

__device__ __forceinline__ void stage_rows_bf16(const NeRows& R, unsigned* __restrict__ blk, int swz)
{
    unsigned hi[4], lo[4];
    bf16_split_pair(R.xD, 0.0, hi[0], lo[0]);
    bf16_split_pair(R.Au[4], R.Av[4], hi[1], lo[1]);
    hi[2] = 0x00003f80u; lo[2] = 0u;                                   // (1 | 0)
    bf16_split_pair(R.Wc[0], R.Wc[3], hi[3], lo[3]);
    stage_chunk(blk, swz, 0, hi, lo);
    bf16_split_pair(0.0, R.yD, hi[0], lo[0]);
    bf16_split_pair(R.Wc[1], R.Wc[4], hi[1], lo[1]);
    hi[2] = 0x3f800000u; lo[2] = 0u;                                   // (0 | 1)
    bf16_split_pair(R.Wc[2], R.Wc[5], hi[3], lo[3]);
    stage_chunk(blk, swz, 1, hi, lo);
    bf16_split_pair(R.Au[0], R.Av[0], hi[0], lo[0]);
    bf16_split_pair(R.Pm[0], R.Pm[3], hi[1], lo[1]);
    bf16_split_pair(R.Au[1], R.Av[1], hi[2], lo[2]);
    bf16_split_pair(R.Pm[1], R.Pm[4], hi[3], lo[3]);
    stage_chunk(blk, swz, 2, hi, lo);
    bf16_split_pair(R.Au[2], R.Av[2], hi[0], lo[0]);
    bf16_split_pair(R.Pm[2], R.Pm[5], hi[1], lo[1]);
    bf16_split_pair(R.Au[3], R.Av[3], hi[2], lo[2]);
    hi[3] = 0u; lo[3] = 0u;                                            // column 15 (the residual column of the FP64 kernel): g is formed in FP64
    stage_chunk(blk, swz, 3, hi, lo);
}

// the lane's 16 FP64 gradient products [J_u[a] r_u + J_v[a] r_v (a = 0..14) | r.r], parked in its row of the table
// (pairs are stored as they are formed, at compile-time offsets)
__device__ __forceinline__ void store_grad_products(const NeRows& R, double* __restrict__ grow)
{
    const double ru = R.res[0], rv = R.res[1];
    double2* g2 = reinterpret_cast<double2*>(grow);
    g2[0] = make_double2(R.xD * ru, ru);
    g2[1] = make_double2(R.yD * rv, rv);
    g2[2] = make_double2(fma(R.Au[0], ru, R.Av[0] * rv), fma(R.Au[1], ru, R.Av[1] * rv));
    g2[3] = make_double2(fma(R.Au[2], ru, R.Av[2] * rv), fma(R.Au[3], ru, R.Av[3] * rv));
    g2[4] = make_double2(fma(R.Au[4], ru, R.Av[4] * rv), fma(R.Wc[0], ru, R.Wc[3] * rv));
    g2[5] = make_double2(fma(R.Wc[1], ru, R.Wc[4] * rv), fma(R.Wc[2], ru, R.Wc[5] * rv));
    g2[6] = make_double2(fma(R.Pm[0], ru, R.Pm[3] * rv), fma(R.Pm[1], ru, R.Pm[4] * rv));
    g2[7] = make_double2(fma(R.Pm[2], ru, R.Pm[5] * rv), fma(ru, ru, rv * rv));
}

template <int CTAS_PER_SM, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, CTAS_PER_SM)
k_normal_mixed(int n_warps, const int64_t* __restrict__ warp_seg, const int32_t* __restrict__ s_cam, const int32_t* __restrict__ s_pose,
               const int32_t* __restrict__ s_key, const double2* __restrict__ s_uv, const int64_t* __restrict__ seg_start,
               const double* __restrict__ camtab, const double* __restrict__ posetab, const double* __restrict__ pts,
               double* __restrict__ U, double* __restrict__ gc, double* __restrict__ cost, double* __restrict__ V,
               double* __restrict__ gp, double* __restrict__ W)
{
    extern __shared__ __align__(16) double ne_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* ws = ne_smem + warp * NEM_WARP_DOUBLES;
    const int wg = blockIdx.x * WARPS + warp;
    pdl_launch_dependents();
    pdl_wait();
    if (wg >= n_warps) return;
    const int64_t sb = warp_seg[wg], se = warp_seg[wg + 1];
    if (sb >= se) return;
    const int64_t begin = seg_start[sb], end = seg_start[se];

    unsigned* const stage = reinterpret_cast<unsigned*>(ws);
    double* const gbuf = ws + NEM_STAGE_DOUBLES;
    double* const scratch = gbuf + NEM_GBUF_DOUBLES;     // Tbar | running camera sums, as in the FP64 kernel
    scratch[lane] = 0.0;
    scratch[32 + lane] = lane == 30 ? 1.0 : 0.0;       // Tbar[7][6] = 1
    for (int e = lane; e < 192; e += 32) scratch[64 + e] = 0.0;
    __syncwarp();

    float D0[4] = {0.f, 0.f, 0.f, 0.f}, D1[4] = {0.f, 0.f, 0.f, 0.f};   // segment Gram: columns 0..7 / 8..15 (FP32)
    double gacc = 0.0;                                                   // lane (a = lane & 15, half = lane >> 4): partial g_s[a]
    int64_t cur_seg = sb - 1;
    int cur_c = -1, cur_m = -1, last_c = -1, last_m = -1;

    const int g8 = lane >> 2, t4 = lane & 3;
    unsigned* const my_blk = stage + lane * 32;
    const int my_swz = nem_swz(lane);
    const int ga = lane & 15, gh = lane >> 4;
    const double* const my_gcol = gbuf + 16 * gh * NEM_GSTRIDE + ga;   // column ga of this lane's half of the table
    // fragment words of k-step 0 (hi / lo words of observations t4 and t4 + 4, columns g8 and g8 + 8); step ks adds 256 ks words
    const int f_ch = g8 >> 1, f_wi = (g8 & 1) << 1, f_s0 = nem_swz(t4), f_s1 = nem_swz(t4 + 4);
    const unsigned* const frag_h0 = stage + t4 * 32 + (((f_ch ^ f_s0) << 2) | f_wi);
    const unsigned* const frag_l0 = stage + t4 * 32 + ((((4 + f_ch) ^ f_s0) << 2) | f_wi);
    const unsigned* const frag_h1 = stage + (t4 + 4) * 32 + (((f_ch ^ f_s1) << 2) | f_wi);
    const unsigned* const frag_l1 = stage + (t4 + 4) * 32 + ((((4 + f_ch) ^ f_s1) << 2) | f_wi);

    auto flush = [&]() {
        // FP32 segment sums -> FP64 fragments of the FP64 kernel's flush (aa = G[0:8,0:8], ab = G[0:8,8:16], bb = G[8:16,8:16]);
        // column 15 (the gradient / cost column) comes from the FP64 sums
        NeAcc S;
        S.aa[0] = D0[0]; S.aa[1] = D0[1]; S.ab[0] = D1[0]; S.ab[1] = D1[1]; S.bb[0] = D1[2]; S.bb[1] = D1[3];
        const double tot = gacc + __shfl_xor_sync(0xffffffffu, gacc, 16);      // lanes a and a + 16: g_s[a]
        const double ga_lo = __shfl_sync(0xffffffffu, tot, g8), ga_hi = __shfl_sync(0xffffffffu, tot, 8 + g8);
        if (t4 == 3) { S.ab[1] = ga_lo; S.bb[1] = ga_hi; }
        flush_segment(S, lane, cur_seg, cur_c, cur_m, camtab, posetab, scratch, scratch + 64, V, gp, W);
#pragma unroll
        for (int i = 0; i < 4; ++i) { D0[i] = 0.f; D1[i] = 0.f; }
        gacc = 0.0;
    };

    NeObs nxt;
    load_obs(nxt, begin + lane, end, s_cam, s_pose, s_key, s_uv);
    for (int64_t base = begin; base < end; base += 32) {
        const NeObs ob = nxt;
        NeRows R;
        eval_rows(ob, camtab, posetab, pts, R);
        load_obs(nxt, base + 32 + lane, end, s_cam, s_pose, s_key, s_uv);   // issued after the evaluation, as in k_normal
        const int cnt = (int)min((int64_t)32, end - base);
        const int c = ob.c, m = ob.m;
        if (lane < cnt) {
            stage_rows_bf16(R, my_blk, my_swz);
            store_grad_products(R, gbuf + lane * NEM_GSTRIDE);
        }
        int pc = __shfl_up_sync(0xffffffffu, c, 1), pm = __shfl_up_sync(0xffffffffu, m, 1);
        if (lane == 0) { pc = last_c; pm = last_m; }
        const unsigned heads = __ballot_sync(0xffffffffu, lane < cnt && (c != pc || m != pm));
        last_c = __shfl_sync(0xffffffffu, c, cnt - 1);
        last_m = __shfl_sync(0xffffffffu, m, cnt - 1);
        __syncwarp();
        unsigned pieces = heads | 1u;
        while (pieces) {
            const int a = __ffs(pieces) - 1;
            pieces &= pieces - 1;
            const int b = pieces ? __ffs(pieces) - 1 : cnt;
            if ((heads >> a) & 1u) {
                if (cur_c >= 0) flush();
                const int nc = __shfl_sync(0xffffffffu, c, a);
                if (nc != cur_c && cur_c >= 0) flush_camera(lane, cur_c, camtab, scratch + 64, U, gc, cost);
                ++cur_seg; cur_c = nc; cur_m = __shfl_sync(0xffffffffu, m, a);
            }
            // gradient column sums of the piece: lane (ga, gh) adds the rows of its half that lie in [a, b) -- in quarters of
            // four predicated loads issued back to back (four partial sums, compile-time offsets), so that the latency of a
            // piece is a few shared-memory round trips instead of one per row
            {
                double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
                for (int q = 0; q < 16; q += 4) {
                    const int lo = 16 * gh + q;
                    if (lo + 4 > a && lo < b) {
                        const double* gq = my_gcol + q * NEM_GSTRIDE;
                        s0 += (lo >= a && lo < b) ? gq[0] : 0.0;
                        s1 += (lo + 1 >= a && lo + 1 < b) ? gq[NEM_GSTRIDE] : 0.0;
                        s2 += (lo + 2 >= a && lo + 2 < b) ? gq[2 * NEM_GSTRIDE] : 0.0;
                        s3 += (lo + 3 >= a && lo + 3 < b) ? gq[3 * NEM_GSTRIDE] : 0.0;
                    }
                }
                gacc += (s0 + s1) + (s2 + s3);
            }
            // Gram k-steps (8 observations each) of the piece, unrolled: the fragment addresses of a step are the lane's four
            // constants plus a compile-time offset.  Steps outside the piece are skipped (warp-uniform), steps shared with a
            // neighbouring piece are masked.
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                if (8 * ks + 8 <= a || 8 * ks >= b) continue;
                uint2 h0 = *reinterpret_cast<const uint2*>(frag_h0 + ks * 256);
                uint2 l0 = *reinterpret_cast<const uint2*>(frag_l0 + ks * 256);
                uint2 h1 = *reinterpret_cast<const uint2*>(frag_h1 + ks * 256);
                uint2 l1 = *reinterpret_cast<const uint2*>(frag_l1 + ks * 256);
                if (8 * ks < a || 8 * ks + 8 > b) {
                    const int o0 = 8 * ks + t4, o1 = o0 + 4;
                    if (o0 < a || o0 >= b) { h0 = make_uint2(0u, 0u); l0 = make_uint2(0u, 0u); }
                    if (o1 < a || o1 >= b) { h1 = make_uint2(0u, 0u); l1 = make_uint2(0u, 0u); }
                }
                // A = J'^T (columns g, g + 8 x 16 staged rows): a0 = (col g, obs o0), a1 = (col g + 8, obs o0), a2 / a3: obs o1;
                // B of column tile h = the same registers: (a0, a2) for columns 0..7, (a1, a3) for columns 8..15
                hmma_bf16(D0, h0.x, h0.y, h1.x, h1.y, h0.x, h1.x);
                hmma_bf16(D1, h0.x, h0.y, h1.x, h1.y, h0.y, h1.y);
                hmma_bf16(D0, h0.x, h0.y, h1.x, h1.y, l0.x, l1.x);
                hmma_bf16(D1, h0.x, h0.y, h1.x, h1.y, l0.y, l1.y);
                hmma_bf16(D0, l0.x, l0.y, l1.x, l1.y, h0.x, h1.x);
                hmma_bf16(D1, l0.x, l0.y, l1.x, l1.y, h0.y, h1.y);
                // lo^T lo: 2^-16 of the result, but without it the sum is (H + L)^T (H + L) MINUS a positive semi-definite
                // matrix -- no longer the Gram matrix of any Jacobian -- and the Schur complement of the LM step, which lives
                // on cancellation between U, W and V, degrades: 66 instead of 17 iterations on the ring5 golden (measured)
                hmma_bf16(D0, l0.x, l0.y, l1.x, l1.y, l0.x, l1.x);
                hmma_bf16(D1, l0.x, l0.y, l1.x, l1.y, l0.y, l1.y);
            }
        }
        __syncwarp();
    }
    if (cur_c >= 0) {
        flush();
        flush_camera(lane, cur_c, camtab, scratch + 64, U, gc, cost);
    }
}

// Segment range of every warp of every part.  The observation range is cut into `n_parts` equal parts and each part
// into `n_warps` equal pieces; piece boundaries are moved to segment starts:
//     warp_seg[part * (n_warps + 1) + w] = lower_bound(seg_start, N part / n_parts + (N / n_parts) w / n_warps).
// Depends only on the static problem structure; evaluated once per (problem, n_warps, n_parts).
__global__ void k_warp_ranges(int64_t N, int64_t n_seg, int n_warps, int n_parts, const int64_t* __restrict__ seg_start,
                              int64_t* __restrict__ warp_seg)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= (int64_t)n_parts * (n_warps + 1)) return;
    const int part = (int)(t / (n_warps + 1)), w = (int)(t % (n_warps + 1));
    const int64_t lo_obs = N * part / n_parts, hi_obs = N * (part + 1) / n_parts;
    const int64_t target = lo_obs + (hi_obs - lo_obs) * w / n_warps;
    int64_t lo = 0, hi = n_seg;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (seg_start[mid] < target) lo = mid + 1; else hi = mid; }
    warp_seg[t] = lo;
}

static int ensure_ranges(pcs_problem* p, int64_t n_ranges, int n_parts)
{
    const int slot = n_parts > 1 ? 1 : 0;
    if (p->ne_warps[slot] == n_ranges && p->ne_parts[slot] == n_parts) return PCS_OK;
    if (p->warp_seg[slot]) cudaFree(p->warp_seg[slot]);
    p->warp_seg[slot] = nullptr;
    p->ne_warps[slot] = 0;
    const int64_t total = (int64_t)n_parts * (n_ranges + 1);
    PCS_CUDA(cudaMalloc((void**)&p->warp_seg[slot], (size_t)total * sizeof(int64_t)));
    k_warp_ranges<<<(int)((total + 127) / 128), 128, 0, p->stream>>>(p->N, p->n_seg, (int)n_ranges, n_parts, p->seg_start,
                                                                     p->warp_seg[slot]);
    PCS_CUDA(cudaGetLastError());
    if (slot == 0) {
        p->ne_warps[0] = n_ranges;
        p->ne_parts[0] = 1;
        return PCS_OK;
    }
    // segment boundaries of the parts, for the host-side pipelining of the W copy-out
    p->h_part_bounds.assign(n_parts + 1, 0);
    for (int k = 0; k < n_parts; ++k)
        PCS_CUDA(cudaMemcpyAsync(&p->h_part_bounds[k], p->warp_seg[1] + (int64_t)k * (n_ranges + 1), sizeof(int64_t),
                                 cudaMemcpyDeviceToHost, p->stream));
    PCS_CUDA(cudaStreamSynchronize(p->stream));
    p->h_part_bounds[n_parts] = p->n_seg;
    p->ne_warps[1] = n_ranges;
    p->ne_parts[1] = n_parts;
    return PCS_OK;
}

// part / n_parts: evaluate only the observations of one part (host path: the copy-out of a part's W segments overlaps
// the evaluation of the next part); n_parts = 1 evaluates everything in one launch.
int launch_normal_blocks(pcs_problem* p, bool targets_cleared, int part, int n_parts)
{
    // zero what is accumulated with reductions: [U | gc | cost | pad | V | gp]; W is fully overwritten
    if (!targets_cleared && part == 0) {
        const int64_t zero_doubles = ne_zero_doubles(p);
        PCS_CUDA(cudaMemsetAsync(p->ne, 0, (size_t)zero_doubles * sizeof(double), p->stream));
    }
    if (p->N == 0) return PCS_OK;
    // FP64 (default): 5 CTAs x 4 warps per SM, 96 registers.  Mixed (pcs_set_normal_precision): BF16-split Gram on HMMA.
    const bool mixed = p->normal_precision == PCS_PRECISION_MIXED;
    // mixed kernel: 4 CTAs per SM (128 registers, no spills; at 5 CTAs it has 96 registers and 80 B of spills)
    const int ctas = mixed ? 4 : 5, warps = 4;
    const size_t smem = (size_t)warps * (mixed ? NEM_WARP_DOUBLES : NE_WARP_DOUBLES) * sizeof(double);
    if (mixed) PCS_CUDA(ensure_dynamic_smem(k_normal_mixed<4, 4>, smem));
    else PCS_CUDA(ensure_dynamic_smem(k_normal<5, 4>, smem));
    // persistent-style grid: `ctas` CTAs of `warps` warps per SM; at least ~64 observations per warp
    const int64_t n_part_obs = p->N / n_parts + 1;
    int64_t n_warps = std::min<int64_t>((n_part_obs + 63) / 64, (int64_t)p->sm_count * ctas * warps);
    n_warps = std::max<int64_t>(1, std::min<int64_t>(n_warps, p->n_seg));
    PCS_TRY(ensure_ranges(p, n_warps, n_parts));
    const int grid = (int)((n_warps + warps - 1) / warps);
    const int tslot = (int)(p->timing_count % (int64_t)std::max<size_t>(p->ev_a.size(), 1));
    if (p->timing) PCS_CUDA(cudaEventRecord(p->ev_a[tslot], p->stream));
    const int64_t* ranges = p->warp_seg[n_parts > 1 ? 1 : 0] + (int64_t)part * (n_warps + 1);
    // programmatic dependent launch: the grid becomes resident while k_prepare_tables drains (pdl_wait inside the kernel)
    PCS_CUDA(launch_pdl(mixed ? k_normal_mixed<4, 4> : k_normal<5, 4>, dim3(grid), dim3(warps * 32), smem, p->stream, (int)n_warps, ranges,
                        (const int32_t*)p->s_cam, (const int32_t*)p->s_pose, (const int32_t*)p->s_key, (const double2*)p->s_uv,
                        (const int64_t*)p->seg_start, (const double*)p->camtab, (const double*)p->posetab, (const double*)p->tmpl4,
                        p->U, p->gc, p->cost, p->V, p->gp, p->W));
    PCS_CUDA(cudaGetLastError());
    ++p->n_launches;
    if (p->timing) {
        PCS_CUDA(cudaEventRecord(p->ev_b[tslot], p->stream));
        ++p->timing_count;
    }
    return PCS_OK;
}

}  // namespace pcs
