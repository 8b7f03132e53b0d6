// pcs_math.cuh -- per-observation device math for the bundle-adjustment chain (FP64).
//
// Mirrors the reference blocks (paths relative to the pyCamSet repository):
//   projection        function_block_implementations.py:21-140  (pinhole + Brown-Conrady, params
//                     [fx, px, fy, py, k1, k2, p1, p2, k3])
//   rigidTform3d / extrinsic3D / template_points   :143-211      (X' = R(rvec) X + t)
//   numba_flat_rodrigues_INPLACE / numba_rodrigues_jac  compiled_helpers.py:197-286
//   chain product (matflow)  matmul_map.py:147-243:  J = [A | Pm [D_c | I] | Pm R_c [D_m | I] (| Pm R_c R_m)]
//
// Not a translation:
//   * rotations are hoisted out of the per-observation path into per-camera / per-pose tables (the reference
//     recomputes sin/cos for every observation);
//   * the rotation derivative uses the SO(3) left Jacobian instead of the 27-entry dR/dr table:
//         d(R(r) X)/dr = -[R X]x Jl(r),      Jl = I + (1 - cos t)/t^2 [r]x + (t - sin t)/t^3 [r]x^2
//     which is the same analytic derivative as the OpenCV formula the reference evaluates
//     (compiled_helpers.py:237-286), needs 9 table entries instead of 27 and turns L * D(X) into
//     (R X  x  L_row)^T Jl.  The normal-equation kernel goes one step further and accumulates J^T J in the
//     tangent parametrisation (rows (R X x L_row)^T), applying Jl once per block afterwards;
//   * the projection Jacobian is evaluated in normalised coordinates instead of the reference's
//     z**7 / z**8 polynomial form (same function, better conditioned).
#pragma once
#include <cuda_runtime.h>

namespace pcs {

// Per-camera table row: [q(9) | R(9) | t(3) | Jl(9) | pad(2)] = 32 doubles.
constexpr int CAM_Q = 0, CAM_R = 9, CAM_T = 18, CAM_JL = 21, CAM_STRIDE = 32;
// Per-pose table row: [R(9) | t(3) | Jl(9) | pad(3)] = 24 doubles.
constexpr int POSE_R = 0, POSE_T = 9, POSE_JL = 12, POSE_STRIDE = 24;
// Per-segment (camera, pose) row of the residual kernel: [R_c R_m (9) | R_c t_m + t_c (3) | intrinsics q (9) | pad] = 22 doubles:
// everything an observation of the segment needs sits in ONE row (one dependent load level after the segment id).
constexpr int SEG_R = 0, SEG_T = 9, SEG_Q = 12, SEG_STRIDE = 22;

__device__ __forceinline__ void rodrigues(const double r[3], double R[9])
{
    const double th2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2];
    const double theta = sqrt(th2);
    if (theta < 1e-10) {  // compiled_helpers.py:205-210
        R[0] = 1; R[1] = 0; R[2] = 0; R[3] = 0; R[4] = 1; R[5] = 0; R[6] = 0; R[7] = 0; R[8] = 1;
        return;
    }
    const double inv = 1.0 / theta;
    double st, ct;
    sincos(theta, &st, &ct);
    const double f = (1.0 - ct) * inv * inv;
    st *= inv;
    R[0] = r[0] * r[0] * f + ct;
    R[4] = r[1] * r[1] * f + ct;
    R[8] = r[2] * r[2] * f + ct;
    const double xy = r[0] * r[1] * f, xz = r[0] * r[2] * f, yz = r[1] * r[2] * f;
    R[1] = xy - r[2] * st; R[3] = xy + r[2] * st;
    R[2] = xz + r[1] * st; R[6] = xz - r[1] * st;
    R[5] = yz - r[0] * st; R[7] = yz + r[0] * st;
}

// out[i*9 + k] = d R_k / d r_i  (OpenCV formula, compiled_helpers.py:237-286)
__device__ __forceinline__ void rodrigues_jac(const double r[3], double out[27])
{
    const double theta = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
#pragma unroll
    for (int k = 0; k < 27; ++k) out[k] = 0.0;
    if (theta < 1e-10) {  // so(3) generators, compiled_helpers.py:246-254
        out[5] = -1; out[7] = 1; out[11] = 1; out[15] = -1; out[19] = -1; out[21] = 1;
        return;
    }
    const double it = 1.0 / theta;
    double st, ct;
    sincos(theta, &st, &ct);
    const double c1 = 1.0 - ct;
    const double n[3] = {r[0] * it, r[1] * it, r[2] * it};
    const double rrt[9] = {n[0] * n[0], n[0] * n[1], n[0] * n[2], n[0] * n[1], n[1] * n[1],
                           n[1] * n[2], n[0] * n[2], n[1] * n[2], n[2] * n[2]};
    const double rx[9] = {0, -n[2], n[1], n[2], 0, -n[0], -n[1], n[0], 0};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double ri = n[i];
        const double a0 = -st * ri, a1 = (st - 2 * c1 * it) * ri, a2 = c1 * it, a3 = (ct - st * it) * ri,
                     a4 = st * it;
        double* o = out + 9 * i;
#pragma unroll
        for (int k = 0; k < 9; ++k) o[k] = a1 * rrt[k] + a3 * rx[k];
        o[0] += a0; o[4] += a0; o[8] += a0;
        // a2 * d(rr^T)/dn_i : row i and column i of the 3x3 get n, the (i,i) entry gets 2 n_i
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            o[3 * i + j] += a2 * n[j];
            o[3 * j + i] += a2 * n[j];
        }
        // a4 * d[n]x/dn_i
        const int j1 = (i + 1) % 3, j2 = (i + 2) % 3;
        o[3 * j2 + j1] += a4;
        o[3 * j1 + j2] -= a4;
    }
}

// Left Jacobian of SO(3), row-major 3x3:  d(R(r) X)/dr_i = Jl[:, i] x (R X).
// theta < 1e-10 -> identity, matching the reference's switch to the so(3) generators (compiled_helpers.py:246-254).
__device__ __forceinline__ void rodrigues_left_jacobian(const double r[3], double Jl[9])
{
    const double th2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2];
    const double theta = sqrt(th2);
    if (theta < 1e-10) {
        Jl[0] = 1; Jl[1] = 0; Jl[2] = 0; Jl[3] = 0; Jl[4] = 1; Jl[5] = 0; Jl[6] = 0; Jl[7] = 0; Jl[8] = 1;
        return;
    }
    double a, b;
    if (theta < 0.05) {  // series: avoids the cancellation in 1 - cos and theta - sin
        a = 0.5 - th2 * (1.0 / 24.0 - th2 * (1.0 / 720.0 - th2 * (1.0 / 40320.0)));
        b = 1.0 / 6.0 - th2 * (1.0 / 120.0 - th2 * (1.0 / 5040.0 - th2 * (1.0 / 362880.0)));
    } else {
        double sh, ch, st, ct;
        sincos(0.5 * theta, &sh, &ch);
        sincos(theta, &st, &ct);
        a = 2.0 * sh * sh / th2;
        b = (theta - st) / (th2 * theta);
    }
    const double x = r[0], y = r[1], z = r[2];
    // [r]x^2 = r r^T - |r|^2 I
    Jl[0] = 1.0 + b * (x * x - th2); Jl[1] = -a * z + b * x * y;      Jl[2] = a * y + b * x * z;
    Jl[3] = a * z + b * x * y;       Jl[4] = 1.0 + b * (y * y - th2); Jl[5] = -a * x + b * y * z;
    Jl[6] = -a * y + b * x * z;      Jl[7] = a * x + b * y * z;       Jl[8] = 1.0 + b * (z * z - th2);
}

// Forward chain up to camera coordinates.
struct ObsGeom {
    double Xt[3], Xw[3], Xc[3];
};

__device__ __forceinline__ void transform(const double* __restrict__ R, const double* __restrict__ t,
                                          const double X[3], double Y[3])
{
#pragma unroll
    for (int a = 0; a < 3; ++a) Y[a] = fma(R[3 * a], X[0], fma(R[3 * a + 1], X[1], fma(R[3 * a + 2], X[2], t[a])));
}

// Projection in normalised coordinates; returns projected (u, v) and the pieces the Jacobian needs.
struct Proj {
    double u, v;          // projected pixel
    double xn, yn, r2;    // normalised coords
    double xD, yD;        // distorted normalised coords
    double iz;            // 1 / z
    double drad;          // d rad / d r2
    double rad;
};

__device__ __forceinline__ Proj project(const double* __restrict__ q, const double Xc[3])
{
    Proj p;
    p.iz = 1.0 / Xc[2];
    p.xn = Xc[0] * p.iz;
    p.yn = Xc[1] * p.iz;
    p.r2 = fma(p.xn, p.xn, p.yn * p.yn);
    const double k1 = q[4], k2 = q[5], p1 = q[6], p2 = q[7], k3 = q[8];
    p.rad = fma(p.r2, fma(p.r2, fma(p.r2, k3, k2), k1), 1.0);
    p.drad = fma(p.r2, fma(p.r2, 3.0 * k3, 2.0 * k2), k1);
    const double xy = p.xn * p.yn;
    p.xD = fma(p.xn, p.rad, fma(2.0 * p1, xy, p2 * fma(2.0 * p.xn, p.xn, p.r2)));
    p.yD = fma(p.yn, p.rad, fma(p1, fma(2.0 * p.yn, p.yn, p.r2), 2.0 * p2 * xy));
    p.u = fma(q[0], p.xD, q[1]);
    p.v = fma(q[2], p.yD, q[3]);
    return p;
}

// Jacobian of one observation in "compressed" form:
//   Au[5] / Av[5]: d u / d(k1,k2,p1,p2,k3), d v / d(k1,k2,p1,p2,k3)
//   du/dfx = xD, du/dpx = 1, dv/dfy = yD, dv/dpy = 1, all other intrinsic entries are structural zeros
//   Pm (2x3) = d(u,v)/dXc;  N (2x3) = Pm R_c
//   Wc (2x3): rows (R_c X_w) x Pm_row   -- camera-rotation block in the tangent parametrisation; Bc = Wc Jl_c
//   Wm (2x3): rows (R_m X_t) x N_row    -- pose-rotation block in the tangent parametrisation;   Bm = Wm Jl_m
// Dense row layout (matflow column order): [fx px fy py k1 k2 p1 p2 k3 | Bc(3) Pm(3) | Bm(3) N(3) | (N R_m)(3)]
struct ObsJac {
    double xD, yD;
    double Au[5], Av[5];
    double Pm[6];
    double Wc[6];
    double N[6];
    double Wm[6];
};

__device__ __forceinline__ void projection_jac(const double* __restrict__ q, const Proj& p, ObsJac& J)
{
    const double fx = q[0], fy = q[2], p1 = q[6], p2 = q[7];
    const double r2 = p.r2, r4 = r2 * r2, r6 = r4 * r2;
    const double xy2 = 2.0 * p.xn * p.yn;
    J.xD = p.xD;
    J.yD = p.yD;
    const double fxx = fx * p.xn, fyy = fy * p.yn;
    J.Au[0] = fxx * r2; J.Au[1] = fxx * r4; J.Au[2] = fx * xy2; J.Au[3] = fx * fma(2.0 * p.xn, p.xn, r2); J.Au[4] = fxx * r6;
    J.Av[0] = fyy * r2; J.Av[1] = fyy * r4; J.Av[2] = fy * fma(2.0 * p.yn, p.yn, r2); J.Av[3] = fy * xy2; J.Av[4] = fyy * r6;
    // d(xD, yD) / d(xn, yn)
    const double d2 = 2.0 * p.drad;
    const double xDx = fma(d2 * p.xn, p.xn, p.rad) + 2.0 * p1 * p.yn + 6.0 * p2 * p.xn;
    const double xDy = d2 * p.xn * p.yn + 2.0 * p1 * p.xn + 2.0 * p2 * p.yn;
    const double yDy = fma(d2 * p.yn, p.yn, p.rad) + 6.0 * p1 * p.yn + 2.0 * p2 * p.xn;
    const double sx = fx * p.iz, sy = fy * p.iz;
    J.Pm[0] = sx * xDx;
    J.Pm[1] = sx * xDy;
    J.Pm[2] = -sx * fma(xDx, p.xn, xDy * p.yn);
    J.Pm[3] = sy * xDy;  // dyD/dxn == dxD/dyn
    J.Pm[4] = sy * yDy;
    J.Pm[5] = -sy * fma(xDy, p.xn, yDy * p.yn);
}

// D[a][i] = sum_j dR[i*9 + 3a + j] X[j]   (rigidTform3d.compute_jac, function_block_implementations.py:161-169)
// out (2x3) = L (2x3) * D (3x3), without materialising D in memory.
__device__ __forceinline__ void left_times_drx(const double L[6], const double* __restrict__ dR, const double X[3],
                                               double out[6])
{
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double d[3];
#pragma unroll
        for (int a = 0; a < 3; ++a)
            d[a] = fma(dR[9 * i + 3 * a], X[0], fma(dR[9 * i + 3 * a + 1], X[1], dR[9 * i + 3 * a + 2] * X[2]));
        out[i] = fma(L[0], d[0], fma(L[1], d[1], L[2] * d[2]));
        out[3 + i] = fma(L[3], d[0], fma(L[4], d[1], L[5] * d[2]));
    }
}

// out rows = Y x L_row  (L is 2x3): the derivative of L (R X) with respect to a left perturbation of R, Y = R X
__device__ __forceinline__ void cross_rows(const double Y[3], const double L[6], double out[6])
{
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const double* p = L + 3 * r;
        out[3 * r + 0] = fma(Y[1], p[2], -(Y[2] * p[1]));
        out[3 * r + 1] = fma(Y[2], p[0], -(Y[0] * p[2]));
        out[3 * r + 2] = fma(Y[0], p[1], -(Y[1] * p[0]));
    }
}

// out (2x3) = L (2x3) * R (3x3 row-major)
__device__ __forceinline__ void left_times_R(const double L[6], const double* __restrict__ R, double out[6])
{
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        out[i] = fma(L[0], R[i], fma(L[1], R[3 + i], L[2] * R[6 + i]));
        out[3 + i] = fma(L[3], R[i], fma(L[4], R[3 + i], L[5] * R[6 + i]));
    }
}

// Y = R X (no translation)
__device__ __forceinline__ void rotate(const double* __restrict__ R, const double X[3], double Y[3])
{
#pragma unroll
    for (int a = 0; a < 3; ++a) Y[a] = fma(R[3 * a], X[0], fma(R[3 * a + 1], X[1], R[3 * a + 2] * X[2]));
}

// Full evaluation of one observation: residual + compressed Jacobian (rotation blocks in tangent form).
__device__ __forceinline__ void eval_obs(const double* __restrict__ cam, const double* __restrict__ pose,
                                         const double Xt[3], double u_obs, double v_obs, double res[2], ObsJac& J)
{
    double Ym[3], Xw[3], Yc[3], Xc[3];
    rotate(pose + POSE_R, Xt, Ym);
#pragma unroll
    for (int a = 0; a < 3; ++a) Xw[a] = Ym[a] + pose[POSE_T + a];
    rotate(cam + CAM_R, Xw, Yc);
#pragma unroll
    for (int a = 0; a < 3; ++a) Xc[a] = Yc[a] + cam[CAM_T + a];
    const Proj p = project(cam + CAM_Q, Xc);
    res[0] = p.u - u_obs;
    res[1] = p.v - v_obs;
    projection_jac(cam + CAM_Q, p, J);
    cross_rows(Yc, J.Pm, J.Wc);
    left_times_R(J.Pm, cam + CAM_R, J.N);
    cross_rows(Ym, J.N, J.Wm);
}

// Camera-side evaluation for the normal-equation kernel: residual, intrinsic entries, Pm and the camera-rotation
// rows in tangent form.  The pose columns are NOT evaluated per observation: within one (camera, pose) segment they
// are the extrinsic columns times a constant 6x6 adjoint (see pcs_normal.cu), so only their segment sums are formed.
struct ObsJacCam {
    double xD, yD;
    double Au[5], Av[5];
    double Pm[6];
    double Wc[6];
};

// Table rows are fetched with 16-byte loads (rows are 16-byte aligned): camera row doubles 0..21 = q(9) R(9) t(3)
// (+1 unused), pose row doubles 0..11 = R(9) t(3); the template row is padded to 4 doubles.
__device__ __forceinline__ void eval_obs_cam(const double* __restrict__ cam, const double* __restrict__ pose,
                                             const double* __restrict__ pt4, double u_obs, double v_obs, double res[2],
                                             ObsJacCam& J)
{
    double cv[22], pv[12], Xt[4];
    const double2* c2 = reinterpret_cast<const double2*>(cam);
    const double2* p2 = reinterpret_cast<const double2*>(pose);
    const double2* x2 = reinterpret_cast<const double2*>(pt4);
#pragma unroll
    for (int k = 0; k < 6; ++k) { const double2 v = p2[k]; pv[2 * k] = v.x; pv[2 * k + 1] = v.y; }
#pragma unroll
    for (int k = 0; k < 2; ++k) { const double2 v = x2[k]; Xt[2 * k] = v.x; Xt[2 * k + 1] = v.y; }
#pragma unroll
    for (int k = 0; k < 11; ++k) { const double2 v = c2[k]; cv[2 * k] = v.x; cv[2 * k + 1] = v.y; }
    double Xw[3], Yc[3], Xc[3];
    transform(pv + POSE_R, pv + POSE_T, Xt, Xw);
    rotate(cv + CAM_R, Xw, Yc);
#pragma unroll
    for (int a = 0; a < 3; ++a) Xc[a] = Yc[a] + cv[CAM_T + a];
    const Proj p = project(cv + CAM_Q, Xc);
    res[0] = p.u - u_obs;
    res[1] = p.v - v_obs;
    ObsJac full;
    projection_jac(cv + CAM_Q, p, full);
    J.xD = full.xD; J.yD = full.yD;
#pragma unroll
    for (int k = 0; k < 5; ++k) { J.Au[k] = full.Au[k]; J.Av[k] = full.Av[k]; }
#pragma unroll
    for (int k = 0; k < 6; ++k) J.Pm[k] = full.Pm[k];
    cross_rows(Yc, J.Pm, J.Wc);
}

// Residual only.
__device__ __forceinline__ void eval_residual(const double* __restrict__ cam, const double* __restrict__ pose,
                                              const double Xt[3], double u_obs, double v_obs, double res[2])
{
    double Xw[3], Xc[3];
    transform(pose + POSE_R, pose + POSE_T, Xt, Xw);
    transform(cam + CAM_R, cam + CAM_T, Xw, Xc);
    const Proj p = project(cam + CAM_Q, Xc);
    res[0] = p.u - u_obs;
    res[1] = p.v - v_obs;
}

// Rotation blocks exactly as the reference evaluates them: Bc = Pm D_c(X_w), Bm = N D_m(X_t) with
// D[a][i] = sum_j dR[i][3a+j] X[j] from the OpenCV dR/dr table (function_block_implementations.py:157-182,
// compiled_helpers.py:237-286).  Used by the explicit-Jacobian (jac_fn drop-in) and dense paths so that their
// entries match the reference's to rounding; the OpenCV formula itself loses ~1e-8 relative accuracy for
// |rvec| ~ 1e-5 (cancellation), which the left-Jacobian form used by the normal-equation kernel does not.
__device__ __forceinline__ void reference_rotation_blocks(const ObsJac& J, const double* __restrict__ pose,
                                                          const double* __restrict__ cam_dR, const double* __restrict__ pose_dR,
                                                          const double Xt[3], double Bc[6], double Bm[6])
{
    double Xw[3];
    transform(pose + POSE_R, pose + POSE_T, Xt, Xw);
    left_times_drx(J.Pm, cam_dR, Xw, Bc);
    left_times_drx(J.N, pose_dR, Xt, Bm);
}

// Expand the compressed Jacobian into dense matflow rows (P = 21, or 24 with the point block).
// row 0 = d u / d(.), row 1 = d v / d(.)
template <int P>
__device__ __forceinline__ void expand_rows(const ObsJac& J, const double Bc[6], const double Bm[6],
                                            const double* __restrict__ pose, double ju[P], double jv[P])
{
    ju[0] = J.xD; ju[1] = 1.0; ju[2] = 0.0; ju[3] = 0.0;
    jv[0] = 0.0; jv[1] = 0.0; jv[2] = J.yD; jv[3] = 1.0;
#pragma unroll
    for (int k = 0; k < 5; ++k) { ju[4 + k] = J.Au[k]; jv[4 + k] = J.Av[k]; }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        ju[9 + k] = Bc[k];    jv[9 + k] = Bc[3 + k];
        ju[12 + k] = J.Pm[k]; jv[12 + k] = J.Pm[3 + k];
        ju[15 + k] = Bm[k];   jv[15 + k] = Bm[3 + k];
        ju[18 + k] = J.N[k];  jv[18 + k] = J.N[3 + k];
    }
    if (P == 24) {
        double Bk[6];
        left_times_R(J.N, pose + POSE_R, Bk);
#pragma unroll
        for (int k = 0; k < 3; ++k) { ju[21 + k] = Bk[k]; jv[21 + k] = Bk[3 + k]; }
    }
}

}  // namespace pcs
