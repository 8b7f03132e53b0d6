// pcs_internal.cuh -- host-side problem state shared by the translation units of libpcs_b200.so
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/pcs_b200.h"

namespace pcs {

void set_error(const std::string& msg);

#define PCS_CUDA(call)                                                                                       \
    do {                                                                                                     \
        cudaError_t e__ = (call);                                                                            \
        if (e__ != cudaSuccess) {                                                                            \
            ::pcs::set_error(std::string(#call) + " -> " + cudaGetErrorString(e__) + " (" __FILE__ ":" +      \
                             std::to_string(__LINE__) + ")");                                                 \
            return PCS_ERR_CUDA;                                                                             \
        }                                                                                                    \
    } while (0)

#define PCS_REQUIRE(cond, msg)                                  \
    do {                                                        \
        if (!(cond)) {                                          \
            ::pcs::set_error(std::string("invalid argument: ") + (msg)); \
            return PCS_ERR_INVALID;                             \
        }                                                       \
    } while (0)

// Opt a kernel in to `bytes` of dynamic shared memory on the CURRENT device, once per (kernel, device): the attribute
// belongs to the device's context, so a process that drives several GPUs has to set it on each of them.
template <typename Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, size_t bytes)
{
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> done;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    size_t& have = done[{reinterpret_cast<const void*>(kernel), dev}];
    if (have >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) have = bytes;
    return e;
}

// Programmatic dependent launch (sm_90+): a kernel launched through launch_pdl may become resident while the kernel
// before it in the stream is still running; it must call pdl_wait() before it touches anything that kernel writes (the
// wait returns once the whole prerequisite grid has completed and flushed).  The earlier kernel allows this by calling
// pdl_launch_dependents().  Net effect: the launch latency and the on-chip prologue of the dependent overlap the tail of
// its predecessor.  Without the launch attribute both instructions are no-ops and the stream serialises as usual.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

#define PCS_TRY(expr)              \
    do {                           \
        int rc__ = (expr);         \
        if (rc__ != PCS_OK) return rc__; \
    } while (0)

}  // namespace pcs

struct pcs_problem {
    int chain = 0, C = 0, M = 0, K = 0, P = 21, device = 0, sm_count = 148;
    int64_t N = 0, L = 0, n_free = 0, nnz = 0, n_seg = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;

    // observations, original (dd) order
    int32_t *cam = nullptr, *pose = nullptr, *key = nullptr;
    double* uv = nullptr;
    // static tables
    double* tmpl = nullptr;        // [K][3] chain 0
    double* tmpl4 = nullptr;       // [K][4] points padded to 16-byte rows: the template (chain 0) or the free points (chain 1; refreshed by k_prepare_tables)
    int32_t* free_map = nullptr;   // [L]
    int32_t* free_idx = nullptr;   // [n_free] parameter-string position of free variable j
    uint16_t* cam_mask = nullptr;  // [C] bit k set = column k of [intr(9) extr(6)] is free
    uint8_t* pose_mask = nullptr;  // [M] 6 bits
    uint8_t* key_mask = nullptr;   // [K] 3 bits (chain 1)
    int64_t* row_prefix = nullptr; // [N+1] free columns per observation, exclusive prefix sum
    // dynamic
    double* params = nullptr;      // [L]
    double* x = nullptr;           // [n_free]
    double* camtab = nullptr;      // [C][32]
    double* posetab = nullptr;     // [M][24]
    double* dRtab = nullptr;       // [C + M][27] OpenCV dR/dr tables (explicit-Jacobian / dense paths; allocated on first use)
    double* resid = nullptr;       // [2N] (allocated on first use)
    double* jvals = nullptr;       // [nnz] (allocated on first use)
    // (camera, pose)-sorted layout for the normal equations
    int32_t *seg_cam = nullptr, *seg_pose = nullptr;  // [S]
    int64_t* seg_start = nullptr;                      // [S+1] into the sorted observation arrays
    int32_t *s_key = nullptr, *s_cam = nullptr, *s_pose = nullptr;  // [N] sorted
    double* s_uv = nullptr;                            // [N][2] sorted
    int32_t* obs_seg = nullptr;                        // [N] dd order: segment of every observation (residual kernel)
    double* segtab = nullptr;                          // [S][SEG_STRIDE] per-segment combined transform (allocated on first use)
    // normal-equation outputs: one allocation [U | gc | cost | pad | V | gp | W]
    double* ne = nullptr;
    double *U = nullptr, *gc = nullptr, *cost = nullptr, *V = nullptr, *gp = nullptr, *W = nullptr;
    // chain 1 (self-calibration), inside the same allocation between gp and W: point blocks Pk [K][3][3], gk [K][3] and the
    // dense coupling tables Xck [C][K][15][3] (camera x point), Ymk [M][K][6][3] (pose x point); nullptr when the tables
    // would be too large (block path unavailable: pcs_normal_dense remains)
    double *Pk = nullptr, *gk = nullptr, *Xck = nullptr, *Ymk = nullptr;
    int64_t ne_doubles = 0;
    // dense path
    double* dense = nullptr;  // [n_free*n_free + n_free + 1]
    // pinned staging
    double* h_pin = nullptr;
    int64_t h_pin_doubles = 0;

    pcs_allreduce_fn allreduce = nullptr;
    void* allreduce_user = nullptr;
    int rank = 0, world = 1;

    // optional event timing of the normal-equation kernel
    // ring of (start, stop) event pairs, one per launch, read back without synchronising inside a timed loop
    bool timing = false;
    std::vector<cudaEvent_t> ev_a, ev_b;
    int64_t timing_count = 0;   // launches recorded since timing was enabled

    // segment range tables of the normal-equation kernel, slot 0: single launch, slot 1: host path in parts
    int64_t* warp_seg[2] = {nullptr, nullptr};  // [ne_parts][ne_warps + 1]
    int64_t ne_warps[2] = {0, 0};
    int ne_parts[2] = {0, 0};
    std::vector<int64_t> h_part_bounds;   // [ne_parts + 1] first segment of every part (host copy)
    cudaStream_t copy_stream = nullptr;    // host path: copy-out of finished parts overlaps the next part's kernel
    cudaEvent_t part_done[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t copy_done = nullptr;
    int normal_precision = 0; // pcs_precision of the fused normal-equation kernel (pcs_set_normal_precision)
    int64_t n_launches = 0;  // kernels launched by this library on behalf of the problem (pcs_launch_count)

    // peer-memory all-reduce state (pcs_p2p.cu)
    void* p2p = nullptr;

    // LM workspace (pcs_solver.cu)
    void* lm_ws = nullptr;
};

namespace pcs {
// kernels / launchers implemented in pcs_core.cu, used by pcs_solver.cu
int launch_scatter_x(pcs_problem* p, const double* x_dev);
int launch_prepare(pcs_problem* p, bool with_dR = false, const double* x_dev = nullptr, double* zero = nullptr,
                   int64_t n_zero = 0, bool with_seg = false);
int launch_residual(pcs_problem* p, double* r_dev);
int launch_cost_only(pcs_problem* p, double* cost_dev);
int launch_normal_blocks(pcs_problem* p, bool targets_cleared = false, int part = 0, int n_parts = 1);
int launch_point_blocks(pcs_problem* p);   // chain 1: Pk, gk, Xck, Ymk (targets cleared by the prepare launch)
inline int64_t ne_zero_doubles(const pcs_problem* p) { return p->W - p->ne; }   // everything accumulated with reductions precedes W
int ensure_pinned(pcs_problem* p, int64_t doubles);
void lm_free(pcs_problem* p);
// pcs_schur.cu: S (n x n, column-major, lower) -= Z Z^T, Z column-major [k][n]; with a plan only the listed non-zero
// (tile, slab) units are visited and pose m's six columns sit at 6 pose_slot[m] .. 6 pose_slot[m] + 5
struct SchurPlan {
    int32_t* pose_slot = nullptr;   // [M] device, nullptr = identity
    void* units = nullptr;          // int2[n_units] device, nullptr = dense iteration space
    int64_t n_units = 0;
    double fraction = 1.0;          // non-zero units / all units
};
int schur_plan_build(pcs_problem* p, int64_t nc, int64_t nl, SchurPlan* plan);
void schur_plan_free(SchurPlan* plan);
int launch_schur_syrk(cudaStream_t st, int sm_count, int64_t n, int64_t k, const double* Z, double* S, const SchurPlan* plan = nullptr);
// pcs_chol.cu: dense SPD solve in one persistent kernel, every factorisation of the library
int chol_prepare(int device, int64_t n, double** Ldiag, unsigned long long** bar, int* grid);
int launch_chol_solve(cudaStream_t st, int grid, int64_t n, double* A, int64_t ld, double* rhs, double* Ldiag,
                      unsigned long long* bar, unsigned long long* bar_base, int* info, long long* trace = nullptr);
int chol_status(int info);   // the kernel's info word as a pcs_status
void p2p_free(pcs_problem* p);
// pcs_cov.cu: covariance from the factored reduced system (S off-diagonal tiles of L, Ldiag its diagonal tiles)
int cov_forward_substitution(cudaStream_t st, int64_t nc, const double* S, double* Ldiag, double* Xi, double* Z, int64_t np);
int cov_reduced_inverse(cudaStream_t st, int sm_count, int64_t nc, double* Xi, double* S);
int cov_block_marginals(cudaStream_t st, int n_blocks, int B, int64_t nc, const double* X, const int32_t* slot, double* L);
int cov_assemble(cudaStream_t st, const pcs_problem* p, int64_t nc, int red_B, int elim_B, const double* S, double* elim,
                 double* out_cam, double* out_red, double* n_observed);
}  // namespace pcs
