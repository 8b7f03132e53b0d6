// pcs_p2p.cu -- one-shot all-reduce of the camera blocks [U | g_c | r.r] over NVLink peer memory.
//
// The per-evaluation exchange of the pose-sharded problem (SURVEY.md 8e) is C * 240 + 1 doubles (61 KB at C = 32):
// a latency problem, not a bandwidth one.  Every rank owns a "symmetric" buffer that all peers have mapped (the
// Python host allocates it with torch's symmetric-memory allocator and passes the peer pointers in): a 256-byte header,
// then two slot sets of `world` blocks each, used alternately so that a rank that races ahead never overwrites a block
// still being read.  The exchange (k_p2p_allreduce_sentinel) pushes a rank's block into its slot at every peer with
// plain posted stores and polls its own buffer until the sentinel NaN in the slots it needs is replaced: no system
// fence, no flag (7.6 us per exchange at N = 2).  The received blocks are summed from LOCAL memory in rank order: the
// result is bitwise identical on every rank.
#include "pcs_internal.cuh"

namespace pcs {

constexpr int P2P_MAX_WORLD = 16;
constexpr int64_t P2P_HEADER_DOUBLES = 32; // 256 bytes; word P2P_MAX_WORLD is the `done` counter of k_p2p_allreduce_sentinel
constexpr int P2P_ILP = 8;                 // push: entries per thread and pass with their loads in flight together
constexpr int P2P_SUM_ILP = 4;             // sum: entries per thread and pass (x world loads each)

struct P2PPeers {
    double* buf[P2P_MAX_WORLD];
};

struct P2PState {
    P2PPeers peers;
    int rank = 0, world = 1;
    int64_t n = 0;          // doubles exchanged
    uint64_t epoch = 0;
    int* err = nullptr;     // device flag: a poll timed out
};

// "The data is the signal": the slots of a buffer hold a sentinel NaN whenever they are empty.  CTA b pushes this rank's
// block into its slot at peer b -- no system fence, no flag -- and every CTA sums its 1 / world share of
// the entries by polling the `world` slots of its OWN buffer until none of the values it needs is the sentinel (8-byte
// stores are atomic, so a value is either the sentinel or complete), in rank order (identical bits on every rank), and
// then puts the sentinel back.  A slot set is reused two exchanges later; the peer's write for that exchange causally
// follows this rank's next push, which is issued by a later kernel of the same stream, i.e. after the reset below is
// complete.  The result may only overwrite `local` once every CTA of this rank has finished reading it for its push:
// a counter in the rank's own buffer (local traffic only).  Chain per exchange: one NVLink one-way trip + local polls.
constexpr unsigned long long P2P_SENTINEL = 0x7ff8dead7ff8deadull;

__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const void* p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__global__ void k_p2p_fill_sentinel(double* __restrict__ slots, int64_t n)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) reinterpret_cast<unsigned long long*>(slots)[i] = P2P_SENTINEL;
}

template <int WORLD>
__global__ void __launch_bounds__(512)
k_p2p_allreduce_sentinel(double* __restrict__ local, int64_t n, int rank, int world_rt, P2PPeers peers, uint64_t epoch, int* __restrict__ err)
{
    const int world = WORLD > 0 ? WORLD : world_rt;
    const int tid = threadIdx.x, b = blockIdx.x;   // gridDim.x == world
    const int64_t data = P2P_HEADER_DOUBLES + (int64_t)(epoch & 1) * world * n;
    pdl_wait();
    {
        double* dst = peers.buf[b] + data + (int64_t)rank * n;
        const bool vec = ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(local)) & 15) == 0;
        const int64_t n2 = vec ? n / 2 : 0;
        for (int64_t i0 = 0; i0 < n2; i0 += (int64_t)P2P_ILP * blockDim.x) {   // loads of a pass in flight together
            double2 v[P2P_ILP];
#pragma unroll
            for (int u = 0; u < P2P_ILP; ++u) {
                const int64_t i = i0 + (int64_t)u * blockDim.x + tid;
                if (i < n2) v[u] = reinterpret_cast<const double2*>(local)[i];
            }
#pragma unroll
            for (int u = 0; u < P2P_ILP; ++u) {
                const int64_t i = i0 + (int64_t)u * blockDim.x + tid;
                if (i < n2) reinterpret_cast<double2*>(dst)[i] = v[u];
            }
        }
        for (int64_t i = 2 * n2 + tid; i < n; i += blockDim.x) dst[i] = local[i];
    }
    __syncthreads();
    double* mine = peers.buf[rank];
    unsigned long long* done = reinterpret_cast<unsigned long long*>(mine) + P2P_MAX_WORLD;
    if (tid == 0) atomicAdd(done, 1ull);             // this CTA has finished reading `local`
    const int64_t e0 = n * b / world, e1 = n * (b + 1) / world;
    bool may_write = false;
    for (int64_t i0 = e0; i0 < e1; i0 += (int64_t)P2P_SUM_ILP * blockDim.x) {
        double s[P2P_SUM_ILP];
#pragma unroll
        for (int u = 0; u < P2P_SUM_ILP; ++u) {
            const int64_t i = i0 + (int64_t)u * blockDim.x + tid;
            s[u] = 0.0;
            if (i < e1) {
                unsigned long long v[WORLD > 0 ? WORLD : P2P_MAX_WORLD];
                int spins = 0;
                bool ready;
                do {
                    ready = true;
#pragma unroll
                    for (int r = 0; r < (WORLD > 0 ? WORLD : P2P_MAX_WORLD); ++r)
                        if (r < world) {
                            v[r] = ld_relaxed_sys_u64(mine + data + (int64_t)r * n + i);
                            ready = ready && v[r] != P2P_SENTINEL;
                        }
                } while (!ready && ++spins < (1 << 24));
                if (!ready) *err = 1;                // a peer never delivered: report instead of hanging
#pragma unroll
                for (int r = 0; r < (WORLD > 0 ? WORLD : P2P_MAX_WORLD); ++r)
                    if (r < world) s[u] += __longlong_as_double((long long)v[r]);   // rank order: identical bits everywhere
            }
        }
        if (!may_write) {                            // before the first result lands in `local`: all CTAs are done reading it
            if (tid == 0) {
                int spins = 0;
                while (ld_relaxed_sys_u64(done) < epoch * (uint64_t)world && ++spins < (1 << 24)) { }
            }
            __syncthreads();
            may_write = true;
        }
#pragma unroll
        for (int u = 0; u < P2P_SUM_ILP; ++u) {
            const int64_t i = i0 + (int64_t)u * blockDim.x + tid;
            if (i < e1) {
                local[i] = s[u];
#pragma unroll
                for (int r = 0; r < (WORLD > 0 ? WORLD : P2P_MAX_WORLD); ++r)
                    if (r < world) reinterpret_cast<unsigned long long*>(mine + data + (int64_t)r * n)[i] = P2P_SENTINEL;
            }
        }
    }
}

}  // namespace pcs

using namespace pcs;

extern "C" {

int64_t pcs_p2p_buffer_bytes(const pcs_problem* p, int world)
{
    if (!p || world < 1) return 0;
    const int64_t n = (int64_t)p->C * 240 + 1;
    return (P2P_HEADER_DOUBLES + 2 * (int64_t)world * n) * (int64_t)sizeof(double);
}

int pcs_p2p_allreduce_setup(pcs_problem* p, int rank, int world, void* const* peer_buffers, int64_t buffer_bytes)
{
    PCS_REQUIRE(p && peer_buffers, "NULL argument");
    PCS_REQUIRE(world >= 1 && world <= P2P_MAX_WORLD && rank >= 0 && rank < world, "rank / world out of range");
    PCS_REQUIRE(buffer_bytes >= pcs_p2p_buffer_bytes(p, world), "symmetric buffer is smaller than pcs_p2p_buffer_bytes()");
    P2PState* st = (P2PState*)p->p2p;
    if (!st) {
        st = new P2PState();
        p->p2p = st;
    }
    for (int r = 0; r < world; ++r) {
        PCS_REQUIRE(peer_buffers[r], "peer buffer pointer is NULL");
        st->peers.buf[r] = (double*)peer_buffers[r];
    }
    st->rank = rank; st->world = world; st->n = (int64_t)p->C * 240 + 1; st->epoch = 0;
    // the slots of THIS rank's buffer are filled with the sentinel here; the caller's barrier after setup -- see
    // pycamset_b200/distributed.py -- keeps any peer from pushing before that
    if (!st->err) PCS_CUDA(cudaMalloc((void**)&st->err, sizeof(int)));
    PCS_CUDA(cudaMemsetAsync(st->err, 0, sizeof(int), p->stream));
    const int64_t n_slots = 2 * (int64_t)world * st->n;
    k_p2p_fill_sentinel<<<(int)((n_slots + 255) / 256), 256, 0, p->stream>>>(st->peers.buf[rank] + P2P_HEADER_DOUBLES, n_slots);
    PCS_CUDA(cudaGetLastError());
    PCS_CUDA(cudaStreamSynchronize(p->stream));
    return PCS_OK;
}

int pcs_p2p_allreduce_camera_blocks(pcs_problem* p)
{
    PCS_REQUIRE(p && p->p2p, "pcs_p2p_allreduce_setup has not been called");
    PCS_CUDA(cudaSetDevice(p->device));
    P2PState* st = (P2PState*)p->p2p;
    ++st->epoch;
    auto kern = st->world == 2 ? k_p2p_allreduce_sentinel<2> : st->world == 4 ? k_p2p_allreduce_sentinel<4>
                : st->world == 8 ? k_p2p_allreduce_sentinel<8> : k_p2p_allreduce_sentinel<0>;
    PCS_CUDA(launch_pdl(kern, dim3(st->world), dim3(512), 0, p->stream, p->U, st->n, st->rank, st->world, st->peers, st->epoch, st->err));
    PCS_CUDA(cudaGetLastError());
    ++p->n_launches;
    return PCS_OK;
}

int pcs_p2p_status(pcs_problem* p, int* timed_out)
{
    PCS_REQUIRE(p && p->p2p && timed_out, "NULL argument or pcs_p2p_allreduce_setup has not been called");
    PCS_CUDA(cudaSetDevice(p->device));
    P2PState* st = (P2PState*)p->p2p;
    *timed_out = 0;
    if (st->err) {
        PCS_CUDA(cudaMemcpyAsync(timed_out, st->err, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
        PCS_CUDA(cudaStreamSynchronize(p->stream));
    }
    return PCS_OK;
}

}  // extern "C"

namespace pcs {
void p2p_free(pcs_problem* p)
{
    if (p->p2p && ((P2PState*)p->p2p)->err) cudaFree(((P2PState*)p->p2p)->err);
    delete (P2PState*)p->p2p;
    p->p2p = nullptr;
}
}  // namespace pcs
