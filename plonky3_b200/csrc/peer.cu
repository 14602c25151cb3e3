// Multi-GPU plumbing of the row-sharded commit (SURVEY.md section 8e) over NVLink peer memory, with no collective library on the
// data path: one process per GPU, buffers shared through CUDA IPC handles (exchanged by the host over any channel), and
// primitives on mapped peer pointers:
//   * the all-to-all of column blocks into row blocks: the LDE's column chunks are copied into the destination ranks' row
//     blocks on the copy engines (ntt.cu, ntt_coset_lde_sharded);
//   * peer_allgather_kernel: every rank stores a small record (a sub-tree root, a FRI final polynomial) into slot `rank` of
//     every rank's table;
//   * peer_barrier_kernel: flag barrier with system-scope release/acquire; stream-ordered, so "all peers' stores have landed"
//     becomes a dependency of the next kernel on this stream without any host round trip.
#include "common.h"

namespace p3 {

// Control block layout (u32 words) of every rank, allocated with p3gpu_malloc (cudaMalloc memory is IPC-shareable), zeroed
// before the handles are exchanged:  flags[16] (one arrival counter per source rank)  |  user area
constexpr int PEER_MAX = 16;

__device__ __forceinline__ void st_release_sys(u32 *p, u32 v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ u32 ld_acquire_sys(const u32 *p) {
    u32 v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

struct PeerPtrs { u32 *p[PEER_MAX]; };

// One warp.  Lane q < world: publish `epoch` in flags[rank] of rank q, then wait until flags[q] of OUR block reached `epoch`.
// Epochs only grow (the caller passes 1, 2, 3, ...), so no reset and no ABA.  All writes of earlier work on this stream
// (the LDE's peer copies) are complete before this kernel starts; the release store orders them before the flag.
__global__ void peer_barrier_kernel(const PeerPtrs ctrl, unsigned world, unsigned rank, u32 epoch, unsigned long long timeout_ns) {
    const unsigned q = threadIdx.x;
    if (q < world) {
        __threadfence_system();
        st_release_sys(ctrl.p[q] + rank, epoch);
        const u32 *mine = ctrl.p[rank] + q;
        unsigned long long t0 = 0;
        u32 spins = 0;
        while ((int)(ld_acquire_sys(mine) - epoch) < 0) {
            if ((++spins & 0x3ffu) == 0) {   // watchdog: a missing peer must become an error, not a hung device
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (t0 == 0) t0 = now;
                else if (now - t0 > timeout_ns) __trap();
            }
        }
    }
    __syncwarp();
    __threadfence_system();
}

// every rank's table[rank * words .. +words) <- src[0 .. words)   (tables = user area of the control blocks, or any mapped buffer)
__global__ void peer_allgather_kernel(const PeerPtrs tables, unsigned world, unsigned rank, const u32 *src, size_t words) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= words) return;
    const u32 v = src[i];
    for (unsigned q = 0; q < world; q++) tables.p[q][(size_t)rank * words + i] = v;
}

int32_t peer_barrier(p3gpu_ctx *ctx, unsigned world, unsigned rank, void *const *ctrl, u32 epoch, double timeout_s) {
    P3_CHECK(world >= 1 && world <= PEER_MAX && rank < world, P3GPU_EINVAL, "bad world/rank %u/%u", world, rank);
    PeerPtrs pp;
    for (unsigned q = 0; q < PEER_MAX; q++) pp.p[q] = q < world ? (u32 *)ctrl[q] : nullptr;
    for (unsigned q = 0; q < world; q++) P3_CHECK(pp.p[q], P3GPU_EINVAL, "null control block for rank %u", q);
    peer_barrier_kernel<<<1, 32, 0, ctx->stream>>>(pp, world, rank, epoch, (unsigned long long)(timeout_s * 1e9));
    ctx->launches++;
    P3_CUDA(cudaGetLastError());
    return P3GPU_OK;
}

int32_t peer_allgather(p3gpu_ctx *ctx, unsigned world, unsigned rank, void *const *tables, const u32 *d_src, size_t words) {
    P3_CHECK(world >= 1 && world <= PEER_MAX && rank < world, P3GPU_EINVAL, "bad world/rank %u/%u", world, rank);
    PeerPtrs pp;
    for (unsigned q = 0; q < PEER_MAX; q++) pp.p[q] = q < world ? (u32 *)tables[q] : nullptr;
    for (unsigned q = 0; q < world; q++) P3_CHECK(pp.p[q], P3GPU_EINVAL, "null table for rank %u", q);
    if (words == 0) return P3GPU_OK;
    peer_allgather_kernel<<<(unsigned)((words + 127) / 128), 128, 0, ctx->stream>>>(pp, world, rank, d_src, words);
    ctx->launches++;
    P3_CUDA(cudaGetLastError());
    return P3GPU_OK;
}

}  // namespace p3
