// Internal declarations shared by the translation units of libp3gpu.
#pragma once
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <tuple>
#include <type_traits>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/p3gpu.h"
#include "field.cuh"
#include "poseidon2_consts.h"

namespace p3 {

void set_error(const char *fmt, ...);

#define P3_CUDA(call)                                                                           \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            p3::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return P3GPU_ECUDA;                                                                 \
        }                                                                                       \
    } while (0)

#define P3_CHECK(cond, code, ...)                 \
    do {                                          \
        if (!(cond)) {                            \
            p3::set_error(__VA_ARGS__);           \
            return (code);                        \
        }                                         \
    } while (0)

// first statement of every extern "C" entry point that takes a context: serialise callers, select the device (CUDA's current
// device is per host thread: callers may come from any thread)
#define P3_ENTER(ctx)                                                        \
    P3_CHECK((ctx) != nullptr, P3GPU_EINVAL, "null context");                \
    std::lock_guard<std::recursive_mutex> p3_lock__((ctx)->call_mu);         \
    P3_CUDA(cudaSetDevice((ctx)->device));                                   \
    (ctx)->tick++

#define P3_TRY(expr)                      \
    do {                                  \
        int32_t rc__ = (expr);            \
        if (rc__ != P3GPU_OK) return rc__; \
    } while (0)


struct TwiddleKey {
    int field, log_n; u32 shift; int inverse;
    bool operator<(const TwiddleKey &o) const {
        return std::tie(field, log_n, shift, inverse) < std::tie(o.field, o.log_n, o.shift, o.inverse);
    }
};

}  // namespace p3

namespace p3 { struct TwiddleEntry { uint2 *ptr; size_t bytes; uint64_t last_use; }; }

struct p3gpu_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t switch_event = nullptr;   // orders work across p3gpu_ctx_set_stream changes (shared scratch / caches)
    int sm_count = 148;
    uint64_t launches = 0;
    // Every extern "C" entry point holds call_mu for its whole duration: the reference's objects are Clone + Sync and may be
    // called through &self from several threads (SURVEY 8b "Threading"); a context serialises such callers (scratch buffers,
    // caches and the stream are per context).  Clones that want concurrency create their own context.
    std::recursive_mutex call_mu;
    uint64_t tick = 0;                    // entry-point counter: LRU clock of the twiddle cache
    // twiddle heaps keyed like the reference's coset_twiddles cache (radix_2_dit_parallel.rs:32-40), bounded by bytes (LRU)
    std::map<p3::TwiddleKey, p3::TwiddleEntry> twiddles;
    size_t twiddle_bytes = 0;
    size_t twiddle_cap_bytes = (size_t)2 << 30;   // P3GPU_TWIDDLE_CACHE_MB
    void *leaf_table = nullptr; size_t leaf_table_bytes = 0;
    // host-pointer entry points: copy streams + events of the chunked H2D || compute || D2H pipeline, double-buffered chunk buffers
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr}, ev_start = nullptr;
    void *chunk_in[2] = {nullptr, nullptr}; size_t chunk_in_bytes[2] = {0, 0};
    void *chunk_out[2] = {nullptr, nullptr}; size_t chunk_out_bytes[2] = {0, 0};
    // staged multi-GPU exchange: staging buffers (one LDE'd column chunk each), exchange stream and events
    cudaStream_t xchg_stream = nullptr;
    cudaStream_t dma_stream[16] = {nullptr}; cudaEvent_t dma_done[16] = {nullptr};   // dma exchange: one copy stream per destination rank
    cudaEvent_t ev_stage_full[2] = {nullptr, nullptr}, ev_stage_free[2] = {nullptr, nullptr};
    void *stage_buf[2] = {nullptr, nullptr}; size_t stage_bytes[2] = {0, 0};   // device copy of the per-height matrix table (> 8 matrices)
    // FRI half-inverse-power tables (bit-reversed), one per field, grown on demand
    uint32_t *fold_table[2] = {nullptr, nullptr};
    size_t fold_table_len[2] = {0, 0};
    // grow-only scratch
    void *scratch = nullptr; size_t scratch_bytes = 0;
    void *scratch2 = nullptr; size_t scratch2_bytes = 0;
    void *pool[4] = {nullptr, nullptr, nullptr, nullptr}; size_t pool_bytes[4] = {0, 0, 0, 0};  // host-pointer wrappers / commit phase
    // Poseidon2 constants: [field][0: width 16, 1: width 24], host copy + device copy
    p3::Poseidon2Consts p2_host[2][2];
    p3::Poseidon2Consts *p2_dev = nullptr;  // 4 entries
    alignas(8) unsigned char air_consts[1024];   // Poseidon2 AIR round constants (air.cu: AirConsts)
    int air_set = 0;
};

namespace p3 {

int32_t ctx_scratch(p3gpu_ctx *ctx, size_t bytes, void **out);
int32_t ctx_scratch2(p3gpu_ctx *ctx, size_t bytes, void **out);
int32_t ctx_pool(p3gpu_ctx *ctx, int slot, size_t bytes, void **out);
int32_t ctx_leaf_table(p3gpu_ctx *ctx, size_t bytes, void **out);  // grow-only cached device buffers (no malloc/free per call)

// ntt.cu
int32_t ntt_dft_batch(p3gpu_ctx *ctx, int field, int kind, const u32 *d_in, u32 *d_out, size_t h, size_t w, u32 shift);
int32_t ntt_coset_lde(p3gpu_ctx *ctx, int field, const u32 *d_in, size_t h, size_t w, unsigned added_bits, u32 shift,
                      u32 *d_out, int bitrev_rows, size_t in_pitch = 0, size_t out_pitch = 0);
// hash.cu
int32_t hash_poseidon2_permute(p3gpu_ctx *ctx, int field, int width, u32 *d_states, size_t n);
int32_t hash_keccak_f(p3gpu_ctx *ctx, u64 *d_states, size_t n);
int32_t hash_merkle_commit(p3gpu_ctx *ctx, int field, int hash, size_t n_mats, const u32 *const *d_mats,
                           const size_t *heights, const size_t *widths, u32 *d_layers, size_t *layer_lens,
                           size_t *n_layers);
int32_t hash_merkle_from_digests(p3gpu_ctx *ctx, int field, int hash, const u32 *d_digests, size_t n, u32 *d_layers,
                                 size_t *layer_lens, size_t *n_layers);
// fri.cu
int32_t fri_fold(p3gpu_ctx *ctx, int field, const u32 *d_in, size_t rows, unsigned log_arity, const u32 beta[4], u32 *d_out);

int32_t fri_ef_axpy(p3gpu_ctx *ctx, int field, u32 *d_acc, const u32 *d_x, size_t n, const u32 s[4]);

// open.cu
int32_t open_inv_denoms(p3gpu_ctx *ctx, int field, unsigned log_h, const u32 *z, const u32 *zinv, u32 *d_out, u32 *d_adj);
int32_t open_columnwise_dot(p3gpu_ctx *ctx, int field, const u32 *d_mat, size_t h, size_t w, const u32 *d_vec, u32 *d_out, const u32 *scale);
int32_t open_rowwise_dot(p3gpu_ctx *ctx, int field, const u32 *d_mat, size_t h, size_t w, const u32 *alpha, u32 *d_out);
int32_t open_reduce(p3gpu_ctx *ctx, int field, u32 *d_ro, const u32 *d_r, const u32 *d_invd, size_t h, const u32 *coeff, const u32 *yred);

// ntt.cu / peer.cu: multi-GPU
int32_t ntt_coset_lde_sharded(p3gpu_ctx *ctx, int field, const u32 *d_in, size_t h, size_t w_local, unsigned added_bits, u32 shift,
                              unsigned world, u32 *const *rank_out, size_t w_total, size_t col_off, int chunk_major = 0);
std::vector<size_t> shard_chunk_bounds(size_t w_local);
int32_t peer_barrier(p3gpu_ctx *ctx, unsigned world, unsigned rank, void *const *ctrl, u32 epoch, double timeout_s);
int32_t peer_allgather(p3gpu_ctx *ctx, unsigned world, unsigned rank, void *const *tables, const u32 *d_src, size_t words);

// air.cu: Poseidon2 AIR trace generation / quotient (SURVEY 8f ranks 2-3)
int32_t air_set_constants(p3gpu_ctx *ctx, int field, const u32 *beg, const u32 *part, int rounds_p, const u32 *end);
int32_t air_generate_trace(p3gpu_ctx *ctx, int field, const u32 *d_inputs, size_t n_perms, u32 *d_trace);
int32_t air_quotient(p3gpu_ctx *ctx, int field, int vec_len, const u32 *d_lde, unsigned log_h, unsigned log_n, const u32 *alpha, u32 *d_q);

// challenger.cu / query.cu: transcript + query-phase gathers of the prove driver (SURVEY 8f rank 4, N1)
int32_t challenger_new(p3gpu_ctx *ctx, int field, int width, int rate, p3gpu_challenger **out);
void challenger_free(p3gpu_ctx *ctx, p3gpu_challenger *ch);
int32_t challenger_clone(p3gpu_ctx *ctx, const p3gpu_challenger *src, p3gpu_challenger **out);
int32_t challenger_observe_dev(p3gpu_ctx *ctx, p3gpu_challenger *ch, const u32 *d_vals, size_t n);
int32_t challenger_observe_host(p3gpu_ctx *ctx, p3gpu_challenger *ch, const u32 *h_vals, size_t n);
int32_t challenger_sample(p3gpu_ctx *ctx, p3gpu_challenger *ch, u32 *h_out, size_t n);
int32_t challenger_grind(p3gpu_ctx *ctx, p3gpu_challenger *ch, unsigned bits, u32 *witness_monty);
int32_t query_gather_rows(p3gpu_ctx *ctx, const u32 *d_mat, size_t h, size_t w, const u32 *h_idx, size_t n, unsigned shift, u32 *d_out);
int32_t query_merkle_paths(p3gpu_ctx *ctx, const u32 *d_layers, const size_t *layer_lens, size_t n_layers, size_t path_len, const u32 *h_idx,
                           size_t n, unsigned shift, u32 *d_out);

static inline unsigned log2_floor(size_t x) { unsigned l = 0; while ((x >> l) > 1) l++; return l; }
static inline bool is_pow2(size_t x) { return x && !(x & (x - 1)); }

}  // namespace p3
