// Batched NTT / coset LDE for row-major matrices over BabyBear / KoalaBear on sm_100a.
//
// Replaces Radix2DitParallel (dft/src/radix_2_dit_parallel.rs:30-515) behind TwoAdicSubgroupDft
// (dft/src/traits.rs:28-291).  Not a port: the reference runs two cache-blocked half networks separated by
// row bit-reversals on CPU threads; here ONE kernel family implements a Cooley-Tukey network that maps
// natural-order input to bit-reversed-order output ("network order"), executed as 1-3 passes over HBM:
//
//   * a pass owns the butterfly layers [l0, l1) of the size-2^n network.  A CTA takes a tile of R = 2^(l1-l0)
//     rows (all rows that agree on the top l0 and the low n-l1 index bits) x CT adjacent columns, stages it in
//     shared memory, runs the layers as radix-16 register steps (4 layers per shared-memory round trip), and
//     writes the tile back.  Row segments of CT*4 bytes are contiguous, so any row permutation (bit reversal on
//     input or output) is free: it only changes which 64/128-byte segments a tile touches.
//   * layer l uses one twiddle per block q (the reference's "twiddles with the coset shift baked in",
//     radix_2_dit_parallel.rs:80-115):  z_l[q] = shift^(N/2^(l+1)) * w_(2^(l+1))^bitrev_l(q).  They live in a
//     heap-ordered table Z[2^l + q]; a tile needs R-1 of them (contiguous runs per layer) and stages them in
//     shared memory next to the data.
//   * butterflies use Shoup multiplication by the precomputed twiddle and lazy [0, 2p) reduction:
//     3 multiply-pipe + 6 ALU-pipe instructions each (field.cuh: ct_butterfly).
//
// Two kernel generations implement a pass: ntt_pass_pipe_kernel (TMA tile loads into an mbarrier stage ring, warp-specialised
// consumer groups; the production path for 16-byte aligned shapes, with column-tile-major intermediates for the LDE) and
// ntt_pass_fast_kernel / ntt_pass_kernel (cp.async or plain loads; every other shape).  P3GPU_NTT_PIPE=0 forces the latter.
//
// coset_lde_batch = inverse network (root^-1, scale 1/h) producing coefficients in network (bit-reversed) order,
// then per coset a forward network reading those coefficients through a bit-reversed row map and leaving the
// evaluations in network order — which is exactly the bit-reversed row order the reference leaves in memory
// (radix_2_dit_parallel.rs:245, fri/src/two_adic_pcs.rs:313-318).  No standalone bit-reversal or scaling pass exists.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda.h>   // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint, no libcuda link)

#include "common.h"

namespace p3 {

static int env_int(const char *name, int dflt) {
    const char *s = getenv(name);
    return s ? atoi(s) : dflt;
}

struct PassArgs {
    const u32 *in;
    u32 *out;
    u32 w;         // row pitch in elements
    u32 col0;      // first column of this launch
    u32 n_ctiles;  // column tiles (of CT columns) in this launch
    u32 ct;        // tile width of the generic-width kernel variant
    u32 n_cosets;  // cosets batched in this launch (fastest-varying part of blockIdx.x)
    u32 vec16;     // fast kernel: row segments are 16-byte aligned (cp.async 16)
    u32 wc;                    // pipelined kernel: columns of this launch (<= w = row pitch of the dense layout)
    u32 in_tiled, out_tiled;   // pipelined kernel: intermediate buffers in column-tile-major layout (see lde_tiled_impl)
    u32 in_blocks;             // pipelined kernel, tiled input: 2^log_n-row blocks per column tile (cosets)
    u32 n_items, csplit, tpi;  // pipelined kernel: work items = (row tile, coset) units x csplit column chunks of tpi tiles
    unsigned long long *prof;  // profiling build only: per CTA/tile phase timestamps (P3GPU_NTT_PROFBUF)
    int log_n, l0, l1;
    const uint2 *tw;  // heap-ordered twiddles of coset 0
    int in_bitrev, out_bitrev;
    int out_sh;
    u32 out_add;  // output row = (maybe_bitrev(i) << out_sh) + out_add
    uint2 scale;
    int has_scale, final_reduce;
    size_t tw_stride;   // uint2 elements between consecutive cosets' heaps
    size_t out_stride;  // u32 elements between consecutive cosets' output blocks
    size_t in_stride;   // u32 elements between consecutive cosets' input blocks
};

template <int LOG_CT> __device__ __forceinline__ u32 sidx(u32 row, u32 c) {
    // XOR swizzle so that narrow column tiles (CT < 32) stay bank-conflict free in the stride-1 radix step
    if (LOG_CT < 5) row ^= (row >> 4) & ((32u >> LOG_CT) - 1u);
    return (row << LOG_CT) + c;
}

template <int F, int LOG_CT, int THREADS, int Q>
__device__ __forceinline__ void radix_step(u32 *data, const uint2 *tws, int r, int lam0) {
    constexpr u32 CT = 1u << LOG_CT;
    constexpr int E = 1 << Q;
    const int logD = r - lam0 - Q;
    const u32 D = 1u << logD;
    const u32 items = (1u << (r - Q)) << LOG_CT;
    for (u32 it = threadIdx.x; it < items; it += THREADS) {
        const u32 c = it & (CT - 1), g = it >> LOG_CT;
        const u32 lo = g & (D - 1), hi = g >> logD;
        const u32 base = (hi << (logD + Q)) + lo;
        const u32 node = (1u << lam0) + hi;
        u32 x[E];
#pragma unroll
        for (int m = 0; m < E; m++) x[m] = data[sidx<LOG_CT>(base + m * D, c)];
#pragma unroll
        for (int j = 0; j < Q; j++) {
            const int half = E >> (j + 1);
#pragma unroll
            for (int grp = 0; grp < (1 << j); grp++) {
                const uint2 z = tws[(node << j) + grp];
#pragma unroll
                for (int t = 0; t < half; t++) ct_butterfly<F>(x[grp * 2 * half + t], x[grp * 2 * half + t + half], z);
            }
        }
#pragma unroll
        for (int m = 0; m < E; m++) data[sidx<LOG_CT>(base + m * D, c)] = x[m];
    }
    __syncthreads();
}

template <int F, int LOG_CT, int THREADS, bool VEC>
__global__ void __launch_bounds__(THREADS) ntt_pass_kernel(const PassArgs a) {
    constexpr u32 CT = 1u << LOG_CT;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int r = a.l1 - a.l0;
    const u32 R = 1u << r;
    u32 *data = reinterpret_cast<u32 *>(smem_raw);
    uint2 *tws = reinterpret_cast<uint2 *>(data + ((size_t)R << LOG_CT));

    const u32 coset = blockIdx.x % a.n_cosets, bx = blockIdx.x / a.n_cosets;
    const u32 ctile = bx % a.n_ctiles, tile = bx / a.n_ctiles;
    const int lowbits = a.log_n - a.l1;
    const u32 L = tile & ((1u << lowbits) - 1u), T = tile >> lowbits;
    const u32 col = a.col0 + ctile * CT;
    const uint2 *tw = a.tw + (size_t)coset * a.tw_stride;
    const u32 *in = a.in + (size_t)coset * a.in_stride;
    u32 *out = a.out + (size_t)coset * a.out_stride;
    const u32 out_add = a.out_add;
    const u32 ibase = (a.l0 == 0 ? 0u : (T << (a.log_n - a.l0))) | L;
    const int brsh = 32 - a.log_n;

    // stage this tile's R-1 twiddles: tws[2^lam + ql] = Z[2^(l0+lam) + T*2^lam + ql]
    for (u32 k = threadIdx.x + 1; k < R; k += THREADS) {
        const int lam = 31 - __clz(k);
        const u32 ql = k - (1u << lam);
        tws[k] = tw[((size_t)1 << (a.l0 + lam)) + ((size_t)T << lam) + ql];
    }
    // gather the tile
    if (VEC) {
        constexpr u32 CV = CT >= 4 ? CT / 4 : 1;
        for (u32 it = threadIdx.x; it < R * CV; it += THREADS) {
            const u32 c4 = it % CV, rho = it / CV;
            const u32 i = ibase | (rho << lowbits);
            const u32 row = a.in_bitrev ? (__brev(i) >> brsh) : i;
            uint4 v = *reinterpret_cast<const uint4 *>(in + (size_t)row * a.w + col + 4 * c4);
            if (a.has_scale) {
                v.x = shoup_mul<F>(v.x, a.scale); v.y = shoup_mul<F>(v.y, a.scale);
                v.z = shoup_mul<F>(v.z, a.scale); v.w = shoup_mul<F>(v.w, a.scale);
            }
            *reinterpret_cast<uint4 *>(data + sidx<LOG_CT>(rho, 4 * c4)) = v;
        }
    } else {
        for (u32 it = threadIdx.x; it < (R << LOG_CT); it += THREADS) {
            const u32 c = it & (CT - 1), rho = it >> LOG_CT;
            const u32 i = ibase | (rho << lowbits);
            const u32 row = a.in_bitrev ? (__brev(i) >> brsh) : i;
            u32 v = in[(size_t)row * a.w + col + c];
            if (a.has_scale) v = shoup_mul<F>(v, a.scale);
            data[sidx<LOG_CT>(rho, c)] = v;
        }
    }
    __syncthreads();

    int lam0 = 0;
    const int q0 = (r & 3) ? (r & 3) : 4;
    switch (q0) {
        case 1: radix_step<F, LOG_CT, THREADS, 1>(data, tws, r, 0); break;
        case 2: radix_step<F, LOG_CT, THREADS, 2>(data, tws, r, 0); break;
        case 3: radix_step<F, LOG_CT, THREADS, 3>(data, tws, r, 0); break;
        default: radix_step<F, LOG_CT, THREADS, 4>(data, tws, r, 0); break;
    }
    for (lam0 = q0; lam0 < r; lam0 += 4) radix_step<F, LOG_CT, THREADS, 4>(data, tws, r, lam0);

    // scatter the tile
    if (VEC) {
        constexpr u32 CV = CT >= 4 ? CT / 4 : 1;
        for (u32 it = threadIdx.x; it < R * CV; it += THREADS) {
            const u32 c4 = it % CV, rho = it / CV;
            const u32 i = ibase | (rho << lowbits);
            const u32 row = ((a.out_bitrev ? (__brev(i) >> brsh) : i) << a.out_sh) + out_add;
            uint4 v = *reinterpret_cast<const uint4 *>(data + sidx<LOG_CT>(rho, 4 * c4));
            if (a.final_reduce) { v.x = fp_reduce<F>(v.x); v.y = fp_reduce<F>(v.y); v.z = fp_reduce<F>(v.z); v.w = fp_reduce<F>(v.w); }
            *reinterpret_cast<uint4 *>(out + (size_t)row * a.w + col + 4 * c4) = v;
        }
    } else {
        for (u32 it = threadIdx.x; it < (R << LOG_CT); it += THREADS) {
            const u32 c = it & (CT - 1), rho = it >> LOG_CT;
            const u32 i = ibase | (rho << lowbits);
            const u32 row = ((a.out_bitrev ? (__brev(i) >> brsh) : i) << a.out_sh) + out_add;
            u32 v = data[sidx<LOG_CT>(rho, c)];
            if (a.final_reduce) v = fp_reduce<F>(v);
            out[(size_t)row * a.w + col + c] = v;
        }
    }
}

// ---- fast path: the whole pass as TWO register networks with one shared-memory exchange ------------------------
// For 7 <= r <= 10 the r layers split as Q1 + Q2 (Q2 = ceil(r/2) <= 5).  Step 1 loads 2^Q1 rows per thread straight from
// global memory (stride 2^Q2 local rows), runs Q1 layers in registers and parks the results in shared memory; step 2
// reads 2^Q2 consecutive local rows, runs Q2 layers and stores straight to global memory.  Per element and pass that is
// one shared store + one shared load (the generic kernel does 2 per radix step plus the staging copy).
// Shared layout: local row rho, column c at (rho >> Q2) * gstride + (rho & (2^Q2-1)) * CT + c with gstride = 2^Q2*CT + pad,
// pad chosen so that gstride = CT (mod 32): both access patterns are bank-conflict free for ANY tile width CT, which lets
// one launch class take a non-power-of-two remainder tile (e.g. 100 = 5 x 16 + 20 columns) without sector over-fetch.
template <int Q> __host__ __device__ constexpr u32 brev_const(u32 m) {
    u32 r = 0;
    for (int b = 0; b < Q; b++) r |= ((m >> b) & 1u) << (Q - 1 - b);
    return r;
}

template <int F, int Q>
__device__ __forceinline__ void reg_network(u32 (&x)[1 << Q], const uint2 *tws, u32 node) {
    constexpr int E = 1 << Q;
#pragma unroll
    for (int j = 0; j < Q; j++) {
        const int half = E >> (j + 1);
#pragma unroll
        for (int grp = 0; grp < (1 << j); grp++) {
            const uint2 z = tws[(node << j) + grp];
#pragma unroll
            for (int t = 0; t < half; t++) ct_butterfly<F>(x[grp * 2 * half + t], x[grp * 2 * half + t + half], z);
        }
    }
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async4(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// Persistent pass kernel.  2-3 CTAs of 256 threads share an SM; each walks over tiles of 2^R_LOG rows x `ct` columns:
//   * the tile (rows as 16-byte cp.async/LDGSTS copies, plus its 2^R_LOG - 1 twiddles) streams into shared memory while
//     the other resident CTAs compute, so HBM latency overlaps the integer work;
//   * step 1 runs Q1 layers in registers IN PLACE in shared memory, step 2 runs Q2 layers and streams the results to
//     global memory (per-row TMA bulk stores were tried and rejected: UBLKCP is a warp-uniform instruction, so one
//     copy per lane serialises into a 32-iteration R2UR/PLOP3 loop per warp: +25 % instructions, profiles/README.md);
//   * all tiles of a pass have the same runtime width ct (16/20/24 columns; w = 100 -> 5 x 20) so that ONE launch covers
//     every column and neighbouring tiles share DRAM bursts through L2.
// Measured on the 2^20 x 100 LDE: 1.82 ms, vs 2.17 ms for one double-buffered 512-thread CTA per SM; block sizes 128/192/320/384
// give 1.88/1.82/1.91/1.92 ms.  Rejected experiments (profiles/README.md): two columns per thread with 64-bit shared accesses
// (2.01 ms), L2 prefetch of the next tile (1.99 ms), three passes of 7+7+6 layers with small tiles (3.1 ms).
constexpr int FAST_THREADS = 256;
template <int F, int R_LOG, int CT_T>   // CT_T: compile-time tile width (16/20/24) or 0 = runtime a.ct
__global__ void __launch_bounds__(FAST_THREADS, CT_T == 16 ? 3 : 2) ntt_pass_fast_kernel(const __grid_constant__ PassArgs a) {
    constexpr int THREADS = FAST_THREADS;
    constexpr int Q2 = (R_LOG + 1) / 2, Q1 = R_LOG - Q2;
    constexpr u32 E1 = 1u << Q1, E2 = 1u << Q2, R = 1u << R_LOG;
    const u32 CT = CT_T ? (u32)CT_T : a.ct;
    const u32 padw = (CT + 32u - ((E2 * CT) & 31u)) & 31u;
    const u32 gstride = E2 * CT + padw;
    const u32 buf_words = (E1 * gstride + 3u) & ~3u;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    u32 *data = reinterpret_cast<u32 *>(smem_raw);
    uint2 *tws = reinterpret_cast<uint2 *>(data + buf_words);

    const int lowbits = a.log_n - a.l1;
    const int brsh = 32 - a.log_n;
    const u32 n_row_tiles = 1u << (a.log_n - R_LOG);
    const u32 total = n_row_tiles * a.n_ctiles * a.n_cosets;
    const bool vec16 = a.vec16 != 0;       // row segments 16-byte aligned in global memory (loads AND stores)
    const bool shared_tw = (a.l0 == 0);    // first pass of a network: every tile uses the same twiddles

    auto decode = [&](u32 t, u32 &coset, u32 &col, u32 &cw, u32 &T, u32 &ibase) {
        coset = t % a.n_cosets;
        const u32 bx = t / a.n_cosets;
        const u32 ctile = bx % a.n_ctiles, tile = bx / a.n_ctiles;
        const u32 L = tile & ((1u << lowbits) - 1u);
        T = tile >> lowbits;
        col = ctile * CT;
        cw = min(CT, a.w - col);
        ibase = (a.l0 == 0 ? 0u : (T << (a.log_n - a.l0))) | L;
    };
    auto issue_twiddles = [&](u32 coset, u32 T) {
        const uint2 *tw = a.tw + (size_t)coset * a.tw_stride;
        for (u32 k = threadIdx.x + 1; k < R; k += THREADS) {
            const int lam = 31 - __clz(k);
            const u32 ql = k - (1u << lam);
            cp_async8(tws + k, tw + ((size_t)1 << (a.l0 + lam)) + ((size_t)T << lam) + ql);
        }
    };
    auto issue = [&](u32 t) {
        u32 coset, col, cw, T, ibase;
        decode(t, coset, col, cw, T, ibase);
        const u32 *in = a.in + (size_t)coset * a.in_stride + col;
        if (!shared_tw || a.n_cosets > 1) issue_twiddles(coset, T);
        // chunk = 16 bytes (4 columns) when aligned, else one element
        const u32 cpr = vec16 ? (cw >> 2) : cw;                  // chunks per row segment
        const u32 rs = (THREADS / cpr) & ~(E2 - 1u);             // rows per sweep: a multiple of E2 keeps the shared address linear
        const u32 nthr = rs * cpr;
        if (rs == 0) {
            // fewer than E2 whole rows per sweep (wide unaligned tiles): plain index arithmetic per chunk
            for (u32 it = threadIdx.x; it < R * cpr; it += THREADS) {
                const u32 rho = it / cpr, ch = it - rho * cpr;
                const u32 e = vec16 ? 4u * ch : ch;
                const u32 i = ibase | (rho << lowbits);
                const u32 row = a.in_bitrev ? (__brev(i) >> brsh) : i;
                u32 *dst = data + (rho >> Q2) * gstride + (rho & (E2 - 1u)) * CT + e;
                const u32 *src = in + (size_t)row * a.w + e;
                if (vec16) cp_async16(dst, src); else cp_async4(dst, src);
            }
        } else if (threadIdx.x < nthr) {
            const u32 rho0 = threadIdx.x / cpr, ch = threadIdx.x - rho0 * cpr;
            const u32 e = vec16 ? 4u * ch : ch;
            u32 *dst = data + (rho0 >> Q2) * gstride + (rho0 & (E2 - 1u)) * CT + e;
            const u32 dstep = (rs >> Q2) * gstride;
            if (!a.in_bitrev) {
                const u32 *src = in + (size_t)(ibase | (rho0 << lowbits)) * a.w + e;
                const size_t sstep = ((size_t)rs << lowbits) * a.w;
                for (u32 rho = rho0; rho < R; rho += rs, dst += dstep, src += sstep) {
                    if (vec16) cp_async16(dst, src); else cp_async4(dst, src);
                }
            } else {
                for (u32 rho = rho0; rho < R; rho += rs, dst += dstep) {
                    const u32 row = __brev(ibase | (rho << lowbits)) >> brsh;
                    const u32 *src = in + (size_t)row * a.w + e;
                    if (vec16) cp_async16(dst, src); else cp_async4(dst, src);
                }
            }
        }
        cp_async_commit();
    };

    u32 t = blockIdx.x;
    if (t >= total) return;
#ifdef P3GPU_NTT_PROFILE
    // 8 slots per (CTA, tile < 16): smid, t_start, t_issued, t_loaded, t_step1, t_step2 (globaltimer ns)
#define P3_STAMP(slot) do { if (a.prof && threadIdx.x == 0 && k < 16) { unsigned long long ts_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts_)); \
        a.prof[((size_t)blockIdx.x * 16 + k) * 8 + (slot)] = ts_; } } while (0)
#else
#define P3_STAMP(slot) do { } while (0)
#endif
    if (shared_tw && a.n_cosets == 1) issue_twiddles(0, 0);   // once per CTA, lands with the first tile's group
    for (u32 k = 0; t < total; t += gridDim.x, k++) {
        __syncthreads();   // every warp is done reading the buffer that is refilled next
#ifdef P3GPU_NTT_PROFILE
        if (a.prof && threadIdx.x == 0 && k < 16) { u32 sm_; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm_)); a.prof[((size_t)blockIdx.x * 16 + k) * 8] = sm_; }
#endif
        P3_STAMP(1);
        issue(t);   // other resident CTAs of this SM compute while this one waits for its tile
        P3_STAMP(2);
        cp_async_wait<0>();
        __syncthreads();
        P3_STAMP(3);
        u32 coset, col, cw, T, ibase;
        decode(t, coset, col, cw, T, ibase);
        const u32 dg = THREADS / cw, dc = THREADS - dg * cw;
        // ---- step 1 (in place in shared memory): item (g, c) holds local rows g + m*E2, m < E1
        {
            u32 g = threadIdx.x / cw, c = threadIdx.x - g * cw;
            for (; g < E2; ) {
                u32 *sp = data + g * CT + c;
                u32 x[E1];
#pragma unroll
                for (u32 m = 0; m < E1; m++) x[m] = sp[m * gstride];
                if (a.has_scale) {
#pragma unroll
                    for (u32 m = 0; m < E1; m++) x[m] = shoup_mul<F>(x[m], a.scale);
                }
                reg_network<F, Q1>(x, tws, 1u);
#pragma unroll
                for (u32 m = 0; m < E1; m++) sp[m * gstride] = x[m];
                c += dc; g += dg;
                if (c >= cw) { c -= cw; g++; }
            }
        }
        __syncthreads();
        P3_STAMP(4);
        // ---- step 2: item (g, c) holds local rows g*E2 + m, m < E2
        {
            u32 *out = a.out + (size_t)coset * a.out_stride + col;
            // out row(m) = ((row0 + K_m * S) << out_sh) + out_add: natural: K_m = m, S = 1 << lowbits;
            //                                                        bit-reversed: K_m = brev_Q2(m), S = 1 << (l0+Q1)
            const size_t sstride = ((size_t)(a.out_bitrev ? (1u << (a.l0 + Q1)) : (1u << lowbits)) << a.out_sh) * a.w;
            u32 g = threadIdx.x / cw, c = threadIdx.x - g * cw;
            for (; g < E1; ) {
                u32 *sp = data + g * gstride + c;
                u32 x[E2];
#pragma unroll
                for (u32 m = 0; m < E2; m++) x[m] = sp[m * CT];
                reg_network<F, Q2>(x, tws, E1 + g);
                if (a.final_reduce) {
#pragma unroll
                    for (u32 m = 0; m < E2; m++) x[m] = fp_reduce<F>(x[m]);
                }
                {
                    const u32 i0 = ibase | (g << (lowbits + Q2));
                    const u32 row0 = ((a.out_bitrev ? (__brev(i0) >> brsh) : i0) << a.out_sh) + a.out_add;
                    u32 *p = out + (size_t)row0 * a.w + c;
                    if (a.out_bitrev) {
#pragma unroll
                        for (u32 m = 0; m < E2; m++) p[brev_const<Q2>(m) * sstride] = x[m];
                    } else {
#pragma unroll
                        for (u32 m = 0; m < E2; m++) p[m * sstride] = x[m];
                    }
                }
                c += dc; g += dg;
                if (c >= cw) { c -= cw; g++; }
            }
        }
        P3_STAMP(5);
    }
}

// ---- pipelined path: TMA tile loads + warp-specialised consumer groups -------------------------------------------
// The cp.async kernel above spends ~5 of its ~17 us per tile issuing and waiting for its own loads (LDGSTS issue is
// back-pressured by HBM latency: ~20 KB in flight per CTA, tools/ntt_timeline.py), and only 2-3 CTAs fit an SM.  This kernel
// keeps ONE CTA per SM and decouples the two jobs:
//   * a producer lane walks the CTA's tile sequence and issues ONE 5-D tiled TMA copy per tile (cp.async.bulk.tensor) into a
//     ring of NSTAGE shared-memory stages, plus the tile row's 2^r - 1 twiddles as 1-D bulk copies; completion is signalled
//     on mbarriers, so up to NSTAGE - NGROUP tiles (~34 KB each) are always in flight per SM at zero issue cost;
//   * NGROUP independent consumer groups (GTHREADS threads, own named barrier) each take every NGROUP-th tile through the same
//     two register networks as above and release the stage as soon as their last shared-memory read is done.
// Tiles are 2^r rows x 8 columns (32-byte row segments = one sector).  The TMA box is (8 cols, GS + 1, NG): asking for one
// row more than the tensor has in the "row within group" dimension makes the copy engine zero-fill a padding row per group,
// which is exactly the skew (group stride = 8 mod 32 words) that keeps both register-network access patterns bank-conflict
// free; no other padding mechanism exists for a dense TMA box.
// A CTA processes all column tiles of one (row tile, coset) unit back to back, so the unit's twiddles are staged once and
// neighbouring 32-byte segments of the same rows are requested within microseconds of each other (L2/DRAM page locality).
// PERM = the pass reads its rows through the bit-reversal map (first forward pass of the LDE): the tile is then a CONTIGUOUS
// block of rows holding local row rho at position bitrev_r(rho); the two steps simply swap their shared-memory access shapes.
__device__ __forceinline__ void mbar_init(u32 bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_wait(u32 bar, u32 parity) {
    u32 done = 0, spins = 0;
    unsigned long long t0 = 0;
    while (true) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        // watchdog: a pass takes milliseconds; a wait of 20 s can only be a protocol error.  Trap (the launch fails with an error the
        // host reports) instead of leaving a hung kernel on the device.
        if ((++spins & 0xfffu) == 0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 20000000000ull) __trap();
        }
    }
}
__device__ __forceinline__ void mbar_arrive(u32 bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_arrive_n(u32 bar, u32 n) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(n) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(u32 bar, u32 bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory"); }

template <int F, int R_LOG, bool PERM, int NSTAGE, int NGROUP, int GTHREADS>
__global__ void __launch_bounds__(NGROUP * GTHREADS + 32, 1) ntt_pass_pipe_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ PassArgs a) {
    constexpr u32 CT = 8;
    constexpr int Q2 = (R_LOG + 1) / 2, Q1 = R_LOG - Q2;
    constexpr u32 E1 = 1u << Q1, E2 = 1u << Q2, R = 1u << R_LOG;
    constexpr u32 GS = PERM ? E1 : E2, NG = PERM ? E2 : E1;   // rows per group, groups per tile (see above)
    constexpr u32 gstride = (GS + 1) * CT;
    constexpr u32 STAGE_WORDS = NG * gstride;
    constexpr u32 BOX_BYTES = STAGE_WORDS * 4;
    static_assert(BOX_BYTES % 128 == 0, "stage alignment");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    u32 *stages = reinterpret_cast<u32 *>(smem_raw);
    uint2 *tws0 = reinterpret_cast<uint2 *>(smem_raw + (size_t)NSTAGE * BOX_BYTES);
    const u32 bar0 = (u32)__cvta_generic_to_shared(smem_raw + (size_t)NSTAGE * BOX_BYTES + 2 * R * sizeof(uint2));
    // barrier slots (8 bytes each): full[s] = s, empty[s] = NSTAGE + s, twfull[b] = 2 NSTAGE + b, twempty[b] = 2 NSTAGE + 2 + b
    auto full_bar = [&](u32 s) { return bar0 + 8u * s; };
    auto empty_bar = [&](u32 s) { return bar0 + 8u * (NSTAGE + s); };
    auto twfull_bar = [&](u32 b) { return bar0 + 8u * (2 * NSTAGE + b); };
    auto twempty_bar = [&](u32 b) { return bar0 + 8u * (2 * NSTAGE + 2 + b); };

    if (threadIdx.x == 0) {
        for (u32 s = 0; s < NSTAGE; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), NGROUP * GTHREADS); }
        for (u32 b = 0; b < 2; b++) { mbar_init(twfull_bar(b), 1); mbar_init(twempty_bar(b), a.tpi * NGROUP * GTHREADS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int lowbits = a.log_n - a.l1;
    const int brsh = 32 - a.log_n;
    auto decode = [&](u32 it, u32 &coset, u32 &L, u32 &T, u32 &ct0, u32 &ct1) {
        const u32 unit = it / a.csplit, chunk = it - unit * a.csplit;
        coset = unit % a.n_cosets;
        const u32 tile = unit / a.n_cosets;
        L = tile & ((1u << lowbits) - 1u);
        T = tile >> lowbits;
        ct0 = chunk * a.tpi;
        ct1 = min(ct0 + a.tpi, a.n_ctiles);
    };

    if (threadIdx.x >= NGROUP * GTHREADS) {
        // ---------------- producer ----------------
        if ((threadIdx.x & 31u) != 0) return;
        u32 q = 0, ui = 0;
        for (u32 it = blockIdx.x; it < a.n_items; it += gridDim.x, ui++) {
            u32 coset, L, T, ct0, ct1;
            decode(it, coset, L, T, ct0, ct1);
            const u32 b = ui & 1u, ph = (ui >> 1) & 1u;
            mbar_wait(twempty_bar(b), ph ^ 1u);   // every tile of unit ui-2 is done with this twiddle buffer
            if (ct1 - ct0 < a.tpi) mbar_arrive_n(twempty_bar(b), (a.tpi - (ct1 - ct0)) * NGROUP * GTHREADS);   // short last chunk
            {
                const uint2 *tw = a.tw + (size_t)coset * a.tw_stride;
                uint2 *tws = tws0 + b * R;
                tws[1] = tw[((size_t)1 << a.l0) + T];   // layer lam = 0 has a single 8-byte entry: too small for a bulk copy
                mbar_expect_tx(twfull_bar(b), 8u * (R - 2u));
#pragma unroll 1
                for (int lam = 1; lam < R_LOG; lam++) {
                    const uint2 *src = tw + ((size_t)1 << (a.l0 + lam)) + ((size_t)T << lam);
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"((u32)__cvta_generic_to_shared(tws + (1u << lam))), "l"(src), "r"(8u << lam), "r"(twfull_bar(b)) : "memory");
                }
            }
            // tensor coordinates: (column, 0, 0, c3, c4); see make_pass_tensor_map
            // tiled input: column tile ct, block cb is the 8-column matrix number ct * in_blocks + cb (blocks fold into dim 4)
            const u32 in_block = (a.in_tiled ? a.in_blocks > 1 : a.in_stride != 0) ? coset : 0u;
            const int blk_sh = PERM ? lowbits : a.l0;   // dim-4 coordinates per 2^log_n-row block
            const int c3 = PERM ? 0 : (int)L;
            const int c4 = (PERM ? (lowbits ? (int)(__brev(L) >> (32 - lowbits)) : 0) : (int)T) + (int)(in_block << blk_sh);
            for (u32 ct = ct0; ct < ct1; ct++, q++) {
                const u32 s = q % NSTAGE, k = q / NSTAGE;
                mbar_wait(empty_bar(s), (k & 1u) ^ 1u);
                mbar_expect_tx(full_bar(s), BOX_BYTES);
                const int cc0 = a.in_tiled ? 0 : (int)(ct * CT);
                const int cc4 = a.in_tiled ? c4 + (int)((ct * a.in_blocks) << blk_sh) : c4;
                asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
                             ::"r"((u32)__cvta_generic_to_shared(stages + (size_t)s * STAGE_WORDS)), "l"(reinterpret_cast<unsigned long long>(&tmap)),
                               "r"(cc0), "r"(0), "r"(0), "r"(c3), "r"(cc4), "r"(full_bar(s)) : "memory");
            }
        }
        return;
    }

    // ---------------- consumers ----------------
    const u32 gid = threadIdx.x / GTHREADS, tg = threadIdx.x - gid * GTHREADS;
    u32 q = 0, ui = 0;
#ifdef P3GPU_NTT_PROFILE
    u32 kk = 0;   // tiles taken by this group; 8 slots per (CTA, group, tile < 16): smid, t_start, t_full, t_step1, t_step2
#define P3_GSTAMP(slot) do { if (a.prof && tg == 0 && kk < 16) { unsigned long long ts_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts_)); \
        a.prof[(((size_t)blockIdx.x * NGROUP + gid) * 16 + kk) * 8 + (slot)] = ts_; } } while (0)
#else
#define P3_GSTAMP(slot) do { } while (0)
#endif
    for (u32 it = blockIdx.x; it < a.n_items; it += gridDim.x, ui++) {
        u32 coset, L, T, ct0, ct1;
        decode(it, coset, L, T, ct0, ct1);
        const u32 b = ui & 1u, ph = (ui >> 1) & 1u;
        const uint2 *tws = tws0 + b * R;
        const u32 ibase = (a.l0 == 0 ? 0u : (T << (a.log_n - a.l0))) | L;
        bool tw_ready = false;
        for (u32 ct = ct0; ct < ct1; ct++, q++) {
            const u32 s = q % NSTAGE, k = q / NSTAGE;
            const u32 col = ct * CT, cw = min(CT, a.wc - col);
            u32 *data = stages + (size_t)s * STAGE_WORDS;
            P3_GSTAMP(1);
            // EVERY group waits for EVERY tile and twiddle buffer in sequence order, also those it does not process, and only then
            // lets the ring advance (empty[s] / twempty[b] count all consumer threads).  A parity wait can only tell the current
            // mbarrier phase from the one before it; a group that skipped a stage's previous use could otherwise run ahead of a
            // load that is still in flight and take the older phase for the one it wants (seen with 128-row tiles, which are
            // processed faster than HBM latency varies: corrupted arrival counts, i.e. hangs and mbarrier traps).
            mbar_wait(full_bar(s), k & 1u);
            if (!tw_ready) { mbar_wait(twfull_bar(b), ph); tw_ready = true; }
            if (q % NGROUP != gid) {
                mbar_arrive(empty_bar(s));
                mbar_arrive(twempty_bar(b));
                continue;
            }
            P3_GSTAMP(2);
            const u32 dg = GTHREADS / cw, dc = GTHREADS - dg * cw;
            // ---- step 1 (in place): E1 values per item, Q1 layers
            {
                u32 g = tg / cw, c = tg - g * cw;
                for (; g < E2; ) {
                    u32 x[E1];
                    if (!PERM) {
                        u32 *sp = data + g * CT + c;           // local rows g + m*E2
#pragma unroll
                        for (u32 m = 0; m < E1; m++) x[m] = sp[m * gstride];
                        if (a.has_scale) {
#pragma unroll
                            for (u32 m = 0; m < E1; m++) x[m] = shoup_mul<F>(x[m], a.scale);
                        }
                        reg_network<F, Q1>(x, tws, 1u);
#pragma unroll
                        for (u32 m = 0; m < E1; m++) sp[m * gstride] = x[m];
                    } else {
                        u32 *sp = data + g * gstride + c;      // g = gamma: local rows bitrev_Q2(gamma) + m*E2 sit in group gamma
#pragma unroll
                        for (u32 m = 0; m < E1; m++) x[m] = sp[brev_const<Q1>(m) * CT];
                        if (a.has_scale) {
#pragma unroll
                            for (u32 m = 0; m < E1; m++) x[m] = shoup_mul<F>(x[m], a.scale);
                        }
                        reg_network<F, Q1>(x, tws, 1u);
#pragma unroll
                        for (u32 m = 0; m < E1; m++) sp[brev_const<Q1>(m) * CT] = x[m];
                    }
                    c += dc; g += dg;
                    if (c >= cw) { c -= cw; g++; }
                }
            }
            asm volatile("bar.sync %0, %1;" ::"r"(gid + 1u), "r"((u32)GTHREADS) : "memory");
            P3_GSTAMP(3);
            // ---- step 2: E2 values per item, Q2 layers, results straight to global memory
            {
                // dense output: row pitch w, this tile at column col of coset block `coset`;
                // tiled output: 8-column matrix number ct * n_cosets + coset, row pitch 8
                const u32 ow = a.out_tiled ? CT : a.w;
                u32 *out = a.out_tiled ? a.out + ((((size_t)ct * a.n_cosets + coset) << a.log_n) << 3) : a.out + (size_t)coset * a.out_stride + col;
                const size_t sstride = ((size_t)(a.out_bitrev ? (1u << (a.l0 + Q1)) : (1u << lowbits)) << a.out_sh) * ow;
                u32 g = tg / cw, c = tg - g * cw;
                bool released = false;
                for (; g < E1; ) {
                    u32 x[E2];
                    u32 gg;   // item = local rows gg*E2 + m
                    if (!PERM) {
                        gg = g;
                        const u32 *sp = data + g * gstride + c;
#pragma unroll
                        for (u32 m = 0; m < E2; m++) x[m] = sp[m * CT];
                    } else {
                        gg = __brev(g) >> (32 - Q1);
                        const u32 *sp = data + g * CT + c;
#pragma unroll
                        for (u32 m = 0; m < E2; m++) x[m] = sp[brev_const<Q2>(m) * gstride];
                    }
                    u32 gn = g + dg, cn = c + dc;
                    if (cn >= cw) { cn -= cw; gn++; }
                    if (gn >= E1) {   // last shared-memory read of this thread for this stage: hand it back to the producer
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        mbar_arrive(empty_bar(s));
                        released = true;
                    }
                    reg_network<F, Q2>(x, tws, E1 + gg);
                    if (a.final_reduce) {
#pragma unroll
                        for (u32 m = 0; m < E2; m++) x[m] = fp_reduce<F>(x[m]);
                    }
                    const u32 i0 = ibase | (gg << (lowbits + Q2));
                    const u32 row0 = ((a.out_bitrev ? (__brev(i0) >> brsh) : i0) << a.out_sh) + a.out_add;
                    u32 *p = out + (size_t)row0 * ow + c;
                    if (a.out_bitrev) {
#pragma unroll
                        for (u32 m = 0; m < E2; m++) p[brev_const<Q2>(m) * sstride] = x[m];
                    } else {
#pragma unroll
                        for (u32 m = 0; m < E2; m++) p[m * sstride] = x[m];
                    }
                    g = gn; c = cn;
                }
                if (!released) {   // threads without a step-2 item (ragged tile)
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    mbar_arrive(empty_bar(s));
                }
            }
            mbar_arrive(twempty_bar(b));
            P3_GSTAMP(4);
#ifdef P3GPU_NTT_PROFILE
            kk++;
#endif
        }
    }
}

// ---- twiddle heaps ---------------------------------------------------------------------------
struct TwGenArgs {
    u32 sigma[32];  // sigma[l] = shift^(N/2^(l+1)), Montgomery
    u32 roots[32];  // roots[k] = primitive 2^k-th root (or its inverse), Montgomery
};
template <int F> __global__ void gen_twiddle_heap(uint2 *Z, int log_n, const TwGenArgs a) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ((size_t)1 << log_n)) return;
    if (idx == 0) { Z[0] = make_uint2(0, 0); return; }
    const int l = 63 - __clzll((long long)idx);
    const u32 q = (u32)(idx - ((size_t)1 << l));
    u32 z = a.sigma[l];
    for (int b = 0; b < l; b++)
        if ((q >> b) & 1u) z = mont_mul<F>(z, a.roots[b + 2]);
    Z[idx] = shoup_pair<F>(from_monty<F>(z));
}

// row i *= base^i  (dft/src/util.rs:32-55 coset_shift_cols), used by coset_idft_batch only
struct PowArgs { u32 pw[32]; };  // pw[k] = base^(2^k), Montgomery
template <int F> __global__ void scale_rows_by_powers(u32 *m, size_t h, size_t w, const PowArgs a) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= h * w) return;
    size_t row = idx / w;
    u32 s = Fp<F>::ONE;
    for (int k = 0; row; k++, row >>= 1)
        if (row & 1) s = mont_mul<F>(s, a.pw[k]);
    m[idx] = mont_mul<F>(m[idx], s);
}
__global__ void broadcast_row(const u32 *in, u32 *out, size_t rows, size_t w) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < rows * w) out[idx] = in[idx % w];
}

// Heap(s) for the size-2^log_n network.  added_bits = 0: one heap for (shift, inverse).  added_bits > 0 (LDE): 2^added_bits
// heaps back to back, block cb for the coset shift * g_big^bitrev(cb).
template <int F>
static int32_t get_twiddles(p3gpu_ctx *ctx, int log_n, int added_bits, u32 shift, int inverse, const uint2 **out) {
    TwiddleKey key{F, log_n, shift, inverse + 2 * added_bits};
    std::lock_guard<std::recursive_mutex> g(ctx->call_mu);   // entry points already hold it; kept for internal callers
    {
        auto it = ctx->twiddles.find(key);
        if (it != ctx->twiddles.end()) { it->second.last_use = ctx->tick; *out = it->second.ptr; return P3GPU_OK; }
    }
    const size_t N = (size_t)1 << log_n, n_cosets = (size_t)1 << added_bits;
    const size_t bytes = n_cosets * N * sizeof(uint2);
    // bounded cache (the reference's map grows without bound; a long-lived prover with many shifts/sizes must not): evict
    // least-recently-used heaps that no call of the current entry point has touched until the new heap fits
    while (ctx->twiddle_bytes + bytes > ctx->twiddle_cap_bytes) {
        auto victim = ctx->twiddles.end();
        for (auto it = ctx->twiddles.begin(); it != ctx->twiddles.end(); ++it)
            if (it->second.last_use < ctx->tick && (victim == ctx->twiddles.end() || it->second.last_use < victim->second.last_use)) victim = it;
        if (victim == ctx->twiddles.end()) break;          // everything left is in use by this call: exceed the cap rather than fail
        P3_CUDA(cudaStreamSynchronize(ctx->stream));       // queued kernels may still read the heap
        P3_CUDA(cudaFree(victim->second.ptr));
        ctx->twiddle_bytes -= victim->second.bytes;
        ctx->twiddles.erase(victim);
    }
    uint2 *Z = nullptr;
    {
        cudaError_t e = cudaMalloc(&Z, bytes);
        if (e != cudaSuccess) { set_error("cudaMalloc(%zu) for a twiddle heap failed: %s", bytes, cudaGetErrorString(e)); cudaGetLastError(); return P3GPU_ENOMEM; }
    }
    const u32 g_big = two_adic_generator<F>((u32)(log_n + added_bits));
    for (size_t cb = 0; cb < n_cosets; cb++) {
        size_t c = 0;
        for (int b = 0; b < added_bits; b++) c |= ((cb >> b) & 1) << (added_bits - 1 - b);
        const u32 s = mont_mul<F>(shift, fp_pow<F>(g_big, c));
        TwGenArgs a;
        for (int l = 0; l < 32; l++) { a.sigma[l] = Fp<F>::ONE; a.roots[l] = Fp<F>::ONE; }
        for (int l = 0; l < log_n; l++) a.sigma[l] = fp_pow<F>(s, (u64)(N >> (l + 1)));
        for (u32 k = 0; k <= (u32)log_n && k <= Fp<F>::TWO_ADICITY; k++) {
            u32 gk = two_adic_generator<F>(k);
            a.roots[k] = inverse ? fp_inv<F>(gk) : gk;
        }
        const unsigned blocks = (unsigned)((N + 255) / 256);
        gen_twiddle_heap<F><<<blocks, 256, 0, ctx->stream>>>(Z + cb * N, log_n, a);
        ctx->launches++;
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { cudaFree(Z); set_error("gen_twiddle_heap launch failed: %s", cudaGetErrorString(e)); return P3GPU_ECUDA; }
    }
    ctx->twiddles.emplace(key, TwiddleEntry{Z, bytes, ctx->tick});
    ctx->twiddle_bytes += bytes;
    *out = Z;
    return P3GPU_OK;
}

template <int F, int LOG_CT, bool VEC>
static int32_t launch_pass_ct(p3gpu_ctx *ctx, const PassArgs &a) {
    constexpr int THREADS = 256;
    const int r = a.l1 - a.l0;
    const size_t smem = (((size_t)1 << r) << LOG_CT) * 4 + ((size_t)1 << r) * sizeof(uint2);
    auto kern = ntt_pass_kernel<F, LOG_CT, THREADS, VEC>;
    if (smem > 48 * 1024) P3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const size_t tiles = ((size_t)1 << (a.log_n - r)) * a.n_ctiles * a.n_cosets;
    P3_CHECK(tiles < (1ull << 31), P3GPU_EINVAL, "ntt: grid too large");
    kern<<<(unsigned)tiles, THREADS, smem, ctx->stream>>>(a);
    ctx->launches++;
    P3_CUDA(cudaGetLastError());
    return P3GPU_OK;
}

template <int F, int R_LOG, int CT_T>
static int32_t launch_fast_rc(p3gpu_ctx *ctx, const PassArgs &a) {
    constexpr int THREADS = FAST_THREADS;
    constexpr int Q2 = (R_LOG + 1) / 2, Q1 = R_LOG - Q2;
    const u32 ct = a.ct;
    const u32 e2 = 1u << Q2, e1 = 1u << Q1;
    const u32 padw = (ct + 32u - ((e2 * ct) & 31u)) & 31u;
    const size_t buf_words = ((size_t)e1 * (e2 * ct + padw) + 3) & ~(size_t)3;
    const size_t smem = buf_words * 4 + ((size_t)1 << R_LOG) * sizeof(uint2);
    auto kern = ntt_pass_fast_kernel<F, R_LOG, CT_T>;
    P3_CHECK(smem <= 227 * 1024, P3GPU_EINVAL, "ntt: tile does not fit shared memory");
    static size_t smem_set[64] = {0};   // per instantiation and device: raise the dynamic shared memory limit once per size
    if (smem > 48 * 1024 && smem > smem_set[ctx->device & 63]) {
        P3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set[ctx->device & 63] = smem;
    }
    const size_t tiles = ((size_t)1 << (a.log_n - R_LOG)) * a.n_ctiles * a.n_cosets;
    P3_CHECK(tiles < (1ull << 31), P3GPU_EINVAL, "ntt: grid too large");
    // persistent grid: as many CTAs per SM as the shared memory and the register file hold (one loads its tile while the others compute)
    size_t per_sm = std::min<size_t>(2048 / THREADS, (227 * 1024) / (smem + 1024));
    static int num_regs = 0;   // per instantiation; benign race (same value)
    if (num_regs == 0) {
        cudaFuncAttributes fa;
        P3_CUDA(cudaFuncGetAttributes(&fa, kern));
        num_regs = std::max(fa.numRegs, 16);
    }
    const size_t by_regs = 65536 / ((size_t)THREADS * (size_t)num_regs);   // register file of the SM
    if (per_sm > by_regs) per_sm = by_regs;
    if (per_sm < 1) per_sm = 1;
    const size_t grid = std::min(tiles, per_sm * (size_t)ctx->sm_count);
    kern<<<(unsigned)grid, THREADS, smem, ctx->stream>>>(a);
    ctx->launches++;
    P3_CUDA(cudaGetLastError());
    return P3GPU_OK;
}
template <int F, int R_LOG>
static int32_t launch_fast_r(p3gpu_ctx *ctx, const PassArgs &a) {
    switch (a.ct) {   // compile-time widths keep every shared-memory offset an immediate
        case 16: return launch_fast_rc<F, R_LOG, 16>(ctx, a);
        case 20: return launch_fast_rc<F, R_LOG, 20>(ctx, a);
        case 24: return launch_fast_rc<F, R_LOG, 24>(ctx, a);
        default: return launch_fast_rc<F, R_LOG, 0>(ctx, a);
    }
}
template <int F>
static int32_t launch_fast(p3gpu_ctx *ctx, const PassArgs &a) {
    switch (a.l1 - a.l0) {
        case 6: return launch_fast_r<F, 6>(ctx, a);
        case 7: return launch_fast_r<F, 7>(ctx, a);
        case 8: return launch_fast_r<F, 8>(ctx, a);
        case 9: return launch_fast_r<F, 9>(ctx, a);
        default: return launch_fast_r<F, 10>(ctx, a);
    }
}

// ---- pipelined kernel: host side -------------------------------------------------------------------------------
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                      const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TensorMapEncodeFn tensor_map_encoder() {
    static TensorMapEncodeFn fn = []() -> TensorMapEncodeFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<TensorMapEncodeFn>(p);
    }();
    return fn;
}

// 5-D view of the pass input for ntt_pass_pipe_kernel: (column, row-in-group, group, L, T) with the tile's local row
// rho = group * GS + row-in-group at global row  T * 2^(n-l0) + rho * 2^lowbits + L   (PERM: block * 2^r + position).
static int32_t make_pass_tensor_map(const PassArgs &a, bool perm, CUtensorMap *tm) {
    TensorMapEncodeFn enc = tensor_map_encoder();
    P3_CHECK(enc != nullptr, P3GPU_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const int r = a.l1 - a.l0, q2 = (r + 1) / 2, q1 = r - q2, lowbits = a.log_n - a.l1;
    const cuuint64_t pitch = a.in_tiled ? 32 : (cuuint64_t)a.w * 4;
    const cuuint64_t n_ctiles = (a.wc + 7) / 8;
    cuuint64_t dims[5], strides[4];
    cuuint32_t box[5] = {8, 0, 0, 1, 1}, es[5] = {1, 1, 1, 1, 1};
    dims[0] = a.in_tiled ? 8 : a.wc;
    const cuuint64_t in_blocks = a.in_tiled ? n_ctiles * a.in_blocks : (a.in_stride ? a.n_cosets : 1);
    if (!perm) {
        dims[1] = 1ull << q2; dims[2] = 1ull << q1; dims[3] = 1ull << lowbits; dims[4] = in_blocks << a.l0;
        strides[0] = pitch << lowbits; strides[1] = pitch << (lowbits + q2); strides[2] = pitch; strides[3] = pitch << (a.log_n - a.l0);
        box[1] = (1u << q2) + 1; box[2] = 1u << q1;
    } else {
        dims[1] = 1ull << q1; dims[2] = 1ull << q2; dims[3] = 1; dims[4] = in_blocks << (a.log_n - r);
        strides[0] = pitch; strides[1] = pitch << q1; strides[2] = pitch; strides[3] = pitch << r;
        box[1] = (1u << q1) + 1; box[2] = 1u << q2;
    }
    const CUresult rc = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, const_cast<u32 *>(a.in), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    P3_CHECK(rc == CUDA_SUCCESS, P3GPU_ECUDA, "cuTensorMapEncodeTiled failed (%d)", (int)rc);
    return P3GPU_OK;
}

static bool pipe_eligible(const PassArgs &a) {
    if (!env_int("P3GPU_NTT_PIPE", 1)) return false;   // read per call: the tests switch between the two kernel families
    const int r = a.l1 - a.l0;
    if (r < 6 || r > 10) return false;
    if (a.in_tiled || a.out_tiled) return true;                                 // set up by lde_tiled_impl, which checked
    if (a.w % 4 != 0 || a.w < 8 || a.w > 8192) return false;                    // TMA: 16-byte global strides; mbarrier count per unit
    if (reinterpret_cast<uintptr_t>(a.in) % 16 != 0) return false;
    if ((((size_t)a.w * 4) << a.log_n) >= (1ull << 40)) return false;           // TMA stride limit
    if (a.in_stride != 0 && a.in_stride != ((size_t)a.w << a.log_n)) return false;
    if (a.in_bitrev && (a.l0 != 0 || (a.in_stride != 0 && a.n_cosets > 1))) return false;
    return true;
}

template <int F, int R_LOG, bool PERM>
static int32_t launch_pipe_r(p3gpu_ctx *ctx, PassArgs a) {
    constexpr int NSTAGE = 6, NGROUP = 4, GTHREADS = 128;
    constexpr int Q2 = (R_LOG + 1) / 2, Q1 = R_LOG - Q2;
    constexpr size_t GS = PERM ? (1u << Q1) : (1u << Q2), NG = PERM ? (1u << Q2) : (1u << Q1);
    constexpr size_t box_bytes = NG * (GS + 1) * 8 * 4;
    constexpr size_t smem = NSTAGE * box_bytes + 2 * ((size_t)1 << R_LOG) * sizeof(uint2) + (2 * NSTAGE + 4) * 8;
    static_assert(smem <= 227 * 1024, "pipelined NTT kernel: shared memory budget");
    CUtensorMap tm;
    if (a.wc == 0) a.wc = a.w;
    if (a.in_blocks == 0) a.in_blocks = 1;
    P3_TRY(make_pass_tensor_map(a, PERM, &tm));
    a.n_ctiles = (a.wc + 7) / 8;
    const size_t units = ((size_t)1 << (a.log_n - R_LOG)) * a.n_cosets;
    // few units (small transforms): split a unit's column tiles over several CTAs so that every SM has work
    size_t csplit = units >= 2 * (size_t)ctx->sm_count ? 1 : std::min<size_t>(a.n_ctiles, (2 * (size_t)ctx->sm_count + units - 1) / units);
    a.tpi = (u32)((a.n_ctiles + csplit - 1) / csplit);
    csplit = (a.n_ctiles + a.tpi - 1) / a.tpi;
    a.csplit = (u32)csplit;
    const size_t items = units * csplit;
    P3_CHECK(items < (1ull << 31), P3GPU_EINVAL, "ntt: too many tiles");
    P3_CHECK((size_t)a.tpi * NGROUP * GTHREADS < (1u << 20), P3GPU_EINVAL, "ntt: too many column tiles per unit for the mbarrier count");
    a.n_items = (u32)items;
    auto kern = ntt_pass_pipe_kernel<F, R_LOG, PERM, NSTAGE, NGROUP, GTHREADS>;
    static bool attr_set[64] = {false};
    if (!attr_set[ctx->device & 63]) {
        P3_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[ctx->device & 63] = true;
    }
    const size_t grid = std::min(items, (size_t)ctx->sm_count);
    kern<<<(unsigned)grid, NGROUP * GTHREADS + 32, smem, ctx->stream>>>(tm, a);
    ctx->launches++;
    P3_CUDA(cudaGetLastError());
    return P3GPU_OK;
}
template <int F, int R_LOG>
static int32_t launch_pipe_p(p3gpu_ctx *ctx, const PassArgs &a) {
    return a.in_bitrev ? launch_pipe_r<F, R_LOG, true>(ctx, a) : launch_pipe_r<F, R_LOG, false>(ctx, a);
}
template <int F>
static int32_t launch_pipe(p3gpu_ctx *ctx, const PassArgs &a) {
    switch (a.l1 - a.l0) {
        case 6: return launch_pipe_p<F, 6>(ctx, a);
        case 7: return launch_pipe_p<F, 7>(ctx, a);
        case 8: return launch_pipe_p<F, 8>(ctx, a);
        case 9: return launch_pipe_p<F, 9>(ctx, a);
        default: return launch_pipe_p<F, 10>(ctx, a);
    }
}

// Column tile width of the fast kernel: all tiles of a launch share one width (a ragged last tile is allowed).
// Prefer exact divisors that keep 16-byte alignment (16, 20, 24 columns = 64/80/96-byte row segments).
static u32 choose_tile_width(u32 w) {
    if (w <= 24) return w;
    for (u32 ct : {16u, 20u, 24u, 12u})
        if (w % ct == 0) return ct;
    const u32 n = (w + 19) / 20;                 // ~20 columns per tile, nearly equal tiles
    u32 ct = (w + n - 1) / n;
    ct = (ct + 3) & ~3u;
    return ct > 24 ? 24 : ct;
}

// One pass over all columns.
//   fast path (7 <= r <= 10): ONE launch, tiles of choose_tile_width(w) columns (16/20/24; ragged last tile allowed).
//   generic path: columns are split greedily into power-of-two tiles of 16, 8, 4, 2, 1 columns.
template <int F>
static int32_t launch_pass(p3gpu_ctx *ctx, PassArgs a, unsigned n_cosets) {
    a.n_cosets = n_cosets;
    const int r = a.l1 - a.l0;
#ifdef P3GPU_NTT_PROFILE
    {   // each launch gets its own 1 MiB window of the timeline buffer
        static int launch_no = 0;
        const char *pb = getenv("P3GPU_NTT_PROFBUF");
        a.prof = pb ? reinterpret_cast<unsigned long long *>(strtoull(pb, nullptr, 0)) + (size_t)(launch_no++ % 8) * (1u << 17) : nullptr;
    }
#endif
    if (pipe_eligible(a)) return launch_pipe<F>(ctx, a);
    if (r >= 6 && r <= 10) {
        const u32 ct = choose_tile_width(a.w);
        // 16-byte cp.async / TMA bulk stores need every row segment of every tile 16-byte aligned on both sides
        const bool al16 = (a.w % 4 == 0) && (ct % 4 == 0) &&
                          ((reinterpret_cast<uintptr_t>(a.in) | reinterpret_cast<uintptr_t>(a.out)) % 16 == 0) &&
                          ((a.in_stride | a.out_stride) % 4 == 0);
        a.col0 = 0; a.ct = ct; a.n_ctiles = (a.w + ct - 1) / ct; a.vec16 = al16;
        return launch_fast<F>(ctx, a);
    }
    const bool aligned = (a.w % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.in) | reinterpret_cast<uintptr_t>(a.out)) % 16 == 0) &&
                         ((a.in_stride | a.out_stride) % 4 == 0);
    u32 col = 0, rem = a.w;
    for (int lct = 4; lct >= 0 && rem; lct--) {
        const u32 ct = 1u << lct;
        const u32 n = rem >> lct;
        if (!n) continue;
        a.col0 = col; a.n_ctiles = n; a.ct = ct;
        const bool vec = aligned && lct >= 2 && (col % 4 == 0);
        int32_t rc;
        switch (lct) {
            case 4: rc = vec ? launch_pass_ct<F, 4, true>(ctx, a) : launch_pass_ct<F, 4, false>(ctx, a); break;
            case 3: rc = vec ? launch_pass_ct<F, 3, true>(ctx, a) : launch_pass_ct<F, 3, false>(ctx, a); break;
            case 2: rc = vec ? launch_pass_ct<F, 2, true>(ctx, a) : launch_pass_ct<F, 2, false>(ctx, a); break;
            case 1: rc = launch_pass_ct<F, 1, false>(ctx, a); break;
            default: rc = launch_pass_ct<F, 0, false>(ctx, a); break;
        }
        P3_TRY(rc);
        col += n * ct; rem -= n * ct;
    }
    return P3GPU_OK;
}

struct NetworkPlan {
    int n_passes;
    int bounds[8];  // layer boundaries: pass k covers [bounds[k], bounds[k+1])
};
// as few passes as possible of at most 10 layers each (the deepest pass the pass kernels are instantiated for), layers spread evenly
static NetworkPlan plan_passes(int log_n) {
    constexpr int max_r = 10;
    NetworkPlan p;
    p.n_passes = (log_n + max_r - 1) / max_r;
    if (p.n_passes < 1) p.n_passes = 1;
    int base = log_n / p.n_passes, extra = log_n % p.n_passes;
    p.bounds[0] = 0;
    for (int k = 0; k < p.n_passes; k++) p.bounds[k + 1] = p.bounds[k] + base + (k < extra ? 1 : 0);
    return p;
}

// Runs the size-2^log_n network on n_cosets (input, output, twiddle heap) triples laid out at fixed strides.
//   src: input rows, natural order unless in_bitrev (then element i of the network is read from row bitrev(i))
//   dst: output.  Default: network order (row i = network position i).  With out_bitrev / out_sh / out_add the last pass
//        writes position i to row (bitrev(i) << out_sh) + out_add, i.e. natural order (optionally interleaved);
//        that remap cannot run in place, so multi-pass plans then keep intermediate data in tmp (h*w words per coset).
template <int F>
static int32_t run_network(p3gpu_ctx *ctx, int log_n, size_t w, const uint2 *tw, size_t tw_stride, unsigned n_cosets,
                           const u32 *src, size_t src_stride, int in_bitrev, u32 *dst, size_t dst_stride, int out_bitrev,
                           int out_sh, u32 out_add, u32 *tmp, bool has_scale, uint2 scale, bool final_reduce) {
    const NetworkPlan plan = plan_passes(log_n);
    const bool remap = out_bitrev || out_sh != 0 || out_add != 0;
    const size_t hw = ((size_t)1 << log_n) * w;
    if (remap && plan.n_passes > 1) P3_CHECK(tmp != nullptr, P3GPU_EINVAL, "ntt: scratch missing");
    for (int k = 0; k < plan.n_passes; k++) {
        PassArgs a;
        memset(&a, 0, sizeof a);
        const bool first = (k == 0), last = (k == plan.n_passes - 1);
        a.w = (u32)w; a.log_n = log_n; a.l0 = plan.bounds[k]; a.l1 = plan.bounds[k + 1];
        a.tw = tw; a.tw_stride = tw_stride;
        u32 *mid = remap ? tmp : dst;
        const size_t mid_stride = remap ? hw : dst_stride;
        a.in = first ? src : mid;
        a.in_stride = first ? src_stride : mid_stride;
        a.in_bitrev = first ? in_bitrev : 0;
        if (last) {
            a.out = dst; a.out_stride = dst_stride;
            a.out_bitrev = out_bitrev; a.out_sh = out_sh; a.out_add = out_add;
            a.final_reduce = final_reduce;
        } else {
            a.out = mid; a.out_stride = mid_stride;
        }
        if (first) { a.has_scale = has_scale; a.scale = scale; }
        P3_TRY(launch_pass<F>(ctx, a, n_cosets));
    }
    return P3GPU_OK;
}

template <int F> static uint2 inv_height_scale(size_t h) {
    return shoup_pair<F>(from_monty<F>(fp_inv<F>(to_monty<F>((u32)(h % Fp<F>::P)))));
}

template <int F>
static int32_t dft_batch_impl(p3gpu_ctx *ctx, int kind, const u32 *d_in, u32 *d_out, size_t h, size_t w, u32 shift) {
    const int log_n = (int)log2_floor(h);
    if (log_n == 0) {  // size-1 transform is the identity for every kind
        if (d_in != d_out) P3_CUDA(cudaMemcpyAsync(d_out, d_in, w * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        return P3GPU_OK;
    }
    const bool inverse = (kind == P3GPU_IDFT || kind == P3GPU_COSET_IDFT);
    const u32 tw_shift = (kind == P3GPU_COSET_DFT) ? shift : Fp<F>::ONE;
    const uint2 *tw = nullptr;
    P3_TRY(get_twiddles<F>(ctx, log_n, 0, tw_shift, inverse, &tw));
    void *tmp = nullptr;
    P3_TRY(ctx_scratch(ctx, h * w * 4, &tmp));
    P3_TRY(run_network<F>(ctx, log_n, w, tw, 0, 1, d_in, 0, 0, d_out, 0, /*out_bitrev=*/1, 0, 0, (u32 *)tmp, inverse,
                          inverse ? inv_height_scale<F>(h) : make_uint2(0, 0), true));
    if (kind == P3GPU_COSET_IDFT) {  // traits.rs:145-155: coefficient i *= shift^-i
        PowArgs pa;
        u32 b = fp_inv<F>(shift);
        for (int k = 0; k < 32; k++) { pa.pw[k] = b; b = mont_mul<F>(b, b); }
        const size_t n = h * w;
        scale_rows_by_powers<F><<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_out, h, w, pa);
        ctx->launches++;
        P3_CUDA(cudaGetLastError());
    }
    return P3GPU_OK;
}

// coset_lde_batch (bit-reversed output rows) on the pipelined kernel with COLUMN-TILE-MAJOR intermediates.
// Between passes the data lives as one 8-column matrix (32-byte rows) per column tile and coset ("tiled" layout): every
// 32-byte row segment a pass touches is then one aligned DRAM sector, and the contiguous passes stream whole 32 KB tiles.
// In the caller's dense layout a 400-byte pitch (w = 100) puts every odd row's segments across two sectors, which cost the
// strided passes ~30 % (profiles/README.md).  Only the first pass (TMA reads) and the last pass (contiguous rows, neighbouring
// column tiles written back to back by the same CTA) touch the dense layout.  Wide matrices go through in column chunks so
// that the two intermediates stay small (and L2-friendly) whatever the width.
//   inverse:  d_in (dense) --pass--> A (tiled) --passes in place--> A = coefficients, network order, lazy range
//   forward:  A --PERM pass, per coset--> B (tiled, 2^added_bits blocks per tile) --passes in place--> last pass --> d_out (dense)
template <int F>
static int32_t lde_tiled_impl(p3gpu_ctx *ctx, const u32 *d_in, size_t h, size_t w, unsigned added_bits, u32 shift, u32 *d_out, bool *done,
                              size_t in_pitch, size_t out_pitch) {
    // in_pitch / out_pitch (elements, 0 = w): the matrix may be a column block of a wider row-major buffer on either side
    if (in_pitch == 0) in_pitch = w;
    if (out_pitch == 0) out_pitch = w;
    *done = false;
    const int log_n = (int)log2_floor(h);
    const NetworkPlan plan = plan_passes(log_n);
    if (!env_int("P3GPU_NTT_PIPE", 1) || plan.n_passes < 2 || plan.n_passes > 6) return P3GPU_OK;
    for (int k = 0; k < plan.n_passes; k++) {
        const int r = plan.bounds[k + 1] - plan.bounds[k];
        if (r < 6 || r > 10) return P3GPU_OK;
    }
    if (w % 4 != 0 || w < 8 || (reinterpret_cast<uintptr_t>(d_in) | reinterpret_cast<uintptr_t>(d_out)) % 16 != 0) return P3GPU_OK;
    if (((in_pitch * 4) << log_n) >= (1ull << 40) || in_pitch % 4 != 0 || tensor_map_encoder() == nullptr) return P3GPU_OK;
    const size_t n_cosets = (size_t)1 << added_bits;
    // column chunk: keep B (n_cosets * h * chunk * 4 bytes) around 1 GiB, at least 64 columns
    size_t chunk = ((size_t)1 << 28) / (n_cosets * h);
    chunk = std::max<size_t>(64, chunk & ~(size_t)7);
    if (const int forced = env_int("P3GPU_NTT_CHUNK", 0)) chunk = (size_t)std::max(8, forced & ~7);   // tests: exercise the chunk loop
    const size_t w8 = (w + 7) & ~(size_t)7;
    chunk = std::min(std::min(chunk, w8), (size_t)8192);
    if (n_cosets * h * chunk * 4 > ((size_t)8 << 30)) return P3GPU_OK;   // huge blow-ups: the 64-column floor would need > 8 GiB of scratch

    const uint2 *tw_inv = nullptr, *tw = nullptr;
    P3_TRY(get_twiddles<F>(ctx, log_n, 0, Fp<F>::ONE, 1, &tw_inv));
    P3_TRY(get_twiddles<F>(ctx, log_n, (int)added_bits, shift, 0, &tw));
    void *A = nullptr, *B = nullptr;
    P3_TRY(ctx_scratch(ctx, h * chunk * 4, &A));
    P3_TRY(ctx_scratch2(ctx, n_cosets * h * chunk * 4, &B));

    // the inverse network runs its passes in reverse plan order so that its LAST pass and the forward network's FIRST pass
    // cover the same number of layers (same tile shape on the coefficient buffer)
    for (size_t col0 = 0; col0 < w; col0 += chunk) {
        const size_t wc = std::min(chunk, w - col0);
        for (int k = 0; k < plan.n_passes; k++) {          // inverse
            PassArgs a;
            memset(&a, 0, sizeof a);
            const int kk = plan.n_passes - 1 - k;            // reversed plan: bounds mirrored
            a.l0 = log_n - plan.bounds[kk + 1]; a.l1 = log_n - plan.bounds[kk];
            a.w = (u32)in_pitch; a.wc = (u32)wc; a.log_n = log_n; a.n_cosets = 1; a.in_blocks = 1;
            a.tw = tw_inv; a.tw_stride = 0;
            if (k == 0) { a.in = d_in + col0; a.in_tiled = 0; a.has_scale = 1; a.scale = inv_height_scale<F>(h); }
            else { a.in = (const u32 *)A; a.in_tiled = 1; }
            a.out = (u32 *)A; a.out_tiled = 1;
            P3_TRY(launch_pipe<F>(ctx, a));
        }
        for (int k = 0; k < plan.n_passes; k++) {          // forward, all cosets per launch
            PassArgs a;
            memset(&a, 0, sizeof a);
            a.l0 = plan.bounds[k]; a.l1 = plan.bounds[k + 1];
            a.w = (u32)out_pitch; a.wc = (u32)wc; a.log_n = log_n; a.n_cosets = (u32)n_cosets;
            a.tw = tw; a.tw_stride = h;
            if (k == 0) { a.in = (const u32 *)A; a.in_tiled = 1; a.in_blocks = 1; a.in_bitrev = 1; }
            else { a.in = (const u32 *)B; a.in_tiled = 1; a.in_blocks = (u32)n_cosets; }
            if (k == plan.n_passes - 1) { a.out = d_out + col0; a.out_tiled = 0; a.out_stride = h * out_pitch; a.final_reduce = 1; }
            else { a.out = (u32 *)B; a.out_tiled = 1; }
            P3_TRY(launch_pipe<F>(ctx, a));
        }
    }
    *done = true;
    return P3GPU_OK;
}

template <int F>
static int32_t coset_lde_impl(p3gpu_ctx *ctx, const u32 *d_in, size_t h, size_t w, unsigned added_bits, u32 shift, u32 *d_out,
                              int bitrev_rows, size_t in_pitch = 0, size_t out_pitch = 0) {
    const int log_n = (int)log2_floor(h);
    const size_t n_cosets = (size_t)1 << added_bits;
    if (log_n == 0) {  // a constant polynomial: every evaluation equals the single input row
        const size_t n = n_cosets * w;
        broadcast_row<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_in, d_out, n_cosets, w);
        ctx->launches++;
        P3_CUDA(cudaGetLastError());
        return P3GPU_OK;
    }
    if (bitrev_rows) {
        bool done = false;
        P3_TRY(lde_tiled_impl<F>(ctx, d_in, h, w, added_bits, shift, d_out, &done, in_pitch, out_pitch));
        if (done) return P3GPU_OK;
    }
    P3_CHECK((in_pitch == 0 || in_pitch == w) && (out_pitch == 0 || out_pitch == w), P3GPU_EUNSUPPORTED,
             "column-block LDE (pitch != width) needs the pipelined tiled path: bit-reversed rows, width %% 4 == 0, width >= 8, height >= 2^12");
    // 1) inverse network: evaluations on H (natural) -> coefficients in network (bit-reversed) order, scaled by 1/h
    const uint2 *tw_inv = nullptr;
    P3_TRY(get_twiddles<F>(ctx, log_n, 0, Fp<F>::ONE, 1, &tw_inv));
    void *coef = nullptr;
    P3_TRY(ctx_scratch(ctx, h * w * 4, &coef));
    P3_TRY(run_network<F>(ctx, log_n, w, tw_inv, 0, 1, d_in, 0, 0, (u32 *)coef, 0, 0, 0, 0, nullptr, true, inv_height_scale<F>(h), false));

    // 2) forward networks, one per coset.  Memory block cb (h rows) holds the coset with natural index c = bitrev(cb):
    //    points shift * g_big^c * H  (radix_2_dit_parallel.rs:226-239).  The heaps of all cosets are one allocation
    //    (block cb at offset cb*h) so that the cosets run as grid.y of a single launch and share the coefficient reads in L2.
    const uint2 *tw = nullptr;
    P3_TRY(get_twiddles<F>(ctx, log_n, (int)added_bits, shift, 0, &tw));
    if (bitrev_rows) {
        P3_TRY(run_network<F>(ctx, log_n, w, tw, h, (unsigned)n_cosets, (const u32 *)coef, 0, 1, d_out, h * w, 0, 0, 0, nullptr, false,
                              make_uint2(0, 0), true));
    } else {
        void *tmp = nullptr;
        P3_TRY(ctx_scratch2(ctx, h * w * 4, &tmp));
        for (size_t cb = 0; cb < n_cosets; cb++) {
            size_t c = 0;
            for (unsigned b = 0; b < added_bits; b++) c |= ((cb >> b) & 1) << (added_bits - 1 - b);
            // natural LDE row of (coset c, evaluation index j) is j * n_cosets + c
            P3_TRY(run_network<F>(ctx, log_n, w, tw + cb * h, 0, 1, (const u32 *)coef, 0, 1, d_out, 0, 1, (int)added_bits, (u32)c,
                                  (u32 *)tmp, false, make_uint2(0, 0), true));
        }
    }
    return P3GPU_OK;
}

static int32_t check_shape(int field, size_t h, size_t w, unsigned extra_bits) {
    P3_CHECK(field == BABY_BEAR || field == KOALA_BEAR, P3GPU_EUNSUPPORTED, "unknown field %d", field);
    P3_CHECK(w >= 1 && w < (1ull << 31), P3GPU_EINVAL, "matrix width %zu out of range", w);
    P3_CHECK(is_pow2(h), P3GPU_EINVAL, "matrix height %zu is not a power of two", h);
    const unsigned adicity = field == BABY_BEAR ? Fp<BABY_BEAR>::TWO_ADICITY : Fp<KOALA_BEAR>::TWO_ADICITY;
    P3_CHECK(log2_floor(h) + extra_bits <= adicity, P3GPU_EINVAL, "height 2^%u (+%u bits) exceeds the field's two-adicity %u",
             log2_floor(h), extra_bits, adicity);
    P3_CHECK((h << extra_bits) * w < (1ull << 40), P3GPU_EINVAL, "matrix too large");
    return P3GPU_OK;
}

int32_t ntt_dft_batch(p3gpu_ctx *ctx, int field, int kind, const u32 *d_in, u32 *d_out, size_t h, size_t w, u32 shift) {
    P3_TRY(check_shape(field, h, w, 0));
    P3_CHECK(kind >= P3GPU_DFT && kind <= P3GPU_COSET_IDFT, P3GPU_EINVAL, "unknown transform kind %d", kind);
    return field == BABY_BEAR ? dft_batch_impl<BABY_BEAR>(ctx, kind, d_in, d_out, h, w, shift)
                              : dft_batch_impl<KOALA_BEAR>(ctx, kind, d_in, d_out, h, w, shift);
}

int32_t ntt_coset_lde(p3gpu_ctx *ctx, int field, const u32 *d_in, size_t h, size_t w, unsigned added_bits, u32 shift, u32 *d_out,
                      int bitrev_rows, size_t in_pitch, size_t out_pitch) {
    P3_CHECK(added_bits <= 8, P3GPU_EINVAL, "added_bits %u too large", added_bits);
    P3_TRY(check_shape(field, h, w, added_bits));
    P3_CHECK(d_in != d_out, P3GPU_EINVAL, "coset_lde_batch cannot run in place");
    P3_CHECK((in_pitch == 0 || in_pitch >= w) && (out_pitch == 0 || out_pitch >= w), P3GPU_EINVAL, "row pitch smaller than the width");
    return field == BABY_BEAR ? coset_lde_impl<BABY_BEAR>(ctx, d_in, h, w, added_bits, shift, d_out, bitrev_rows, in_pitch, out_pitch)
                              : coset_lde_impl<KOALA_BEAR>(ctx, d_in, h, w, added_bits, shift, d_out, bitrev_rows, in_pitch, out_pitch);
}

// Column-sharded coset LDE whose result lands row-sharded on all ranks (SURVEY 8e: column blocks -> all-to-all -> row blocks).
// Column chunks a rank's block of w_local columns is exchanged in (about 64 columns each, boundaries multiples of 8 columns).
// Every rank computes the same list for every source rank: the chunk-major row-block layout depends on it.
std::vector<size_t> shard_chunk_bounds(size_t w_local) {
    constexpr size_t chunk = 64;
    const size_t n_chunks = std::max<size_t>(1, (w_local + chunk / 2) / chunk);
    std::vector<size_t> cb{0};
    for (size_t c = 1; c <= n_chunks; c++) {
        const size_t b = c == n_chunks ? w_local : (w_local * c / n_chunks) & ~(size_t)7;
        if (b > cb.back()) cb.push_back(b);
    }
    if (cb.back() != w_local) cb.push_back(w_local);
    return cb;
}

int32_t ntt_coset_lde_sharded(p3gpu_ctx *ctx, int field, const u32 *d_in, size_t h, size_t w_local, unsigned added_bits, u32 shift,
                              unsigned world, u32 *const *rank_out, size_t w_total, size_t col_off, int chunk_major) {
    P3_CHECK(added_bits <= 8, P3GPU_EINVAL, "added_bits %u too large", added_bits);
    if (w_local == 0) {   // a rank without columns (more ranks than column units) only takes part in the barriers and the hashing
        P3_TRY(check_shape(field, h, 1, added_bits));
        return P3GPU_OK;
    }
    P3_TRY(check_shape(field, h, w_local, added_bits));
    P3_CHECK(world >= 1 && world <= 16 && (world & (world - 1)) == 0, P3GPU_EINVAL, "world size %u must be a power of two <= 16", world);
    P3_CHECK(col_off + w_local <= w_total && w_total < (1ull << 31), P3GPU_EINVAL, "column block [%zu, %zu) outside the trace width %zu", col_off, col_off + w_local, w_total);
    const size_t H = h << added_bits;
    P3_CHECK(H % world == 0, P3GPU_EINVAL, "LDE height %zu not divisible by %u ranks", H, world);
    const unsigned log_rows = log2_floor(H / world);
    P3_CHECK(log_rows >= 10 && log_rows <= 31, P3GPU_EUNSUPPORTED, "sharded LDE needs at least 1024 rows per rank (have 2^%u)", log_rows);
    for (unsigned g = 0; g < world; g++) P3_CHECK(rank_out[g] != nullptr, P3GPU_EINVAL, "null output block for rank %u", g);
    P3_CHECK(w_local % 4 == 0 && w_total % 4 == 0 && col_off % 4 == 0, P3GPU_EUNSUPPORTED, "sharded LDE: column blocks must be multiples of 4 columns");
    if (world == 1)   // a single rank owns every row: the LDE stores straight into its block, nothing to exchange
        return ntt_coset_lde(ctx, field, d_in, h, w_local, added_bits, shift, rank_out[0] + col_off, 1, w_local, w_total);
    // The LDE runs column chunk by column chunk into a staging buffer while the copy engines move the previous chunk's row blocks
    // to their owners, taking no SM time from the transform (fastest of the exchanges measured in profiles/README.md, "Multi-GPU exchange").
    if (!ctx->xchg_stream) {
        P3_CUDA(cudaStreamCreateWithFlags(&ctx->xchg_stream, cudaStreamNonBlocking));
        for (int b = 0; b < 2; b++) {
            P3_CUDA(cudaEventCreateWithFlags(&ctx->ev_stage_full[b], cudaEventDisableTiming));
            P3_CUDA(cudaEventCreateWithFlags(&ctx->ev_stage_free[b], cudaEventDisableTiming));
        }
    }
    const unsigned sh_rank_hint = (unsigned)((col_off * world) / std::max<size_t>(w_total, 1));   // ~ my rank: staggers the peers' copy order
    const std::vector<size_t> cb = shard_chunk_bounds(w_local);
    size_t wmax = 0;
    for (size_t c = 0; c + 1 < cb.size(); c++) wmax = std::max(wmax, cb[c + 1] - cb[c]);
    for (int b = 0; b < 2; b++) {
        if (ctx->stage_bytes[b] < H * wmax * 4) {
            if (ctx->stage_buf[b]) { P3_CUDA(cudaDeviceSynchronize()); P3_CUDA(cudaFree(ctx->stage_buf[b])); ctx->stage_buf[b] = nullptr; ctx->stage_bytes[b] = 0; }
            cudaError_t e = cudaMalloc(&ctx->stage_buf[b], H * wmax * 4);
            if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", H * wmax * 4, cudaGetErrorString(e)); cudaGetLastError(); return P3GPU_ENOMEM; }
            ctx->stage_bytes[b] = H * wmax * 4;
        }
    }
    const size_t R = (size_t)1 << log_rows;
    for (size_t c = 0; c + 1 < cb.size(); c++) {
        const int b = (int)(c & 1);
        const size_t c0 = cb[c], wc = cb[c + 1] - c0;
        if (wc == 0) continue;
        if (c >= 2) P3_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_stage_free[b], 0));      // the copies of chunk c-2 have drained this buffer
        u32 *S = (u32 *)ctx->stage_buf[b];
        if (field == BABY_BEAR) P3_TRY(coset_lde_impl<BABY_BEAR>(ctx, d_in + c0, h, wc, added_bits, shift, S, 1, w_local, wc));
        else P3_TRY(coset_lde_impl<KOALA_BEAR>(ctx, d_in + c0, h, wc, added_bits, shift, S, 1, w_local, wc));
        P3_CUDA(cudaEventRecord(ctx->ev_stage_full[b], ctx->stream));
        P3_CUDA(cudaStreamWaitEvent(ctx->xchg_stream, ctx->ev_stage_full[b], 0));
        // one peer copy per destination rank, each on its own stream so that the copies to the different peers run concurrently
        // (serialised on one stream they reached 180 GB/s per GPU at N = 8); the exchange stream joins them
        for (unsigned q = 0; q < world; q++) {
            const unsigned dq = (q + sh_rank_hint) % world;            // start with a different peer on every rank
            if (!ctx->dma_stream[dq]) {
                P3_CUDA(cudaStreamCreateWithFlags(&ctx->dma_stream[dq], cudaStreamNonBlocking));
                P3_CUDA(cudaEventCreateWithFlags(&ctx->dma_done[dq], cudaEventDisableTiming));
            }
            P3_CUDA(cudaStreamWaitEvent(ctx->dma_stream[dq], ctx->ev_stage_full[b], 0));
            if (chunk_major)   // the chunk is one contiguous (R x wc) matrix on both sides: a plain copy at link rate
                P3_CUDA(cudaMemcpyAsync(rank_out[dq] + R * (col_off + c0), S + (size_t)dq * R * wc, R * wc * 4, cudaMemcpyDeviceToDevice, ctx->dma_stream[dq]));
            else
                P3_CUDA(cudaMemcpy2DAsync(rank_out[dq] + col_off + c0, w_total * 4, S + (size_t)dq * R * wc, wc * 4, wc * 4, R, cudaMemcpyDeviceToDevice,
                                          ctx->dma_stream[dq]));
            P3_CUDA(cudaEventRecord(ctx->dma_done[dq], ctx->dma_stream[dq]));
            P3_CUDA(cudaStreamWaitEvent(ctx->xchg_stream, ctx->dma_done[dq], 0));
        }
        P3_CUDA(cudaEventRecord(ctx->ev_stage_free[b], ctx->xchg_stream));
    }
    // whatever follows on the context's stream (the barrier) comes after the last copies
    for (int b = 0; b < 2; b++) P3_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_stage_free[b], 0));
    return P3GPU_OK;
}

}  // namespace p3
