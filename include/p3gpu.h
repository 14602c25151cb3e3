/*
 * p3gpu.h — C ABI of libp3gpu: the B200 (sm_100a) backend for Plonky3's prover hot path
 * (batched NTT / coset LDE  ->  Merkle-tree commitment  ->  FRI fold/commit loop).
 *
 * This is the drop-in boundary: the entry points are what a Rust FFI shim implementing the reference's
 * trait surfaces would bind (the shim is shown in INTEGRATION.md):
 *     TwoAdicSubgroupDft   dft/src/traits.rs:28-291                  -> p3gpu_dft_batch*, p3gpu_coset_lde_batch*
 *     Mmcs::commit         commit/src/mmcs.rs:42, merkle-tree/src/mmcs/batch.rs:42-64 -> p3gpu_merkle_commit*
 *     FriFoldingStrategy   fri/src/config.rs:147-169, two_adic_pcs.rs:134-213          -> p3gpu_fri_fold*
 *     Pcs::commit / commit_phase  fri/src/two_adic_pcs.rs:300-324, fri/src/prover.rs:192-286
 *                                                                   -> p3gpu_pcs_commit*, p3gpu_fri_commit_phase*
 *
 * Conventions
 *   - Field elements are uint32_t in MONTGOMERY form, bit-identical to MontyField31.value
 *     (monty-31/src/monty_31.rs:34-44), so RowMajorMatrix<F>.values.as_ptr() can be passed unchanged.
 *   - Matrices are row-major: element (r, c) at m[r * width + c] (matrix/src/dense.rs:23-33).
 *   - A digest is 8 x uint32_t (Poseidon2: [F; 8]; Keccak: [u64; 4] little-endian).
 *   - Every function returns 0 on success and a negative P3GPU_E* code otherwise; p3gpu_last_error()
 *     describes the most recent failure of the calling thread.  The reference's prover-side trait methods
 *     panic on shape violations (dft: log2_strict_usize; mmcs/batch.rs:50-54); the shim turns non-zero into panic!.
 *   - "_dev" variants take DEVICE pointers and run asynchronously on the context's stream; the plain variants
 *     take HOST pointers and include the host<->device copies (they synchronise before returning).
 *   - There is no CPU fallback: without a CUDA device p3gpu_ctx_create fails with P3GPU_ECUDA.
 *   - Threads and devices: a context belongs to one device and serialises its work on one stream; every entry point makes
 *     that device current for the calling host thread, so calls may come from any thread (the reference's DFT / MMCS
 *     objects are Clone + Sync, radix_2_dit_parallel.rs:32-40).  A context is RE-ENTRANT: every entry point holds the
 *     context's internal mutex for its whole duration, so several threads may share one context (their calls are
 *     serialised); use one context per thread (each has its own stream, scratch buffers and twiddle cache) to keep
 *     several calls in flight.  The twiddle cache is bounded (LRU by bytes, P3GPU_TWIDDLE_CACHE_MB, default 2048).
 */
#ifndef P3GPU_H
#define P3GPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct p3gpu_ctx p3gpu_ctx;
typedef struct p3gpu_challenger p3gpu_challenger;

enum { P3GPU_BABY_BEAR = 0, P3GPU_KOALA_BEAR = 1 };

enum {
    P3GPU_OK = 0,
    P3GPU_EINVAL = -1,       /* bad shape (non power-of-two height, height above the field's two-adicity, ...) */
    P3GPU_EUNSUPPORTED = -2, /* unsupported field / width / hash */
    P3GPU_ECUDA = -3,        /* CUDA runtime error (incl. no device) */
    P3GPU_ENOMEM = -4,
    P3GPU_ESTATE = -5        /* missing configuration (e.g. Poseidon2 constants not set) */
};

/* which transform p3gpu_dft_batch computes (dft/src/traits.rs) */
enum {
    P3GPU_DFT = 0,        /* dft_batch            traits.rs:62    */
    P3GPU_IDFT = 1,       /* idft_batch           traits.rs:112   */
    P3GPU_COSET_DFT = 2,  /* coset_dft_batch      traits.rs:84    */
    P3GPU_COSET_IDFT = 3  /* coset_idft_batch     traits.rs:145   */
};

/* hash configurations of MerkleTreeMmcs (examples/src/types.rs:19-53, merkle-tree/benches/merkle_tree.rs:38) */
enum {
    P3GPU_HASH_POSEIDON2_W16 = 0, /* leaf PaddingFreeSponge<Perm16,16,8,8>,  node TruncatedPermutation<Perm16,2,8,16> */
    P3GPU_HASH_POSEIDON2_W24 = 1, /* leaf PaddingFreeSponge<Perm24,24,16,8>, node TruncatedPermutation<Perm16,2,8,16> */
    P3GPU_HASH_KECCAK = 2         /* leaf SerializingHasher<PaddingFreeSponge<KeccakF,25,17,4>>, node CompressionFunctionFromHasher<_,2,4> */
};

/* ---- context ---------------------------------------------------------------------------------- */
int32_t p3gpu_ctx_create(int device, p3gpu_ctx **out);
void p3gpu_ctx_destroy(p3gpu_ctx *ctx);
/* run subsequent calls on this cudaStream_t (e.g. torch's current stream); NULL = the legacy default stream.
 * A fresh context uses a private non-blocking stream; p3gpu_ctx_use_own_stream switches back to it. */
int32_t p3gpu_ctx_set_stream(p3gpu_ctx *ctx, void *cuda_stream);
int32_t p3gpu_ctx_use_own_stream(p3gpu_ctx *ctx);
int32_t p3gpu_ctx_sync(p3gpu_ctx *ctx);
const char *p3gpu_last_error(void);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t p3gpu_launch_count(const p3gpu_ctx *ctx);

/* device memory helpers for hosts that do not bring their own allocator */
int32_t p3gpu_malloc(p3gpu_ctx *ctx, size_t bytes, void **dptr);
int32_t p3gpu_free(p3gpu_ctx *ctx, void *dptr);
int32_t p3gpu_memcpy_h2d(p3gpu_ctx *ctx, void *dst, const void *src, size_t bytes);
int32_t p3gpu_memcpy_d2h(p3gpu_ctx *ctx, void *dst, const void *src, size_t bytes);
/* page-lock / unlock a host buffer so the host-pointer entry points copy at full PCIe rate */
int32_t p3gpu_host_register(void *ptr, size_t bytes);
int32_t p3gpu_host_unregister(void *ptr);

/* ---- TwoAdicSubgroupDft ----------------------------------------------------------------------- */
/* In-place capable (d_out may equal d_in).  kind: P3GPU_DFT..P3GPU_COSET_IDFT; shift (Montgomery) is used by the
 * coset kinds.  Result rows are in natural order (what `.to_row_major_matrix()` of the reference's result yields).
 * h must be a power of two <= 2^TWO_ADICITY; w >= 1. */
int32_t p3gpu_dft_batch_dev(p3gpu_ctx *ctx, int field, int kind, const uint32_t *d_in, uint32_t *d_out,
                            size_t h, size_t w, uint32_t shift);
int32_t p3gpu_dft_batch(p3gpu_ctx *ctx, int field, int kind, uint32_t *h_inout, size_t h, size_t w, uint32_t shift);

/* coset_lde_batch (traits.rs:227-234; Radix2DitParallel: radix_2_dit_parallel.rs:181-246).
 * in:  h x w evaluations over H (natural order).   out: (h << added_bits) x w evaluations over shift*K.
 * bitrev_rows != 0: memory row m holds the evaluation at shift * w_K^bitrev(m) — exactly the buffer
 *   Radix2DitParallel returns inside its BitReversedMatrixView and TwoAdicFriPcs::commit commits
 *   (fri/src/two_adic_pcs.rs:313-318).  bitrev_rows == 0: natural row order.
 * d_out must not alias d_in. */
int32_t p3gpu_coset_lde_batch_dev(p3gpu_ctx *ctx, int field, const uint32_t *d_in, size_t h, size_t w,
                                  unsigned added_bits, uint32_t shift, uint32_t *d_out, int bitrev_rows);
/* Host-pointer variant (page-lock the buffers with p3gpu_host_register for full PCIe rate).  With P3GPU_E2E_CHUNKS = n > 1 the call
 * is pipelined internally in n column chunks on three streams — H2D(chunk i+1) || LDE(chunk i) || D2H(chunk i-1); the default is
 * 1 (strictly serial, contiguous copies) because 2-D copies of narrow chunks run at 60-75 % of the contiguous PCIe rate on the
 * measured hosts (profiles/r02_pcie_probe.txt), which cancels the overlap for matrices of a few hundred bytes per row. */
int32_t p3gpu_coset_lde_batch(p3gpu_ctx *ctx, int field, const uint32_t *h_in, size_t h, size_t w,
                              unsigned added_bits, uint32_t shift, uint32_t *h_out, int bitrev_rows);

/* ---- Poseidon2 / hashing ---------------------------------------------------------------------- */
/* Poseidon2::new (poseidon2/src/lib.rs:50-87): round constants cross the boundary in Montgomery form.
 * width 16 or 24; rc_initial / rc_terminal: 4 x width; rc_internal: rounds_p scalars. */
int32_t p3gpu_poseidon2_set_constants(p3gpu_ctx *ctx, int field, int width, const uint32_t *rc_initial,
                                      const uint32_t *rc_terminal, const uint32_t *rc_internal, int rounds_p);
/* Permutation::permute_mut on n independent states (n x width, device memory) — used by KAT tests/benches. */
int32_t p3gpu_poseidon2_permute_dev(p3gpu_ctx *ctx, int field, int width, uint32_t *d_states, size_t n);
/* Keccak-f[1600] on n independent states (n x 25 u64, device memory). */
int32_t p3gpu_keccak_f_dev(p3gpu_ctx *ctx, uint64_t *d_states, size_t n);

/* ---- Mmcs::commit ----------------------------------------------------------------------------- */
/* total digests in all layers of a tree whose tallest matrix has max_height rows (layers padded as the
 * reference pads them, merkle_tree.rs:473-481) */
size_t p3gpu_merkle_total_digests(size_t max_height);
/* MerkleTree::new with arity 2 over n_mats matrices (merkle_tree.rs:95-178; mixed heights allowed if they sit
 * on the reference's height ladder, mmcs/geometry.rs:83-124).  d_layers receives every digest layer
 * back to back (layer 0 = leaf digests); layer_lens[k] its length in digests; *n_layers the layer count
 * (layer_lens must have room for 65 entries).  The cap of height c is the first 2^c digests of layer n_layers-1-c. */
int32_t p3gpu_merkle_commit_dev(p3gpu_ctx *ctx, int field, int hash, size_t n_mats, const uint32_t *const *d_mats,
                                const size_t *heights, const size_t *widths, uint32_t *d_layers,
                                size_t *layer_lens, size_t *n_layers);
int32_t p3gpu_merkle_commit(p3gpu_ctx *ctx, int field, int hash, size_t n_mats, const uint32_t *const *h_mats,
                            const size_t *heights, const size_t *widths, uint32_t *h_layers,
                            size_t *layer_lens, size_t *n_layers);

/* Digest layers ABOVE an existing layer of n digests (d_digests, device): d_layers receives the (padded) copy of the input
 * layer followed by every layer up to the root, p3gpu_merkle_total_digests(n) digests in all.  Used to finish a tree whose
 * sub-tree roots were produced elsewhere (multi-GPU row sharding, DESIGN.md section 5). */
int32_t p3gpu_merkle_from_digests_dev(p3gpu_ctx *ctx, int field, int hash, const uint32_t *d_digests, size_t n,
                                      uint32_t *d_layers, size_t *layer_lens, size_t *n_layers);

/* ---- FRI -------------------------------------------------------------------------------------- */
/* TwoAdicFriFolding::fold_matrix (two_adic_pcs.rs:134-213): rows x 2^log_arity EF4 values in bit-reversed
 * evaluation order -> rows EF4 values.  beta: 4 Montgomery words. */
int32_t p3gpu_fri_fold_dev(p3gpu_ctx *ctx, int field, const uint32_t *d_in, size_t rows, unsigned log_arity,
                           const uint32_t beta[4], uint32_t *d_out);
int32_t p3gpu_fri_fold(p3gpu_ctx *ctx, int field, const uint32_t *h_in, size_t rows, unsigned log_arity,
                       const uint32_t beta[4], uint32_t *h_out);

/* acc[i] += s * x[i] over EF4 (n elements, device memory): the roll-in of a shorter FRI input, folded += beta^arity * input
 * (fri/src/prover.rs:258-265). */
int32_t p3gpu_ef_axpy_dev(p3gpu_ctx *ctx, int field, uint32_t *d_acc, const uint32_t *d_x, size_t n, const uint32_t s[4]);

/* BENCHMARK / TEST ONLY — not the Fiat-Shamir flow of fri/src/prover.rs:237-248: all betas are supplied up front, so no beta
 * depends on the cap of its round, and a single input vector is supported (no roll-in of shorter inputs).  A prover
 * drives the transcript per round: p3gpu_merkle_commit_dev -> cap to the host -> challenger -> p3gpu_fri_fold_dev
 * (-> p3gpu_ef_axpy_dev for the roll-in); plonky3_b200.fri.commit_phase does exactly that and is what bench.py times.
 * commit_phase (fri/src/prover.rs:192-286) for ONE input vector with caller-supplied betas (the Fiat-Shamir
 * transcript stays on the host; with commit_proof_of_work_bits = 0 a round's beta depends only on that round's cap,
 * so a host driving the transcript calls p3gpu_merkle_commit_dev / p3gpu_fri_fold_dev per round instead).
 * d_vec: len EF4 values (bit-reversed), consumed.  Rounds use compute_log_arity_for_round (fri/src/config.rs:180-207).
 * caps: per round 2^min(cap_height, layers-1) digests written back to back into h_caps (host), cap_lens[k] digests;
 * h_final: the folded vector of length 2^(log_blowup+log_final_poly_len) EF4 (before the final-poly iDFT). */
int32_t p3gpu_fri_commit_phase_dev(p3gpu_ctx *ctx, int field, int hash, uint32_t *d_vec, size_t len,
                                   unsigned log_blowup, unsigned log_final_poly_len, unsigned max_log_arity,
                                   unsigned cap_height, const uint32_t *betas /* rounds x 4 */, size_t n_betas,
                                   uint32_t *h_caps, size_t *cap_lens, unsigned *log_arities, size_t *n_rounds,
                                   uint32_t *h_final);

/* ---- Pcs::open, pre-FRI part (fri/src/two_adic_pcs.rs:413-662; SURVEY.md 8f rank 1) ---------------- */
/* compute_inverse_denominators (:743-780): d_inv_denoms[i] = 1/(z - x_i) for x_i = GENERATOR * w^bitrev(i), i < 2^log_height
 * (EF4, bit-reversed coset order, so a prefix serves every smaller height).  If d_adjusted != NULL it receives
 * 1/(z - x_i) - 1/z (compute_adjusted_weights) and zinv = 1/z must be supplied. */
int32_t p3gpu_open_inv_denoms_dev(p3gpu_ctx *ctx, int field, unsigned log_height, const uint32_t z[4], const uint32_t *zinv,
                                  uint32_t *d_inv_denoms, uint32_t *d_adjusted);
/* Matrix::columnwise_dot_product: d_out[j] = scale * sum_i mat[i][j] * vec[i]  (vec: h EF4 values, out: w EF4 values; scale may be
 * NULL).  With vec = adjusted weights and scale = z (z^N - g^N) / (N g^N) this is interpolate_coset_with_precomputation
 * (matrix/src/interpolation.rs:161-193) on the first h rows of a committed bit-reversed LDE. */
int32_t p3gpu_columnwise_dot_dev(p3gpu_ctx *ctx, int field, const uint32_t *d_mat, size_t h, size_t w, const uint32_t *d_vec_ef,
                                 const uint32_t *scale, uint32_t *d_out);
/* rowwise_packed_dot_product with the powers of alpha (:622-626): d_out[i] = sum_j alpha^j * mat[i][j]  (h EF4 values). */
int32_t p3gpu_rowwise_dot_dev(p3gpu_ctx *ctx, int field, const uint32_t *d_mat, size_t h, size_t w, const uint32_t alpha[4],
                              uint32_t *d_out);
/* reduced-opening accumulation (:640-657): d_ro[i] += coeff * (yred - d_r[i]) * d_inv_denoms[i], i < h. */
int32_t p3gpu_open_reduce_dev(p3gpu_ctx *ctx, int field, uint32_t *d_ro, const uint32_t *d_r, const uint32_t *d_inv_denoms, size_t h,
                              const uint32_t coeff[4], const uint32_t yred[4]);

/* ---- Pcs::commit ------------------------------------------------------------------------------ */
/* TwoAdicFriPcs::commit for one matrix whose domain is the subgroup H (shift = GENERATOR / 1):
 * LDE onto GENERATOR*K with K = |H| << log_blowup, bit-reversed rows, then MerkleTreeMmcs::commit.
 * d_lde ((h<<log_blowup) x w) and d_layers stay resident for get_evaluations_on_domain / open. */
int32_t p3gpu_pcs_commit_dev(p3gpu_ctx *ctx, int field, int hash, const uint32_t *d_evals, size_t h, size_t w,
                             unsigned log_blowup, uint32_t *d_lde, uint32_t *d_layers, size_t *layer_lens,
                             size_t *n_layers);

/* The same commit with the trace in HOST memory (pinned for full PCIe rate): the realistic drop-in point of a GpuFriPcs (the
 * reference's Pcs::commit receives host matrices, two_adic_pcs.rs:300-324).  The trace crosses PCIe once, in column chunks
 * whose copies overlap the LDE of the previous chunk; LDE and digest layers stay resident in d_lde / d_layers; only the cap
 * (2^min(cap_height, layers-1) digests) is copied back to h_cap.  Synchronous. */
int32_t p3gpu_pcs_commit(p3gpu_ctx *ctx, int field, int hash, const uint32_t *h_evals, size_t h, size_t w, unsigned log_blowup,
                         unsigned cap_height, uint32_t *d_lde, uint32_t *d_layers, size_t *layer_lens, size_t *n_layers,
                         uint32_t *h_cap, size_t *cap_len);

/* ---- Poseidon2 AIR (SURVEY.md 8f ranks 2-3): the AIR of prove_prime_field_31 -o poseidon-2-permutations ---------------
 * VectorizedPoseidon2Air<KoalaBear, width 16, S-box degree 3, 0 S-box registers, 4 + rounds_p + 4 rounds> (poseidon2-air/src/
 * air.rs, vectorized.rs).  Only the KoalaBear instance is built (BabyBear's degree-7 S-box needs register columns).
 * RoundConstants::new (poseidon2-air/src/constants.rs:47-57): 4 x 16 beginning, rounds_p partial, 4 x 16 ending, Montgomery. */
int32_t p3gpu_p2air_set_constants(p3gpu_ctx *ctx, int field, const uint32_t *beginning_full, const uint32_t *partial, int rounds_p,
                                  const uint32_t *ending_full);
/* columns of ONE permutation: 16 inputs + 4*16 + rounds_p + 4*16 (columns.rs:11-48) */
size_t p3gpu_p2air_columns(int rounds_p);
/* generate_vectorized_trace_rows (poseidon2-air/src/generation.rs:14-70): d_inputs n_perms x 16 -> d_trace n_perms x columns,
 * i.e. the (n_perms / VECTOR_LEN) x (VECTOR_LEN * columns) row-major trace. */
int32_t p3gpu_p2air_generate_trace_dev(p3gpu_ctx *ctx, int field, const uint32_t *d_inputs, size_t n_perms, uint32_t *d_trace);
/* quotient_values (uni-stark/src/prover.rs:462-827) of that AIR over the quotient domain GENERATOR * K with |K| = the LDE height
 * (log_quotient_degree == log_blowup: the truncation fast path of get_evaluations_on_domain, two_adic_pcs.rs:376-385).
 * d_lde: the committed trace LDE, 2^log_lde_height rows in bit-reversed order, vector_len * columns wide.
 * d_quotient: 2^log_lde_height EF4 values in NATURAL order (what commit_quotient / split_evals consume). */
int32_t p3gpu_p2air_quotient_dev(p3gpu_ctx *ctx, int field, int vector_len, const uint32_t *d_lde, unsigned log_lde_height,
                                 unsigned log_trace_height, const uint32_t alpha[4], uint32_t *d_quotient);

/* ---- transcript and query phase of the prove driver (SURVEY.md 8f rank 4 / N1) ----------------------------------------
 * DuplexChallenger<F, Poseidon2<width>, width, rate> (challenger/src/duplex_challenger.rs:60-300) with its state resident on the
 * device, so that caps and opened values produced on the GPU are absorbed without a PCIe round trip per duplexing.  The
 * Poseidon2 constants of (field, width) must have been set.  Values are Montgomery words; `observe` of an EF4 element = its 4
 * coefficients in order; sampled elements pop from the END of the rate (duplex_challenger.rs:255-268). */
int32_t p3gpu_challenger_new(p3gpu_ctx *ctx, int field, int width, int rate, p3gpu_challenger **out);
void p3gpu_challenger_free(p3gpu_ctx *ctx, p3gpu_challenger *ch);
int32_t p3gpu_challenger_clone(p3gpu_ctx *ctx, const p3gpu_challenger *src, p3gpu_challenger **out);
int32_t p3gpu_challenger_observe_dev(p3gpu_ctx *ctx, p3gpu_challenger *ch, const uint32_t *d_values, size_t n);
int32_t p3gpu_challenger_observe(p3gpu_ctx *ctx, p3gpu_challenger *ch, const uint32_t *h_values, size_t n);
int32_t p3gpu_challenger_sample(p3gpu_ctx *ctx, p3gpu_challenger *ch, uint32_t *h_out, size_t n);   /* synchronous */
/* GrindingChallenger::grind (grinding_challenger.rs:100-232): parallel search on the device, returns the SMALLEST witness (what a
 * serial reference build returns), observes it and consumes the checked sample. */
int32_t p3gpu_challenger_grind(p3gpu_ctx *ctx, p3gpu_challenger *ch, unsigned bits, uint32_t *witness);
/* Mmcs::open_batch for n indices at once (merkle-tree/src/mmcs/batch.rs:75-121): d_out[q] = row (h_indices[q] >> index_shift) of a
 * device matrix; and the authentication paths: d_out[q][l] = sibling digest at layer l, l < path_len = layers - 1 - cap_height. */
int32_t p3gpu_gather_rows_dev(p3gpu_ctx *ctx, const uint32_t *d_mat, size_t h, size_t w, const uint32_t *h_indices, size_t n, unsigned index_shift,
                              uint32_t *d_out);
int32_t p3gpu_merkle_paths_dev(p3gpu_ctx *ctx, const uint32_t *d_layers, const size_t *layer_lens, size_t n_layers, size_t path_len,
                               const uint32_t *h_indices, size_t n, unsigned index_shift, uint32_t *d_out);

/* ---- multi-GPU: one process per GPU, peer memory over NVLink (SURVEY.md 8e; DESIGN.md section 5) ------------------
 * The path shards by COLUMN for the LDE (every column is an independent polynomial, dft/src/traits.rs:22-24) and by
 * ROW RANGE for the Merkle tree (a leaf is a sequential sponge over the whole row, merkle_tree.rs:309-317; rows
 * [k*H/G, (k+1)*H/G) of the bit-reversed LDE are a complete sub-tree).  The re-sharding all-to-all copies the LDE's
 * column chunks into the destination ranks' row blocks through CUDA-IPC-mapped peer pointers on the copy engines.
 * No collective library is involved; the host only exchanges 64-byte IPC handles once (any channel: MPI, sockets,
 * torch.distributed, ...) and fills a p3gpu_peer_group. */
#define P3GPU_PEER_CTRL_BYTES 65536   /* size of every rank's control block (p3gpu_malloc'ed, zeroed, IPC-exported) */
#define P3GPU_PEER_CTRL_USER 256      /* byte offset of its user area (all-gather tables); the first 64 bytes are barrier flags */
typedef struct p3gpu_peer_group {
    uint32_t world, rank;             /* ranks (power of two, <= 16), my rank */
    void *ctrl[16];                   /* control block of every rank: own pointer at [rank], IPC-mapped pointers elsewhere */
    uint32_t *rows[16];               /* row block of every rank: (H / world) x w_total u32, row-major (NULL if unused) */
    double timeout_s;                 /* barrier watchdog (0 = 20 s): a missing peer traps the kernel instead of hanging */
} p3gpu_peer_group;

/* cudaIpcGetMemHandle / cudaIpcOpenMemHandle / cudaIpcCloseMemHandle on a p3gpu_malloc'ed buffer (64-byte handle) */
int32_t p3gpu_ipc_export(p3gpu_ctx *ctx, void *dptr, uint8_t handle[64]);
int32_t p3gpu_ipc_import(p3gpu_ctx *ctx, const uint8_t handle[64], void **dptr);
int32_t p3gpu_ipc_close(p3gpu_ctx *ctx, void *dptr);
int32_t p3gpu_memset_dev(p3gpu_ctx *ctx, void *dptr, int value, size_t bytes);

/* Stream-ordered flag barrier across the group (system-scope release/acquire on the control blocks).  `epoch` must be
 * the same on all ranks and strictly increasing from call to call (1, 2, 3, ...). */
int32_t p3gpu_peer_barrier_dev(p3gpu_ctx *ctx, const p3gpu_peer_group *grp, uint32_t epoch);
/* Every rank stores `words` u32 from d_src into slot `rank` of the table at user-area offset table_offset_bytes of EVERY
 * rank's control block (replaces the all-gather of Merkle roots / FRI final polynomials; pair with a barrier). */
int32_t p3gpu_peer_allgather_dev(p3gpu_ctx *ctx, const p3gpu_peer_group *grp, size_t table_offset_bytes, const uint32_t *d_src, size_t words);

/* coset_lde_batch of this rank's column block [col_off, col_off + w_local) of a trace of width w_total; the
 * bit-reversed-row result is scattered by row range: LDE row r goes to grp->rows[r / (H/world)] (local row r % (H/world),
 * columns col_off.., pitch w_total).  Needs w_local, w_total and col_off to be multiples of 4 (16-byte aligned rows;
 * column blocks that are multiples of 8 keep every 32-byte row segment sector-aligned) and H / world >= 1024.  Complete on
 * all ranks only after a following barrier. */
int32_t p3gpu_coset_lde_batch_sharded_dev(p3gpu_ctx *ctx, int field, const p3gpu_peer_group *grp, const uint32_t *d_in, size_t h,
                                          size_t w_local, unsigned added_bits, uint32_t shift, size_t w_total, size_t col_off);

/* TwoAdicFriPcs::commit (two_adic_pcs.rs:300-324) of ONE trace sharded by column block over the group; bit-identical to
 * the single-GPU commitment: sharded LDE -> barrier -> leaf hashing + sub-tree over grp->rows[rank] -> exchange
 * of the cap slices -> barrier -> (cap_height < log2(world): top levels compressed redundantly on every rank).
 * col_starts: world + 1 column offsets, rank g holds columns [col_starts[g], col_starts[g+1]) of the trace (every rank passes the
 *   same array; blocks that are multiples of 8 columns keep all copies sector aligned; a block may be empty); d_evals_local: my
 *   block, h x (col_starts[rank+1] - col_starts[rank]).
 * *epoch: the group's barrier epoch counter (start at 0; same variable for every collective call of this group).
 * Row-block layout after the call (world > 1): CHUNK-MAJOR — for every source rank g and every column chunk [b, b') of its block
 *   (p3gpu_shard_chunk_bounds of the block width) one contiguous (H/world) x (b' - b) row-major matrix at element offset
 *   (H/world) * (col_starts[g] + b); with world == 1 the block is the dense (H x w_total) LDE.
 * d_sub_layers: p3gpu_merkle_total_digests(H / world) digests = this rank's sub-tree (kept for openings);
 * h_cap: 2^cap_height digests (host), identical on every rank.  phase_ms (NULL or 4 floats): device time of
 * [LDE + exchange, barrier wait, hashing, cap exchange]. */
int32_t p3gpu_commit_sharded_dev(p3gpu_ctx *ctx, int field, int hash, const p3gpu_peer_group *grp, uint32_t *epoch,
                                 const uint32_t *d_evals_local, size_t h, const size_t *col_starts,
                                 unsigned log_blowup, unsigned cap_height, uint32_t *d_sub_layers, size_t *layer_lens,
                                 size_t *n_layers, uint32_t *h_cap, size_t *cap_len, float *phase_ms);
/* the column chunk boundaries (0 = first, w_local = last) a block of w_local columns is exchanged in; returns their number */
size_t p3gpu_shard_chunk_bounds(size_t w_local, size_t *bounds, size_t max_bounds);

#ifdef __cplusplus
}
#endif
#endif /* P3GPU_H */
