/*
 * dmv_b200.h -- C ABI of libdmv_b200.so: the B200-native distributed matrix-free H.x hot path.
 *
 * This is the drop-in boundary for the reference's hot path (SURVEY.md section 8b).  Plain pointers
 * and sizes only; no torch / C++ types.  Every entry point names the reference interface it replaces.
 * All functions returning int return 0 on success and a non-zero code on failure, with a message
 * available from dmv_last_error() (the reference halts instead: src/DistributedMatrixVector.chpl:116,
 * 1099-1102; the ls_chpl_* wrappers below abort() on failure to stay drop-in).
 *
 * Threading: one context per GPU; a context is not thread-safe; dmv_matvec() is collective over the
 * ranks of the communicator (like the reference's allLocalesBarrier use, DMV:895,954,1013).
 */
#ifndef DMV_B200_H
#define DMV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dmv_context dmv_context;

/* Element type of x / y.  The reference's vectors are real(64) (DMV:1095-1096); complex128 is the
 * extension BASELINE.json asks for. */
enum { DMV_F64 = 1, DMV_C128 = 2 };

/* Flat description of a spin basis: the visible part of `ls_hs_basis` (reference src/FFI.chpl:94-105)
 * plus the symmetry group the third-party library keeps opaque.  Group element g maps a state s to
 * g.s with (g.s) bit i = s bit perms[g*number_sites + i], followed by a global spin flip when
 * flips[g] != 0.  characters are interleaved (re, im).  group_order == 0: no projection. */
typedef struct {
  int32_t number_sites;      /* <= 64 (DMV:1099: numberWords == 1) */
  int32_t hamming_weight;    /* -1: not fixed */
  int32_t spin_inversion;    /* 0, +1, -1 */
  int32_t has_permutations;  /* basis.hasPermutationSymmetries(), src/ForeignTypes.chpl:96-98 */
  int64_t group_order;       /* all elements, including the inversion-doubled ones */
  const int32_t *perms;
  const uint8_t *flips;
  const double *characters;
} dmv_basis_desc;

/* Flat non-branching term tables: <beta|t|alpha> = v [alpha & m == r] (-1)^popcount(alpha & s),
 * beta = alpha ^ x (the content of `ls_hs_nonbranching_terms`, reference src/FFI.chpl:109-113, whose
 * tail is opaque there).  v interleaved (re, im).  Diagonal terms have x == 0 and carry no x array. */
typedef struct {
  int64_t n_off;
  const double *off_v;
  const uint64_t *off_m, *off_r, *off_x, *off_s;
  int64_t n_diag;
  const double *diag_v;
  const uint64_t *diag_m, *diag_r, *diag_s;
} dmv_operator_desc;

/* ---- library lifetime: replaces ls_chpl_init / ls_chpl_finalize (reference src/library.c:19-34) */
void ls_chpl_init(void);
void ls_chpl_finalize(void);
const char *dmv_last_error(void);
int dmv_version(void);
/* number of kernel launches issued by this library since load (evidence for bench.py's gpu_launches) */
int64_t dmv_launch_count(void);

/* ---- context: replaces the per-call setup of matrixVectorProduct (DMV:1077-1084: operator clone,
 * uncheckedSetRepresentatives) and of localOffDiagonalNoQueue (DMV:864-955: buffers, pointer wiring)
 * with a persistent object.  `device` is the CUDA device ordinal; rank / num_ranks define the hash
 * partition  owner(s) = hash64_01(s) % num_ranks  (reference src/StatesEnumeration.chpl:122-136). */
int dmv_context_create(const dmv_basis_desc *basis, const dmv_operator_desc *op, int device, int rank,
                       int num_ranks, dmv_context **out);
int dmv_context_destroy(dmv_context *ctx);
/* launch on `cuda_stream` (a cudaStream_t; NULL is the legacy default stream), or on the context's own
 * non-blocking stream when use_own_stream != 0 (the initial state) */
int dmv_set_stream(dmv_context *ctx, void *cuda_stream, int use_own_stream);
int dmv_synchronize(dmv_context *ctx);
/* options: "mode"     = -1 auto (row traversal on one rank when a row kernel applies -- k_gather: bit-parallel operator on a
 *                        basis without permutation symmetries; k_rows: real bit-parallel operator on a basis with
 *                        permutation symmetries and trivial characters -- else push) | 0 push: scatter with FP64
 *                        atomics, the reference's traversal (DMV:73-127) | 1 rows (k_gather / k_rows, else the queued
 *                        k_pull); one rank only
 *          "gather"   = -1 auto | 0 use the queued k_pull instead of k_gather when "mode" selects rows
 *          "rows"     = -1 auto | 0 use the queued k_pull instead of k_rows
 *          "rows_index" = -1 auto, 0 open-addressing table with the vector element in the slot | 1 dense table behind a
 *                        two-level perfect hash (5 bits per state; measured slower, kept for reference)
 *          "rows_ctas" = 3 (default) | 2 | 4 resident CTAs per SM of k_rows (k_rows_batch: always 2) (registers per thread 80 | 122 |
 *                        64; at 80 a few words of the pipeline state spill and the extra warps more than pay for it)
 *          "rows_batch" = -1 auto, 1: dmv_matvec_batch on bases with permutation symmetries takes up to six doubles per
 *                        state (six real / three complex vectors) through k_rows_batch | 0 vector by vector;
 *                        "rows_batch_min" = doubles per state (vectors x element width, default 2) from which it is used
 *                        (1: a single real vector goes through k_rows_batch too)
 *          "rows_table_per_state" = 0 auto (complex128 k_rows table and k_rows_batch table: 8 buckets per state, 4 or 2
 *                        when the table would take more than a quarter of the free memory) | 2 | 4 | 8 forced; the
 *                        float64 k_rows table always has 2 two-slot buckets per state
 *          "gather_walk" = 0 every lane walks its emitting groups from the top bit | 1 group-major warp-uniform walk
 *                        (measured slower) | 2 from the bottom bit (round 1)
 *          "index"    = -1 auto (identity / Lin tables / directory) | 0 directory + binary search | 2 combinadic rank
 *                        | 3 Lin tables (full fixed-Hamming bases)
 *          "bitparallel" = 1 | 0 walk the flip-mask groups one by one
 *          "canon"    = -1 auto (orbit minima through canonical forms: full space group of a torus, rotations x mirror x
 *                        flip of a chain) | 1 the round-1 forms (block rotations + coset chain; four run searches)
 *                        | 2 single-block LUT + independent networks | 0 walk the chain of group elements
 *          "exchange" = -1 auto (replicated x when the whole basis fits, else peer-direct records, else NCCL buckets)
 *                        | 0 NCCL send/recv of record buckets | 1 peer-direct records over NVLink | 2 replicated x
 *          "peer_gather" = -1 auto (replicated x: all-gather of x as peer-direct NVLink stores + flags) | 0 ncclAllGather
 *          "rounds"   = -1 auto (peer-direct records in 4 overlapped rounds for blocks of >= 2^18 states) | 0, 1 one shot
 *                        (generate everything, fence, accumulate) | R <= 64 rounds
 * dmv_get_info: "index_mode", "pull", "gather", "rows", "rows_ok", "projection", "n_groups", "orbit_n_q", "orbit_n_t",
 *               "canon_mode", "torus_mode", "peer_direct", "replicated", "replicated_block", "peer_gather", "rounds",
 *               "global_states", "complex_coefficients", "rows_kernel" (instantiation of the last k_rows launch:
 *               100 CTAS + 10 TK + MPH, CTAS = resident CTAs per SM, TK = torus block size of the canonical form or 0,
 *               MPH = 1 with the dense index; 0 before the first launch), "rows_batch_kernel" (the same for the last
 *               k_rows_batch launch), "rows_table_buckets" / "rows_batch_buckets" (buckets of the k_rows / k_rows_batch
 *               open-addressing table as last built; 0 before), ... (-1: unknown) */
int dmv_set_option(dmv_context *ctx, const char *name, int64_t value);
int64_t dmv_get_info(const dmv_context *ctx, const char *name);

/* ---- basis
 * dmv_basis_build: replaces Basis.build() / enumerateStates for this rank (reference
 *   src/ForeignTypes.chpl:72, src/StatesEnumeration.chpl:516-603): enumerates on the GPU the ascending
 *   representatives owned by this rank and their norms, and installs them.
 * dmv_set_representatives: replaces Basis.uncheckedSetRepresentatives (src/ForeignTypes.chpl:74-77,
 *   DMV:1084).  `representatives` must be ascending and owned by this rank; `norms` may be NULL (they
 *   are then computed on the GPU when the basis needs them).  Host or device pointers.
 * dmv_get_representatives copies them out (host or device destination); pass NULL to query the count. */
int dmv_basis_build(dmv_context *ctx);
int dmv_set_representatives(dmv_context *ctx, const uint64_t *representatives, int64_t count,
                            const double *norms);
int64_t dmv_number_states(const dmv_context *ctx);
int dmv_get_representatives(dmv_context *ctx, uint64_t *representatives, double *norms);

/* ---- third-party kernels the path consumes, now on the GPU (host or device pointers)
 * dmv_state_index: ls_hs_state_index (reference src/FFI.chpl:173-175; call DMV:102); -1 when absent.
 * dmv_state_info:  ls_hs_state_info  (src/FFI.chpl:181-184; call src/BatchedOperator.chpl:188-194).
 * dmv_locale_idx_of: localeIdxOf     (src/StatesEnumeration.chpl:129-136). */
int dmv_state_index(dmv_context *ctx, int64_t count, const uint64_t *spins, int64_t *indices);
int dmv_state_info(dmv_context *ctx, int64_t count, const uint64_t *alphas, uint64_t *betas,
                   double *characters, double *norms);
int dmv_locale_idx_of(dmv_context *ctx, int64_t count, const uint64_t *states, int num_locales,
                      uint8_t *keys);

/* ---- BatchedOperator.computeOffDiag (reference src/BatchedOperator.chpl:82-213)
 * Generates, for alphas[0..count) with values xs, the flat list (betas, coeffs, keys) after
 * projection; *n receives the number of entries.  Output arrays must hold count * max_off_diag
 * entries (dmv_max_number_off_diag).  Entry ORDER is unspecified (the reference's is row-major;
 * consumers only bucket and accumulate).  coeffs interleaved complex128.  Host or device pointers. */
int64_t dmv_max_number_off_diag(const dmv_context *ctx);
int dmv_compute_off_diag(dmv_context *ctx, int64_t count, const uint64_t *alphas, const void *xs,
                         int elt, int64_t *n, uint64_t *betas, double *coeffs, uint8_t *keys);

/* ---- the hot path
 * dmv_local_matvec: localMatrixVector(matrix, x, y, representatives) (DMV:1055-1070) on this rank's
 *   block when num_ranks == 1.  y = D x + O x if the operator has diagonal terms, else y += O x
 *   (DMV:1062-1069: without diagonal terms y is not cleared).  x, y: host or device pointers of
 *   dmv_number_states() elements of type `elt`.
 * dmv_matvec: matrixVectorProduct (DMV:1072-1093), collective over the communicator: generation,
 *   hash bucketing, all-to-all exchange (peer-direct NVLink stores or NCCL) and owner-side search +
 *   accumulate -- or the replicated-x form below when it applies. */
int dmv_local_matvec(dmv_context *ctx, int elt, const void *x, void *y);
int dmv_matvec(dmv_context *ctx, int elt, const void *x, void *y);

/* ---- stepwise form of the distributed product, for hosts that own the exchange themselves (a Chapel
 * host with GASNet PUTs as in DMV:361-371, torch.distributed, or several logical ranks on one GPU):
 *   dmv_plan:      one counting pass; fills send_counts[num_ranks] (records this rank emits for each
 *                  destination in one product; the own entry is processed locally and reported too).
 *   dmv_generate:  y (+)= D x; emits all records; own bucket is searched + accumulated into y at once,
 *                  the others are left in the context's outgoing buckets.
 *   dmv_outgoing:  device pointers + count of the bucket for `dest` (valid until the next generate).
 *   dmv_accumulate: localProcess (DMV:73-127) on `count` received records (device or host pointers):
 *                  y[index(beta)] += coeff (* norm).  A record that is non-zero and not in the basis
 *                  is an error (DMV:115-118). */
int dmv_plan(dmv_context *ctx, int64_t *send_counts);
int dmv_generate(dmv_context *ctx, int elt, const void *x, void *y);
int dmv_outgoing(dmv_context *ctx, int dest, const uint64_t **betas, const double **coeffs,
                 int64_t *count);
int dmv_accumulate(dmv_context *ctx, int elt, int64_t count, const uint64_t *betas,
                   const double *coeffs, void *y);

/* ---- replicated-x form of the distributed product (B200-first alternative to the record exchange of DMV:313-436,
 * chosen automatically by dmv_matvec -- option "exchange" = -1 / 2 -- when the whole basis fits on one device): every
 * rank keeps the whole sorted basis, x is all-gathered (E bytes per state instead of 8 + E bytes per off-diagonal term
 * over NVLink) into slots of dmv_get_info(ctx, "replicated_block") elements per rank, and each rank computes ITS rows by
 * the row traversal (k_gather, or the queued k_pull for bases with permutation symmetries): no records, no atomics on y.
 * The hash partition of x, y and the representatives seen by the caller (SE:129-156) is unchanged.
 * Inside dmv_matvec the all-gather of x is one kernel of peer-direct NVLink stores into the CUDA-IPC-mapped gathered
 * vectors of all ranks plus release / acquire flags (option "peer_gather"; ncclAllGather when IPC mapping is impossible).
 * Bases with permutation symmetries run k_rows on a hash table over the whole basis, refilled from the gathered x.
 *   dmv_replicated_setup:   local set-up (whole basis, slot table); no communication.
 *   dmv_replicated_product: y <- rows of this rank applied to a caller-assembled gathered x (device pointers); for
 *                           hosts that own the all-gather themselves (several logical ranks on one GPU, tests). */
int dmv_replicated_setup(dmv_context *ctx);
int dmv_replicated_product(dmv_context *ctx, int elt, const void *x_cat, void *y);

/* ---- block <-> hashed redistribution of vectors (arrFromBlockToHashed, reference src/BlockToHashed.chpl:87-208;
 * arrFromHashedToBlock, src/HashedToBlock.chpl:67-153): how vectors in file (sorted-state) order enter and leave the
 * hash partition (test/TestMatrixVectorProduct.chpl:35,45).  "Block": the global array cut into contiguous chunks,
 * one per rank, with masks[i] = owner of element i (SE:138-156); "hashed": each rank holds the elements it owns,
 * ascending.  elt = 8-byte words per element (1: real(64) / uint(64), 2: complex128).  Host or device pointers.
 *   dmv_hashed_positions: positions[i] = slot of chunk element i in the ordering "grouped by owner, stable";
 *                         counts[r] = elements owned by r.  Building block of the two conversions.
 *   dmv_permute:          out[positions[i]] = in[i] (gather == 0) or out[i] = in[positions[i]] (gather != 0).
 *   dmv_block_to_hashed / dmv_hashed_to_block: the conversions, collective over the communicator (NCCL
 *                         all-to-all-v of the grouped chunks); with one rank they are the permutation alone. */
int dmv_hashed_positions(dmv_context *ctx, int64_t count, const uint8_t *masks, int num_ranks, int64_t *counts,
                         uint32_t *positions);
int dmv_permute(dmv_context *ctx, int elt, int64_t count, const uint32_t *positions, const void *in, void *out,
                int gather);
int dmv_block_to_hashed(dmv_context *ctx, int elt, int64_t chunk_count, const uint8_t *masks_chunk,
                        const void *block_chunk, void *hashed, int64_t hashed_count);
int dmv_hashed_to_block(dmv_context *ctx, int elt, int64_t chunk_count, const uint8_t *masks_chunk,
                        const void *hashed, int64_t hashed_count, void *block_chunk);

/* ---- communicator (NCCL over NVLink): 128-byte unique id made on rank 0, shared by the host */
int dmv_comm_unique_id(void *id128);
int dmv_comm_init(dmv_context *ctx, const void *id128);

/* ---- several vectors per call: numVectors > 1 of ls_chpl_matrix_vector_product, which the reference itself does not
 * implement (DMV:1101-1102 halts; its eigensolver loops over columns, src/Diagonalize.chpl:154-158).  x, y hold
 * num_vectors vectors of dmv_number_states elements one after the other (the [numVectors, N] layout of BlockVector).
 * On one rank: with device pointers and an operator k_gather applies to, four vectors at a time share the term walk and the
 * index look-ups; on bases with permutation symmetries (k_rows) up to six doubles per state -- six real or three complex
 * vectors -- share the orbit minimum and ONE 64-byte look-up per term (k_rows_batch; host vectors are staged a batch at a
 * time).  Everything else is the loop over dmv_local_matvec / dmv_matvec.  Semantics per vector as for a single product.
 * (The ls_chpl_* entry keeps the reference's behaviour and halts for numVectors != 1.) */
int dmv_matvec_batch(dmv_context *ctx, int elt, int num_vectors, const void *x, void *y);

/* ---- Lanczos ground state on the device ("next" row f3; the reference gives its product to PRIMME as the matvec
 * callback, src/Diagonalize.chpl:134-225).  Three-term recurrence with the vectors resident in HBM, dot products reduced
 * over the ranks with NCCL; converged when |beta_k s_k| <= tol * max(1, |theta|).  Collective when num_ranks > 1.
 * eigenvector (optional, host or device, dmv_number_states elements of type elt) is rebuilt in a second pass.
 * The start vector is a deterministic function of `seed`. */
int dmv_lanczos(dmv_context *ctx, int elt, int max_iters, double tol, uint64_t seed, double *eigenvalue,
                void *eigenvector, int *iterations, double *residual);

/* ---- per-stage timings of the last product, in milliseconds (the reference's timing tree,
 * DMV:1028-1052).  names: see dmv_timing_name(i); returns the number of stages. */
int dmv_last_timings(dmv_context *ctx, double *ms, int capacity);
const char *dmv_timing_name(int i);
/* algorithmic counters of the last plan: number of emitted off-diagonal terms of this rank */
int64_t dmv_number_terms(const dmv_context *ctx);

/* ---- the reference's plugin surface (src/FFI.chpl:233-239, DMV:1095-1110).  `op` is the
 * ls_hs_operator* the Haskell library hands out; it must have been bound to a context with
 * dmv_bind_operator (see INTEGRATION.md for the shim that extracts the flat tables). */
int dmv_bind_operator(const void *ls_hs_operator_ptr, dmv_context *ctx);
void ls_chpl_matrix_vector_product(const void *ls_hs_operator_ptr, int num_vectors, double *x, double *y);

/* PRIMME's matrix-vector callback (reference src/Diagonalize.chpl:134-162: `primme.matrixMatvec = ls_chpl_primme_matvec`):
 * y[:, k] = H x[:, k] for k < *block_size, real(64) columns with leading dimensions *ldx, *ldy >= dmv_number_states.
 * The reference finds the operator through primme->matrix; here the primme_params pointer is the handle and must have
 * been bound with dmv_bind_operator(primme, ctx).  Host or device columns; collective when the context has several
 * ranks; sets *ierr = 0 and halts on failure like the reference. */
void ls_chpl_primme_matvec(void *x, int64_t *ldx, void *y, int64_t *ldy, int *block_size, void *primme, int *ierr);

/* The other three entries of `ls_chpl_kernels` (src/FFI.chpl:233-239).  Outputs are returned the way Chapel's
 * convertToExternalArray does (BO:232,265-272): allocated by the callee, released by the caller through `freer`.
 * Layout of chpl_external_array (Chapel runtime, chpl-external-array.h): {void *elts; uint64_t num_elts; void *freer}.
 *   ls_chpl_operator_apply_diag      BO:217-234: coeffs[i] = <alpha_i|H|alpha_i> (real(64)), no projection
 *   ls_chpl_operator_apply_off_diag  BO:236-275: CSR by row: betas / coeffs (complex128) hold count * T entries of
 *                                    which offsets[count] are used, offsets = row pointer; terms with the same flip
 *                                    mask are merged into one entry; within a row entries are ordered by flip-mask
 *                                    group (the third-party kernel's order is not specified in the reference tree)
 *   ls_chpl_enumerate_representatives SE:588-603: this rank's block of representatives; `handle` is the ls_hs_basis*
 *                                    (bound with dmv_bind_operator like an operator handle); bounds are ignored
 *                                    exactly as in the reference
 * dmv_apply_diag / dmv_apply_off_diag are the same kernels on caller-owned arrays (host or device pointers;
 * betas: count * dmv_max_number_off_diag entries, coeffs: twice that many doubles, offsets: count + 1). */
typedef struct {
  void *elts;
  uint64_t num_elts;
  void (*freer)(void *);
} dmv_external_array;
int dmv_apply_diag(dmv_context *ctx, int64_t count, const uint64_t *alphas, double *coeffs);
int dmv_apply_off_diag(dmv_context *ctx, int64_t count, const uint64_t *alphas, uint64_t *betas, double *coeffs,
                       int64_t *offsets);
void ls_chpl_operator_apply_diag(const void *ls_hs_operator_ptr, int64_t count, const uint64_t *alphas,
                                 dmv_external_array *coeffs, int64_t num_tasks);
void ls_chpl_operator_apply_off_diag(const void *ls_hs_operator_ptr, int64_t count, const uint64_t *alphas,
                                     dmv_external_array *betas, dmv_external_array *coeffs,
                                     dmv_external_array *offsets, int64_t num_tasks);
void ls_chpl_enumerate_representatives(const void *ls_hs_basis_ptr, uint64_t lower, uint64_t upper,
                                       dmv_external_array *dest);

/* ---- host-side pieces exposed for the CPU tests (no device needed; NOT on the product path).
 * dmv_debug_tridiagonal_lowest: lowest eigenpair of a symmetric tridiagonal matrix, the host half of dmv_lanczos.
 * dmv_debug_compile_group: compiles the symmetry group of `basis` into the device orbit program, verifies it against
 *   bit-by-bit permutation and evaluates the compiled program (the device functions themselves, compiled for the host)
 *   for `count` states: reps[k] = min_g g(s_k), stab[k] = |{g : g(s_k) = s_k}|.
 *   info[0..5] = {n_q, n_stages, n_t, n_left, n_right, has_flip}. */
int dmv_debug_tridiagonal_lowest(int k, const double *diag, const double *offdiag, double *eigenvalue, double *vector);
int dmv_debug_compile_group(const dmv_basis_desc *basis, int64_t *info, int64_t count,
                            const uint64_t *states, uint64_t *reps, int32_t *stab);

#ifdef __cplusplus
}
#endif
#endif /* DMV_B200_H */
