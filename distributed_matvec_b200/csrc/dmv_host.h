// dmv_host.h -- host-side declarations shared by the translation units of libdmv_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "dmv_device.cuh"

namespace dmv {

struct HostOrbitProgram {
  int32_t n_sites = 0, n_q = 0, n_stages = 0, n_t = 0, n_left = 0, n_right = 0;
  int32_t has_flip = 0, trivial_characters = 1;
  uint64_t site_mask = 0;
  int64_t group_order = 0;
  std::vector<uint64_t> benes_mask;
  std::vector<int32_t> benes_delta;
  std::vector<uint64_t> step_mask;
  std::vector<int32_t> step_shift;
  std::vector<double> characters;  // interleaved, [n_q][n_t][2][2]
  std::vector<uint32_t> step_pack32;  // 4 words per step (empty unless simple and n_sites <= 32)
  std::vector<uint64_t> step_pack64;  // 3 words per step (empty unless simple)
  int32_t simple = 0;
  int32_t canon_mode = 0, canon_k = 0, canon_r = 0;   // block-rotation canonical form of the chain subgroup
  int32_t chain_dihedral = 0;
  std::vector<uint16_t> canon_lut;
  std::vector<uint64_t> canon_masks;
  std::vector<uint32_t> canon_lut2;      // pair LUT (empty: single-block LUT)
  int32_t canon_div = 0;
  std::vector<int32_t> cc_begin, cc_delta;   // coset chain of the canonical-form scan
  std::vector<uint64_t> cc_mask;
  int32_t tor_mode = 0, tor_rho_n = 0, tor_tau_n = 0, tor_div_r = 0;   // full-space-group canonical form of a torus
  std::vector<uint16_t> tor_lutm;
  std::vector<uint32_t> tor_luts;
  std::vector<uint8_t> tor_frow;
  std::vector<uint64_t> tor_net_mask;
  std::vector<int32_t> tor_net_delta;
  OrbitProgram view() const;       // pointers into the host vectors
};

HostOrbitProgram compile_orbit_program(int n_sites, int64_t group_order, const int32_t *perms,
                                       const uint8_t *flips, const double *characters);

// projection mode of the basis: which branch of BatchedOperator.computeOffDiag applies
// (reference src/BatchedOperator.chpl:89, 119, 163)
enum Projection { PROJ_NONE = 0, PROJ_INVERSION = 1, PROJ_GROUP = 2 };

// Everything a kernel needs, passed by value (fits the 4 KB kernel-parameter space).
struct KernelParams {
  // basis block of this rank
  StateIndex index;
  const double *norms;        // [n] (PROJ_GROUP only)
  // operator
  // (the host points these at the column-traversal (push) or row-traversal (pull) tables, see k_pull)
  const LutGroup *groups;  int32_t n_groups;
  const double *lut;       int32_t n_lut;     // real table (CV = false) or interleaved complex (CV = true)
  const OffTerm *terms;    int32_t n_terms;   // only read by groups with the generic flag
  int32_t any_generic, any_s_out;
  const BpWord *bp; int32_t n_bp;   // bit-parallel emit test (n_bp == 0: walk the groups one by one)
  uint64_t rank_total;        // INDEX_RANK: C(n_sites, weight)
  const DiagTerm *diag;    int32_t n_diag;       // all diagonal terms (n_diag > 0 <=> the operator has a diagonal)
  const DiagClass *diag_classes; int32_t n_diag_classes;   // bit-parallel part
  int32_t n_diag_rest;        // terms diag[0 .. n_diag_rest) are NOT covered by the classes (evaluated one by one)
  // symmetry
  OrbitProgram orbit;         // device pointers (PROJ_GROUP)
  uint64_t site_mask;
  double inversion_character; // PROJ_INVERSION: spin_inversion as a double
  // partition
  int32_t rank, num_ranks;
  // vectors
  const void *x; void *y;
  // outgoing buckets (num_ranks > 1): records for destination d go to out_betas + out_offset[d]
  uint64_t *out_betas; double *out_coeffs;
  const int64_t *out_offset;      // [num_ranks + 1] device
  unsigned long long *out_count;  // [num_ranks] device, reset before each generate
  // exact warp-private regions (num_ranks <= 32): the grid-stride tile loop is deterministic, so the
  // counting pass records how many records every warp emits per destination and the real pass starts
  // each warp at the prefix sum -- no slot-claim atomics, no slack, deterministic bucket layout.
  int32_t grid_blocks;              // 0: size the grid from occupancy; else exactly this many CTAs
  int32_t row_split;                // lanes sharing one source state (1, 2, 4, ... 32), see k_generate
  const int64_t *warp_offsets;      // [grid_blocks * 8][num_ranks]
  unsigned long long *warp_counts;  // counting pass output, same shape
  uint64_t *const *out_betas_ptr;   // [num_ranks]: base of MY region in the destination's record buffer
  double *const *out_coeffs_ptr;    //              (a local bucket, or the peer's incoming buffer over NVLink)
  const int64_t *out_capacity;      // [num_ranks]
  // emit_all: computeOffDiag mode -- every record goes to one flat output with its locale key
  int32_t emit_all; uint8_t *out_keys;
  // error reporting: status[0] = number of bad records, status[1] = first bad state, status[2] = overflow
  unsigned long long *status;
  // source range of this launch
  int64_t row_begin, row_end;
  // k_gather: the coefficient shared by every emitting (group, support bits) pair, when there is one
  double uni_re, uni_im;
  // k_gather / k_pull, replicated-x product (several ranks, every rank holds the whole basis and an all-gathered x):
  //   rows come from row_states (this rank's block) while `index` describes the GLOBAL basis; global index g lives
  //   at x[pos[g]]; the row's own element is x[x_row_offset + i].  All null / zero on one rank.
  const uint64_t *row_states;
  const double *row_norms;     // norms of the rows (k_pull on bases with permutation symmetries); `norms` is then global
  const uint32_t *pos;
  int64_t x_row_offset;
  // k_gather on several vectors at once: vector k of x / y starts batch_stride elements after vector k - 1
  int32_t gather_walk;         // k_gather: 0 per-lane walk from the top bit (default), 1 group-major, 2 per-lane from the bottom
  int32_t batch;               // 0 / 1: one vector; 4: four vectors per launch (k_gather); 2 .. 6: k_rows_batch
  int32_t batch_elt;           // k_rows_batch: doubles per vector element (1 | 2); batch * batch_elt <= 6
  int64_t batch_stride;
  // k_rows (row traversal of bases with permutation symmetries): hash table over the representatives with the scaled
  // vector element in the slot (see table_slot in dmv_device.cuh)
  const void *table;
  uint32_t table_slots;
  // ... or, with a dense index: perfect hash -> slot of `dense` (32 bytes: {key, spare, re, im} / 16 bytes: {key, value});
  // `table` then only holds the few per cent of the states the two levels could not place
  PerfectHash mph;
  const void *dense;
  int32_t rows_ctas;           // k_rows / k_rows_batch: resident CTAs per SM the kernel is compiled for (3 default | 2 | 4)
};

// launchers (dmv_kernels.cu)
struct LaunchConfig { int blocks; int threads; size_t smem; };
void launch_generate(const KernelParams &p, Projection proj, bool complex_values, bool complex_elements,
                     bool count_only, cudaStream_t stream);
void launch_pull(const KernelParams &p, Projection proj, bool complex_values, bool complex_elements,
                 cudaStream_t stream);
// row traversal without queue / atomics for bit-parallel operators on unprojected or inversion-only bases
void launch_gather(const KernelParams &p, bool inversion, bool complex_values, bool complex_elements,
                   bool narrow, bool lin, bool uniform, cudaStream_t stream);
// k_rows applies to real operators with a bit-parallel emit test on bases with trivial characters; returns the
// instantiation it launched as 100 CTAS + 10 TK + MPH (0: nothing launched)
int launch_rows(const KernelParams &p, bool complex_elements, cudaStream_t stream);
// hash table of k_rows: insert every state (slot_of[i] = its slot), then per product table[slot_of[i]] = x[src(i)] * norm[i]
// with src(i) = pos ? pos[i] : i
void launch_table_insert(const uint64_t *reps, int64_t n, void *table, uint32_t n_buckets, int slots_per_bucket,
                         uint32_t *slot_of, cudaStream_t stream, int bucket_bytes = 32);
// k_rows on several vectors at once: 64-byte buckets { key, six doubles, spare } shared by the vectors of the batch
int launch_rows_batch(const KernelParams &p, cudaStream_t stream);   // -> 100 CTAS + 10 TK (0: nothing launched)
void launch_table_fill_batch(int64_t n, int num_vectors, int elt, const void *x, int64_t stride, const double *norms,
                             const uint32_t *slot_of, const uint64_t *reps, void *table, cudaStream_t stream);
void launch_table_fill(int64_t n, bool complex_elements, const void *x, const double *norms, const uint32_t *pos,
                       const uint32_t *slot_of, const uint64_t *reps, void *table, void *dense, cudaStream_t stream);
// perfect-hash set-up (k_rows dense index): mark the positions of `n` states at a level in seen / collide bit arrays
// (192 bits per block, 3 words each), and compact the states whose position collided into `next`
void launch_mph_mark(const uint64_t *keys, int64_t n, int level, uint32_t n_blocks, unsigned long long *seen,
                     unsigned long long *collide, cudaStream_t stream);
void launch_mph_compact(const uint64_t *keys, int64_t n, int level, uint32_t n_blocks, const unsigned long long *collide,
                        uint64_t *next, unsigned long long *next_count, cudaStream_t stream);
// slot of every state: dense slot through the perfect hash, or 0x80000000 | (slot in the open-addressing table)
void launch_mph_slots(const uint64_t *keys, int64_t n, PerfectHash mph, const void *table, uint32_t n_buckets,
                      int slots_per_bucket, uint32_t *slot_of, unsigned long long *status, cudaStream_t stream);
void launch_accumulate(const KernelParams &p, Projection proj, bool complex_values, bool complex_elements,
                       int64_t count, const uint64_t *betas, const double *coeffs, cudaStream_t stream);
// plugin kernels (BO:217-275): diagonal coefficients / CSR list of off-diagonal terms of caller-given states
void launch_apply_diag(const KernelParams &p, int64_t count, const uint64_t *alphas, double *coeffs, cudaStream_t stream);
void launch_apply_off_diag(const KernelParams &p, int64_t count, const uint64_t *alphas, const int64_t *offsets,
                           int64_t *counts, uint64_t *betas, double *coeffs, bool write_pass, cudaStream_t stream);
void launch_build_directory(const uint64_t *reps, int64_t n, uint32_t *dir, uint64_t n_buckets, int shift,
                            cudaStream_t stream);
void launch_state_index(const StateIndex &ix, int64_t count, const uint64_t *spins, int64_t *indices,
                        cudaStream_t stream);
void launch_state_info(const OrbitProgram &P, Projection proj, uint64_t site_mask, double inv_char,
                       int64_t count, const uint64_t *alphas, uint64_t *betas, double *characters,
                       double *norms, cudaStream_t stream);
void launch_verify_rank(const StateIndex &ix, unsigned long long *status, cudaStream_t stream);
void launch_locale_idx(int64_t count, const uint64_t *states, int num_ranks, uint8_t *keys, cudaStream_t stream);
void launch_compute_norms(const OrbitProgram &P, int64_t count, const uint64_t *reps, double *norms,
                          cudaStream_t stream);
// enumeration: chunk c covers candidates [chunk_first[c], chunk_first[c] + chunk_len[c]) in the
// combinadic (fixed Hamming weight) or plain integer order; pass 0 counts, pass 1 writes.
void launch_enumerate(const OrbitProgram &P, Projection proj, uint64_t site_mask, bool fixed_hamming,
                      int rank, int num_ranks, int64_t n_chunks, const uint64_t *chunk_first,
                      const uint64_t *chunk_last, unsigned long long *chunk_count,
                      const unsigned long long *chunk_offset, uint64_t *out, double *out_norms,
                      bool write_pass, cudaStream_t stream);
// replicated-x set-up: owner and position of every global state in the all-gathered x.
//   pass 0: chunk_counts[c * P + r] = states of chunk c owned by r;  pass 1: pos[g] = r * block + chunk_base[c * P + r] + k
// (owners from hash64_01(states[g]) % P, or from masks[g] when masks != nullptr)
void launch_owner_positions(const uint64_t *states, const uint8_t *masks, int64_t n, int num_ranks, int64_t chunk,
                            bool write_pass, unsigned long long *chunk_counts, const unsigned long long *chunk_base,
                            int64_t block, uint32_t *pos, cudaStream_t stream);
// out[pos[i]] = in[i] (gather == false) or out[i] = in[pos[i]]; elt = 8-byte words per element (1 or 2)
void launch_permute(int64_t n, int elt, const uint32_t *pos, const void *in, void *out, bool gather, cudaStream_t stream);
// peer-direct all-gather of x (replicated-x product): my block into slot `rank` of every rank's gathered vector over
// NVLink, then my flag in every peer; the consumer waits for all flags of the epoch
void launch_push_block(const void *x, int64_t n_doubles, int num_ranks, void *const *peer_slot, unsigned *done,
                       unsigned *const *peer_flags, int rank, unsigned epoch, bool wide, cudaStream_t stream);
void launch_raise_flags(unsigned *const *peer_flags, int num_ranks, int rank, unsigned value, cudaStream_t stream);
void launch_wait_flags(const unsigned *flags, int num_ranks, unsigned epoch, unsigned long long *status,
                       cudaStream_t stream);
// Lanczos vector kernels (dmv_solver.cu); n = elements, words = 8-byte words
void launch_dot(int64_t n, bool complex_elements, const double *a, const double *b, double *out2, cudaStream_t s);
void launch_lanczos_update(int64_t n, bool complex_elements, double *w, const double *v, const double *u,
                           const double *coef2, double *out1, cudaStream_t s);
void launch_scale(int64_t words, double scale, const double *x, double *y, bool accumulate, cudaStream_t s);
void launch_fill(int64_t words, uint64_t seed, uint64_t offset, double *x, cudaStream_t s);
int64_t launch_counter();
int planned_grid(int64_t rows, int row_split);
int choose_row_split(int64_t rows, int n_groups);
constexpr int kWarpsPerCta = 8;

}  // namespace dmv
