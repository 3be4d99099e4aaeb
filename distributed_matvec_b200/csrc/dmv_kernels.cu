// dmv_kernels.cu -- hand-written sm_100a kernels of the distributed matrix-free H.x product.
//
//   k_generate   : diagonal + off-diagonal term generation (BatchedOperator.computeOffDiag, reference
//                  src/BatchedOperator.chpl:82-213) fused with the destination hash (localeIdxOf,
//                  src/StatesEnumeration.chpl:129-136), the per-destination bucketing (radixOneStep,
//                  DMV:265-311) and -- for the records this rank owns -- the index search and atomic
//                  accumulate (localProcess, DMV:73-127).
//   k_accumulate : localProcess for records received from other ranks.
//
// Work decomposition of k_generate: a warp owns 32 consecutive source states (one per lane, coalesced
// 8-byte loads of sigma_i and x_i), walks the flip-mask groups of the operator in lock step (tables in
// shared memory, broadcast reads), and compacts the emitted (beta, c*x_i) pairs into a warp-private
// ring buffer in shared memory.  Whenever 32 entries are queued the warp drains them with all lanes
// busy: symmetry projection (orbit scan in registers), hash, directory + bounded binary search in the
// sorted representatives, FP64 atomic add.  This keeps the expensive part (projection, search,
// atomics) at full lane occupancy although only ~half of the (state, bond) pairs emit a term.
#include <cuda_runtime.h>

#include <atomic>
#include <stdexcept>
#include <string>

#include "dmv_host.h"

namespace dmv {

static std::atomic<int64_t> g_launches{0};
int64_t launch_counter() { return g_launches.load(); }
void count_launch() { g_launches++; }

#define DMV_CUDA_CHECK(expr)                                                                    \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      throw std::runtime_error(std::string(#expr) + ": " + cudaGetErrorString(_e));            \
  } while (0)

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kQueue = 128;  // ring capacity per warp (>= 63 pending + 32 appended)

// ---- value helpers: V = double (real coefficients and real x) or double2 (complex) -------------
template <bool CV> struct ValT { using type = double; };
template <> struct ValT<true> { using type = double2; };

__device__ __forceinline__ double v_make(double re, double, double *) { return re; }
__device__ __forceinline__ double2 v_make(double re, double im, double2 *) { return make_double2(re, im); }
__device__ __forceinline__ double v_mul(double a, double b) { return a * b; }
__device__ __forceinline__ double2 v_mul(double2 a, double2 b) {
  return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double v_scale(double a, double s) { return a * s; }
__device__ __forceinline__ double2 v_scale(double2 a, double s) { return make_double2(a.x * s, a.y * s); }
__device__ __forceinline__ bool v_nonzero(double a) { return a != 0.0; }
__device__ __forceinline__ bool v_nonzero(double2 a) { return a.x != 0.0 || a.y != 0.0; }
__device__ __forceinline__ void v_acc(double &a, double re, double) { a += re; }
__device__ __forceinline__ void v_acc(double2 &a, double re, double im) { a.x += re; a.y += im; }

template <bool CE>
__device__ __forceinline__ void atomic_accumulate(void *y, int64_t idx, double re, double im) {
  if (CE) {
    double *p = reinterpret_cast<double *>(y) + 2 * idx;
    atomicAdd(p, re);
    atomicAdd(p + 1, im);
  } else {
    atomicAdd(reinterpret_cast<double *>(y) + idx, re);
  }
}
__device__ __forceinline__ double v_re(double a) { return a; }
__device__ __forceinline__ double v_re(double2 a) { return a.x; }
__device__ __forceinline__ double v_im(double) { return 0.0; }
__device__ __forceinline__ double v_im(double2 a) { return a.y; }

// ---- shared-memory staging of the operator / orbit tables ---------------------------------------
struct SmemLayout {
  size_t groups, gx, bp, lut, terms, diag, dclass, orbit64, orbit32, canon, binom, queues, total;
};
__host__ __device__ inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
__host__ __device__ inline SmemLayout smem_layout(const KernelParams &p, int proj, size_t val_bytes,
                                                  bool queues = true) {
  SmemLayout L;
  size_t off = 0;
  // bit-parallel mode keeps only the flip masks (compact) and the word descriptors; the full group
  // records are needed when groups are walked one by one or carry an outside sign mask
  const bool full_groups = p.n_bp == 0 || p.any_s_out;
  L.groups = off; off += full_groups ? sizeof(LutGroup) * p.n_groups : 0;
  L.gx = off; off += 8 * (size_t)p.n_groups;
  L.bp = off; off += sizeof(BpWord) * p.n_bp;
  off = align_up(off, 16);
  L.lut = off; off += val_bytes * p.n_lut;
  off = align_up(off, 8);
  L.terms = off; off += p.any_generic ? sizeof(OffTerm) * p.n_terms : 0;
  L.diag = off; off += sizeof(DiagTerm) * p.n_diag_rest;
  L.dclass = off; off += sizeof(DiagClass) * p.n_diag_classes;
  off = align_up(off, 16);   // packed orbit steps are read with 16-byte loads
  L.orbit64 = off;
  size_t n64 = 0, n32 = 0;
  if (proj == PROJ_GROUP) {
    const int np = p.orbit.n_left + p.orbit.n_right;
    const size_t steps = (size_t)(p.orbit.n_t - 1);
    n64 = (size_t)p.orbit.n_q * p.orbit.n_stages;
    if (n64 & 1) ++n64;   // keep the packed steps 16-byte aligned
    n32 = (size_t)p.orbit.n_stages;
    if (p.orbit.simple) n64 += p.orbit.step_pack32 ? 2 * steps : 3 * steps;   // packed steps only
    else { n64 += steps * np; n32 += steps * np; }
  }
  off += 8 * n64;
  L.orbit32 = off; off += 4 * n32;
  // canonical-form scan: coset chain (masks, then begin / delta) and the pair LUT
  off = align_up(off, 8);
  L.canon = off;
  if (proj == PROJ_GROUP && p.orbit.canon_mode != 0 && p.orbit.tor_mode != 0) {
    // full-space-group canonical form: delta-swap stages of rho / tau and the 16-bit pair table
    const size_t n_st = (size_t)(p.orbit.tor_rho_n + p.orbit.tor_tau_n);
    off += 8 * n_st + 4 * n_st;
    off = align_up(off, 16);                                    // bulk copies need 16-byte aligned destinations
    off += 2 * ((size_t)1 << (2 * p.orbit.canon_k));            // tor_lutm
    off += align_up((size_t)4 * p.orbit.canon_k << p.orbit.canon_k, 16);   // tor_frow
    off += 16;                                                  // mbarrier of the bulk copies
    off = align_up(off, 8);
  } else if (proj == PROJ_GROUP && p.orbit.canon_mode != 0) {
    const size_t n_st = p.orbit.cc_n > 0 ? (size_t)p.orbit.cc_stages : 0;
    off += 8 * n_st + 4 * (n_st + (p.orbit.cc_n > 0 ? (size_t)p.orbit.cc_n + 1 : 0));
    off = align_up(off, 4);
    if (p.orbit.canon_lut2) off += 4 * ((size_t)1 << (2 * p.orbit.canon_k));
  }
  L.binom = off;
  if (p.index.mode == INDEX_RANK) off += 4 * (size_t)p.index.n_sites * p.index.stride;
  off = align_up(off, 16);
  // per warp: ring of (beta, value) + (pull mode) source lane and a row accumulator
  L.queues = off; off += queues ? (size_t)kWarps * (kQueue * (8 + val_bytes) + kQueue + 32 * val_bytes) : 0;
  L.total = off;
  return L;
}

template <typename T>
__device__ __forceinline__ void stage(T *dst, const T *src, int count) {
  for (int i = threadIdx.x; i < count; i += blockDim.x) dst[i] = src[i];
}

// Two global -> shared bulk copies through the TMA engine (cp.async.bulk; sizes multiples of 16, 16-byte aligned), issued
// by one thread and awaited by the whole CTA on an mbarrier.  The source buffers are over-allocated to the padded size.
__device__ __forceinline__ void bulk_stage2(void *dst0, const void *src0, uint32_t bytes0, void *dst1, const void *src1,
                                            uint32_t bytes1, uint64_t *mbar) {
  const uint32_t bar = (uint32_t)__cvta_generic_to_shared(mbar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes0 + bytes1) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(dst0)), "l"(src0), "r"(bytes0), "r"(bar) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(dst1)), "l"(src1), "r"(bytes1), "r"(bar) : "memory");
  }
  uint32_t done = 0;
  while (!done) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar) : "memory");
  }
}

// Everything a CTA keeps in shared memory, set up once per CTA.
template <bool CV>
struct Tables {
  using V = typename ValT<CV>::type;
  const LutGroup *groups;
  const uint64_t *gx;   // flip mask of every group
  const BpWord *bp;
  int n_bp;
  const V *lut;
  const OffTerm *terms;
  const DiagTerm *diag;
  const DiagClass *dclass;
  int n_diag_rest, n_dclass;
  OrbitProgram orbit;
  StateIndex index;
};

template <int PROJ, bool CV>
__device__ __forceinline__ Tables<CV> stage_tables(const KernelParams &p, unsigned char *smem, const SmemLayout &L) {
  using V = typename ValT<CV>::type;
  Tables<CV> T;
  LutGroup *s_groups = reinterpret_cast<LutGroup *>(smem + L.groups);
  V *s_lut = reinterpret_cast<V *>(smem + L.lut);
  OffTerm *s_terms = reinterpret_cast<OffTerm *>(smem + L.terms);
  DiagTerm *s_diag = reinterpret_cast<DiagTerm *>(smem + L.diag);
  uint64_t *s_gx = reinterpret_cast<uint64_t *>(smem + L.gx);
  BpWord *s_bp = reinterpret_cast<BpWord *>(smem + L.bp);
  if (p.n_bp == 0 || p.any_s_out) stage(s_groups, p.groups, p.n_groups);
  for (int i = threadIdx.x; i < p.n_groups; i += blockDim.x) s_gx[i] = p.groups[i].x;
  stage(reinterpret_cast<uint64_t *>(s_bp), reinterpret_cast<const uint64_t *>(p.bp),
        p.n_bp * (int)(sizeof(BpWord) / 8));
  T.gx = s_gx; T.bp = s_bp; T.n_bp = p.n_bp;
  stage(s_lut, reinterpret_cast<const V *>(p.lut), p.n_lut);
  if (p.any_generic) stage(s_terms, p.terms, p.n_terms);
  stage(s_diag, p.diag, p.n_diag_rest);
  DiagClass *s_dclass = reinterpret_cast<DiagClass *>(smem + L.dclass);
  stage(reinterpret_cast<uint64_t *>(s_dclass), reinterpret_cast<const uint64_t *>(p.diag_classes),
        p.n_diag_classes * (int)(sizeof(DiagClass) / 8));
  T.groups = s_groups; T.lut = s_lut; T.terms = s_terms; T.diag = s_diag;
  T.dclass = s_dclass; T.n_diag_rest = p.n_diag_rest; T.n_dclass = p.n_diag_classes;
  T.orbit = p.orbit;
  if (PROJ == PROJ_GROUP) {
    const int np = T.orbit.n_left + T.orbit.n_right;
    uint64_t *s64 = reinterpret_cast<uint64_t *>(smem + L.orbit64);
    int32_t *s32 = reinterpret_cast<int32_t *>(smem + L.orbit32);
    const int nb = T.orbit.n_q * T.orbit.n_stages, steps = T.orbit.n_t - 1;
    const int nb_pad = nb + (nb & 1);
    stage(s64, p.orbit.benes_mask, nb);
    stage(s32, p.orbit.benes_delta, T.orbit.n_stages);
    T.orbit.benes_mask = s64;
    T.orbit.benes_delta = s32;
    if (T.orbit.simple) {
      // only the packed steps live in shared memory; the general arrays (rare paths) stay in global
      if (p.orbit.step_pack32) {
        stage(s64 + nb_pad, reinterpret_cast<const uint64_t *>(p.orbit.step_pack32), 2 * steps);
        T.orbit.step_pack32 = reinterpret_cast<const uint4 *>(s64 + nb_pad);
      } else {
        stage(s64 + nb_pad, p.orbit.step_pack64, 3 * steps);
        T.orbit.step_pack64 = s64 + nb_pad;
      }
    } else {
      stage(s64 + nb_pad, p.orbit.step_mask, steps * np);
      stage(s32 + T.orbit.n_stages, p.orbit.step_shift, steps * np);
      T.orbit.step_mask = s64 + nb_pad;
      T.orbit.step_shift = s32 + T.orbit.n_stages;
    }
  }
  if (PROJ == PROJ_GROUP && T.orbit.canon_mode != 0 && T.orbit.tor_mode != 0) {
    unsigned char *base = smem + L.canon;
    const int n_st = T.orbit.tor_rho_n + T.orbit.tor_tau_n;
    uint64_t *nm = reinterpret_cast<uint64_t *>(base);
    int32_t *nd = reinterpret_cast<int32_t *>(base + 8 * (size_t)n_st);
    uint16_t *lm = reinterpret_cast<uint16_t *>(smem + align_up((size_t)(base - smem) + 12 * (size_t)n_st, 16));
    stage(nm, p.orbit.tor_net_mask, n_st);
    stage(nd, p.orbit.tor_net_delta, n_st);
    // the pair table (8 KB for k = 6) and the row table arrive as two TMA bulk copies (cp.async.bulk, one elected
    // thread, completion on an mbarrier) instead of a strided loop of every thread
    const uint32_t lut_bytes = 2u << (2 * T.orbit.canon_k);
    const uint32_t frow_bytes = (uint32_t)align_up((size_t)4 * T.orbit.canon_k << T.orbit.canon_k, 16);
    uint8_t *fr = reinterpret_cast<uint8_t *>(lm) + lut_bytes;
    uint64_t *mbar = reinterpret_cast<uint64_t *>(fr + frow_bytes);
    bulk_stage2(lm, p.orbit.tor_lutm, lut_bytes, fr, p.orbit.tor_frow, frow_bytes, mbar);
    T.orbit.tor_net_mask = nm; T.orbit.tor_net_delta = nd; T.orbit.tor_lutm = lm; T.orbit.tor_frow = fr;
  } else if (PROJ == PROJ_GROUP && T.orbit.canon_mode != 0) {
    unsigned char *base = smem + L.canon;
    if (T.orbit.cc_n > 0) {
      const int n_st = T.orbit.cc_stages;
      uint64_t *cm = reinterpret_cast<uint64_t *>(base);
      int32_t *cb = reinterpret_cast<int32_t *>(base + 8 * (size_t)n_st);
      int32_t *cd = cb + (T.orbit.cc_n + 1);
      stage(cm, p.orbit.cc_mask, n_st);
      stage(cb, p.orbit.cc_begin, T.orbit.cc_n + 1);
      stage(cd, p.orbit.cc_delta, n_st);
      T.orbit.cc_mask = cm; T.orbit.cc_begin = cb; T.orbit.cc_delta = cd;
      base += 8 * (size_t)n_st + 4 * ((size_t)n_st + T.orbit.cc_n + 1);
    }
    base = smem + align_up((size_t)(base - smem), 4);
    if (T.orbit.canon_lut2) {
      uint32_t *l2 = reinterpret_cast<uint32_t *>(base);
      stage(l2, p.orbit.canon_lut2, 1 << (2 * T.orbit.canon_k));
      T.orbit.canon_lut2 = l2;
    }
  }
  T.index = p.index;
  if (T.index.mode == INDEX_RANK) {
    uint32_t *sb = reinterpret_cast<uint32_t *>(smem + L.binom);
    stage(sb, p.index.binom, T.index.n_sites * T.index.stride);
    T.index.binom = sb;
  }
  return T;
}

// ---- term generation ----------------------------------------------------------------------------
// generic (term by term) evaluation of one group: c = sum_t v_t [a & m == r] (-1)^popc(a & s)
template <bool CV>
__device__ __noinline__ typename ValT<CV>::type generic_coefficient(const OffTerm *terms, int first, int count,
                                                                     uint64_t a, bool *hit) {
  using V = typename ValT<CV>::type;
  V c = v_make(0.0, 0.0, (V *)nullptr);
  bool any = false;
  for (int t = first; t < first + count; ++t) {
    const OffTerm term = terms[t];
    if ((a & term.m) == term.r) {
      const double sg = (__popcll(a & term.s) & 1) ? -1.0 : 1.0;
      v_acc(c, sg * term.v_re, sg * term.v_im);
      any = true;
    }
  }
  *hit = any;
  return c;
}

// The terms one row emits within a word of <= 64 groups.
struct RowTerms {
  uint64_t mask;     // bit g - g0 set <=> group g emits
  uint64_t a0, a1;   // bit-parallel mode: the two support bits of every group (for the LUT index)
};

// All lanes evaluate the same word in lock step (table reads are shared-memory broadcasts).
template <bool CV>
__device__ __forceinline__ RowTerms row_terms(const Tables<CV> &T, int w, int g0, int g1, uint64_t a) {
  RowTerms rt;
  rt.mask = 0; rt.a0 = 0; rt.a1 = 0;
  if (T.n_bp > 0) {
    const BpWord &W = T.bp[w];
#pragma unroll 1
    for (int k = 0; k < W.n0; ++k) { const BpPair q = W.p0[k]; rt.a0 |= ((a << q.l) >> q.r) & q.m; }
#pragma unroll 1
    for (int k = 0; k < W.n1; ++k) { const BpPair q = W.p1[k]; rt.a1 |= ((a << q.l) >> q.r) & q.m; }
    rt.mask = (~rt.a0 & ~rt.a1 & W.tt[0]) | (rt.a0 & ~rt.a1 & W.tt[1]) | (~rt.a0 & rt.a1 & W.tt[2]) |
              (rt.a0 & rt.a1 & W.tt[3]);
    return rt;
  }
  for (int g = g0; g < g1; ++g) {
    const uint64_t posk = T.groups[g].posk;
    bool emit;
    if (posk >> 56) {
      bool hit;
      const auto c = generic_coefficient<CV>(T.terms, T.groups[g].first, T.groups[g].count, a, &hit);
      emit = hit && v_nonzero(c);   // same decision in the counting pass: the plan is exact
    } else {
      emit = (T.groups[g].emit_bits >> lut_index(posk, a)) & 1ull;
    }
    rt.mask |= (uint64_t)emit << (g - g0);
  }
  return rt;
}

// Pops the lowest emitting group of the row: returns its flip mask and coefficient for state a.
template <bool CV>
__device__ __forceinline__ typename ValT<CV>::type pop_term(const Tables<CV> &T, RowTerms &rt, int g0, uint64_t a,
                                                             bool any_s_out, uint64_t &flip) {
  using V = typename ValT<CV>::type;
  const int gl = __ffsll((long long)rt.mask) - 1;
  rt.mask &= rt.mask - 1;
  const int g = g0 + gl;
  flip = T.gx[g];
  V c;
  if (T.n_bp > 0) {
    const unsigned idx = (unsigned)((rt.a0 >> gl) & 1ull) | ((unsigned)((rt.a1 >> gl) & 1ull) << 1);
    c = T.lut[4 * g + idx];
    if (any_s_out && (__popcll(a & T.groups[g].s_out) & 1)) c = v_scale(c, -1.0);
    return c;
  }
  const LutGroup grp = T.groups[g];
  if (grp.posk >> 56) {
    bool hit;
    return generic_coefficient<CV>(T.terms, grp.first, grp.count, a, &hit);
  }
  c = T.lut[grp.lut_offset + lut_index(grp.posk, a)];
  if (any_s_out && (__popcll(a & grp.s_out) & 1)) c = v_scale(c, -1.0);
  return c;
}

template <bool CV>
__device__ __forceinline__ void diagonal(const Tables<CV> &T, int /*n_diag*/, uint64_t a, double &dre, double &dim) {
  dre = 0.0; dim = 0.0;
  // zz-like couplings, one class per distinct coefficient: count - 2 popc(antiparallel bonds)
  for (int c = 0; c < T.n_dclass; ++c) {
    const DiagClass &D = T.dclass[c];
    uint64_t a0 = 0, a1 = 0;
#pragma unroll 1
    for (int k = 0; k < D.n0; ++k) { const BpPair q = D.p0[k]; a0 |= ((a << q.l) >> q.r) & q.m; }
#pragma unroll 1
    for (int k = 0; k < D.n1; ++k) { const BpPair q = D.p1[k]; a1 |= ((a << q.l) >> q.r) & q.m; }
    const double w = (double)(D.count - 2 * __popcll((a0 ^ a1) & D.mask));
    dre += w * D.v_re;
    dim += w * D.v_im;
  }
  for (int t = 0; t < T.n_diag_rest; ++t) {
    const DiagTerm d = T.diag[t];
    if ((a & d.m) == d.r) {
      const double sg = (__popcll(a & d.s) & 1) ? -1.0 : 1.0;
      dre += sg * d.v_re;
      dim += sg * d.v_im;
    }
  }
}

// ---- the consumer side: one record per lane -----------------------------------------------------
// route(): projects beta (inversion / full group) and appends the record to the bucket of its owner when
// that is another rank.  Returns true when the record is this rank's own (to be searched + accumulated).
// All 32 lanes must call it (warp collectives); `active` lanes carry a record.
template <int PROJ, bool CV, bool CE, bool COUNT_ONLY>
__device__ __forceinline__ bool route(const KernelParams &p, const OrbitProgram &orbit, bool active,
                                      uint64_t &beta, typename ValT<CV>::type &c, unsigned long long &cur) {
  using V = typename ValT<CV>::type;
  const unsigned lane = threadIdx.x & 31u;
  if (PROJ == PROJ_INVERSION) {
    // reference src/BatchedOperator.chpl:145-152
    const uint64_t inv = beta ^ p.site_mask;
    if (inv < beta) { beta = inv; c = v_scale(c, p.inversion_character); }
  } else if (PROJ == PROJ_GROUP) {
    if (active) {
      if (orbit.trivial_characters) {
        beta = orbit_representative(orbit, beta);
      } else {
        const OrbitResult r = orbit_scan<false, false>(orbit, beta);
        beta = r.rep;
        const double2 chi = __ldg(orbit.characters + r.arg);   // state_info returns conj(chi)
        c = v_mul(c, v_make(chi.x, -chi.y, (V *)nullptr));
      }
    }
  }
  int owner = p.rank;
  if (p.num_ranks > 1) owner = locale_idx_of(beta, p.num_ranks);

  if (p.emit_all) {   // BatchedOperator.computeOffDiag output: (beta, coeff, key) flat, unordered
    if (active && !COUNT_ONLY) {
      if (PROJ == PROJ_GROUP) {   // norm of the representative: BO:200 `norms[k]`
        const double stab = orbit.trivial_characters ? (double)orbit_scan<true, false>(orbit, beta).stab
                                                     : orbit_stabiliser_sum(orbit, beta);
        const double nn = stab / (double)orbit.group_order;
        c = v_scale(c, nn > 1e-12 ? sqrt(nn) : 0.0);
      }
      const unsigned long long pos = atomicAdd(p.out_count, 1ull);
      if ((int64_t)pos < p.out_offset[1]) {
        p.out_betas[pos] = beta;
        reinterpret_cast<V *>(p.out_coeffs)[pos] = c;
        p.out_keys[pos] = (uint8_t)owner;
      }
    }
    return false;
  }

  if (p.num_ranks <= 32 && (p.num_ranks > 1 || COUNT_ONLY)) {
    // ---- remote records: lane d keeps this warp's cursor into destination d's region (exact regions
    // from the plan: no atomics).  In the counting pass every record (own ones too) is counted.
    const bool remote = active && (COUNT_ONLY || owner != p.rank);
    for (int d = 0; d < p.num_ranks; ++d) {   // warp-uniform
      const bool mine = remote && owner == d;
      const unsigned m = __ballot_sync(0xffffffffu, mine);
      if (m) {
        const unsigned long long base = __shfl_sync(0xffffffffu, cur, d);
        if (!COUNT_ONLY && mine) {
          const int64_t slot = (int64_t)base + __popc(m & ((1u << lane) - 1u));
          if (slot < p.out_capacity[d]) {
            p.out_betas_ptr[d][slot] = beta;
            reinterpret_cast<V *>(p.out_coeffs_ptr[d])[slot] = c;
          } else {
            atomicAdd(p.status + 2, 1ull);
          }
        }
        if ((int)lane == d) cur += __popc(m);
      }
    }
    if (COUNT_ONLY) return false;
    return active && owner == p.rank;
  }
  if (p.num_ranks > 1) {
    // ---- more than 32 ranks: warp-aggregated slot claim per destination with global atomics
    const bool remote = active && (COUNT_ONLY || owner != p.rank);
    const unsigned remote_mask = __ballot_sync(0xffffffffu, remote);
    if (remote) {
      const unsigned peers = __match_any_sync(remote_mask, owner);
      const int leader = __ffs(peers) - 1;
      unsigned long long base = 0;
      if ((int)lane == leader) base = atomicAdd(p.out_count + owner, (unsigned long long)__popc(peers));
      base = __shfl_sync(peers, base, leader);
      if (!COUNT_ONLY) {
        const int64_t pos = (int64_t)base + __popc(peers & ((1u << lane) - 1u));
        const int64_t cap = p.out_offset[owner + 1] - p.out_offset[owner];
        if (pos < cap) {
          const int64_t slot = p.out_offset[owner] + pos;
          p.out_betas[slot] = beta;
          reinterpret_cast<V *>(p.out_coeffs)[slot] = c;
        } else {
          atomicAdd(p.status + 2, 1ull);
        }
      }
    }
    if (COUNT_ONLY) return false;
    return active && owner == p.rank;
  }
  return active;
}

// finish(): localProcess (reference DMV:73-127) for one located record
template <int PROJ, bool CV, bool CE>
__device__ __forceinline__ void finish(const KernelParams &p, const OrbitProgram &orbit, bool active,
                                       uint64_t beta, typename ValT<CV>::type c, int64_t idx) {
  if (!active) return;
  if (idx >= 0) {
    if (PROJ == PROJ_GROUP) c = v_scale(c, __ldg(p.norms + idx));
    if (v_nonzero(c)) atomic_accumulate<CE>(p.y, idx, v_re(c), v_im(c));   // DMV:110: skip c == 0
  } else if (v_nonzero(c)) {
    bool fatal = true;
    if (PROJ == PROJ_GROUP && !orbit.trivial_characters)
      fatal = orbit_stabiliser_sum(orbit, beta) > 1e-12 * (double)orbit.group_order;  // zero-norm orbit
    if (fatal) {                                                             // DMV:115-118
      if (atomicAdd(p.status, 1ull) == 0) p.status[1] = beta;
    }
  }
}

// Two independent searches advanced in lock step: both directory loads, then both probes of every
// level, are in flight together (the search is a chain of dependent L2 accesses; this doubles the
// memory-level parallelism of a warp).
__device__ __forceinline__ void locate2(const StateIndex &ix, bool a0, uint64_t k0, bool a1, uint64_t k1,
                                        int64_t &i0, int64_t &i1) {
  if (ix.mode != INDEX_DIRECTORY) {
    i0 = a0 ? locate(ix, k0) : -1;
    i1 = a1 ? locate(ix, k1) : -1;
    return;
  }
  i0 = -1; i1 = -1;
  const uint64_t b0 = k0 >> ix.shift, b1 = k1 >> ix.shift;
  a0 = a0 && b0 < ix.n_buckets;
  a1 = a1 && b1 < ix.n_buckets;
  uint2 r0 = make_uint2(0, 0), r1 = make_uint2(0, 0);
  if (a0) r0 = __ldg(reinterpret_cast<const uint2 *>(ix.dir) + b0);
  if (a1) r1 = __ldg(reinterpret_cast<const uint2 *>(ix.dir) + b1);
  uint32_t lo0 = r0.x, hi0 = r0.y, lo1 = r1.x, hi1 = r1.y;
  while (lo0 < hi0 || lo1 < hi1) {
    const bool s0 = lo0 < hi0, s1 = lo1 < hi1;
    const uint32_t m0 = (lo0 + hi0) >> 1, m1 = (lo1 + hi1) >> 1;
    uint64_t v0 = 0, v1 = 0;
    if (s0) v0 = __ldg(ix.reps + m0);
    if (s1) v1 = __ldg(ix.reps + m1);
    if (s0) {
      if (v0 == k0) { i0 = m0; lo0 = hi0; }
      else if (v0 < k0) lo0 = m0 + 1; else hi0 = m0;
    }
    if (s1) {
      if (v1 == k1) { i1 = m1; lo1 = hi1; }
      else if (v1 < k1) lo1 = m1 + 1; else hi1 = m1;
    }
  }
}

// Drain up to 64 queued records of this warp: lane handles entries `lane` and `lane + 32`.
template <int PROJ, bool CV, bool CE, bool COUNT_ONLY>
__device__ __forceinline__ void drain(const KernelParams &p, const OrbitProgram &orbit, const StateIndex &index,
                                      const uint64_t *qb, const typename ValT<CV>::type *qc, unsigned head,
                                      unsigned n, unsigned long long &cur) {
  using V = typename ValT<CV>::type;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned p0 = (head + lane) & (kQueue - 1), p1 = (head + lane + 32) & (kQueue - 1);
  bool a0 = lane < n, a1 = lane + 32 < n;
  uint64_t k0 = a0 ? qb[p0] : 0ull, k1 = a1 ? qb[p1] : 0ull;
  V c0 = a0 ? qc[p0] : v_make(0.0, 0.0, (V *)nullptr), c1 = a1 ? qc[p1] : v_make(0.0, 0.0, (V *)nullptr);
  a0 = route<PROJ, CV, CE, COUNT_ONLY>(p, orbit, a0, k0, c0, cur);
  if (n > 32) a1 = route<PROJ, CV, CE, COUNT_ONLY>(p, orbit, a1, k1, c1, cur);   // n is warp-uniform
  else a1 = false;
  if (COUNT_ONLY) return;
  int64_t i0, i1;
  locate2(index, a0, k0, a1, k1, i0, i1);
  finish<PROJ, CV, CE>(p, orbit, a0, k0, c0, i0);
  finish<PROJ, CV, CE>(p, orbit, a1, k1, c1, i1);
}

// (symmetric bases: the orbit scan wants > 100 registers; three resident CTAs per SM hide its latencies better than
// two, at the price of a few spills outside the scan)
template <int PROJ, bool CV, bool CE, bool COUNT_ONLY>
__global__ void __launch_bounds__(kThreads, PROJ == PROJ_GROUP ? 3 : 1) k_generate(const KernelParams p) {
  using V = typename ValT<CV>::type;
  extern __shared__ __align__(16) unsigned char smem[];
  const SmemLayout L = smem_layout(p, PROJ, sizeof(V));
  const Tables<CV> T = stage_tables<PROJ, CV>(p, smem, L);
  __syncthreads();

  const unsigned lane = threadIdx.x & 31u;
  const unsigned warp = threadIdx.x >> 5;
  uint64_t *qb = reinterpret_cast<uint64_t *>(smem + L.queues) + warp * kQueue;
  V *qc = reinterpret_cast<V *>(smem + L.queues + (size_t)kWarps * kQueue * 8) + warp * kQueue;
  unsigned head = 0, count = 0;  // warp-uniform
  const bool any_s_out = p.any_s_out != 0;
  // lane d: cursor of this warp in destination d's region (see route())
  const int64_t gw = (int64_t)blockIdx.x * kWarps + warp;
  unsigned long long cur = 0;
  if (!COUNT_ONLY && p.num_ranks > 1 && p.num_ranks <= 32 && (int)lane < p.num_ranks)
    cur = (unsigned long long)p.warp_offsets[gw * p.num_ranks + lane];

  // row_split = S lanes share one source state (each takes every S-th flip-mask group): small bases get
  // S times more warps and S times shorter per-warp latency chains; large ones run with S = 1
  const int S = p.row_split > 1 ? p.row_split : 1;
  const int rows_per_tile = 32 / S;
  const unsigned slice = lane & (unsigned)(S - 1);
  uint64_t slice_mask = ~0ull;
  if (S > 1) {
    slice_mask = 0;
    for (int g = (int)slice; g < 64; g += S) slice_mask |= 1ull << g;
  }
  const int64_t n_rows = p.row_end - p.row_begin;
  const int64_t n_tiles = (n_rows + rows_per_tile - 1) / rows_per_tile;
  const int64_t warps_total = (int64_t)gridDim.x * kWarps;
  for (int64_t tile = (int64_t)blockIdx.x * kWarps + warp; tile < n_tiles; tile += warps_total) {
    const int64_t i = p.row_begin + tile * rows_per_tile + lane / S;
    const bool valid = i < p.row_end;
    uint64_t alpha = 0;
    V xi = v_make(0.0, 0.0, (V *)nullptr);
    if (valid) {
      alpha = __ldg(p.index.reps + i);
      if (!COUNT_ONLY) {
        if (CE) {
          const double2 t = __ldg(reinterpret_cast<const double2 *>(p.x) + i);
          xi = v_make(t.x, t.y, (V *)nullptr);
        } else {
          xi = v_make(__ldg(reinterpret_cast<const double *>(p.x) + i), 0.0, (V *)nullptr);
        }
      }
    }
    // ---- diagonal: y[i] += x[i] * sum_t v_t [alpha & m == r] (-1)^popc(alpha & s)   (DMV:36-53)
    if (!COUNT_ONLY && !p.emit_all && p.n_diag > 0 && valid && slice == 0) {
      double dre, dim;
      diagonal<CV>(T, p.n_diag, alpha, dre, dim);
      if (CE) {
        const double2 t = __ldg(reinterpret_cast<const double2 *>(p.x) + i);
        atomic_accumulate<true>(p.y, i, dre * t.x - dim * t.y, dre * t.y + dim * t.x);
      } else {
        // real vectors take the real part of the diagonal (ls_internal_operator_apply_diag_x1 on real(64))
        atomic_accumulate<false>(p.y, i, dre * __ldg(reinterpret_cast<const double *>(p.x) + i), 0.0);
      }
    }
    if (PROJ == PROJ_GROUP && valid && !COUNT_ONLY)
      xi = v_scale(xi, 1.0 / __ldg(p.norms + i));   // 1 / norm(alpha): BO:200

    // ---- off-diagonal: which groups emit (bit mask), then compact the emitted terms into the ring
    for (int g0 = 0, w = 0; g0 < p.n_groups; g0 += 64, ++w) {
      const int g1 = min(g0 + 64, p.n_groups);
      RowTerms rt = row_terms<CV>(T, w, g0, g1, alpha);
      rt.mask &= slice_mask;
      if (!valid) rt.mask = 0;
      for (;;) {
        const bool has = rt.mask != 0;
        const unsigned m = __ballot_sync(0xffffffffu, has);
        if (m == 0) break;
        if (has) {
          uint64_t flip;
          const V c = pop_term<CV>(T, rt, g0, alpha, any_s_out, flip);
          const unsigned pos = (head + count + __popc(m & ((1u << lane) - 1u))) & (kQueue - 1);
          qb[pos] = alpha ^ flip;
          if (!COUNT_ONLY) qc[pos] = v_mul(c, xi);
        }
        count += __popc(m);
        if (count >= 64) {
          __syncwarp();
          drain<PROJ, CV, CE, COUNT_ONLY>(p, T.orbit, T.index, qb, qc, head, 64, cur);
          head = (head + 64) & (kQueue - 1);
          count -= 64;
          __syncwarp();
        }
      }
    }
  }
  if (count > 0) {
    __syncwarp();
    drain<PROJ, CV, CE, COUNT_ONLY>(p, T.orbit, T.index, qb, qc, head, count, cur);
  }
  if (COUNT_ONLY && p.num_ranks <= 32 && (int)lane < p.num_ranks)
    p.warp_counts[gw * p.num_ranks + lane] = cur;
}

// -------------------------------------------------------------------------------------------------
// k_pull: the same product traversed by ROWS (gather) -- used when one rank owns the whole basis.
//   y[b] = D(b) x[b] + sum_t <b|t|b^x_t> chi(g) n_a / n_b x[index(a)],   a = rep(b ^ x_t), g(b^x_t) = a
// with <b|t|b^x> = v (-1)^popc(x&s) [b & m == r ^ (x & m)] (-1)^popc(b & s): the term table is
// transformed once on the host (terms_adj).  Same generate -> project -> search pipeline as
// k_generate, but the scattered FP64 atomics of localProcess (DMV:107-120) become scattered loads of x
// and every y element is written exactly once (deterministic, no memset, half the L2 traffic).
// -------------------------------------------------------------------------------------------------
template <bool CE>
__device__ __forceinline__ typename ValT<CE>::type load_x(const void *x, int64_t i) {
  if (CE) {
    const double2 t = __ldg(reinterpret_cast<const double2 *>(x) + i);
    return v_make(t.x, t.y, (typename ValT<CE>::type *)nullptr);
  }
  return v_make(__ldg(reinterpret_cast<const double *>(x) + i), 0.0, (typename ValT<CE>::type *)nullptr);
}
__device__ __forceinline__ double to_v(double a, double *) { return a; }
__device__ __forceinline__ double2 to_v(double a, double2 *) { return make_double2(a, 0.0); }
__device__ __forceinline__ double2 to_v(double2 a, double2 *) { return a; }
__device__ __forceinline__ void v_add(double &a, double b) { a += b; }
__device__ __forceinline__ void v_add(double2 &a, double2 b) { a.x += b.x; a.y += b.y; }
__device__ __forceinline__ void smem_add(double *p, double v) { atomicAdd(p, v); }
__device__ __forceinline__ void smem_add(double2 *p, double2 v) { atomicAdd(&p->x, v.x); atomicAdd(&p->y, v.y); }

template <int PROJ, bool CV, bool CE>
__global__ void __launch_bounds__(kThreads) k_pull(const KernelParams p) {
  using V = typename ValT<CV>::type;
  using E = typename ValT<CE>::type;
  extern __shared__ __align__(16) unsigned char smem[];
  const SmemLayout L = smem_layout(p, PROJ, sizeof(V));
  const Tables<CV> T = stage_tables<PROJ, CV>(p, smem, L);   // p.groups / p.lut / p.terms: row-traversal tables
  const OrbitProgram &orbit = T.orbit;
  const StateIndex &index = T.index;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned warp = threadIdx.x >> 5;
  unsigned char *qbase = smem + L.queues;
  uint64_t *qb = reinterpret_cast<uint64_t *>(qbase) + warp * kQueue;
  V *qc = reinterpret_cast<V *>(qbase + (size_t)kWarps * kQueue * 8) + warp * kQueue;
  V *acc_s = reinterpret_cast<V *>(qbase + (size_t)kWarps * kQueue * (8 + sizeof(V))) + warp * 32;
  unsigned char *ql = qbase + (size_t)kWarps * (kQueue * (8 + sizeof(V)) + 32 * sizeof(V)) + warp * kQueue;
  if (PROJ == PROJ_GROUP) acc_s[lane] = v_make(0.0, 0.0, (V *)nullptr);
  __syncthreads();
  unsigned head = 0, count = 0;
  const bool any_s_out = p.any_s_out != 0;
  // replicated-x product: rows are this rank's block, `index` / `norms` describe the global basis, global index g
  // lives at x[pos[g]] (see dmv_host.h)
  const uint64_t *__restrict__ row_states = p.row_states ? p.row_states : p.index.reps;
  const double *__restrict__ row_norms = p.row_norms ? p.row_norms : p.norms;
  const uint32_t *__restrict__ xslot = p.pos;

  // drains `k` queued entries (PROJ_GROUP): orbit scan, search, gather, add into the owner row's slot
  auto drain = [&](unsigned k) {
    const bool active = lane < k;
    if (active) {
      const unsigned pos = (head + lane) & (kQueue - 1);
      const uint64_t raw = qb[pos];
      V h = qc[pos];
      const unsigned src = ql[pos];
      OrbitResult r;
      if (orbit.trivial_characters) {
        r.rep = orbit_representative(orbit, raw);
      } else {
        r = orbit_scan<false, false>(orbit, raw);
        const double2 chi = __ldg(orbit.characters + r.arg);   // chi(g), not conjugated (see header)
        h = v_mul(h, v_make(chi.x, chi.y, (V *)nullptr));
      }
      const int64_t idx = locate(index, r.rep);
      if (idx >= 0) {
        h = v_scale(h, __ldg(p.norms + idx));
        const int64_t xi = xslot ? (int64_t)__ldg(xslot + idx) : idx;
        const V val = v_mul(h, to_v(load_x<CE>(p.x, xi), (V *)nullptr));
        smem_add(acc_s + src, val);
      } else if (v_nonzero(h)) {
        bool fatal = true;
        if (!orbit.trivial_characters)
          fatal = orbit_stabiliser_sum(orbit, r.rep) > 1e-12 * (double)orbit.group_order;
        if (fatal && atomicAdd(p.status, 1ull) == 0) p.status[1] = r.rep;
      }
    }
  };

  const int64_t n_rows = p.row_end - p.row_begin;
  const int64_t n_tiles = (n_rows + 31) / 32;
  const int64_t warps_total = (int64_t)gridDim.x * kWarps;
  for (int64_t tile = (int64_t)blockIdx.x * kWarps + warp; tile < n_tiles; tile += warps_total) {
    const int64_t i = p.row_begin + tile * 32 + lane;
    const bool valid = i < p.row_end;
    const uint64_t b = valid ? __ldg(row_states + i) : 0ull;
    V acc = v_make(0.0, 0.0, (V *)nullptr);
    double inv_nb = 1.0;
    if (PROJ == PROJ_GROUP && valid) inv_nb = 1.0 / __ldg(row_norms + i);

    for (int g0 = 0, w = 0; g0 < p.n_groups; g0 += 64, ++w) {
      const int g1 = min(g0 + 64, p.n_groups);
      RowTerms rt = row_terms<CV>(T, w, g0, g1, b);
      if (!valid) rt.mask = 0;
      if (PROJ != PROJ_GROUP) {
        // every lane walks the set bits of ITS row: no lane idles on a bond that does not emit
        while (rt.mask) {
          uint64_t flip;
          V h = pop_term<CV>(T, rt, g0, b, any_s_out, flip);
          uint64_t a = b ^ flip;
          bool flipped = false;
          if (PROJ == PROJ_INVERSION) {
            const uint64_t inv = a ^ p.site_mask;
            flipped = inv < a;
            if (flipped) h = v_scale(h, p.inversion_character);
          }
          int64_t idx;
          if (index.mode == INDEX_RANK) {
            // rank over the full fixed-weight set, incrementally from rank(b) = i
            const int lo = __ffsll((long long)flip) - 1;
            const int hi = 63 - __clzll((long long)flip);
            const uint64_t span = ((hi == 63) ? ~0ull : ((1ull << (hi + 1)) - 1)) & ~((1ull << lo) - 1);
            const uint64_t ob = b & span, nb = a & span;
            idx = -1;
            if ((a & ~index.site_mask) == 0 && __popcll(ob) == __popcll(nb)) {
              const int k0 = __popcll(b & ((1ull << lo) - 1));
              int64_t r = i - (int64_t)combinadic_sum(index.binom, index.stride, ob, k0) +
                          (int64_t)combinadic_sum(index.binom, index.stride, nb, k0);
              if (flipped) r = (int64_t)p.rank_total - 1 - r;   // complement reverses the order
              if (r >= 0 && r < index.n) idx = r;
            }
          } else {
            idx = locate(index, flipped ? (a ^ p.site_mask) : a);
          }
          if (idx >= 0) {
            const int64_t xi = xslot ? (int64_t)__ldg(xslot + idx) : idx;
            v_add(acc, v_mul(h, to_v(load_x<CE>(p.x, xi), (V *)nullptr)));
          } else if (v_nonzero(h) && atomicAdd(p.status, 1ull) == 0) {
            p.status[1] = a;
          }
        }
      } else {
        for (;;) {
          const bool has = rt.mask != 0;
          const unsigned m = __ballot_sync(0xffffffffu, has);
          if (m == 0) break;
          if (has) {
            uint64_t flip;
            const V c = pop_term<CV>(T, rt, g0, b, any_s_out, flip);
            const unsigned pos = (head + count + __popc(m & ((1u << lane) - 1u))) & (kQueue - 1);
            qb[pos] = b ^ flip;
            qc[pos] = v_scale(c, inv_nb);
            ql[pos] = (unsigned char)lane;
          }
          count += __popc(m);
          if (count >= 32) {
            __syncwarp();
            drain(32);
            head = (head + 32) & (kQueue - 1);
            count -= 32;
            __syncwarp();
          }
        }
      }
    }
    if (PROJ == PROJ_GROUP) {
      if (count > 0) {
        __syncwarp();
        drain(count);
        head = (head + count) & (kQueue - 1);
        count = 0;
      }
      __syncwarp();
      acc = acc_s[lane];
      acc_s[lane] = v_make(0.0, 0.0, (V *)nullptr);
      __syncwarp();
    }
    if (valid) {
      // diagonal (DMV:36-53) and the single store of y[i]; without diagonal terms y is accumulated into
      E out;
      if (p.n_diag > 0) {
        double dre, dim;
        diagonal<CV>(T, p.n_diag, b, dre, dim);
        const E xi = load_x<CE>(p.x, p.x_row_offset + i);
        if (CE) out = v_make(dre * v_re(xi) - dim * v_im(xi), dre * v_im(xi) + dim * v_re(xi), (E *)nullptr);
        else out = v_make(dre * v_re(xi), 0.0, (E *)nullptr);
      } else {
        out = reinterpret_cast<const E *>(p.y)[i];
      }
      out = v_make(v_re(out) + v_re(acc), v_im(out) + v_im(acc), (E *)nullptr);
      reinterpret_cast<E *>(p.y)[i] = out;
    }
  }
}

// -------------------------------------------------------------------------------------------------
// k_rows: the row traversal for bases with permutation symmetries, real operators with a bit-parallel emit test and
// trivial characters (every symmetric model input of the reference) -- the product kernel of one rank and of the
// replicated-x form on several ranks.
//   y[b] = D(b) x[b] + 1/n_b sum_t h_t(b) (n x)[rep(b ^ x_t)]
// One lane owns one row and walks ITS emitting groups: no warp queue, no shared-memory atomics, y written once.  Per term:
// orbit minimum in registers (canonical form, dmv_device.cuh), then ONE dependent memory access -- the slot of the
// representative in a hash table that carries the scaled vector element (table_slot) -- and that access is software
// pipelined: the slot of term j is requested right after its orbit minimum and consumed after the orbit minimum of
// term j + 2, so its latency hides behind ~10^3 integer instructions of the same lane.  (Deeper pipelines were measured
// and are slower -- four requests per lane through prefetch.global.L2 or through cp.async into shared memory: 58 / 46 ms
// against 29 ms on the 6x6 square; the look-ups are bound by the rate of random 64-byte requests the memory system takes,
// not by their latency: profiles/r02_rows_pipelines.md.)
// -------------------------------------------------------------------------------------------------
// one bucket = two slots (layout: table_slot in dmv_device.cuh); all loads of a bucket are independent
// 256-bit loads (sm_100: LDG.E.256), not allocated in L1: a bucket is touched once per product, and 50 GB of them
// streaming through L1 would evict the small tables the orbit minimum reads from global memory
__device__ __forceinline__ void load256(const unsigned char *q, uint64_t &a, uint64_t &b, uint64_t &c, uint64_t &d) {
  asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(q));
}
// the same through L1 (perfect-hash blocks: a few bits per state, read by every look-up)
__device__ __forceinline__ void load256_cached(const unsigned char *q, uint64_t &a, uint64_t &b, uint64_t &c, uint64_t &d) {
  asm volatile("ld.global.nc.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(q));
}
template <bool CE>
__device__ __forceinline__ void bucket_load(const unsigned char *__restrict__ table, uint32_t b, ulonglong2 &keys,
                                            typename ValT<CE>::type &v0, typename ValT<CE>::type &v1) {
  uint64_t w0, w1, w2, w3;
  load256(table + (size_t)b * 32, w0, w1, w2, w3);   // one bucket = one 32-byte sector = one request
  if constexpr (CE) {   // { key, spare, re, im }
    keys = make_ulonglong2(w0, w1);                  // (one slot: the second word is spare)
    v0 = make_double2(__longlong_as_double((long long)w2), __longlong_as_double((long long)w3));
    v1 = v0;
  } else {              // { key0, key1, value0, value1 }
    keys = make_ulonglong2(w0, w1);
    v0 = __longlong_as_double((long long)w2);
    v1 = __longlong_as_double((long long)w3);
  }
}
__device__ __forceinline__ void axpy(double &acc, double c, double v) { acc = fma(c, v, acc); }
__device__ __forceinline__ void axpy(double2 &acc, double c, double2 v) { acc.x = fma(c, v.x, acc.x); acc.y = fma(c, v.y, acc.y); }

// two CTAs per SM: the pipeline state must stay in registers (a spilled request waits for its load at once), and the
// latency is hidden inside the lane, not by occupancy
template <bool CE, int TK, bool MPH, int CTAS>
__global__ void __launch_bounds__(kThreads, CTAS) k_rows(const KernelParams p) {
  using E = typename ValT<CE>::type;
  extern __shared__ __align__(16) unsigned char smem[];
  const SmemLayout L = smem_layout(p, PROJ_GROUP, sizeof(double), false);
  const Tables<false> T = stage_tables<PROJ_GROUP, false>(p, smem, L);   // p.groups / p.lut: row-traversal tables
  __syncthreads();
  const OrbitProgram &orbit = T.orbit;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned warp = threadIdx.x >> 5;
  const bool any_s_out = p.any_s_out != 0;
  const unsigned char *__restrict__ table = reinterpret_cast<const unsigned char *>(p.table);
  const uint32_t n_buckets = p.table_slots;
  const uint64_t *__restrict__ row_states = p.row_states ? p.row_states : p.index.reps;
  const double *__restrict__ row_norms = p.row_norms ? p.row_norms : p.norms;
  unsigned long long bad = 0, bad_state = 0;
  const E zero = v_make(0.0, 0.0, (E *)nullptr);
  const PerfectHash H = p.mph;
  const unsigned char *__restrict__ dense = reinterpret_cast<const unsigned char *>(p.dense);

  const int64_t n_rows = p.row_end - p.row_begin;
  const int64_t n_tiles = (n_rows + 31) / 32;
  const int64_t warps_total = (int64_t)gridDim.x * kWarps;
  for (int64_t tile = (int64_t)blockIdx.x * kWarps + warp; tile < n_tiles; tile += warps_total) {
    const int64_t i = p.row_begin + tile * 32 + lane;
    const bool valid = i < p.row_end;
    const uint64_t b = valid ? __ldg(row_states + i) : 0ull;
    E acc = zero;
    int w = 0;
    RowTerms rt = row_terms<false>(T, 0, 0, min(64, p.n_groups), b);
    if (!valid) rt.mask = 0;
    if constexpr (MPH) {
      // ---- dense index: request 0 holds the two perfect-hash blocks of its state (L2 hits), request 1 the slot of
      // the dense table (or, for the few states the two levels could not place, a bucket of the open-addressing table)
      bool live0 = false, live1 = false, in_table1 = false;
      uint64_t want0 = 0, want1 = 0;
      double c0 = 0.0, c1 = 0.0;
      uint32_t bits0 = 0, b1 = 0;
      uint64_t A0 = 0, A1 = 0, A2 = 0, A3 = 0, B0 = 0, B1 = 0, B2 = 0, B3 = 0;
      ulonglong2 k1 = make_ulonglong2(0, 0);
      E v10 = zero, v11 = zero;
      for (;;) {
        while (valid && rt.mask == 0 && 64 * (w + 1) < p.n_groups) {
          ++w;
          rt = row_terms<false>(T, w, 64 * w, min(64 * w + 64, p.n_groups), b);
        }
        const bool has = rt.mask != 0;
        if (!has && !live0 && !live1) break;
        // ---- consume request 1
        bool retry = false;
        if (live1) {
          if (!in_table1) {
            if (k1.x == want1) axpy(acc, c1, v10);
            else if (c1 != 0.0) { ++bad; bad_state = want1; }   // the slot belongs to another state: not in the basis
          } else {
            const bool hit0 = k1.x == want1, hit1 = !CE && k1.y == want1;
            if (hit0 | hit1) axpy(acc, c1, hit0 ? v10 : v11);
            else if (k1.x == kEmptyKey || (!CE && k1.y == kEmptyKey)) { if (c1 != 0.0) { ++bad; bad_state = want1; } }
            else retry = true;
          }
        }
        if (retry) {   // next bucket of the open-addressing table; request 0 and the row wait one trip
          b1 = b1 + 1 == n_buckets ? 0 : b1 + 1;
          bucket_load<CE>(table, b1, k1, v10, v11);
          continue;
        }
        // ---- request 0 -> request 1: resolve the slot, ask for it
        live1 = live0;
        if (live0) {
          want1 = want0; c1 = c0;
          uint32_t slot = mph_rank(A0, A1, A2, A3, bits0 & 0xffu);
          if (slot == kMphMissing && H.n_blocks1 != 0) slot = mph_rank(B0, B1, B2, B3, bits0 >> 8);
          in_table1 = slot == kMphMissing;
          if (!in_table1) {
            if constexpr (CE) {
              uint64_t u0, u1, u2, u3;
              load256(dense + (size_t)slot * 32, u0, u1, u2, u3);
              k1 = make_ulonglong2(u0, u1);
              v10 = make_double2(__longlong_as_double((long long)u2), __longlong_as_double((long long)u3));
            } else {
              const ulonglong2 t = __ldg(reinterpret_cast<const ulonglong2 *>(dense + (size_t)slot * 16));
              k1 = make_ulonglong2(t.x, 0);
              v10 = __longlong_as_double((long long)t.y);
            }
          } else {
            b1 = table_slot(want1, n_buckets);
            bucket_load<CE>(table, b1, k1, v10, v11);
          }
        }
        // ---- a new request 0: the next term of the row
        live0 = has;
        if (has) {
          uint64_t flip;
          c0 = pop_term<false>(T, rt, 64 * w, b, any_s_out, flip);
          const uint64_t raw = b ^ flip;
          if constexpr (TK > 0) want0 = orbit_min_torus_sq<TK>(orbit, raw);
          else want0 = orbit_representative(orbit, raw);
          uint32_t blk, bit, blk1 = 0, bit1 = 0;
          mph_position(want0, 0, H.n_blocks0, blk, bit);
          load256_cached(H.blocks + (size_t)blk * 32, A0, A1, A2, A3);
          if (H.n_blocks1 != 0) {
            mph_position(want0, 1, H.n_blocks1, blk1, bit1);
            load256_cached(H.blocks + ((size_t)H.n_blocks0 + blk1) * 32, B0, B1, B2, B3);
          }
          bits0 = bit | (bit1 << 8);
        }
      }
    } else {
    // two requests in flight per lane: wanted key, coefficient, bucket, and what the bucket held
    bool live0 = false, live1 = false;
    uint64_t want0 = 0, want1 = 0;
    double c0 = 0.0, c1 = 0.0;
    uint32_t b0 = 0, b1 = 0;
    ulonglong2 k0 = make_ulonglong2(0, 0), k1 = k0;
    E v00 = zero, v01 = zero, v10 = zero, v11 = zero;
    for (;;) {
      while (valid && rt.mask == 0 && 64 * (w + 1) < p.n_groups) {
        ++w;
        rt = row_terms<false>(T, w, 64 * w, min(64 * w + 64, p.n_groups), b);
      }
      const bool has = rt.mask != 0;
      if (!has && !live0 && !live1) break;
      // ---- consume the older request
      bool retry = false;
      if (live1) {
        const bool hit0 = k1.x == want1, hit1 = !CE && k1.y == want1;
        if (hit0 | hit1) {
          axpy(acc, c1, hit0 ? v10 : v11);
        } else if (k1.x == kEmptyKey || (!CE && k1.y == kEmptyKey)) {   // a free slot in the bucket: not a basis state
          if (c1 != 0.0) { ++bad; bad_state = want1; }         // DMV:115-118
        } else {
          retry = true;                                        // both slots taken by other states: next bucket
        }
      }
      const uint64_t want_r = want1;
      const double c_r = c1;
      const uint32_t b_r = b1 + 1 == n_buckets ? 0 : b1 + 1;
      live1 = live0; want1 = want0; c1 = c0; b1 = b0; k1 = k0; v10 = v00; v11 = v01;
      // ---- issue a new request: the continuation of a missed one, else the next term of the row
      if (retry) {
        want0 = want_r; c0 = c_r; b0 = b_r;
        bucket_load<CE>(table, b0, k0, v00, v01);
        live0 = true;
      } else if (has) {
        uint64_t flip;
        c0 = pop_term<false>(T, rt, 64 * w, b, any_s_out, flip);
        const uint64_t raw = b ^ flip;
        if constexpr (TK > 0) want0 = orbit_min_torus_sq<TK>(orbit, raw);
        else want0 = orbit_representative(orbit, raw);
        b0 = table_slot(want0, n_buckets);
        bucket_load<CE>(table, b0, k0, v00, v01);
        live0 = true;
      } else {
        live0 = false;
      }
    }
    }
    if (valid) {
      const double inv_nb = 1.0 / __ldg(row_norms + i);
      E out;
      if (p.n_diag > 0) {
        double dre, dim;
        diagonal<false>(T, p.n_diag, b, dre, dim);
        const E xi = load_x<CE>(p.x, p.x_row_offset + i);
        out = v_scale(xi, dre);   // real operator: the diagonal is real
      } else {
        out = reinterpret_cast<const E *>(p.y)[i];
      }
      axpy(out, inv_nb, acc);
      reinterpret_cast<E *>(p.y)[i] = out;
    }
  }
  if (bad) {
    if (atomicAdd(p.status, bad) == 0) p.status[1] = bad_state;
  }
}

// -------------------------------------------------------------------------------------------------
// k_rows_batch: k_rows on up to six real (three complex) vectors at once -- the product the block eigensolver asks for
// (reference src/Diagonalize.chpl:134-162: PRIMME hands `blockSize` vectors to one matvec call).  The orbit minimum and the
// look-up of a term are shared by the vectors: one bucket = 64 bytes = { key, d[0..5], spare }, d = the scaled elements of
// the vectors at that state (three (re, im) pairs or six reals: the operator is real, so every double is treated alike),
// fetched with two independent 256-bit loads.  One request per lane in flight, consumed after the orbit minimum of the
// NEXT term; a bucket taken by another state continues with the next bucket through the same slot.
// Cost model: one 64-byte request per term (17.8 G/s for tables >> L2, profiles/r02_random_access.md) against one 32-byte
// request per term AND vector in k_rows.
// -------------------------------------------------------------------------------------------------
template <int TK, int CTAS>
__global__ void __launch_bounds__(kThreads, CTAS) k_rows_batch(const KernelParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const SmemLayout L = smem_layout(p, PROJ_GROUP, sizeof(double), false);
  const Tables<false> T = stage_tables<PROJ_GROUP, false>(p, smem, L);
  __syncthreads();
  const OrbitProgram &orbit = T.orbit;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned warp = threadIdx.x >> 5;
  const bool any_s_out = p.any_s_out != 0;
  const unsigned char *__restrict__ table = reinterpret_cast<const unsigned char *>(p.table);
  const uint32_t n_buckets = p.table_slots;
  const int elt = p.batch_elt;            // doubles per vector element (1 | 2)
  const int nd = p.batch * elt;           // doubles per state in use (<= 6)
  const int64_t stride = p.batch_stride;  // elements between consecutive vectors
  const double *__restrict__ xd = reinterpret_cast<const double *>(p.x);
  double *__restrict__ yd = reinterpret_cast<double *>(p.y);
  unsigned long long bad = 0, bad_state = 0;

  const int64_t n_rows = p.row_end - p.row_begin;
  const int64_t n_tiles = (n_rows + 31) / 32;
  const int64_t warps_total = (int64_t)gridDim.x * kWarps;
  for (int64_t tile = (int64_t)blockIdx.x * kWarps + warp; tile < n_tiles; tile += warps_total) {
    const int64_t i = p.row_begin + tile * 32 + lane;
    const bool valid = i < p.row_end;
    const uint64_t b = valid ? __ldg(p.index.reps + i) : 0ull;
    double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    int w = 0;
    RowTerms rt = row_terms<false>(T, 0, 0, min(64, p.n_groups), b);
    if (!valid) rt.mask = 0;
    bool live = false, held = false;       // a request in flight; a term popped but not yet requested
    uint64_t want = 0, want_n = 0;
    double c = 0.0, c_n = 0.0;
    uint32_t bk = 0;
    uint64_t q0 = 0, q1 = 0, q2 = 0, q3 = 0, q4 = 0, q5 = 0, q6 = 0, q7 = 0;
    for (;;) {
      while (valid && rt.mask == 0 && 64 * (w + 1) < p.n_groups) {
        ++w;
        rt = row_terms<false>(T, w, 64 * w, min(64 * w + 64, p.n_groups), b);
      }
      const bool has = rt.mask != 0;
      if (!has && !live && !held) break;
      // ---- the next term of the row (its orbit minimum covers the latency of the request in flight)
      if (has && !held) {
        uint64_t flip;
        c_n = pop_term<false>(T, rt, 64 * w, b, any_s_out, flip);
        const uint64_t raw = b ^ flip;
        if constexpr (TK > 0) want_n = orbit_min_torus_sq<TK>(orbit, raw);
        else want_n = orbit_representative(orbit, raw);
        held = true;
      }
      // ---- consume the request in flight
      bool retry = false;
      if (live) {
        if (q0 == want) {
          acc[0] = fma(c, __longlong_as_double((long long)q1), acc[0]);
          acc[1] = fma(c, __longlong_as_double((long long)q2), acc[1]);
          acc[2] = fma(c, __longlong_as_double((long long)q3), acc[2]);
          acc[3] = fma(c, __longlong_as_double((long long)q4), acc[3]);
          acc[4] = fma(c, __longlong_as_double((long long)q5), acc[4]);
          acc[5] = fma(c, __longlong_as_double((long long)q6), acc[5]);
        } else if (q0 == kEmptyKey) {
          if (c != 0.0) { ++bad; bad_state = want; }       // not a basis state (DMV:115-118)
        } else {
          retry = true;
        }
      }
      // ---- issue: the continuation of a missed request, else the held term
      if (retry) {
        bk = bk + 1 == n_buckets ? 0 : bk + 1;
      } else if (held) {
        want = want_n; c = c_n; held = false;
        bk = table_slot(want, n_buckets);
        live = true;
      } else {
        live = false;
      }
      if (live) {
        const unsigned char *q = table + (size_t)bk * 64;
        load256(q, q0, q1, q2, q3);
        load256(q + 32, q4, q5, q6, q7);
      }
    }
    if (valid) {
      const double inv_nb = 1.0 / __ldg(p.norms + i);
      double dre = 0.0, dim = 0.0;
      if (p.n_diag > 0) diagonal<false>(T, p.n_diag, b, dre, dim);
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        if (j < nd) {
          const int64_t at = ((int64_t)(j / elt) * stride + i) * elt + (j % elt);
          const double base = p.n_diag > 0 ? dre * __ldg(xd + at) : yd[at];
          yd[at] = fma(inv_nb, acc[j], base);
        }
      }
    }
  }
  if (bad) {
    if (atomicAdd(p.status, bad) == 0) p.status[1] = bad_state;
  }
}

// hash table set-up: claim a slot per state (keys pre-set to kEmptyKey; slot 0 of a bucket, then slot 1 when the bucket
// has two, then the next bucket), remember it in slot_of (= 2 bucket + slot)
__global__ void k_table_insert(const uint64_t *__restrict__ reps, int64_t n, unsigned char *table, uint32_t n_buckets,
                               int slots_per_bucket, uint32_t *slot_of, int bucket_bytes) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t key = reps[i];
  uint32_t b = table_slot(key, n_buckets);
  for (;;) {
    unsigned long long *q = reinterpret_cast<unsigned long long *>(table + (size_t)b * bucket_bytes);
    if (atomicCAS(q, (unsigned long long)kEmptyKey, (unsigned long long)key) == (unsigned long long)kEmptyKey) {
      slot_of[i] = 2 * b;
      return;
    }
    if (slots_per_bucket == 2 &&
        atomicCAS(q + 1, (unsigned long long)kEmptyKey, (unsigned long long)key) == (unsigned long long)kEmptyKey) {
      slot_of[i] = 2 * b + 1;
      return;
    }
    b = b + 1 == n_buckets ? 0 : b + 1;
  }
}

// per product: value of slot_of[i] = x[src(i)] * norm[i]   (src(i) = pos ? pos[i] : i).  complex128 rewrites the WHOLE
// 32-byte slot {key, spare, re, im} with one 256-bit store: a full-sector write needs no read-modify-write in DRAM.
// slot_of[i] < 2^31: slot of the dense table (perfect hash); else 0x80000000 | slot of the open-addressing table.
template <bool CE>
__global__ void k_table_fill(int64_t n, const void *__restrict__ x, const double *__restrict__ norms,
                             const uint32_t *__restrict__ pos, const uint32_t *__restrict__ slot_of,
                             const uint64_t *__restrict__ reps, unsigned char *table, unsigned char *dense) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int64_t src = pos ? (int64_t)__ldg(pos + i) : i;
    const double nrm = __ldg(norms + i);
    uint32_t s = __ldg(slot_of + i);
    const bool in_table = dense == nullptr || (s & 0x80000000u);
    s &= 0x7fffffffu;
    const uint64_t key = __ldg(reps + i);
    if constexpr (CE) {
      const double2 v = __ldg(reinterpret_cast<const double2 *>(x) + src);
      const uint64_t re = (uint64_t)__double_as_longlong(v.x * nrm), im = (uint64_t)__double_as_longlong(v.y * nrm);
      unsigned char *q = in_table ? table + (size_t)(s >> 1) * 32 : dense + (size_t)s * 32;
      asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(q), "l"(key), "l"(0ull), "l"(re), "l"(im) : "memory");
    } else {
      const double v = __ldg(reinterpret_cast<const double *>(x) + src) * nrm;
      if (in_table) *reinterpret_cast<double *>(table + (size_t)(s >> 1) * 32 + 16 + 8 * (s & 1)) = v;
      else *reinterpret_cast<ulonglong2 *>(dense + (size_t)s * 16) = make_ulonglong2(key, (uint64_t)__double_as_longlong(v));
    }
  }
}

// per batched product: bucket slot_of[i] / 2 of the 64-byte table <- { key, x_v[i] * norm[i] for the vectors v, 0 ... }
// (two 256-bit stores = two full sectors)
__global__ void k_table_fill_batch(int64_t n, int nd, int elt, const double *__restrict__ x, int64_t stride,
                                   const double *__restrict__ norms, const uint32_t *__restrict__ slot_of,
                                   const uint64_t *__restrict__ reps, unsigned char *table) {
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
    const double nrm = __ldg(norms + i);
    uint64_t d[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      double v = 0.0;
      if (j < nd) v = __ldg(x + ((int64_t)(j / elt) * stride + i) * elt + (j % elt)) * nrm;
      d[j] = (uint64_t)__double_as_longlong(v);
    }
    unsigned char *q = table + (size_t)(__ldg(slot_of + i) >> 1) * 64;
    const uint64_t key = __ldg(reps + i);
    asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(q), "l"(key), "l"(d[0]), "l"(d[1]), "l"(d[2]) : "memory");
    asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(q + 32), "l"(d[3]), "l"(d[4]), "l"(d[5]), "l"(0ull) : "memory");
  }
}

// ---- perfect-hash set-up (see PerfectHash in dmv_device.cuh) ----
__global__ void k_mph_mark(const uint64_t *__restrict__ keys, int64_t n, int level, uint32_t n_blocks,
                           unsigned long long *seen, unsigned long long *collide) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t block, bit;
  mph_position(keys[i], level, n_blocks, block, bit);
  const size_t w = (size_t)block * 3 + (bit >> 6);
  const unsigned long long m = 1ull << (bit & 63u);
  if (atomicOr(seen + w, m) & m) atomicOr(collide + w, m);
}
__global__ void k_mph_compact(const uint64_t *__restrict__ keys, int64_t n, int level, uint32_t n_blocks,
                              const unsigned long long *__restrict__ collide, uint64_t *next,
                              unsigned long long *next_count) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t block, bit;
  mph_position(keys[i], level, n_blocks, block, bit);
  if ((collide[(size_t)block * 3 + (bit >> 6)] >> (bit & 63u)) & 1ull) next[atomicAdd(next_count, 1ull)] = keys[i];
}
__device__ __forceinline__ uint32_t mph_lookup(const PerfectHash &H, uint64_t key) {
  uint32_t block, bit;
  mph_position(key, 0, H.n_blocks0, block, bit);
  const unsigned long long *q = reinterpret_cast<const unsigned long long *>(H.blocks) + (size_t)block * 4;
  uint32_t r = mph_rank(q[0], q[1], q[2], q[3], bit);
  if (r != kMphMissing || H.n_blocks1 == 0) return r;
  mph_position(key, 1, H.n_blocks1, block, bit);
  q = reinterpret_cast<const unsigned long long *>(H.blocks) + ((size_t)H.n_blocks0 + block) * 4;
  return mph_rank(q[0], q[1], q[2], q[3], bit);
}
__global__ void k_mph_slots(const uint64_t *__restrict__ keys, int64_t n, PerfectHash H, const unsigned char *table,
                            uint32_t n_buckets, int slots_per_bucket, uint32_t *slot_of, unsigned long long *status) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t key = keys[i];
  const uint32_t r = mph_lookup(H, key);
  if (r != kMphMissing) { slot_of[i] = r; return; }
  uint32_t b = table_slot(key, n_buckets);
  for (uint32_t tries = 0; tries <= n_buckets; ++tries) {   // the state was inserted before: the probe sequence finds it
    const unsigned long long *q = reinterpret_cast<const unsigned long long *>(table + (size_t)b * 32);
    if (q[0] == key) { slot_of[i] = 0x80000000u | (2 * b); return; }
    if (slots_per_bucket == 2 && q[1] == key) { slot_of[i] = 0x80000000u | (2 * b + 1); return; }
    b = b + 1 == n_buckets ? 0 : b + 1;
  }
  atomicAdd(status + 2, 1ull);
}

// localProcess for records that arrived from other ranks: already projected and hashed by the sender.
// Two records per thread with their searches advanced in lock step (see locate2).
template <int PROJ, bool CV, bool CE>
__global__ void __launch_bounds__(kThreads) k_accumulate(const KernelParams p, int64_t count,
                                                         const uint64_t *__restrict__ betas,
                                                         const double *__restrict__ coeffs) {
  using V = typename ValT<CV>::type;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t half = (count + 1) / 2;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < half; k += stride) {
    const int64_t k1 = k + half;
    const bool a1 = k1 < count;
    const uint64_t b0 = __ldg(betas + k), b1 = a1 ? __ldg(betas + k1) : 0ull;
    const V c0 = __ldg(reinterpret_cast<const V *>(coeffs) + k);
    const V c1 = a1 ? __ldg(reinterpret_cast<const V *>(coeffs) + k1) : v_make(0.0, 0.0, (V *)nullptr);
    int64_t i0, i1;
    locate2(p.index, true, b0, a1, b1, i0, i1);
    finish<PROJ, CV, CE>(p, p.orbit, true, b0, c0, i0);
    finish<PROJ, CV, CE>(p, p.orbit, a1, b1, c1, i1);
  }
}

// ls_chpl_operator_apply_diag / ls_chpl_operator_apply_off_diag (reference src/BatchedOperator.chpl:217-275):
// the term kernels applied to caller-given states with xs = nil ("times one", BO:230,263), no projection.
//   apply_diag:     coeffs[i] = Re sum_t v_t [alpha_i & m == r] (-1)^popc(alpha_i & s)
//   apply_off_diag: CSR by row -- pass 0 counts the emitting groups of every row, the host turns the counts into
//                   the row pointer `offsets`, pass 1 writes (beta, coefficient) of row i at offsets[i]...
// One lane per state; tables in shared memory as in k_generate.
__global__ void __launch_bounds__(kThreads) k_apply_diag(const KernelParams p, int64_t count,
                                                         const uint64_t *__restrict__ alphas, double *coeffs) {
  extern __shared__ __align__(16) unsigned char smem[];
  const SmemLayout L = smem_layout(p, PROJ_NONE, sizeof(double2));
  const Tables<true> T = stage_tables<PROJ_NONE, true>(p, smem, L);
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
    double dre, dim;
    diagonal<true>(T, p.n_diag, alphas[i], dre, dim);
    coeffs[i] = dre;
  }
}

template <bool WRITE>
__global__ void __launch_bounds__(kThreads) k_apply_off_diag(const KernelParams p, int64_t count,
                                                             const uint64_t *__restrict__ alphas,
                                                             const int64_t *__restrict__ offsets, int64_t *counts,
                                                             uint64_t *betas, double2 *coeffs) {
  extern __shared__ __align__(16) unsigned char smem[];
  const SmemLayout L = smem_layout(p, PROJ_NONE, sizeof(double2));
  const Tables<true> T = stage_tables<PROJ_NONE, true>(p, smem, L);
  __syncthreads();
  const bool any_s_out = p.any_s_out != 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
    const uint64_t alpha = alphas[i];
    int64_t o = WRITE ? offsets[i] : 0;
    for (int g0 = 0, w = 0; g0 < p.n_groups; g0 += 64, ++w) {
      RowTerms rt = row_terms<true>(T, w, g0, min(g0 + 64, p.n_groups), alpha);
      if (!WRITE) { o += __popcll(rt.mask); continue; }
      while (rt.mask) {
        uint64_t flip;
        const double2 c = pop_term<true>(T, rt, g0, alpha, any_s_out, flip);
        betas[o] = alpha ^ flip;
        coeffs[o] = c;
        ++o;
      }
    }
    if (!WRITE) counts[i] = o;
  }
}

// dir[2b] = lower_bound(reps, b << shift), dir[2b+1] = lower_bound(reps, (b+1) << shift) for b in [0, n_buckets)
__global__ void k_build_directory(const uint64_t *__restrict__ reps, int64_t n, uint32_t *dir,
                                  uint64_t n_buckets, int shift) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 2 * n_buckets) return;
  const uint64_t b = (t >> 1) + (t & 1);
  int64_t lo = 0, hi = n;
  const bool past_end = shift > 0 ? (b > (~0ull >> shift)) : false;
  if (past_end) lo = n;
  const uint64_t key = b << shift;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (reps[mid] < key) lo = mid + 1; else hi = mid;
  }
  dir[t] = (uint32_t)lo;
}

__global__ void k_state_index(const StateIndex ix, int64_t count, const uint64_t *__restrict__ spins,
                              int64_t *indices) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < count) indices[k] = locate(ix, spins[k]);
}

__global__ void k_verify_rank(const StateIndex ix, unsigned long long *status) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < ix.n && locate(ix, ix.reps[k]) != k) atomicAdd(status, 1ull);
}

__global__ void k_locale_idx(int64_t count, const uint64_t *__restrict__ states, int num_ranks, uint8_t *keys) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < count) keys[k] = (uint8_t)locale_idx_of(states[k], num_ranks);
}

// ls_hs_state_info (reference src/FFI.chpl:181-184): representative, conj(character), norm
template <int PROJ>
__global__ void k_state_info(const OrbitProgram P, uint64_t site_mask, double inv_char, int64_t count,
                             const uint64_t *__restrict__ alphas, uint64_t *betas, double2 *characters,
                             double *norms) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  const uint64_t a = alphas[k];
  if (PROJ == PROJ_NONE) {
    betas[k] = a; characters[k] = make_double2(1.0, 0.0); norms[k] = 1.0;
  } else if (PROJ == PROJ_INVERSION) {
    const uint64_t inv = a ^ site_mask;
    const bool flip = inv < a;
    betas[k] = flip ? inv : a;
    characters[k] = make_double2(flip ? inv_char : 1.0, 0.0);
    norms[k] = sqrt(0.5);   // stabiliser = {identity}: |Stab| / |G| = 1/2
    if (inv == a) norms[k] = (inv_char > 0) ? 1.0 : 0.0;
  } else {
    const OrbitResult r = orbit_scan<true, false>(P, a);
    betas[k] = r.rep;
    double2 chi = make_double2(1.0, 0.0);
    double stab = (double)r.stab;
    if (!P.trivial_characters) {
      chi = P.characters[r.arg];
      stab = orbit_stabiliser_sum(P, a);
    }
    characters[k] = make_double2(chi.x, -chi.y);
    const double nn = stab / (double)P.group_order;
    norms[k] = nn > 1e-12 ? sqrt(nn) : 0.0;
  }
}

__global__ void k_compute_norms(const OrbitProgram P, int64_t count, const uint64_t *__restrict__ reps,
                                double *norms) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  double stab;
  if (P.trivial_characters) stab = (double)orbit_scan<true, false>(P, reps[k]).stab;
  else stab = orbit_stabiliser_sum(P, reps[k]);
  const double nn = stab / (double)P.group_order;
  norms[k] = nn > 1e-12 ? sqrt(nn) : 0.0;
}

// nextStateFixedHamming (reference src/StatesEnumeration.chpl:31-34)
__device__ __forceinline__ uint64_t next_state_fixed_hamming(uint64_t v) {
  const uint64_t t = v | (v - 1);
  return (t + 1) | (((~t & (t + 1)) - 1) >> (__ffsll((long long)v)));
}

// One thread per chunk of consecutive candidates [first, last]; keeps a candidate iff it is owned by
// this rank, is the minimum of its orbit and has non-zero norm (reference
// src/StatesEnumeration.chpl:158-224).  Pass 0 counts, pass 1 writes at chunk_offset[c].
template <int PROJ, bool WRITE>
__global__ void k_enumerate(const OrbitProgram P, uint64_t site_mask, bool fixed_hamming, int rank,
                            int num_ranks, int64_t n_chunks, const uint64_t *__restrict__ chunk_first,
                            const uint64_t *__restrict__ chunk_last, unsigned long long *chunk_count,
                            const unsigned long long *__restrict__ chunk_offset, uint64_t *out,
                            double *out_norms) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_chunks) return;
  uint64_t v = chunk_first[c];
  const uint64_t last = chunk_last[c];
  unsigned long long n = 0;
  unsigned long long base = WRITE ? chunk_offset[c] : 0ull;
  for (;;) {
    bool keep = (num_ranks <= 1) || (locale_idx_of(v, num_ranks) == rank);
    double norm = 1.0;
    if (keep) {
      if (PROJ == PROJ_INVERSION) {
        keep = v < (v ^ site_mask);
      } else if (PROJ == PROJ_GROUP) {
        const OrbitResult r = orbit_scan<true, true>(P, v);
        keep = (r.rep == v);
        if (keep) {
          const double stab = P.trivial_characters ? (double)r.stab : orbit_stabiliser_sum(P, v);
          const double nn = stab / (double)P.group_order;
          norm = nn > 1e-12 ? sqrt(nn) : 0.0;
          keep = norm > 0.0;
        }
      }
    }
    if (keep) {
      if (WRITE) { out[base + n] = v; if (out_norms) out_norms[base + n] = norm; }
      ++n;
    }
    if (v == last) break;
    v = fixed_hamming ? next_state_fixed_hamming(v) : v + 1;
  }
  if (!WRITE) chunk_count[c] = n;
}

int grid_for(int64_t work_items, int per_block, int max_blocks) {
  int64_t b = (work_items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return (int)b;
}

}  // namespace
// lanes per source state: enough warps to fill the machine (>= 8 per SM) on small bases, never more than the
// number of flip-mask groups
int choose_row_split(int64_t rows, int n_groups) {
  int dev = 0, n = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  if (n <= 0) n = 148;
  int s = 1;
  while (s < 32 && 2 * s <= n_groups && (rows * s) / 32 < (int64_t)n * 16) s *= 2;
  return s;
}

int planned_grid(int64_t rows, int row_split) {   // grid of the planned launches: fixed, not occupancy-derived
  int dev = 0, n = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  if (n <= 0) n = 148;
  const int rows_per_tile = 32 / (row_split > 1 ? row_split : 1);
  int64_t b = ((rows + rows_per_tile - 1) / rows_per_tile + kWarps - 1) / kWarps;
  if (b < 1) b = 1;
  if (b > (int64_t)n * 4) b = (int64_t)n * 4;
  return (int)b;
}
namespace {

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int PROJ, bool CV, bool CE, bool COUNT_ONLY>
void launch_generate_t(const KernelParams &p, cudaStream_t stream) {
  using V = typename ValT<CV>::type;
  const SmemLayout L = smem_layout(p, PROJ, sizeof(V));
  auto kernel = k_generate<PROJ, CV, CE, COUNT_ONLY>;
  if (L.total > 48 * 1024)
    DMV_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
  if (L.total > 40 * 1024)   // let several CTAs with large tables share the SM
    DMV_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  int per_sm = 0;
  DMV_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, L.total));
  if (per_sm < 1) per_sm = 1;
  const int rpt = 32 / (p.row_split > 1 ? p.row_split : 1);
  const int64_t tiles = (p.row_end - p.row_begin + rpt - 1) / rpt;
  // grid = a whole number of waves of resident CTAs (148 SMs x per_sm), or fewer when the work is small
  const int blocks = p.grid_blocks > 0 ? p.grid_blocks : grid_for(tiles, kWarps, sm_count() * per_sm);
  kernel<<<blocks, kThreads, L.total, stream>>>(p);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

template <int PROJ, bool CV, bool CE>
void launch_generate_c(const KernelParams &p, bool count_only, cudaStream_t s) {
  if (count_only) launch_generate_t<PROJ, CV, CE, true>(p, s);
  else launch_generate_t<PROJ, CV, CE, false>(p, s);
}
template <int PROJ>
void launch_generate_p(const KernelParams &p, bool cv, bool ce, bool count_only, cudaStream_t s) {
  if (!cv && !ce) launch_generate_c<PROJ, false, false>(p, count_only, s);
  else if (cv && ce) launch_generate_c<PROJ, true, true>(p, count_only, s);
  else if (cv && !ce) launch_generate_c<PROJ, true, false>(p, count_only, s);
  else throw std::runtime_error("complex vectors need complex values");
}


template <int PROJ, bool CV, bool CE>
void launch_pull_t(const KernelParams &p, cudaStream_t stream) {
  using V = typename ValT<CV>::type;
  const SmemLayout L = smem_layout(p, PROJ, sizeof(V));
  auto kernel = k_pull<PROJ, CV, CE>;
  if (L.total > 48 * 1024)
    DMV_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
  int per_sm = 0;
  DMV_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, L.total));
  if (per_sm < 1) per_sm = 1;
  const int64_t tiles = (p.row_end - p.row_begin + 31) / 32;
  const int blocks = grid_for(tiles, kWarps, sm_count() * per_sm);
  kernel<<<blocks, kThreads, L.total, stream>>>(p);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}
template <int PROJ>
void launch_pull_p(const KernelParams &p, bool cv, bool ce, cudaStream_t s) {
  if (!cv && !ce) launch_pull_t<PROJ, false, false>(p, s);
  else if (cv && ce) launch_pull_t<PROJ, true, true>(p, s);
  else if (cv && !ce) launch_pull_t<PROJ, true, false>(p, s);
  else throw std::runtime_error("complex vectors need complex values");
}

template <int PROJ>
void launch_accumulate_p(const KernelParams &p, bool cv, bool ce, int64_t count, const uint64_t *b,
                         const double *c, cudaStream_t s) {
  const int blocks = grid_for((count + 1) / 2, kThreads, sm_count() * 8);
  if (!cv && !ce) k_accumulate<PROJ, false, false><<<blocks, kThreads, 0, s>>>(p, count, b, c);
  else if (cv && ce) k_accumulate<PROJ, true, true><<<blocks, kThreads, 0, s>>>(p, count, b, c);
  else if (cv && !ce) k_accumulate<PROJ, true, false><<<blocks, kThreads, 0, s>>>(p, count, b, c);
  else throw std::runtime_error("complex vectors need complex values");
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

}  // namespace

namespace {
template <bool CE, int TK, bool MPH, int CTAS = 2>
int launch_rows_t(const KernelParams &p, cudaStream_t stream) {
  const SmemLayout L = smem_layout(p, PROJ_GROUP, sizeof(double), false);
  const size_t smem_bytes = L.total;
  auto kernel = k_rows<CE, TK, MPH, CTAS>;
  if (smem_bytes > 48 * 1024)
    DMV_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  int per_sm = 0;
  DMV_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem_bytes));
  if (per_sm < 1) per_sm = 1;
  const int64_t tiles = (p.row_end - p.row_begin + 31) / 32;
  const int blocks = grid_for(tiles, kWarps, sm_count() * per_sm);
  kernel<<<blocks, kThreads, smem_bytes, stream>>>(p);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
  return 100 * CTAS + 10 * TK + (MPH ? 1 : 0);
}
template <bool CE>
int launch_rows_e(const KernelParams &p, cudaStream_t stream) {
  const OrbitProgram &o = p.orbit;
  const int k = (o.canon_mode != 0 && o.tor_mode == 2 && o.canon_k == o.canon_r) ? o.canon_k : 0;
  if (p.dense != nullptr) {   // dense index (perfect hash)
    if (k == 6) return launch_rows_t<CE, 6, true>(p, stream);
    if (k == 4) return launch_rows_t<CE, 4, true>(p, stream);
    return launch_rows_t<CE, 0, true>(p, stream);
  }
  if (p.rows_ctas == 2) {   // two CTAs per SM: 122 registers, nothing spills
    if (k == 6) return launch_rows_t<CE, 6, false>(p, stream);
    if (k == 4) return launch_rows_t<CE, 4, false>(p, stream);
    return launch_rows_t<CE, 0, false>(p, stream);
  }
  if (p.rows_ctas == 4) {   // four CTAs per SM: 64 registers
    if (k == 6) return launch_rows_t<CE, 6, false, 4>(p, stream);
    return launch_rows_t<CE, 0, false, 4>(p, stream);
  }
  // default: three CTAs per SM (80 registers; a few words of the pipeline state spill, 24 warps per SM more than pay for it:
  // 6x6 24.9 -> 22.3 ms, chain_36_symm 53.5 -> 44.0 ms, profiles/r02_rows_pipelines.md)
  if (k == 6) return launch_rows_t<CE, 6, false, 3>(p, stream);
  if (k == 4) return launch_rows_t<CE, 4, false, 3>(p, stream);
  return launch_rows_t<CE, 0, false, 3>(p, stream);
}
}  // namespace

namespace {
template <int TK, int CTAS>
int launch_rows_batch_t(const KernelParams &p, cudaStream_t stream) {
  const SmemLayout L = smem_layout(p, PROJ_GROUP, sizeof(double), false);
  const size_t smem_bytes = L.total;
  auto kernel = k_rows_batch<TK, CTAS>;
  if (smem_bytes > 48 * 1024)
    DMV_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  int per_sm = 0;
  DMV_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem_bytes));
  if (per_sm < 1) per_sm = 1;
  const int64_t tiles = (p.row_end - p.row_begin + 31) / 32;
  const int blocks = grid_for(tiles, kWarps, sm_count() * per_sm);
  kernel<<<blocks, kThreads, smem_bytes, stream>>>(p);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
  return 100 * CTAS + 10 * TK;
}
}  // namespace

// p.batch vectors of p.batch_elt doubles per element (p.batch * p.batch_elt <= 6), p.table = the 64-byte-bucket table
int launch_rows_batch(const KernelParams &p, cudaStream_t stream) {
  if (p.row_end <= p.row_begin) return 0;
  if (p.batch < 1 || (p.batch_elt != 1 && p.batch_elt != 2) || p.batch * p.batch_elt > 6)
    throw std::runtime_error("k_rows_batch: at most six doubles per state");
  const OrbitProgram &o = p.orbit;
  const int k = (o.canon_mode != 0 && o.tor_mode == 2 && o.canon_k == o.canon_r) ? o.canon_k : 0;
  // two CTAs per SM (120-128 registers: the eight words of the request stay in registers; at 80 registers part of them
  // spills and the batch is 4 % slower: profiles/r02_rows_batch_6x6.md)
  if (k == 6) return launch_rows_batch_t<6, 2>(p, stream);
  if (k == 4) return launch_rows_batch_t<4, 2>(p, stream);
  return launch_rows_batch_t<0, 2>(p, stream);
}

void launch_table_fill_batch(int64_t n, int num_vectors, int elt, const void *x, int64_t stride, const double *norms,
                             const uint32_t *slot_of, const uint64_t *reps, void *table, cudaStream_t stream) {
  if (n <= 0) return;
  const int blocks = grid_for(n, 256, sm_count() * 16);
  k_table_fill_batch<<<blocks, 256, 0, stream>>>(n, num_vectors * elt, elt, reinterpret_cast<const double *>(x), stride, norms,
                                                 slot_of, reps, reinterpret_cast<unsigned char *>(table));
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

int launch_rows(const KernelParams &p, bool complex_elements, cudaStream_t stream) {
  if (p.row_end <= p.row_begin) return 0;
  return complex_elements ? launch_rows_e<true>(p, stream) : launch_rows_e<false>(p, stream);
}

void launch_table_insert(const uint64_t *reps, int64_t n, void *table, uint32_t n_buckets, int slots_per_bucket,
                         uint32_t *slot_of, cudaStream_t stream, int bucket_bytes) {
  if (n <= 0) return;
  k_table_insert<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(reps, n, reinterpret_cast<unsigned char *>(table),
                                                                 n_buckets, slots_per_bucket, slot_of, bucket_bytes);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_table_fill(int64_t n, bool complex_elements, const void *x, const double *norms, const uint32_t *pos,
                       const uint32_t *slot_of, const uint64_t *reps, void *table, void *dense, cudaStream_t stream) {
  if (n <= 0) return;
  const int blocks = grid_for(n, 256, sm_count() * 16);
  unsigned char *t = reinterpret_cast<unsigned char *>(table), *d = reinterpret_cast<unsigned char *>(dense);
  if (complex_elements) k_table_fill<true><<<blocks, 256, 0, stream>>>(n, x, norms, pos, slot_of, reps, t, d);
  else k_table_fill<false><<<blocks, 256, 0, stream>>>(n, x, norms, pos, slot_of, reps, t, d);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_mph_mark(const uint64_t *keys, int64_t n, int level, uint32_t n_blocks, unsigned long long *seen,
                     unsigned long long *collide, cudaStream_t stream) {
  if (n <= 0) return;
  k_mph_mark<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(keys, n, level, n_blocks, seen, collide);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}
void launch_mph_compact(const uint64_t *keys, int64_t n, int level, uint32_t n_blocks, const unsigned long long *collide,
                        uint64_t *next, unsigned long long *next_count, cudaStream_t stream) {
  if (n <= 0) return;
  k_mph_compact<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(keys, n, level, n_blocks, collide, next, next_count);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}
void launch_mph_slots(const uint64_t *keys, int64_t n, PerfectHash mph, const void *table, uint32_t n_buckets,
                      int slots_per_bucket, uint32_t *slot_of, unsigned long long *status, cudaStream_t stream) {
  if (n <= 0) return;
  k_mph_slots<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(keys, n, mph, reinterpret_cast<const unsigned char *>(table),
                                                              n_buckets, slots_per_bucket, slot_of, status);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_generate(const KernelParams &p, Projection proj, bool cv, bool ce, bool count_only,
                     cudaStream_t stream) {
  if (p.row_end <= p.row_begin) return;
  switch (proj) {
    case PROJ_NONE: launch_generate_p<PROJ_NONE>(p, cv, ce, count_only, stream); break;
    case PROJ_INVERSION: launch_generate_p<PROJ_INVERSION>(p, cv, ce, count_only, stream); break;
    case PROJ_GROUP: launch_generate_p<PROJ_GROUP>(p, cv, ce, count_only, stream); break;
  }
}

void launch_pull(const KernelParams &p, Projection proj, bool cv, bool ce, cudaStream_t stream) {
  if (p.row_end <= p.row_begin) return;
  switch (proj) {
    case PROJ_NONE: launch_pull_p<PROJ_NONE>(p, cv, ce, stream); break;
    case PROJ_INVERSION: launch_pull_p<PROJ_INVERSION>(p, cv, ce, stream); break;
    case PROJ_GROUP: launch_pull_p<PROJ_GROUP>(p, cv, ce, stream); break;
  }
}

void launch_accumulate(const KernelParams &p, Projection proj, bool cv, bool ce, int64_t count,
                       const uint64_t *betas, const double *coeffs, cudaStream_t stream) {
  if (count <= 0) return;
  switch (proj) {
    case PROJ_NONE: launch_accumulate_p<PROJ_NONE>(p, cv, ce, count, betas, coeffs, stream); break;
    case PROJ_INVERSION: launch_accumulate_p<PROJ_INVERSION>(p, cv, ce, count, betas, coeffs, stream); break;
    case PROJ_GROUP: launch_accumulate_p<PROJ_GROUP>(p, cv, ce, count, betas, coeffs, stream); break;
  }
}

void launch_apply_diag(const KernelParams &p, int64_t count, const uint64_t *alphas, double *coeffs,
                       cudaStream_t stream) {
  if (count <= 0) return;
  const SmemLayout L = smem_layout(p, PROJ_NONE, sizeof(double2));
  if (L.total > 48 * 1024)
    DMV_CUDA_CHECK(cudaFuncSetAttribute(k_apply_diag, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
  k_apply_diag<<<grid_for(count, kThreads, sm_count() * 4), kThreads, L.total, stream>>>(p, count, alphas, coeffs);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_apply_off_diag(const KernelParams &p, int64_t count, const uint64_t *alphas, const int64_t *offsets,
                           int64_t *counts, uint64_t *betas, double *coeffs, bool write_pass, cudaStream_t stream) {
  if (count <= 0) return;
  const SmemLayout L = smem_layout(p, PROJ_NONE, sizeof(double2));
  const int blocks = grid_for(count, kThreads, sm_count() * 4);
  if (write_pass) {
    if (L.total > 48 * 1024)
      DMV_CUDA_CHECK(cudaFuncSetAttribute(k_apply_off_diag<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    k_apply_off_diag<true><<<blocks, kThreads, L.total, stream>>>(p, count, alphas, offsets, counts, betas,
                                                                   reinterpret_cast<double2 *>(coeffs));
  } else {
    if (L.total > 48 * 1024)
      DMV_CUDA_CHECK(cudaFuncSetAttribute(k_apply_off_diag<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    k_apply_off_diag<false><<<blocks, kThreads, L.total, stream>>>(p, count, alphas, offsets, counts, betas,
                                                                    reinterpret_cast<double2 *>(coeffs));
  }
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_build_directory(const uint64_t *reps, int64_t n, uint32_t *dir, uint64_t n_buckets, int shift,
                            cudaStream_t stream) {
  const int64_t items = 2 * (int64_t)n_buckets;
  k_build_directory<<<(unsigned)((items + 255) / 256), 256, 0, stream>>>(reps, n, dir, n_buckets, shift);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_state_index(const StateIndex &ix, int64_t count, const uint64_t *spins, int64_t *indices,
                        cudaStream_t stream) {
  if (count <= 0) return;
  k_state_index<<<(unsigned)((count + 255) / 256), 256, 0, stream>>>(ix, count, spins, indices);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_verify_rank(const StateIndex &ix, unsigned long long *status, cudaStream_t stream) {
  if (ix.n <= 0) return;
  k_verify_rank<<<(unsigned)((ix.n + 255) / 256), 256, 0, stream>>>(ix, status);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_locale_idx(int64_t count, const uint64_t *states, int num_ranks, uint8_t *keys, cudaStream_t stream) {
  if (count <= 0) return;
  k_locale_idx<<<(unsigned)((count + 255) / 256), 256, 0, stream>>>(count, states, num_ranks, keys);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_state_info(const OrbitProgram &P, Projection proj, uint64_t site_mask, double inv_char,
                       int64_t count, const uint64_t *alphas, uint64_t *betas, double *characters,
                       double *norms, cudaStream_t stream) {
  if (count <= 0) return;
  const unsigned blocks = (unsigned)((count + 127) / 128);
  double2 *ch = reinterpret_cast<double2 *>(characters);
  switch (proj) {
    case PROJ_NONE: k_state_info<PROJ_NONE><<<blocks, 128, 0, stream>>>(P, site_mask, inv_char, count, alphas, betas, ch, norms); break;
    case PROJ_INVERSION: k_state_info<PROJ_INVERSION><<<blocks, 128, 0, stream>>>(P, site_mask, inv_char, count, alphas, betas, ch, norms); break;
    case PROJ_GROUP: k_state_info<PROJ_GROUP><<<blocks, 128, 0, stream>>>(P, site_mask, inv_char, count, alphas, betas, ch, norms); break;
  }
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_compute_norms(const OrbitProgram &P, int64_t count, const uint64_t *reps, double *norms,
                          cudaStream_t stream) {
  if (count <= 0) return;
  k_compute_norms<<<(unsigned)((count + 127) / 128), 128, 0, stream>>>(P, count, reps, norms);
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

void launch_enumerate(const OrbitProgram &P, Projection proj, uint64_t site_mask, bool fixed_hamming,
                      int rank, int num_ranks, int64_t n_chunks, const uint64_t *chunk_first,
                      const uint64_t *chunk_last, unsigned long long *chunk_count,
                      const unsigned long long *chunk_offset, uint64_t *out, double *out_norms,
                      bool write_pass, cudaStream_t stream) {
  if (n_chunks <= 0) return;
  const unsigned blocks = (unsigned)((n_chunks + 127) / 128);
#define DMV_ENUM(PR)                                                                                      \
  if (write_pass)                                                                                         \
    k_enumerate<PR, true><<<blocks, 128, 0, stream>>>(P, site_mask, fixed_hamming, rank, num_ranks,       \
                                                      n_chunks, chunk_first, chunk_last, chunk_count,     \
                                                      chunk_offset, out, out_norms);                      \
  else                                                                                                    \
    k_enumerate<PR, false><<<blocks, 128, 0, stream>>>(P, site_mask, fixed_hamming, rank, num_ranks,      \
                                                       n_chunks, chunk_first, chunk_last, chunk_count,    \
                                                       chunk_offset, out, out_norms)
  switch (proj) {
    case PROJ_NONE: DMV_ENUM(PROJ_NONE); break;
    case PROJ_INVERSION: DMV_ENUM(PROJ_INVERSION); break;
    case PROJ_GROUP: DMV_ENUM(PROJ_GROUP); break;
  }
#undef DMV_ENUM
  DMV_CUDA_CHECK(cudaGetLastError());
  g_launches++;
}

}  // namespace dmv
