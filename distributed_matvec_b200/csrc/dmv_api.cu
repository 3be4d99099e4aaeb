// dmv_api.cu -- the C ABI of libdmv_b200.so (see include/dmv_b200.h): context, basis, the single-rank product and the
// stepwise pieces of the distributed one.  Exchanges: dmv_exchange.cu; eigensolver: dmv_lanczos.cu; plugin table: dmv_plugin.cu.
#include "dmv_context.h"

namespace dmv { namespace host {
thread_local std::string g_last_error;
} }

namespace dmv { namespace host {


// support of a group: union of the masks of its terms
uint64_t support_of(const std::vector<OffTerm> &terms) {
  uint64_t m = 0;
  for (const auto &t : terms) m |= t.m;
  return m;
}

HostTables build_tables(const std::map<uint64_t, std::vector<OffTerm>> &by_x) {
  HostTables H;
  // ---- can the whole operator use the bit-parallel emit test?  (every group: support <= 2 bits and a
  // common sign mask outside the support)
  struct Item { uint64_t x; const std::vector<OffTerm> *terms; int p0, p1; };
  std::vector<Item> items;
  bool bp_ok = !by_x.empty();
  for (const auto &kv : by_x) {
    const uint64_t sup = support_of(kv.second);
    const int k = __builtin_popcountll(sup);
    Item it{kv.first, &kv.second, 0, 0};
    if (k > 2) bp_ok = false;
    if (k >= 1) it.p0 = __builtin_ctzll(sup);
    it.p1 = (k == 2) ? 63 - __builtin_clzll(sup) : it.p0;
    const uint64_t s_out = kv.second.front().s & ~sup;
    for (const auto &t : kv.second) if ((t.s & ~sup) != s_out) bp_ok = false;
    items.push_back(it);
  }
  if (bp_ok) {
    // Two orders of the groups are tried.  (1) by the LOWEST site they act on: the groups acting only on high sites get
    // the high bits of the emit mask -- the 32 consecutive rows of a warp share their high bits, so k_gather, walking the
    // mask from the top, keeps its lanes in step (chains: two shifts per operand).  (2) by the distance between the two
    // sites, then position: few distinct shifts "group index - bit position" on two-dimensional lattices, where (1)
    // needs more than kBpPairs of them.
    const int n_words = (int)((items.size() + 63) / 64);
    std::vector<BpWord> words;
    for (int order = 0; order < 2; ++order) {
      std::stable_sort(items.begin(), items.end(), [order](const Item &a, const Item &b) {
        if (order == 0) return a.p0 != b.p0 ? a.p0 < b.p0 : a.p1 < b.p1;
        if (a.p1 - a.p0 != b.p1 - b.p0) return a.p1 - a.p0 < b.p1 - b.p0;
        return a.p0 < b.p0;
      });
      bp_ok = true;
      words.assign((size_t)n_words, BpWord{});
      for (auto &w : words) memset(&w, 0, sizeof(w));
      for (size_t g = 0; g < items.size() && bp_ok; ++g) {
        BpWord &W = words[g / 64];
        const int gl = (int)(g % 64);
        auto add = [&](int pos, BpPair *pairs, int32_t &n) {
          const int d = gl - pos;
          const uint32_t sl = d >= 0 ? (uint32_t)d : 0u, sr = d >= 0 ? 0u : (uint32_t)(-d);
          for (int k = 0; k < n; ++k)
            if (pairs[k].l == sl && pairs[k].r == sr) { pairs[k].m |= 1ull << gl; return; }
          if (n == kBpPairs) { bp_ok = false; return; }
          pairs[n].l = sl; pairs[n].r = sr; pairs[n].m = 1ull << gl; ++n;
        };
        add(items[g].p0, W.p0, W.n0);
        add(items[g].p1, W.p1, W.n1);
      }
      if (bp_ok) break;
    }
    if (bp_ok) {
      for (size_t g = 0; g < items.size(); ++g) {
        const Item &it = items[g];
        LutGroup grp{};
        grp.x = it.x;
        grp.first = (int32_t)H.terms.size();
        grp.count = (int32_t)it.terms->size();
        const uint64_t sup = support_of(*it.terms);
        grp.s_out = it.terms->front().s & ~sup;
        if (grp.s_out) H.any_s_out = true;
        grp.posk = (2ull << 48) | ((uint64_t)it.p1 << 8) | (uint64_t)it.p0;
        grp.lut_offset = (uint32_t)(4 * g);
        for (const auto &t : *it.terms) H.terms.push_back(t);
        for (int idx = 0; idx < 4; ++idx) {
          const int b0 = idx & 1, b1 = idx >> 1;
          double re = 0.0, im = 0.0;
          bool hit = false;
          if (!(it.p0 == it.p1 && b0 != b1)) {
            const uint64_t a = ((uint64_t)b0 << it.p0) | ((uint64_t)b1 << it.p1);
            for (const auto &t : *it.terms)
              if ((a & t.m) == t.r) {
                const double sg = (__builtin_popcountll(a & t.s & sup) & 1) ? -1.0 : 1.0;
                re += sg * t.v_re; im += sg * t.v_im; hit = true;
              }
          }
          if (hit && (re != 0.0 || im != 0.0)) {
            grp.emit_bits |= 1ull << idx;
            words[g / 64].tt[idx] |= 1ull << (g % 64);
          }
          H.lut_re.push_back(re);
          H.lut_c.push_back(re); H.lut_c.push_back(im);
        }
        H.groups.push_back(grp);
      }
      H.bp = words;
      return H;
    }
  }
  // ---- general layout: one LUT of 2^k entries per group (k <= 6), term-by-term evaluation otherwise
  for (const auto &kv : by_x) {
    LutGroup g{};
    g.x = kv.first;
    g.first = (int32_t)H.terms.size();
    g.count = (int32_t)kv.second.size();
    for (const auto &t : kv.second) H.terms.push_back(t);
    const uint64_t support = support_of(kv.second);
    const int k = __builtin_popcountll(support);
    bool lutable = k <= 6;
    const uint64_t s_out = kv.second.front().s & ~support;
    for (const auto &t : kv.second) lutable &= ((t.s & ~support) == s_out);
    if (lutable) {
      int pos[6] = {0, 0, 0, 0, 0, 0}, nb = 0;
      for (int b = 0; b < 64; ++b) if ((support >> b) & 1) pos[nb++] = b;
      g.posk = (uint64_t)k << 48;
      for (int b = 0; b < k; ++b) g.posk |= (uint64_t)pos[b] << (8 * b);
      g.s_out = s_out;
      g.lut_offset = (uint32_t)H.lut_re.size();
      for (int idx = 0; idx < (1 << k); ++idx) {
        uint64_t a = 0;
        for (int b = 0; b < k; ++b) if ((idx >> b) & 1) a |= 1ull << pos[b];
        double re = 0.0, im = 0.0;
        bool hit = false;
        for (const auto &t : kv.second)
          if ((a & t.m) == t.r) {
            const double sg = (__builtin_popcountll(a & t.s & support) & 1) ? -1.0 : 1.0;
            re += sg * t.v_re; im += sg * t.v_im; hit = true;
          }
        if (hit && (re != 0.0 || im != 0.0)) g.emit_bits |= 1ull << idx;
        H.lut_re.push_back(re);
        H.lut_c.push_back(re); H.lut_c.push_back(im);
      }
      if (s_out) H.any_s_out = true;
    } else {
      g.posk = 1ull << 56;
      H.any_generic = true;
    }
    H.groups.push_back(g);
  }
  return H;
}

bool use_gather(const dmv_context *ctx) {   // the lean row-gather kernel applies and is not switched off
  return ctx->gather_ok && ctx->opt_gather != 0 && ctx->opt_bitparallel != 0 && ctx->proj != PROJ_GROUP;
}
bool use_rows(const dmv_context *ctx) {   // the pipelined row kernel for bases with permutation symmetries
  return ctx->rows_ok && ctx->opt_rows != 0 && ctx->opt_bitparallel != 0 && ctx->orbit.trivial_characters;
}
bool use_pull(const dmv_context *ctx) {
  // auto: one rank, bit-parallel operator, no permutation symmetries -> k_gather (rows, no atomics, see
  // dmv_gather.cu); everything else -> push (k_generate).  "mode" = 1 forces the row traversal (k_gather
  // when it applies, else the queued k_pull), "mode" = 0 the scatter form.
  if (ctx->num_ranks != 1) return false;
  if (ctx->opt_mode == 1) return true;
  return ctx->opt_mode == -1 && (use_gather(ctx) || use_rows(ctx));
}

void use_device(const dmv_context *ctx) { CUDA_CHECK(cudaSetDevice(ctx->device)); }

bool complex_values(const dmv_context *ctx, int elt) { return elt == DMV_C128 || ctx->complex_coefficients; }

KernelParams base_params(dmv_context *ctx) {
  KernelParams p{};
  p.index.reps = ctx->d_reps.ptr;
  p.index.n = ctx->n_states;
  p.index.dir = ctx->d_dir.ptr;
  p.index.n_buckets = ctx->n_buckets;
  p.index.shift = ctx->dir_shift;
  p.index.mode = ctx->index_mode;
  p.index.binom = ctx->d_binom.ptr;
  p.index.stride = ctx->binom_stride;
  p.index.n_sites = ctx->n_sites;
  p.index.weight = ctx->hamming_weight;
  p.index.site_mask = ctx->site_mask;
  p.index.lin_a = ctx->d_lin_a.ptr;
  p.index.lin_b = ctx->d_lin_b.ptr;
  p.index.lin_bits = ctx->lin_bits;
  p.rank_total = ctx->rank_total;
  p.norms = ctx->d_norms.ptr;
  p.diag = ctx->d_diag.ptr;     p.n_diag = (int)ctx->h_diag_kept;
  p.diag_classes = ctx->d_diag_classes.ptr; p.n_diag_classes = (int)ctx->h_diag_classes.size();
  p.n_diag_rest = ctx->n_diag_rest;
  p.orbit = ctx->orbit;
  p.site_mask = ctx->site_mask;
  p.inversion_character = (double)ctx->spin_inversion;
  p.rank = ctx->rank;
  p.num_ranks = ctx->num_ranks;
  p.out_betas = ctx->d_out_betas.ptr;
  p.out_coeffs = ctx->d_out_coeffs.ptr;
  p.out_offset = ctx->d_out_offset.ptr;
  p.out_count = ctx->d_out_count.ptr;
  p.grid_blocks = ctx->num_ranks > 1 ? ctx->plan_grid : 0;
  p.row_split = ctx->row_split;
  p.warp_offsets = ctx->d_warp_offsets.ptr;
  p.warp_counts = ctx->d_warp_counts.ptr;
  p.out_betas_ptr = ctx->d_out_betas_ptr.ptr;
  p.out_coeffs_ptr = ctx->d_out_coeffs_ptr.ptr;
  p.out_capacity = ctx->d_out_capacity.ptr;
  p.status = ctx->d_status.ptr;
  p.row_begin = 0;
  p.row_end = ctx->n_states;
  p.gather_walk = ctx->opt_gather_walk;
  p.rows_ctas = ctx->opt_rows_ctas;
  return p;
}

// Split the diagonal into bit-parallel classes (m =, two sign bits, equal coefficient) and the rest.
void build_diag_classes(dmv_context *ctx) {
  std::vector<DiagTerm> rest;
  std::map<std::pair<double, double>, std::vector<DiagTerm>> by_v;
  for (const auto &d : ctx->h_diag) {
    if (d.m == 0 && d.r == 0 && __builtin_popcountll(d.s) == 2) by_v[{d.v_re, d.v_im}].push_back(d);
    else rest.push_back(d);
  }
  for (auto &kv : by_v) {
    auto &terms = kv.second;
    std::stable_sort(terms.begin(), terms.end(), [](const DiagTerm &a, const DiagTerm &b) {
      const int a0 = __builtin_ctzll(a.s), a1 = 63 - __builtin_clzll(a.s);
      const int b0 = __builtin_ctzll(b.s), b1 = 63 - __builtin_clzll(b.s);
      if (a1 - a0 != b1 - b0) return a1 - a0 < b1 - b0;
      return a0 < b0;
    });
    for (size_t first = 0; first < terms.size(); first += 64) {
      const size_t n = std::min<size_t>(64, terms.size() - first);
      DiagClass D;
      memset(&D, 0, sizeof(D));
      D.v_re = kv.first.first; D.v_im = kv.first.second;
      bool ok = true;
      for (size_t t = 0; t < n && ok; ++t) {
        const uint64_t sbits = terms[first + t].s;
        const int pos[2] = {__builtin_ctzll(sbits), 63 - __builtin_clzll(sbits)};
        BpPair *pairs[2] = {D.p0, D.p1};
        int32_t *cnt[2] = {&D.n0, &D.n1};
        for (int b = 0; b < 2 && ok; ++b) {
          const int d = (int)t - pos[b];
          const uint32_t sl = d >= 0 ? (uint32_t)d : 0u, sr = d >= 0 ? 0u : (uint32_t)(-d);
          int k = 0;
          for (; k < *cnt[b]; ++k)
            if (pairs[b][k].l == sl && pairs[b][k].r == sr) break;
          if (k == *cnt[b]) {
            if (k == kBpPairs) { ok = false; break; }
            pairs[b][k].l = sl; pairs[b][k].r = sr; pairs[b][k].m = 0; ++*cnt[b];
          }
          pairs[b][k].m |= 1ull << t;
        }
      }
      if (ok) {
        D.count = (int32_t)n;
        D.mask = n == 64 ? ~0ull : ((1ull << n) - 1);
        ctx->h_diag_classes.push_back(D);
      } else {
        for (size_t t = 0; t < n; ++t) rest.push_back(terms[first + t]);
      }
    }
  }
  // reorder: the terms evaluated one by one come first
  ctx->n_diag_rest = (int)rest.size();
  std::vector<DiagTerm> reordered = rest;
  ctx->h_diag_kept = ctx->h_diag.size();
  ctx->h_diag = reordered;
}

// point the kernel at the column-traversal (push) or row-traversal (pull) tables
void select_tables(dmv_context *ctx, KernelParams &p, bool pull, bool complex_vals) {
  const HostTables &h = pull ? ctx->h_pull : ctx->h_push;
  DevTables &d = pull ? ctx->d_pull : ctx->d_push;
  p.groups = d.groups.ptr; p.n_groups = (int)h.groups.size();
  p.lut = complex_vals ? d.lut_c.ptr : d.lut_re.ptr; p.n_lut = (int)h.lut_re.size();
  p.terms = d.terms.ptr; p.n_terms = (int)h.terms.size();
  p.any_generic = h.any_generic ? 1 : 0;
  p.any_s_out = h.any_s_out ? 1 : 0;
  p.bp = d.bp.ptr; p.n_bp = (ctx->opt_bitparallel != 0) ? (int)h.bp.size() : 0;
}

void require_states(const dmv_context *ctx) {
  if (ctx->n_states < 0) throw std::runtime_error("basis is not built");  // src/ForeignTypes.chpl:113-114
}

void check_status(dmv_context *ctx) {
  unsigned long long st[4];
  CUDA_CHECK(cudaMemcpyAsync(st, ctx->d_status.ptr, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (st[0] != 0 || st[2] != 0 || st[3] != 0) {
    CUDA_CHECK(cudaMemsetAsync(ctx->d_status.ptr, 0, 4 * sizeof(unsigned long long), ctx->stream));
    char buf[256];
    if (st[3] != 0)
      snprintf(buf, sizeof(buf), "peer-direct all-gather of x: a rank did not raise its flag within the time limit");
    else if (st[2] != 0)
      snprintf(buf, sizeof(buf), "outgoing bucket overflow (%llu records): plan is stale", st[2]);
    else  // message of the reference: DMV:116-118
      snprintf(buf, sizeof(buf), "invalid index: -1 for state %llu (%llu such records): the operator does "
               "not respect the basis symmetries or the representatives are incomplete", st[1], st[0]);
    throw std::runtime_error(buf);
  }
}
const Binomials &binom() { static Binomials b; return b; }

// Which state -> index kernel applies (the reference's per-basis `state_index_kernel`, FFI:90-93).
//   auto (-1): identity when it applies; two-table Lin lookup for full fixed-Hamming bases on one rank
//   (<= 40 sites); directory search otherwise.  0 forces the directory, 2 the combinadic rank, 3 Lin.
void select_index_mode(dmv_context *ctx) {
  ctx->index_mode = INDEX_DIRECTORY;
  if (ctx->identity_index && ctx->num_ranks == 1) { ctx->index_mode = INDEX_IDENTITY; return; }
  const int n = ctx->n_sites, w = ctx->hamming_weight;
  const int want = ctx->opt_index;
  if (want == 0) return;
  const bool eligible = ctx->num_ranks == 1 && w >= 0 && ctx->proj != PROJ_GROUP;
  if (!eligible) return;
  const uint64_t total = binom().c[n][w];
  const uint64_t expect = (ctx->proj == PROJ_INVERSION) ? total / 2 : total;
  if ((uint64_t)ctx->n_states != expect || total >= (1ull << 32)) return;
  StateIndex ix{};
  ix.reps = ctx->d_reps.ptr; ix.n = ctx->n_states; ix.n_sites = n; ix.weight = w; ix.site_mask = ctx->site_mask;
  if (want == 2) {
    const int stride = w + 2;
    std::vector<uint32_t> table((size_t)n * stride);
    for (int pos = 0; pos < n; ++pos)
      for (int k = 0; k < stride; ++k)
        table[(size_t)pos * stride + k] = (uint32_t)std::min<uint64_t>(binom().c[pos][k], 0xffffffffull);
    ctx->d_binom.upload(table, ctx->stream);
    ctx->binom_stride = stride;
    ix.mode = INDEX_RANK; ix.binom = ctx->d_binom.ptr; ix.stride = stride;
  } else {
    if (n > 40) return;
    // Lin tables: states ascending = (hi, lo) lexicographic; index = Ja[hi] + Jb[lo]
    const int lb = n / 2, hb = n - lb;
    std::vector<uint32_t> ja((size_t)1 << hb), jb((size_t)1 << lb);
    uint64_t running = 0;
    for (uint64_t hi = 0; hi < (1ull << hb); ++hi) {
      const int k = w - __builtin_popcountll(hi);
      ja[hi] = (uint32_t)std::min<uint64_t>(running, 0xffffffffull);
      if (k >= 0 && k <= lb) running += binom().c[lb][k];
    }
    std::vector<uint32_t> counter(lb + 1, 0);
    for (uint64_t lo = 0; lo < (1ull << lb); ++lo) jb[lo] = counter[__builtin_popcountll(lo)]++;
    ctx->d_lin_a.upload(ja, ctx->stream);
    ctx->d_lin_b.upload(jb, ctx->stream);
    ctx->lin_bits = lb;
    ix.mode = INDEX_LIN; ix.lin_a = ctx->d_lin_a.ptr; ix.lin_b = ctx->d_lin_b.ptr; ix.lin_bits = lb;
  }
  ctx->rank_total = total;
  // the block must be exactly the first `expect` fixed-weight states: index(reps[i]) == i for all i
  CUDA_CHECK(cudaMemsetAsync(ctx->d_status.ptr, 0, 4 * sizeof(unsigned long long), ctx->stream));
  launch_verify_rank(ix, ctx->d_status.ptr, ctx->stream);
  unsigned long long bad = 0;
  CUDA_CHECK(cudaMemcpyAsync(&bad, ctx->d_status.ptr, sizeof(bad), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  CUDA_CHECK(cudaMemsetAsync(ctx->d_status.ptr, 0, 4 * sizeof(unsigned long long), ctx->stream));
  if (bad == 0) ctx->index_mode = ix.mode;
}

void install_directory(dmv_context *ctx) {
  const int64_t n = ctx->n_states;
  uint64_t max_rep = 0;
  if (n > 0) CUDA_CHECK(cudaMemcpyAsync(&max_rep, ctx->d_reps.ptr + (n - 1), 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  int bits = 0;
  while (bits < 64 && (max_rep >> bits) != 0) ++bits;
  // about 4 states per bucket on average, at least 2^10 and at most 2^26 buckets
  int want = 10;
  while (want < 26 && (1ll << (want + 2)) < n) ++want;
  int shift = bits > want ? bits - want : 0;
  ctx->dir_shift = shift;
  ctx->n_buckets = (max_rep >> shift) + 1;
  ctx->d_dir.alloc(2 * ctx->n_buckets + 2);
  launch_build_directory(ctx->d_reps.ptr, n, ctx->d_dir.ptr, ctx->n_buckets, shift, ctx->stream);
  ctx->planned = false;
  ctx->table_elt = 0;
  ctx->table_batch_slots = 0;
  // a new block also invalidates the exchange set-up: the replicated-x twin / slot table and the record plan
  ctx->exchange_decided = false;
  ctx->replicated = false;
  ctx->repl_block = 0;
  if (ctx->global) { delete ctx->global; ctx->global = nullptr; }
  ctx->d_pos.release();
  for (auto &q : ctx->peer_xcat) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
  for (auto &q : ctx->peer_flagmem) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
  ctx->peer_gather = false;
  ctx->peer_slot_elt = 0;
  ctx->d_xcat.release();
  for (auto *v : {&ctx->rounds.peer_betas, &ctx->rounds.peer_coeffs, &ctx->rounds.peer_flags})
    for (auto &q : *v) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
  ctx->rounds.ready = false;
  ctx->rounds.tried = false;
  std::fill(ctx->recv_counts.begin(), ctx->recv_counts.end(), -1);
  select_index_mode(ctx);
}

void upload_orbit(dmv_context *ctx) {
  const HostOrbitProgram &H = ctx->host_orbit;
  std::vector<uint64_t> h64 = H.benes_mask;
  h64.insert(h64.end(), H.step_mask.begin(), H.step_mask.end());
  if (h64.size() & 1) h64.push_back(0);   // 16-byte alignment of the packed 32-bit steps
  const size_t off_pack64 = h64.size();
  h64.insert(h64.end(), H.step_pack64.begin(), H.step_pack64.end());
  if (h64.size() & 1) h64.push_back(0);
  const size_t off_pack32 = h64.size();
  for (size_t i = 0; i + 1 < H.step_pack32.size(); i += 2)
    h64.push_back((uint64_t)H.step_pack32[i] | ((uint64_t)H.step_pack32[i + 1] << 32));
  std::vector<int32_t> h32 = H.benes_delta;
  h32.insert(h32.end(), H.step_shift.begin(), H.step_shift.end());
  ctx->d_orbit64.upload(h64, ctx->stream);
  ctx->d_orbit32.upload(h32, ctx->stream);
  ctx->d_chars.upload(H.characters, ctx->stream);
  OrbitProgram P = H.view();
  P.benes_mask = ctx->d_orbit64.ptr;
  P.step_mask = ctx->d_orbit64.ptr + H.benes_mask.size();
  P.benes_delta = ctx->d_orbit32.ptr;
  P.step_shift = ctx->d_orbit32.ptr + H.benes_delta.size();
  P.characters = reinterpret_cast<const double2 *>(ctx->d_chars.ptr);
  P.simple = H.simple;
  P.step_pack64 = ctx->d_orbit64.ptr + off_pack64;
  P.step_pack32 = H.step_pack32.empty() ? nullptr : reinterpret_cast<const uint4 *>(ctx->d_orbit64.ptr + off_pack32);
  ctx->d_canon_lut.upload(H.canon_lut, ctx->stream);
  ctx->d_canon_masks.upload(H.canon_masks, ctx->stream);
  P.canon_lut = ctx->d_canon_lut.ptr;
  P.canon_masks = ctx->d_canon_masks.ptr;
  ctx->d_canon_lut2.upload(H.canon_lut2, ctx->stream);
  ctx->d_cc_begin.upload(H.cc_begin, ctx->stream);
  ctx->d_cc_mask.upload(H.cc_mask, ctx->stream);
  ctx->d_cc_delta.upload(H.cc_delta, ctx->stream);
  P.canon_lut2 = H.canon_lut2.empty() ? nullptr : ctx->d_canon_lut2.ptr;
  P.cc_begin = ctx->d_cc_begin.ptr;
  P.cc_mask = ctx->d_cc_mask.ptr;
  P.cc_delta = ctx->d_cc_delta.ptr;
  ctx->d_tor_lutm.upload(H.tor_lutm, ctx->stream);
  ctx->d_tor_luts.upload(H.tor_luts, ctx->stream);
  ctx->d_tor_net_mask.upload(H.tor_net_mask, ctx->stream);
  ctx->d_tor_net_delta.upload(H.tor_net_delta, ctx->stream);
  P.tor_lutm = ctx->d_tor_lutm.ptr;
  P.tor_luts = ctx->d_tor_luts.ptr;
  ctx->d_tor_frow.upload(H.tor_frow, ctx->stream);
  P.tor_frow = ctx->d_tor_frow.ptr;
  P.tor_net_mask = ctx->d_tor_net_mask.ptr;
  P.tor_net_delta = ctx->d_tor_net_delta.ptr;
  if (ctx->opt_canon >= 0) { P.tor_mode = 0; P.chain_dihedral = 0; }   // 1: round-1 forms (coset chain / four run searches)
  if (ctx->opt_canon == 2) { P.canon_lut2 = nullptr; P.cc_n = 0; P.cc_stages = 0; }   // first version: single-block LUT, independent networks
  if (ctx->opt_canon == 0) P.canon_mode = 0;
  ctx->orbit = P;
}

// rank of a fixed-weight state among states of the same weight in ascending order
// (what ls_hs_fixed_hamming_state_to_index computes, reference src/FFI.chpl:165)
uint64_t fixed_hamming_rank(uint64_t s) {
  uint64_t r = 0;
  int k = 0;
  while (s) {
    const int pos = __builtin_ctzll(s);
    ++k;
    r += binom().c[pos][k];
    s &= s - 1;
  }
  return r;
}
uint64_t fixed_hamming_unrank(uint64_t r, int weight) {  // ls_hs_fixed_hamming_index_to_state
  uint64_t s = 0;
  for (int k = weight; k >= 1; --k) {
    int pos = k - 1;
    while (pos + 1 <= 63 && binom().c[pos + 1][k] <= r) ++pos;
    r -= binom().c[pos][k];
    s |= 1ull << pos;
  }
  return s;
}

void zero_y_if_diag(dmv_context *ctx, int elt, void *y) {
  // DMV:1062-1063: with diagonal terms y is overwritten by D x, otherwise it is accumulated into
  if (ctx->h_diag_kept > 0)
    CUDA_CHECK(cudaMemsetAsync(y, 0, (size_t)ctx->n_states * 8 * elt, ctx->stream));
}
VecStage stage_vectors(dmv_context *ctx, int elt, const void *x, void *y) {
  VecStage v{};
  v.bytes = (size_t)ctx->n_states * 8 * elt;
  CUDA_CHECK(cudaEventRecord(ctx->ev[0], ctx->stream));
  if (is_device_pointer(x)) v.x_dev = x;
  else {
    ctx->d_x.alloc((size_t)ctx->n_states * elt);
    v.x_dev = ctx->d_x.ptr;
    // the column traversal only reads x[i] of the rows it is generating: upload in row chunks on a copy
    // stream and start generating as soon as the first chunk has landed (see do_generate)
    if (!use_pull(ctx) && ctx->num_ranks == 1 && ctx->n_states >= (1 << 16)) v.x_host_pending = x;
    else CUDA_CHECK(cudaMemcpyAsync(ctx->d_x.ptr, x, v.bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (is_device_pointer(y)) { v.y_dev = y; v.y_host = false; }
  else {
    ctx->d_y.alloc((size_t)ctx->n_states * elt);
    v.y_dev = ctx->d_y.ptr; v.y_host = true; v.y_user = y;
    if (ctx->h_diag_kept == 0)  // y is accumulated into: bring the caller's y over
      CUDA_CHECK(cudaMemcpyAsync(ctx->d_y.ptr, y, v.bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  CUDA_CHECK(cudaEventRecord(ctx->ev[1], ctx->stream));
  return v;
}
void finish_vectors(dmv_context *ctx, const VecStage &v) {
  CUDA_CHECK(cudaEventRecord(ctx->ev[4], ctx->stream));
  if (v.y_host) CUDA_CHECK(cudaMemcpyAsync(v.y_user, v.y_dev, v.bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaEventRecord(ctx->ev[5], ctx->stream));
}

void upload_out_pointers(dmv_context *ctx) {
  ctx->d_out_betas_ptr.upload(ctx->h_out_betas_ptr, ctx->stream);
  ctx->d_out_coeffs_ptr.upload(ctx->h_out_coeffs_ptr, ctx->stream);
}

// One counting pass.  Record counts do not depend on x, and the grid-stride tile loop is deterministic,
// so the pass yields (a) the exact number of records for every destination and (b) for num_ranks <= 32
// the exact share of every warp, from which each warp gets a private, exactly sized slice of every
// destination region (prefix sums): the real pass needs no slot-claim atomics at all.
void do_plan(dmv_context *ctx) {
  require_states(ctx);
  const int P = ctx->num_ranks;
  const bool exact_regions = P <= 32;
  ctx->row_split = choose_row_split(ctx->n_states, (int)ctx->h_push.groups.size());
  ctx->plan_grid = planned_grid(ctx->n_states, ctx->row_split);
  const size_t n_warps = (size_t)ctx->plan_grid * kWarpsPerCta;
  ctx->d_out_count.alloc(P);
  ctx->d_warp_counts.alloc(n_warps * P);
  CUDA_CHECK(cudaMemsetAsync(ctx->d_out_count.ptr, 0, sizeof(unsigned long long) * P, ctx->stream));
  CUDA_CHECK(cudaMemsetAsync(ctx->d_warp_counts.ptr, 0, sizeof(unsigned long long) * n_warps * P, ctx->stream));
  KernelParams p = base_params(ctx);
  p.grid_blocks = ctx->plan_grid;
  select_tables(ctx, p, false, ctx->complex_coefficients);
  // counting pass: element type does not matter
  launch_generate(p, ctx->proj, ctx->complex_coefficients, false, /*count_only=*/true, ctx->stream);
  std::vector<unsigned long long> counts(P, 0);
  std::vector<int64_t> warp_offsets(n_warps * P, 0);
  if (exact_regions) {
    std::vector<unsigned long long> wc(n_warps * P);
    CUDA_CHECK(cudaMemcpyAsync(wc.data(), ctx->d_warp_counts.ptr, sizeof(unsigned long long) * wc.size(),
                               cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    for (int d = 0; d < P; ++d)
      for (size_t w = 0; w < n_warps; ++w) {
        warp_offsets[w * P + d] = (int64_t)counts[d];
        counts[d] += wc[w * P + d];
      }
  } else {
    CUDA_CHECK(cudaMemcpyAsync(counts.data(), ctx->d_out_count.ptr, sizeof(unsigned long long) * P,
                               cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  }
  ctx->d_warp_offsets.upload(warp_offsets, ctx->stream);
  ctx->send_counts.assign(P, 0);
  ctx->number_terms = 0;
  for (int d = 0; d < P; ++d) { ctx->send_counts[d] = (int64_t)counts[d]; ctx->number_terms += (int64_t)counts[d]; }
  ctx->h_out_offset.assign(P + 1, 0);
  std::vector<int64_t> capacity(P, 0);
  for (int d = 0; d < P; ++d) {
    capacity[d] = (d == ctx->rank) ? 0 : ctx->send_counts[d];
    ctx->h_out_offset[d + 1] = ctx->h_out_offset[d] + capacity[d];
  }
  ctx->d_out_offset.upload(ctx->h_out_offset, ctx->stream);
  ctx->d_out_capacity.upload(capacity, ctx->stream);
  const int64_t total_out = ctx->h_out_offset[P];
  ctx->d_out_betas.alloc((size_t)total_out);
  ctx->d_out_coeffs.alloc((size_t)total_out * 2);
  // by default the records of destination d go to the local bucket d (sent with NCCL afterwards);
  // the coefficient base assumes the widest record (re-derived per product, see do_generate)
  ctx->h_out_betas_ptr.assign(P, nullptr);
  ctx->h_out_coeffs_ptr.assign(P, nullptr);
  ctx->peer_direct = false;
  ctx->ptr_width = 0;
  ctx->recv_counts.assign(P, -1);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  ctx->planned = true;
}

// hash table of k_rows over ctx's representatives: keys once per basis and element type, values once per product
void ensure_table(dmv_context *ctx, int elt) {
  if (ctx->table_elt == elt) return;
  const int64_t n = ctx->n_states;
  cudaStream_t st = ctx->stream;
  const bool ce = elt == DMV_C128;
  // ---- dense index: two perfect-hash levels of 4 bits per state; what they cannot place goes to the table below
  const uint64_t *left_keys = ctx->d_reps.ptr;
  int64_t n_left = n;
  DevBuf<uint64_t> d_left[2];
  ctx->dense_index = ctx->opt_rows_index == 1 && n >= 1;
  ctx->mph = PerfectHash{};
  if (ctx->dense_index) {
    if (n >= 2147483647ll) throw std::runtime_error("k_rows: more than 2^31 states");
    std::vector<unsigned long long> bits;      // seen & ~collide of both levels, 3 words per block
    uint32_t nb[2] = {0, 0};
    DevBuf<unsigned long long> d_count;
    d_count.alloc(1);
    for (int level = 0; level < 2 && n_left > 0; ++level) {
      nb[level] = (uint32_t)std::max<int64_t>(1, (4 * n_left + kMphBits - 1) / kMphBits);
      const size_t words = (size_t)nb[level] * 3;
      DevBuf<unsigned long long> d_seen, d_coll;
      d_seen.alloc(words); d_coll.alloc(words);
      CUDA_CHECK(cudaMemsetAsync(d_seen.ptr, 0, words * 8, st));
      CUDA_CHECK(cudaMemsetAsync(d_coll.ptr, 0, words * 8, st));
      CUDA_CHECK(cudaMemsetAsync(d_count.ptr, 0, 8, st));
      launch_mph_mark(left_keys, n_left, level, nb[level], d_seen.ptr, d_coll.ptr, st);
      d_left[level].alloc((size_t)std::max<int64_t>(1, n_left));
      launch_mph_compact(left_keys, n_left, level, nb[level], d_coll.ptr, d_left[level].ptr, d_count.ptr, st);
      std::vector<unsigned long long> seen(words), coll(words);
      unsigned long long cnt = 0;
      CUDA_CHECK(cudaMemcpyAsync(seen.data(), d_seen.ptr, words * 8, cudaMemcpyDeviceToHost, st));
      CUDA_CHECK(cudaMemcpyAsync(coll.data(), d_coll.ptr, words * 8, cudaMemcpyDeviceToHost, st));
      CUDA_CHECK(cudaMemcpyAsync(&cnt, d_count.ptr, 8, cudaMemcpyDeviceToHost, st));
      CUDA_CHECK(cudaStreamSynchronize(st));
      for (size_t w = 0; w < words; ++w) bits.push_back(seen[w] & ~coll[w]);
      left_keys = d_left[level].ptr;
      n_left = (int64_t)cnt;
    }
    // blocks { w0, w1, w2, prefix }: prefix = number of set bits before the block, over both levels
    const size_t n_blocks = (size_t)nb[0] + nb[1];
    std::vector<unsigned long long> blocks(n_blocks * 4);
    unsigned long long prefix = 0;
    for (size_t b = 0; b < n_blocks; ++b) {
      blocks[4 * b + 3] = prefix;
      for (int k = 0; k < 3; ++k) {
        blocks[4 * b + k] = bits[3 * b + k];
        prefix += (unsigned long long)__builtin_popcountll(bits[3 * b + k]);
      }
    }
    if ((int64_t)prefix + n_left != n) throw std::runtime_error("k_rows: perfect hash lost states");
    ctx->d_mph_blocks.alloc(blocks.size() * 8);
    CUDA_CHECK(cudaMemcpyAsync(ctx->d_mph_blocks.ptr, blocks.data(), blocks.size() * 8, cudaMemcpyHostToDevice, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    ctx->mph.blocks = ctx->d_mph_blocks.ptr;
    ctx->mph.n_blocks0 = nb[0];
    ctx->mph.n_blocks1 = nb[1];
    ctx->mph.n_dense = (uint32_t)prefix;
    const size_t dense_bytes = (size_t)std::max<unsigned long long>(1, prefix) * (ce ? 32 : 16);
    ctx->d_dense.alloc(dense_bytes);
    CUDA_CHECK(cudaMemsetAsync(ctx->d_dense.ptr, 0xff, dense_bytes, st));
  }
  // ---- open-addressing table over the states that are left (all of them without the dense index)
  // complex128: one-slot buckets, 8 per state (1.07 probes per look-up) while the table stays below a quarter of the
  // free memory, else 4 or 2 per state; float64: two-slot buckets, 2 per state
  size_t free_b = 0, total_b = 0;
  CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  int64_t per_state = ce ? 8 : 2;
  while (per_state > 2 && (double)per_state * n_left * 32.0 > 0.25 * (double)free_b) per_state /= 2;
  if (ce && ctx->opt_table_per_state > 0) per_state = ctx->opt_table_per_state;
  if (per_state * n_left + 16 >= 2147483647ll) throw std::runtime_error("k_rows: table of more than 2^31 buckets");
  const uint32_t slots = (uint32_t)std::max<int64_t>(16, per_state * n_left);
  ctx->d_table.alloc((size_t)slots * 32);
  ctx->d_slot_of.alloc((size_t)std::max<int64_t>(1, n));
  CUDA_CHECK(cudaMemsetAsync(ctx->d_table.ptr, 0xff, (size_t)slots * 32, st));
  if (ctx->dense_index) {
    DevBuf<uint32_t> d_tmp;
    d_tmp.alloc((size_t)std::max<int64_t>(1, n_left));
    launch_table_insert(left_keys, n_left, ctx->d_table.ptr, slots, ce ? 1 : 2, d_tmp.ptr, st);
    launch_mph_slots(ctx->d_reps.ptr, n, ctx->mph, ctx->d_table.ptr, slots, ce ? 1 : 2, ctx->d_slot_of.ptr,
                     ctx->d_status.ptr, st);
    CUDA_CHECK(cudaStreamSynchronize(st));
  } else {
    launch_table_insert(ctx->d_reps.ptr, n, ctx->d_table.ptr, slots, ce ? 1 : 2, ctx->d_slot_of.ptr, st);
  }
  ctx->table_slots = slots;
  ctx->table_elt = elt;
}

// y[rows] <- rows of H through k_rows.  `basis` owns the table (this rank's context, or the twin holding the whole
// basis in the replicated-x product), x_all is indexed like basis' states (through pos when given), p names the rows.
void rows_product(dmv_context *basis, KernelParams &p, int elt, const void *x_all, const uint32_t *pos,
                  cudaStream_t stream, bool fill, dmv_context *timer) {
  if (!timer) timer = basis;   // whose event timeline the refill belongs to (the rank's context in the replicated form)
  cudaStream_t keep = basis->stream;
  basis->stream = stream;
  ensure_table(basis, elt);
  basis->stream = keep;
  if (fill) {   // (a product cut into row chunks refreshes the values once, with its first chunk)
    CUDA_CHECK(cudaEventRecord(timer->ev_fill[0], stream));
    launch_table_fill(basis->n_states, elt == DMV_C128, x_all, basis->d_norms.ptr, pos, basis->d_slot_of.ptr,
                      basis->d_reps.ptr, basis->d_table.ptr, basis->dense_index ? basis->d_dense.ptr : nullptr, stream);
    CUDA_CHECK(cudaEventRecord(timer->ev_fill[1], stream));
    timer->fill_timed = true;
  }
  select_tables(basis, p, true, false);
  p.uni_re = basis->gather_uni[0]; p.uni_im = basis->gather_uni[1];
  p.table = basis->d_table.ptr;
  p.table_slots = basis->table_slots;
  p.mph = basis->mph;
  p.dense = basis->dense_index ? basis->d_dense.ptr : nullptr;
  p.row_split = 1;
  const int launched = launch_rows(p, elt == DMV_C128, stream);
  if (launched) basis->rows_kernel = timer->rows_kernel = launched;
}

// the same for `nv` vectors at once (single rank; x / y: nv device vectors `stride` elements apart): k_rows_batch
void rows_product_batch(dmv_context *ctx, int elt, int nv, const void *x, void *y, int64_t stride) {
  const int64_t n = ctx->n_states;
  cudaStream_t st = ctx->stream;
  if (ctx->table_batch_slots == 0) {
    // one-slot buckets, 8 per state (1.07 probes per look-up; at 2 per state linear probing needs 1.5, and every extra
    // probe is a trip of the lane without a new term: measured 46.7 ms instead of the single product's 22.4 on the 6x6
    // square) while the table stays below a quarter of the free memory, else 4 or 2 per state
    size_t free_b = 0, total_b = 0;
    CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    int64_t per_state = 8;
    while (per_state > 2 && (double)per_state * n * 64.0 > 0.25 * (double)free_b) per_state /= 2;
    if (ctx->opt_table_per_state > 0) per_state = ctx->opt_table_per_state;
    if (per_state * n + 16 >= 2147483647ll) throw std::runtime_error("k_rows_batch: table of more than 2^31 buckets");
    const uint32_t buckets = (uint32_t)std::max<int64_t>(16, per_state * n);
    ctx->d_table_batch.alloc((size_t)buckets * 64);
    ctx->d_slot_of_batch.alloc((size_t)std::max<int64_t>(1, n));
    CUDA_CHECK(cudaMemsetAsync(ctx->d_table_batch.ptr, 0xff, (size_t)buckets * 64, st));
    launch_table_insert(ctx->d_reps.ptr, n, ctx->d_table_batch.ptr, buckets, 1, ctx->d_slot_of_batch.ptr, st, 64);
    ctx->table_batch_slots = buckets;
  }
  launch_table_fill_batch(n, nv, elt, x, stride, ctx->d_norms.ptr, ctx->d_slot_of_batch.ptr, ctx->d_reps.ptr,
                          ctx->d_table_batch.ptr, st);
  KernelParams p = base_params(ctx);
  p.x = x;
  p.y = y;
  select_tables(ctx, p, true, false);
  p.uni_re = ctx->gather_uni[0]; p.uni_im = ctx->gather_uni[1];
  p.table = ctx->d_table_batch.ptr;
  p.table_slots = ctx->table_batch_slots;
  p.batch = nv;
  p.batch_elt = elt;
  p.batch_stride = stride;
  p.row_split = 1;
  const int launched = launch_rows_batch(p, st);
  if (launched) ctx->rows_batch_kernel = launched;
}

void do_generate(dmv_context *ctx, int elt, const void *x_dev, void *y_dev,
                 const void *x_host_pending, int64_t row_begin, int64_t row_end) {
  if (use_pull(ctx)) {   // one rank owns the basis: traverse by rows (gather), see k_gather / k_pull
    KernelParams p = base_params(ctx);
    p.x = x_dev;
    p.y = y_dev;
    if (row_end > row_begin) { p.row_begin = row_begin; p.row_end = row_end; }
    if (use_gather(ctx)) {
      select_tables(ctx, p, true, ctx->complex_coefficients);
      p.row_split = choose_row_split(ctx->n_states, (int)ctx->h_pull.groups.size());
      p.uni_re = ctx->gather_uni[0]; p.uni_im = ctx->gather_uni[1];
      launch_gather(p, ctx->proj == PROJ_INVERSION, ctx->complex_coefficients, elt == DMV_C128,
                    ctx->gather_narrow, ctx->index_mode == INDEX_LIN, ctx->gather_uniform, ctx->stream);
      return;
    }
    if (use_rows(ctx)) {
      rows_product(ctx, p, elt, x_dev, nullptr, ctx->stream, /*fill=*/row_begin == 0);
      return;
    }
    select_tables(ctx, p, true, complex_values(ctx, elt));
    launch_pull(p, ctx->proj, complex_values(ctx, elt), elt == DMV_C128, ctx->stream);
    return;
  }
  if (!ctx->planned) do_plan(ctx);
  zero_y_if_diag(ctx, elt, y_dev);
  if (ctx->num_ranks > 1)
    CUDA_CHECK(cudaMemsetAsync(ctx->d_out_count.ptr, 0, sizeof(unsigned long long) * ctx->num_ranks, ctx->stream));
  KernelParams p = base_params(ctx);
  p.x = x_dev;
  p.y = y_dev;
  const bool cv = complex_values(ctx, elt);
  if (ctx->num_ranks > 1 && ctx->peer_direct && ctx->ptr_width != (cv ? 2 : 1)) {
    // peer-direct: destination d's records are stored straight into d's incoming buffer over NVLink
    const int width = cv ? 2 : 1;
    for (int d = 0; d < ctx->num_ranks; ++d) {
      if (d == ctx->rank) { ctx->h_out_betas_ptr[d] = nullptr; ctx->h_out_coeffs_ptr[d] = nullptr; continue; }
      ctx->h_out_betas_ptr[d] = reinterpret_cast<uint64_t *>(ctx->peer_betas[d]) + ctx->my_offset_in_peer[d];
      ctx->h_out_coeffs_ptr[d] = reinterpret_cast<double *>(ctx->peer_coeffs[d]) + ctx->my_offset_in_peer[d] * width;
    }
    upload_out_pointers(ctx);
    p.out_betas_ptr = ctx->d_out_betas_ptr.ptr;
    p.out_coeffs_ptr = ctx->d_out_coeffs_ptr.ptr;
    ctx->ptr_width = width;
  }
  if (ctx->num_ranks > 1 && !ctx->peer_direct && ctx->ptr_width != (cv ? 2 : 1)) {
    // local buckets: destination d's records start at out_offset[d] (coefficients: width doubles each)
    const int width = cv ? 2 : 1;
    for (int d = 0; d < ctx->num_ranks; ++d) {
      ctx->h_out_betas_ptr[d] = ctx->d_out_betas.ptr + ctx->h_out_offset[d];
      ctx->h_out_coeffs_ptr[d] = ctx->d_out_coeffs.ptr + ctx->h_out_offset[d] * width;
    }
    upload_out_pointers(ctx);
    p.out_betas_ptr = ctx->d_out_betas_ptr.ptr;
    p.out_coeffs_ptr = ctx->d_out_coeffs_ptr.ptr;
    ctx->ptr_width = width;
  }
  ctx->record_width = cv ? 2 : 1;
  select_tables(ctx, p, false, cv);
  if (!x_host_pending) {
    launch_generate(p, ctx->proj, cv, elt == DMV_C128, false, ctx->stream);
    return;
  }
  // pipelined: chunk k of x is copied while chunk k-1 is being generated
  const int chunks = dmv_context::kCopyChunks;
  const int64_t n = ctx->n_states, per = ((n + chunks - 1) / chunks + 31) / 32 * 32;
  const size_t esz = (size_t)8 * elt;
  CUDA_CHECK(cudaEventRecord(ctx->ev_chunk[0], ctx->stream));       // copy stream starts after prior work
  CUDA_CHECK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_chunk[0], 0));
  for (int k = 0; k < chunks; ++k) {
    const int64_t b = std::min<int64_t>(n, (int64_t)k * per), e = std::min<int64_t>(n, b + per);
    if (e <= b) break;
    CUDA_CHECK(cudaMemcpyAsync(reinterpret_cast<char *>(ctx->d_x.ptr) + b * esz,
                               reinterpret_cast<const char *>(x_host_pending) + b * esz, (size_t)(e - b) * esz,
                               cudaMemcpyHostToDevice, ctx->copy_stream));
    CUDA_CHECK(cudaEventRecord(ctx->ev_chunk[k], ctx->copy_stream));
    CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, ctx->ev_chunk[k], 0));
    p.row_begin = b;
    p.row_end = e;
    launch_generate(p, ctx->proj, cv, elt == DMV_C128, false, ctx->stream);
  }
}

void do_accumulate(dmv_context *ctx, int elt, int64_t count, const uint64_t *betas, const double *coeffs,
                   void *y_dev) {
  KernelParams p = base_params(ctx);
  p.y = y_dev;
  launch_accumulate(p, ctx->proj, complex_values(ctx, elt), elt == DMV_C128, count, betas, coeffs, ctx->stream);
}

void collect_timings(dmv_context *ctx) {
  auto ms = [&](int a, int b) { float t = 0; cudaEventElapsedTime(&t, ctx->ev[a], ctx->ev[b]); return (double)t; };
  ctx->timings[T_H2D] = ms(0, 1);
  if (ctx->timeline_replicated) {   // the exchange (all-gather of x) comes first, then the row gather
    ctx->timings[T_EXCHANGE] = ms(1, 6);
    ctx->timings[T_GENERATE] = ms(6, 2);
    ctx->timings[T_ACCUMULATE] = 0.0;
  } else {
  ctx->timings[T_GENERATE] = ms(1, 2);
  ctx->timings[T_EXCHANGE] = ms(2, 3);
  ctx->timings[T_ACCUMULATE] = ms(3, 4);
  }
  ctx->timings[T_D2H] = ms(4, 5);
  ctx->timings[T_TOTAL] = ms(0, 5);
  if (ctx->fill_timed) {   // (kept until the next refill: dmv_last_timings may collect twice)
    float t = 0;
    if (cudaEventElapsedTime(&t, ctx->ev_fill[0], ctx->ev_fill[1]) == cudaSuccess) ctx->timings[T_TABLE_FILL] = t;
    ctx->fill_timed = false;
  }
}

} }  // namespace dmv::host

extern "C" {


const char *dmv_last_error(void) { return g_last_error.c_str(); }
int dmv_version(void) { return 100; }
int64_t dmv_launch_count(void) { return launch_counter(); }

int dmv_context_create(const dmv_basis_desc *basis, const dmv_operator_desc *op, int device, int rank,
                       int num_ranks, dmv_context **out) {
  API_BEGIN
  if (!basis || !op || !out) throw std::runtime_error("null argument");
  if (basis->number_sites <= 0 || basis->number_sites > 64)
    throw std::runtime_error("bases with more than 64 bits are not yet implemented");  // DMV:1099-1100
  if (num_ranks < 1 || num_ranks > 256 || rank < 0 || rank >= num_ranks)
    throw std::runtime_error("need 0 <= rank < num_ranks <= 256");                     // DMV:664: uint8 keys
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0) {
    cudaGetLastError();
    throw std::runtime_error("no CUDA device: libdmv_b200 has no CPU fallback");
  }
  if (device < 0 || device >= n_dev) throw std::runtime_error("bad device ordinal");
  std::unique_ptr<dmv_context> ctx(new dmv_context());
  ctx->device = device; ctx->rank = rank; ctx->num_ranks = num_ranks;
  use_device(ctx.get());
  CUDA_CHECK(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
  ctx->stream = ctx->own_stream;
  CUDA_CHECK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  for (auto &e : ctx->ev) CUDA_CHECK(cudaEventCreate(&e));
  for (auto &e : ctx->ev_fill) CUDA_CHECK(cudaEventCreate(&e));
  for (auto &e : ctx->ev_chunk) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  ctx->n_sites = basis->number_sites;
  ctx->hamming_weight = basis->hamming_weight;
  ctx->spin_inversion = basis->spin_inversion;
  ctx->has_permutations = basis->has_permutations != 0;
  ctx->site_mask = basis->number_sites == 64 ? ~0ull : ((1ull << basis->number_sites) - 1);
  if (ctx->has_permutations) ctx->proj = PROJ_GROUP;                   // BO:163
  else if (ctx->spin_inversion != 0) ctx->proj = PROJ_INVERSION;       // BO:119
  else ctx->proj = PROJ_NONE;                                          // BO:89
  ctx->identity_index = (ctx->proj == PROJ_NONE && ctx->hamming_weight < 0);

  ctx->k_off_v.assign(op->off_v, op->off_v + 2 * op->n_off);
  ctx->k_off_m.assign(op->off_m, op->off_m + op->n_off); ctx->k_off_r.assign(op->off_r, op->off_r + op->n_off);
  ctx->k_off_x.assign(op->off_x, op->off_x + op->n_off); ctx->k_off_s.assign(op->off_s, op->off_s + op->n_off);
  ctx->k_diag_v.assign(op->diag_v, op->diag_v + 2 * op->n_diag);
  ctx->k_diag_m.assign(op->diag_m, op->diag_m + op->n_diag); ctx->k_diag_r.assign(op->diag_r, op->diag_r + op->n_diag);
  ctx->k_diag_s.assign(op->diag_s, op->diag_s + op->n_diag);
  if (basis->has_permutations && basis->group_order > 0 && basis->perms && basis->flips && basis->characters) {
    ctx->k_group_order = basis->group_order;
    ctx->k_perms.assign(basis->perms, basis->perms + basis->group_order * basis->number_sites);
    ctx->k_flips.assign(basis->flips, basis->flips + basis->group_order);
    ctx->k_chars.assign(basis->characters, basis->characters + 2 * basis->group_order);
  }
  bool cplx = false;
  // ---- operator: group off-diagonal terms by flip mask
  std::map<uint64_t, std::vector<OffTerm>> by_x;
  for (int64_t t = 0; t < op->n_off; ++t) {
    OffTerm o{op->off_m[t], op->off_r[t], op->off_s[t], op->off_v[2 * t], op->off_v[2 * t + 1]};
    if (op->off_x[t] == 0) throw std::runtime_error("off-diagonal term with zero flip mask");
    if (o.v_im != 0.0) cplx = true;
    by_x[op->off_x[t]].push_back(o);
  }
  std::map<uint64_t, std::vector<OffTerm>> by_x_rows;
  for (auto &kv : by_x)
    for (auto &o : kv.second) {
      // row traversal: <b|t|b^x> = v (-1)^popc(x&s) [b & m == r ^ (x & m)] (-1)^popc(b & s)
      const uint64_t x = kv.first;
      const double sg = (__builtin_popcountll(x & o.s) & 1) ? -1.0 : 1.0;
      by_x_rows[x].push_back(OffTerm{o.m, o.r ^ (x & o.m), o.s, sg * o.v_re, sg * o.v_im});
    }
  ctx->h_push = build_tables(by_x);
  ctx->h_pull = build_tables(by_x_rows);
  for (int64_t t = 0; t < op->n_diag; ++t) {
    DiagTerm d{op->diag_m[t], op->diag_r[t], op->diag_s[t], op->diag_v[2 * t], op->diag_v[2 * t + 1]};
    if (d.v_im != 0.0) cplx = true;
    ctx->h_diag.push_back(d);
  }
  {
    // k_gather needs the bit-parallel emit test on the row tables and coefficients that depend on the support
    // bits only; it runs in 32-bit registers when sites and groups fit, and skips the LUT when every emitting
    // (group, support bits) pair carries the same coefficient (every Heisenberg-type operator)
    const HostTables &H = ctx->h_pull;
    ctx->gather_ok = !H.bp.empty() && !H.any_s_out && !H.any_generic;
    ctx->gather_narrow = basis->number_sites <= 32 && H.groups.size() <= 32;
    bool first = true, uniform = ctx->gather_ok;
    for (size_t g = 0; g < H.groups.size() && uniform; ++g)
      for (int idx = 0; idx < 4; ++idx)
        if ((H.groups[g].emit_bits >> idx) & 1ull) {
          const double re = H.lut_c[2 * (4 * g + idx)], im = H.lut_c[2 * (4 * g + idx) + 1];
          if (first) { ctx->gather_uni[0] = re; ctx->gather_uni[1] = im; first = false; }
          else if (re != ctx->gather_uni[0] || im != ctx->gather_uni[1]) { uniform = false; break; }
        }
    ctx->gather_uniform = uniform && !first;
  }
  build_diag_classes(ctx.get());
  ctx->d_diag_classes.upload(ctx->h_diag_classes, ctx->stream);
  ctx->d_push.upload(ctx->h_push, ctx->stream);
  ctx->d_pull.upload(ctx->h_pull, ctx->stream);
  ctx->d_diag.upload(ctx->h_diag, ctx->stream);

  // ---- symmetry group
  if (ctx->proj == PROJ_GROUP) {
    if (basis->group_order <= 0 || !basis->perms || !basis->flips || !basis->characters)
      throw std::runtime_error("basis with permutation symmetries needs the group tables");
    ctx->host_orbit = compile_orbit_program(basis->number_sites, basis->group_order, basis->perms,
                                            basis->flips, basis->characters);
    for (double v : ctx->host_orbit.characters) (void)v;
    for (size_t e = 0; e < ctx->host_orbit.characters.size(); e += 2)
      if (ctx->host_orbit.characters[e + 1] != 0.0) cplx = true;
    upload_orbit(ctx.get());
  }
  ctx->complex_coefficients = cplx;
  ctx->rows_ok = ctx->proj == PROJ_GROUP && !cplx && ctx->host_orbit.trivial_characters &&
                 !ctx->h_pull.bp.empty() && !ctx->h_pull.any_generic;
  ctx->d_status.alloc(4);
  CUDA_CHECK(cudaMemsetAsync(ctx->d_status.ptr, 0, 4 * sizeof(unsigned long long), ctx->stream));
  ctx->d_out_count.alloc(num_ranks);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  *out = ctx.release();
  API_END
}

int dmv_context_destroy(dmv_context *ctx) {
  API_BEGIN
  if (ctx) {
    {
      std::lock_guard<std::mutex> lock(g_bind_mutex);
      for (auto it = g_bindings.begin(); it != g_bindings.end();)
        it = (it->second == ctx) ? g_bindings.erase(it) : std::next(it);
    }
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    delete ctx;
  }
  API_END
}

int dmv_set_stream(dmv_context *ctx, void *cuda_stream, int use_own_stream) {
  API_BEGIN
  use_device(ctx);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  // a NULL handle is the legacy default stream, which is what torch's default stream is
  ctx->stream = use_own_stream ? ctx->own_stream : reinterpret_cast<cudaStream_t>(cuda_stream);
  API_END
}

int dmv_set_option(dmv_context *ctx, const char *name, int64_t value) {
  API_BEGIN
  use_device(ctx);
  const std::string key(name ? name : "");
  if (key == "mode") {
    if (value < -1 || value > 1) throw std::runtime_error("mode: -1 auto, 0 push, 1 pull");
    ctx->opt_mode = (int)value;
  } else if (key == "index") {
    if (value != -1 && value != 0 && value != 2 && value != 3)
      throw std::runtime_error("index: -1 auto, 0 directory, 2 combinadic rank, 3 Lin tables");
    ctx->opt_index = (int)value;
    if (ctx->n_states >= 0) { CUDA_CHECK(cudaStreamSynchronize(ctx->stream)); select_index_mode(ctx); }
  } else if (key == "exchange") {
    if (value < -1 || value > 2)
      throw std::runtime_error("exchange: -1 auto, 0 NCCL send/recv, 1 peer-direct records, 2 replicated x (all-gather)");
    ctx->opt_exchange = (int)value;
    ctx->planned = false;
    ctx->exchange_decided = false;
    ctx->replicated = false;
    ctx->rounds.tried = false;
    ctx->rounds.ready = false;
  } else if (key == "gather") {
    if (value < -1 || value > 0) throw std::runtime_error("gather: -1 auto, 0 off (queued k_pull for mode = 1)");
    ctx->opt_gather = (int)value;
  } else if (key == "rows_batch_min") {
    if (value < 1 || value > 6) throw std::runtime_error("rows_batch_min: 1 .. 6 doubles per state");
    ctx->opt_rows_batch_min = (int)value;
  } else if (key == "rows_table_per_state") {
    if (value != 0 && value != 2 && value != 4 && value != 8)
      throw std::runtime_error("rows_table_per_state: 0 auto, or 2 / 4 / 8 buckets per state");
    ctx->opt_table_per_state = (int)value;
    ctx->table_elt = 0;
    ctx->table_batch_slots = 0;
    if (ctx->global) { ctx->global->opt_table_per_state = (int)value; ctx->global->table_elt = 0; }
  } else if (key == "rows_batch") {
    if (value < -1 || value > 1) throw std::runtime_error("rows_batch: -1 auto / 1 k_rows_batch for batched products, 0 vector by vector");
    ctx->opt_rows_batch = (int)value;
  } else if (key == "rows_ctas") {
    ctx->opt_rows_ctas = (value == 2 || value == 4) ? (int)value : 3;
    if (ctx->global) ctx->global->opt_rows_ctas = ctx->opt_rows_ctas;
  } else if (key == "rows_index") {
    if (value < -1 || value > 1) throw std::runtime_error("rows_index: -1 auto / 0 open-addressing table, 1 dense index (perfect hash)");
    ctx->opt_rows_index = (int)value;
    ctx->table_elt = 0;
    if (ctx->global) { ctx->global->opt_rows_index = (int)value; ctx->global->table_elt = 0; }
  } else if (key == "rounds") {
    if (value < -1 || value > 64) throw std::runtime_error("rounds: -1 auto, 0 / 1 one-shot exchange, R <= 64 overlapped rounds");
    ctx->opt_rounds = (int)value;
    ctx->rounds.tried = false;
    ctx->rounds.ready = false;
  } else if (key == "gather_walk") {
    ctx->opt_gather_walk = (value >= 0 && value <= 2) ? (int)value : 0;
    if (ctx->global) ctx->global->opt_gather_walk = ctx->opt_gather_walk;
  } else if (key == "peer_gather") {
    if (value < -1 || value > 0) throw std::runtime_error("peer_gather: -1 auto, 0 NCCL all-gather of x");
    ctx->opt_peer_gather = (int)value;
    ctx->exchange_decided = false;
  } else if (key == "rows") {
    if (value < -1 || value > 0) throw std::runtime_error("rows: -1 auto, 0 off (queued k_pull / k_generate for symmetric bases)");
    ctx->opt_rows = (int)value;
    if (ctx->global) ctx->global->opt_rows = (int)value;
  } else if (key == "canon") {
    ctx->opt_canon = (value >= 0 && value <= 2) ? (int)value : -1;
    if (ctx->proj == PROJ_GROUP) { CUDA_CHECK(cudaStreamSynchronize(ctx->stream)); upload_orbit(ctx); }
  } else if (key == "bitparallel") {
    ctx->opt_bitparallel = value != 0;
    ctx->planned = false;
  } else {
    throw std::runtime_error("unknown option '" + key + "'");
  }
  API_END
}

int64_t dmv_get_info(const dmv_context *ctx, const char *name) {
  const std::string key(name ? name : "");
  if (!ctx) return -1;
  if (key == "index_mode") return ctx->index_mode;
  if (key == "pull") return use_pull(ctx) ? 1 : 0;
  if (key == "gather")
    return ((use_pull(ctx) && use_gather(ctx)) || (ctx->replicated && ctx->global && use_gather(ctx->global))) ? 1 : 0;
  if (key == "gather_narrow") return ctx->gather_narrow ? 1 : 0;
  if (key == "gather_uniform") return ctx->gather_uniform ? 1 : 0;
  if (key == "peer_direct") return ctx->peer_direct ? 1 : 0;
  if (key == "replicated") return ctx->replicated ? 1 : 0;
  if (key == "replicated_block") return ctx->repl_block;
  if (key == "global_states") return ctx->global ? ctx->global->n_states : -1;
  if (key == "projection") return (int64_t)ctx->proj;
  if (key == "n_groups") return (int64_t)ctx->h_push.groups.size();
  if (key == "bp_words") return (int64_t)ctx->h_push.bp.size();
  if (key == "bp_pairs") { int64_t n = 0; for (auto &w : ctx->h_push.bp) n += w.n0 + w.n1; return n; }
  if (key == "canon_mode") return ctx->orbit.canon_mode;
  if (key == "torus_mode") return ctx->orbit.tor_mode;
  if (key == "rows")
    return ((use_pull(ctx) && !use_gather(ctx) && use_rows(ctx)) ||
            (ctx->replicated && ctx->global && !use_gather(ctx->global) && use_rows(ctx->global))) ? 1 : 0;
  if (key == "rows_ok") return ctx->rows_ok ? 1 : 0;
  if (key == "rows_kernel") return ctx->rows_kernel;
  if (key == "rows_batch_kernel") return ctx->rows_batch_kernel;
  if (key == "rows_table_buckets") return (int64_t)ctx->table_slots;
  if (key == "rows_batch_buckets") return (int64_t)ctx->table_batch_slots;
  if (key == "rows_dense") return ctx->dense_index ? (int64_t)ctx->mph.n_dense : (ctx->global && ctx->global->dense_index ? (int64_t)ctx->global->mph.n_dense : 0);
  if (key == "rounds") return ctx->rounds.ready ? ctx->rounds.R : 0;
  if (key == "peer_gather") return (ctx->replicated && ctx->peer_gather) ? 1 : 0;
  if (key == "complex_coefficients") return ctx->complex_coefficients ? 1 : 0;
  if (key == "canon_k") return ctx->host_orbit.canon_k;
  if (key == "orbit_n_q") return ctx->host_orbit.n_q;
  if (key == "orbit_n_t") return ctx->host_orbit.n_t;
  if (key == "orbit_n_stages") return ctx->host_orbit.n_stages;
  if (key == "group_order") return ctx->host_orbit.group_order;
  if (key == "n_buckets") return (int64_t)ctx->n_buckets;
  return -1;
}

int dmv_synchronize(dmv_context *ctx) {
  API_BEGIN
  use_device(ctx);
  check_status(ctx);   // synchronises the stream and surfaces device-side errors (DMV:115-118)
  API_END
}

int dmv_set_representatives(dmv_context *ctx, const uint64_t *representatives, int64_t count,
                            const double *norms) {
  API_BEGIN
  use_device(ctx);
  if (count < 0 || (count > 0 && !representatives)) throw std::runtime_error("bad representatives");
  if (count >= (1ll << 32)) throw std::runtime_error("more than 2^32 states per rank are not supported");
  ctx->d_reps.alloc((size_t)count);
  if (count > 0)
    CUDA_CHECK(cudaMemcpyAsync(ctx->d_reps.ptr, representatives, (size_t)count * 8, cudaMemcpyDefault, ctx->stream));
  ctx->n_states = count;
  if (ctx->proj == PROJ_GROUP) {
    ctx->d_norms.alloc((size_t)count);
    if (norms) {
      if (count > 0)
        CUDA_CHECK(cudaMemcpyAsync(ctx->d_norms.ptr, norms, (size_t)count * 8, cudaMemcpyDefault, ctx->stream));
    } else {
      launch_compute_norms(ctx->orbit, count, ctx->d_reps.ptr, ctx->d_norms.ptr, ctx->stream);
    }
  }
  install_directory(ctx);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_basis_build(dmv_context *ctx) {
  API_BEGIN
  use_device(ctx);
  const int n = ctx->n_sites, w = ctx->hamming_weight;
  const bool fixed = w >= 0;
  // candidate range (mirror of ls_hs_min/max_state_estimate, reference src/ForeignTypes.chpl:102-109);
  // with spin inversion the top site is never set in a representative (SURVEY.md App. A.2)
  uint64_t lo, hi;
  const bool inv = ctx->spin_inversion != 0;
  if (fixed) {
    if (w > n) throw std::runtime_error("hamming weight exceeds the number of sites");
    lo = w == 0 ? 0 : ((w == 64) ? ~0ull : ((1ull << w) - 1));
    const int top = (inv && n - 1 >= w) ? n - 1 : n;
    hi = w == 0 ? 0 : (((w == 64) ? ~0ull : ((1ull << w) - 1)) << (top - w));
  } else {
    lo = 0;
    hi = inv ? (ctx->site_mask >> 1) : ctx->site_mask;
  }
  const uint64_t first_rank = fixed ? fixed_hamming_rank(lo) : lo;
  const uint64_t last_rank = fixed ? fixed_hamming_rank(hi) : hi;
  const uint64_t total = last_rank - first_rank + 1;
  uint64_t chunk_len = total / (148ull * 128 * 16);
  chunk_len = std::min<uint64_t>(std::max<uint64_t>(chunk_len, 64), 4096);
  const int64_t n_chunks = (int64_t)((total + chunk_len - 1) / chunk_len);
  std::vector<uint64_t> h_first((size_t)n_chunks), h_last((size_t)n_chunks);
  for (int64_t c = 0; c < n_chunks; ++c) {
    const uint64_t r0 = first_rank + (uint64_t)c * chunk_len;
    const uint64_t r1 = std::min(r0 + chunk_len - 1, last_rank);
    h_first[c] = fixed ? fixed_hamming_unrank(r0, w) : r0;
    h_last[c] = fixed ? fixed_hamming_unrank(r1, w) : r1;
  }
  DevBuf<uint64_t> d_first, d_last;
  DevBuf<unsigned long long> d_count, d_offset;
  d_first.upload(h_first, ctx->stream);
  d_last.upload(h_last, ctx->stream);
  d_count.alloc((size_t)n_chunks);
  d_offset.alloc((size_t)n_chunks);
  launch_enumerate(ctx->orbit, ctx->proj, ctx->site_mask, fixed, ctx->rank, ctx->num_ranks, n_chunks,
                   d_first.ptr, d_last.ptr, d_count.ptr, d_offset.ptr, nullptr, nullptr, false, ctx->stream);
  std::vector<unsigned long long> h_count((size_t)n_chunks), h_offset((size_t)n_chunks);
  CUDA_CHECK(cudaMemcpyAsync(h_count.data(), d_count.ptr, sizeof(unsigned long long) * n_chunks,
                             cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  unsigned long long acc = 0;
  for (int64_t c = 0; c < n_chunks; ++c) { h_offset[c] = acc; acc += h_count[c]; }
  if (acc >= (1ull << 32)) throw std::runtime_error("more than 2^32 states per rank are not supported");
  d_offset.upload(h_offset, ctx->stream);
  ctx->d_reps.alloc((size_t)acc);
  if (ctx->proj == PROJ_GROUP) ctx->d_norms.alloc((size_t)acc);
  launch_enumerate(ctx->orbit, ctx->proj, ctx->site_mask, fixed, ctx->rank, ctx->num_ranks, n_chunks,
                   d_first.ptr, d_last.ptr, d_count.ptr, d_offset.ptr, ctx->d_reps.ptr,
                   ctx->proj == PROJ_GROUP ? ctx->d_norms.ptr : nullptr, true, ctx->stream);
  ctx->n_states = (int64_t)acc;
  install_directory(ctx);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int64_t dmv_number_states(const dmv_context *ctx) { return ctx ? ctx->n_states : -1; }

int dmv_get_representatives(dmv_context *ctx, uint64_t *representatives, double *norms) {
  API_BEGIN
  use_device(ctx);
  require_states(ctx);
  if (representatives && ctx->n_states > 0)
    CUDA_CHECK(cudaMemcpyAsync(representatives, ctx->d_reps.ptr, (size_t)ctx->n_states * 8, cudaMemcpyDefault, ctx->stream));
  if (norms && ctx->n_states > 0) {
    if (ctx->proj == PROJ_GROUP)
      CUDA_CHECK(cudaMemcpyAsync(norms, ctx->d_norms.ptr, (size_t)ctx->n_states * 8, cudaMemcpyDefault, ctx->stream));
    else {
      std::vector<double> ones((size_t)ctx->n_states, ctx->proj == PROJ_INVERSION ? std::sqrt(0.5) : 1.0);
      CUDA_CHECK(cudaMemcpyAsync(norms, ones.data(), ones.size() * 8, cudaMemcpyDefault, ctx->stream));
      CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    }
  }
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_state_index(dmv_context *ctx, int64_t count, const uint64_t *spins, int64_t *indices) {
  API_BEGIN
  use_device(ctx);
  require_states(ctx);
  InArg<uint64_t> in(spins, (size_t)count, ctx->stream);
  OutArg<int64_t> out(indices, (size_t)count);
  KernelParams p = base_params(ctx);
  launch_state_index(p.index, count, in.ptr, out.ptr, ctx->stream);
  out.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_state_info(dmv_context *ctx, int64_t count, const uint64_t *alphas, uint64_t *betas,
                   double *characters, double *norms) {
  API_BEGIN
  use_device(ctx);
  InArg<uint64_t> in(alphas, (size_t)count, ctx->stream);
  OutArg<uint64_t> ob(betas, (size_t)count);
  OutArg<double> oc(characters, (size_t)count * 2);
  OutArg<double> on(norms, (size_t)count);
  launch_state_info(ctx->orbit, ctx->proj, ctx->site_mask, (double)ctx->spin_inversion, count, in.ptr,
                    ob.ptr, oc.ptr, on.ptr, ctx->stream);
  ob.finish(ctx->stream); oc.finish(ctx->stream); on.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_locale_idx_of(dmv_context *ctx, int64_t count, const uint64_t *states, int num_locales, uint8_t *keys) {
  API_BEGIN
  use_device(ctx);
  InArg<uint64_t> in(states, (size_t)count, ctx->stream);
  OutArg<uint8_t> out(keys, (size_t)count);
  launch_locale_idx(count, in.ptr, num_locales, out.ptr, ctx->stream);
  out.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int64_t dmv_max_number_off_diag(const dmv_context *ctx) { return ctx ? (int64_t)ctx->h_push.groups.size() : -1; }

int dmv_plan(dmv_context *ctx, int64_t *send_counts) {
  API_BEGIN
  use_device(ctx);
  do_plan(ctx);
  if (send_counts) std::copy(ctx->send_counts.begin(), ctx->send_counts.end(), send_counts);
  API_END
}

int64_t dmv_number_terms(const dmv_context *ctx) { return ctx ? ctx->number_terms : -1; }

int dmv_generate(dmv_context *ctx, int elt, const void *x, void *y) {
  API_BEGIN
  use_device(ctx);
  require_states(ctx);
  if (elt != DMV_F64 && elt != DMV_C128) throw std::runtime_error("elt must be DMV_F64 or DMV_C128");
  if (!is_device_vector(x, ctx->n_states) || !is_device_vector(y, ctx->n_states))
    throw std::runtime_error("dmv_generate needs device pointers (y is accumulated into by later steps)");
  do_generate(ctx, elt, x, y);
  check_status(ctx);
  API_END
}

int dmv_outgoing(dmv_context *ctx, int dest, const uint64_t **betas, const double **coeffs, int64_t *count) {
  API_BEGIN
  if (!ctx->planned) throw std::runtime_error("no plan");
  if (dest < 0 || dest >= ctx->num_ranks) throw std::runtime_error("bad destination");
  const int64_t off = ctx->h_out_offset[dest];
  if (betas) *betas = ctx->d_out_betas.ptr + off;
  if (coeffs) *coeffs = ctx->d_out_coeffs.ptr + off * ctx->record_width;
  if (count) *count = ctx->h_out_offset[dest + 1] - off;
  API_END
}

int dmv_accumulate(dmv_context *ctx, int elt, int64_t count, const uint64_t *betas, const double *coeffs, void *y) {
  API_BEGIN
  use_device(ctx);
  require_states(ctx);
  if (!is_device_vector(y, ctx->n_states)) throw std::runtime_error("dmv_accumulate needs a device y");
  const int width = complex_values(ctx, elt) ? 2 : 1;
  InArg<uint64_t> b(betas, (size_t)count, ctx->stream);
  InArg<double> c(coeffs, (size_t)count * width, ctx->stream);
  do_accumulate(ctx, elt, count, b.ptr, c.ptr, y);
  check_status(ctx);
  API_END
}

int dmv_local_matvec(dmv_context *ctx, int elt, const void *x, void *y) {
  API_BEGIN
  use_device(ctx);
  require_states(ctx);
  if (ctx->num_ranks != 1) throw std::runtime_error("dmv_local_matvec needs num_ranks == 1; use dmv_matvec");
  if (elt != DMV_F64 && elt != DMV_C128) throw std::runtime_error("elt must be DMV_F64 or DMV_C128");
  if (x == y) throw std::runtime_error("x and y must not alias");
  VecStage v = stage_vectors(ctx, elt, x, y);
  const bool host_result = v.y_host;
  if (use_pull(ctx) && (use_gather(ctx) || use_rows(ctx)) && v.y_host && ctx->n_states >= (1 << 16)) {
    // row traversal into a host y: every row chunk is final as soon as its launch ends, so its D2H copy
    // (copy stream) overlaps the gather of the next chunk
    const int chunks = dmv_context::kCopyChunks;
    const int64_t n = ctx->n_states, per = ((n + chunks - 1) / chunks + 31) / 32 * 32;
    const size_t esz = (size_t)8 * elt;
    for (int k = 0; k < chunks; ++k) {
      const int64_t b = std::min<int64_t>(n, (int64_t)k * per), e = std::min<int64_t>(n, b + per);
      if (e <= b) break;
      do_generate(ctx, elt, v.x_dev, v.y_dev, nullptr, b, e);
      CUDA_CHECK(cudaEventRecord(ctx->ev_chunk[k], ctx->stream));
      CUDA_CHECK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_chunk[k], 0));
      CUDA_CHECK(cudaMemcpyAsync(reinterpret_cast<char *>(v.y_user) + b * esz,
                                 reinterpret_cast<const char *>(v.y_dev) + b * esz, (size_t)(e - b) * esz,
                                 cudaMemcpyDeviceToHost, ctx->copy_stream));
    }
    CUDA_CHECK(cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_CHECK(cudaEventRecord(ctx->ev[3], ctx->stream));
    CUDA_CHECK(cudaEventRecord(ctx->ev[4], ctx->stream));
    CUDA_CHECK(cudaEventRecord(ctx->ev_chunk[0], ctx->copy_stream));
    CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, ctx->ev_chunk[0], 0));
    CUDA_CHECK(cudaEventRecord(ctx->ev[5], ctx->stream));
  } else {
  do_generate(ctx, elt, v.x_dev, v.y_dev, v.x_host_pending);
  CUDA_CHECK(cudaEventRecord(ctx->ev[2], ctx->stream));
  CUDA_CHECK(cudaEventRecord(ctx->ev[3], ctx->stream));
  finish_vectors(ctx, v);
  }
  if (host_result || !is_device_pointer(x)) {
    // host callers get a finished result (and the error check) on return
    check_status(ctx);
    collect_timings(ctx);
  }
  API_END
}

// ---- several vectors per call (the reference's numVectors > 1, "not yet implemented" there: DMV:1101-1102, and what
// PRIMME's blockSize > 1 would use, src/Diagonalize.chpl:154-158).  x, y: num_vectors arrays of dmv_number_states
// elements, one after the other (the [numVectors, N] layout of the reference's BlockVector).  On one rank with device
// pointers and an operator k_gather applies to, four vectors share one walk over the terms and one index look-up per
// term; every other case is the loop over single products.
int dmv_matvec_batch(dmv_context *ctx, int elt, int num_vectors, const void *x, void *y) {
  API_BEGIN
  use_device(ctx);
  require_states(ctx);
  if (elt != DMV_F64 && elt != DMV_C128) throw std::runtime_error("elt must be DMV_F64 or DMV_C128");
  if (num_vectors < 1) throw std::runtime_error("num_vectors must be positive");
  if (x == y) throw std::runtime_error("x and y must not alias");
  const size_t vec_bytes = (size_t)ctx->n_states * 8 * elt;
  const char *xb = reinterpret_cast<const char *>(x);
  char *yb = reinterpret_cast<char *>(y);
  int k = 0;
  if (ctx->num_ranks == 1 && use_pull(ctx) && use_gather(ctx) && is_device_pointer(x) && is_device_pointer(y)) {
    for (; k + 4 <= num_vectors; k += 4) {
      KernelParams p = base_params(ctx);
      p.x = xb + (size_t)k * vec_bytes;
      p.y = yb + (size_t)k * vec_bytes;
      p.batch = 4;
      p.batch_stride = ctx->n_states;
      select_tables(ctx, p, true, ctx->complex_coefficients);
      p.row_split = choose_row_split(ctx->n_states, (int)ctx->h_pull.groups.size());
      p.uni_re = ctx->gather_uni[0]; p.uni_im = ctx->gather_uni[1];
      launch_gather(p, ctx->proj == PROJ_INVERSION, ctx->complex_coefficients, elt == DMV_C128, ctx->gather_narrow,
                    ctx->index_mode == INDEX_LIN, ctx->gather_uniform, ctx->stream);
    }
  }
  if (ctx->num_ranks == 1 && use_pull(ctx) && !use_gather(ctx) && use_rows(ctx) && ctx->opt_rows_batch != 0 &&
      is_device_pointer(x) == is_device_pointer(y)) {
    // bases with permutation symmetries: up to six doubles per state share one orbit minimum and one look-up per term
    // (host vectors -- what PRIMME hands over -- are staged a batch at a time)
    const int per = 6 / elt;
    const bool on_host = !is_device_pointer(x);
    // (a batch costs 1.5 - 1.6 single products on the 6x6 square -- 64-byte buckets, one request per lane in flight:
    // profiles/r02_rows_batch_6x6.md -- so it pays from two vectors on)
    // (rows_batch_min = 1 sends a single vector through k_rows_batch as well)
    while ((num_vectors - k) * elt >= ctx->opt_rows_batch_min && num_vectors - k >= std::min(2, ctx->opt_rows_batch_min)) {
      const int nv = std::min(per, num_vectors - k);
      const void *xk = xb + (size_t)k * vec_bytes;
      void *yk = yb + (size_t)k * vec_bytes;
      if (on_host) {
        ctx->d_x.alloc((size_t)ctx->n_states * elt * nv);
        ctx->d_y.alloc((size_t)ctx->n_states * elt * nv);
        CUDA_CHECK(cudaMemcpyAsync(ctx->d_x.ptr, xk, vec_bytes * nv, cudaMemcpyHostToDevice, ctx->stream));
        if (ctx->h_diag_kept == 0)   // no diagonal: the product accumulates into y (DMV:1062-1069)
          CUDA_CHECK(cudaMemcpyAsync(ctx->d_y.ptr, yk, vec_bytes * nv, cudaMemcpyHostToDevice, ctx->stream));
        rows_product_batch(ctx, elt, nv, ctx->d_x.ptr, ctx->d_y.ptr, ctx->n_states);
        CUDA_CHECK(cudaMemcpyAsync(yk, ctx->d_y.ptr, vec_bytes * nv, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        check_status(ctx);
      } else {
        rows_product_batch(ctx, elt, nv, xk, yk, ctx->n_states);
      }
      k += nv;
    }
  }
  for (; k < num_vectors; ++k) {
    const int rc = ctx->num_ranks == 1 ? dmv_local_matvec(ctx, elt, xb + (size_t)k * vec_bytes, yb + (size_t)k * vec_bytes)
                                       : dmv_matvec(ctx, elt, xb + (size_t)k * vec_bytes, yb + (size_t)k * vec_bytes);
    if (rc) throw std::runtime_error(g_last_error);
  }
  API_END
}

int dmv_last_timings(dmv_context *ctx, double *ms, int capacity) {
  if (!ctx) return 0;
  cudaSetDevice(ctx->device);
  if (cudaStreamSynchronize(ctx->stream) == cudaSuccess) {
    try { collect_timings(ctx); } catch (...) {}
  }
  for (int i = 0; i < T_COUNT && i < capacity; ++i) ms[i] = ctx->timings[i];
  return T_COUNT;
}
const char *dmv_timing_name(int i) { return (i >= 0 && i < T_COUNT) ? kTimingNames[i] : ""; }

int dmv_compute_off_diag(dmv_context *ctx, int64_t count, const uint64_t *alphas, const void *xs, int elt,
                         int64_t *n, uint64_t *betas, double *coeffs, uint8_t *keys) {
  API_BEGIN
  // BatchedOperator.computeOffDiag (reference src/BatchedOperator.chpl:82-213) through the same kernel
  // as the product: the given alphas play the role of the source block and every record is written to
  // one flat output (emit_all) together with its locale key.
  use_device(ctx);
  if (elt != DMV_F64 && elt != DMV_C128) throw std::runtime_error("elt must be DMV_F64 or DMV_C128");
  const size_t cap = (size_t)count * std::max<size_t>(1, ctx->h_push.groups.size());
  InArg<uint64_t> a(alphas, (size_t)count, ctx->stream);
  InArg<double> x(reinterpret_cast<const double *>(xs), (size_t)count * elt, ctx->stream);
  OutArg<uint64_t> ob(betas, cap);
  OutArg<double> oc(coeffs, cap * 2);
  OutArg<uint8_t> ok(keys, cap);
  DevBuf<double> d_src_norms;
  DevBuf<int64_t> d_off;
  DevBuf<unsigned long long> d_cnt;
  std::vector<int64_t> off = {0, (int64_t)cap};
  d_off.upload(off, ctx->stream);
  d_cnt.alloc(1);
  CUDA_CHECK(cudaMemsetAsync(d_cnt.ptr, 0, sizeof(unsigned long long), ctx->stream));
  KernelParams p = base_params(ctx);
  p.index.reps = a.ptr; p.index.n = count; p.index.mode = INDEX_DIRECTORY;
  if (ctx->proj == PROJ_GROUP) {  // norms of the sources: BO:178-194 appends the alphas to state_info
    d_src_norms.alloc((size_t)count);
    launch_compute_norms(ctx->orbit, count, a.ptr, d_src_norms.ptr, ctx->stream);
    p.norms = d_src_norms.ptr;
  }
  p.x = x.ptr; p.y = nullptr;
  p.emit_all = 1;
  p.out_betas = ob.ptr; p.out_coeffs = oc.ptr; p.out_keys = ok.ptr;
  p.out_offset = d_off.ptr; p.out_count = d_cnt.ptr;
  p.row_begin = 0; p.row_end = count;
  select_tables(ctx, p, false, true);
  launch_generate(p, ctx->proj, /*complex values*/ true, elt == DMV_C128, false, ctx->stream);
  unsigned long long total = 0;
  CUDA_CHECK(cudaMemcpyAsync(&total, d_cnt.ptr, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (total > cap) throw std::runtime_error("dmv_compute_off_diag: output overflow");
  ob.finish(ctx->stream, (size_t)total); oc.finish(ctx->stream, (size_t)total * 2); ok.finish(ctx->stream, (size_t)total);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (n) *n = (int64_t)total;
  API_END
}

// ---- plugin kernels: ls_chpl_operator_apply_diag / _apply_off_diag (reference src/BatchedOperator.chpl:217-275)
int dmv_apply_diag(dmv_context *ctx, int64_t count, const uint64_t *alphas, double *coeffs) {
  API_BEGIN
  use_device(ctx);
  if (ctx->proj != PROJ_NONE) throw std::runtime_error("bases that require projection are not yet supported");  // BO:226-227
  if (count < 0) throw std::runtime_error("negative count");
  InArg<uint64_t> a(alphas, (size_t)count, ctx->stream);
  OutArg<double> out(coeffs, (size_t)count);
  KernelParams p = base_params(ctx);
  select_tables(ctx, p, false, true);
  launch_apply_diag(p, count, a.ptr, out.ptr, ctx->stream);
  out.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_apply_off_diag(dmv_context *ctx, int64_t count, const uint64_t *alphas, uint64_t *betas, double *coeffs,
                       int64_t *offsets) {
  API_BEGIN
  use_device(ctx);
  if (ctx->proj != PROJ_NONE) throw std::runtime_error("bases that require projection are not yet supported");  // BO:247-248
  if (count < 0) throw std::runtime_error("negative count");
  const size_t cap = (size_t)count * std::max<size_t>(1, ctx->h_push.groups.size());
  InArg<uint64_t> a(alphas, (size_t)count, ctx->stream);
  OutArg<uint64_t> ob(betas, cap);
  OutArg<double> oc(coeffs, cap * 2);
  OutArg<int64_t> oo(offsets, (size_t)count + 1);
  DevBuf<int64_t> d_counts;
  d_counts.alloc((size_t)count + 1);
  KernelParams p = base_params(ctx);
  select_tables(ctx, p, false, true);
  launch_apply_off_diag(p, count, a.ptr, nullptr, d_counts.ptr, nullptr, nullptr, false, ctx->stream);
  std::vector<int64_t> h((size_t)count + 1, 0);
  if (count > 0)
    CUDA_CHECK(cudaMemcpyAsync(h.data(), d_counts.ptr, (size_t)count * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  int64_t acc = 0;
  for (int64_t i = 0; i < count; ++i) { const int64_t c = h[i]; h[i] = acc; acc += c; }   // CSR row pointer (BO:109)
  h[count] = acc;
  CUDA_CHECK(cudaMemcpyAsync(oo.ptr, h.data(), ((size_t)count + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  launch_apply_off_diag(p, count, a.ptr, oo.ptr, nullptr, ob.ptr, oc.ptr, true, ctx->stream);
  ob.finish(ctx->stream, (size_t)acc); oc.finish(ctx->stream, (size_t)acc * 2); oo.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_debug_compile_group(const dmv_basis_desc *basis, int64_t *info, int64_t count,
                            const uint64_t *states, uint64_t *reps, int32_t *stab) {
  API_BEGIN
  HostOrbitProgram H = compile_orbit_program(basis->number_sites, basis->group_order, basis->perms,
                                             basis->flips, basis->characters);
  if (info) {
    info[0] = H.n_q; info[1] = H.n_stages; info[2] = H.n_t; info[3] = H.n_left; info[4] = H.n_right;
    info[5] = H.has_flip;
    if (count < 0) {   // extended query (count = -1): info must hold 12 entries
      info[6] = H.canon_mode; info[7] = H.canon_k; info[8] = H.canon_r;
      info[9] = H.canon_lut2.empty() ? 0 : 1;
      info[10] = H.cc_begin.empty() ? 0 : (int64_t)H.cc_begin.size() - 1;
      info[11] = (int64_t)H.cc_mask.size();
    }
    if (count < -1) {  // count = -2: info holds 16 entries
      info[12] = H.tor_mode; info[13] = H.tor_rho_n; info[14] = H.tor_tau_n; info[15] = H.chain_dihedral;
    }
  }
  OrbitProgram P = H.view();
  for (int64_t k = 0; k < count; ++k) {
    const OrbitResult r = orbit_scan<true, false>(P, states[k]);
    if (P.canon_mode && orbit_min_canon(P, states[k]) != r.rep)
      throw std::runtime_error("canonical form disagrees with the chain walk");
    if (P.tor_mode == 2 && P.canon_k == P.canon_r && (P.canon_k == 4 || P.canon_k == 6)) {
      const uint64_t got = P.canon_k == 6 ? orbit_min_torus_sq<6>(P, states[k]) : orbit_min_torus_sq<4>(P, states[k]);
      if (got != r.rep) throw std::runtime_error("square-torus canonical form disagrees with the chain walk");
    }
    if (P.tor_mode || P.chain_dihedral) {
      OrbitProgram P1 = P;
      P1.tor_mode = 0;
      P1.chain_dihedral = 0;
      if (orbit_min_canon(P1, states[k]) != r.rep)
        throw std::runtime_error("block-rotation canonical form disagrees with the chain walk");
    }
    if (reps) reps[k] = r.rep;
    if (stab) stab[k] = r.stab;
  }
  API_END
}

}  // extern "C"
