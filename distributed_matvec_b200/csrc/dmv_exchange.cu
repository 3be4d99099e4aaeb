// dmv_exchange.cu -- the collective product dmv_matvec (matrixVectorProduct, reference src/DistributedMatrixVector.chpl:1072-1093)
// and its three exchanges: replicated x with the peer-direct all-gather, peer-direct records in overlapped rounds, NCCL buckets;
// the block <-> hashed redistribution of vectors.
#include "dmv_context.h"

namespace dmv { namespace host {




// One-time exchange of the plan: every rank learns how many records each peer sends it; then, when
// possible, the peers' incoming buffers are mapped (CUDA IPC over NVLink) so that k_generate can store
// remote records directly where the owner will read them.
void setup_exchange(dmv_context *ctx) {
  NcclApi &N = nccl();
  const int P = ctx->num_ranks;
  for (auto &q : ctx->peer_betas) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
  for (auto &q : ctx->peer_coeffs) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
  DevBuf<int64_t> d_send, d_all;
  d_send.upload(ctx->send_counts, ctx->stream);
  d_all.alloc((size_t)P * P);
  NCCL_CHECK(N.AllGather(d_send.ptr, d_all.ptr, (size_t)P, ncclInt64, ctx->comm, ctx->stream));
  std::vector<int64_t> all((size_t)P * P);   // all[r * P + q]: records r emits for q (own ones included)
  CUDA_CHECK(cudaMemcpyAsync(all.data(), d_all.ptr, all.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  int64_t total_in = 0;
  for (int q = 0; q < P; ++q) {
    ctx->recv_counts[q] = (q == ctx->rank) ? 0 : all[(size_t)q * P + ctx->rank];
    total_in += ctx->recv_counts[q];
  }
  ctx->d_in_betas.alloc((size_t)total_in);
  ctx->d_in_coeffs.alloc((size_t)total_in * 2);
  ctx->d_barrier.alloc(1);
  CUDA_CHECK(cudaMemsetAsync(ctx->d_barrier.ptr, 0, sizeof(int), ctx->stream));
  ctx->peer_direct = false;
  if (ctx->opt_exchange == 0 || P > 32) return;

  // ---- try to map the peers' incoming buffers
  struct Handles { cudaIpcMemHandle_t betas, coeffs; int ok; int pad[15]; };
  static_assert(sizeof(Handles) % 8 == 0, "handle block");
  Handles mine{};
  mine.ok = (cudaIpcGetMemHandle(&mine.betas, ctx->d_in_betas.ptr) == cudaSuccess &&
             cudaIpcGetMemHandle(&mine.coeffs, ctx->d_in_coeffs.ptr) == cudaSuccess) ? 1 : 0;
  cudaGetLastError();
  DevBuf<char> d_mine, d_handles;
  d_mine.alloc(sizeof(Handles));
  d_handles.alloc(sizeof(Handles) * P);
  CUDA_CHECK(cudaMemcpyAsync(d_mine.ptr, &mine, sizeof(Handles), cudaMemcpyHostToDevice, ctx->stream));
  NCCL_CHECK(N.AllGather(d_mine.ptr, d_handles.ptr, sizeof(Handles), ncclChar, ctx->comm, ctx->stream));
  std::vector<Handles> handles(P);
  CUDA_CHECK(cudaMemcpyAsync(handles.data(), d_handles.ptr, sizeof(Handles) * P, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  int ok = 1;
  for (int q = 0; q < P; ++q) ok &= handles[q].ok;
  ctx->peer_betas.assign(P, nullptr);
  ctx->peer_coeffs.assign(P, nullptr);
  if (ok) {
    for (int q = 0; q < P && ok; ++q) {
      if (q == ctx->rank) continue;
      if (cudaIpcOpenMemHandle(&ctx->peer_betas[q], handles[q].betas, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
          cudaIpcOpenMemHandle(&ctx->peer_coeffs[q], handles[q].coeffs, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        ok = 0;
        cudaGetLastError();
      }
    }
  }
  // everybody must agree
  int agree = ok;
  CUDA_CHECK(cudaMemcpyAsync(ctx->d_barrier.ptr, &agree, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  NCCL_CHECK(N.AllReduce(ctx->d_barrier.ptr, ctx->d_barrier.ptr, 1, ncclInt32, ncclMin, ctx->comm, ctx->stream));
  CUDA_CHECK(cudaMemcpyAsync(&agree, ctx->d_barrier.ptr, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (!agree) {
    for (auto &q : ctx->peer_betas) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
    for (auto &q : ctx->peer_coeffs) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
    if (ctx->opt_exchange == 1) throw std::runtime_error("peer-direct exchange requested but CUDA IPC mapping failed");
    return;
  }
  // my region inside peer q's incoming buffer: after the regions of the ranks before me (q itself sends nothing)
  ctx->my_offset_in_peer.assign(P, 0);
  for (int q = 0; q < P; ++q) {
    int64_t off = 0;
    for (int r = 0; r < ctx->rank; ++r)
      if (r != q) off += all[(size_t)r * P + q];
    ctx->my_offset_in_peer[q] = off;
  }
  ctx->peer_direct = true;
  ctx->ptr_width = 0;
}

// -------------------------------------------------------------------------------------------------
// Replicated-x product.  With 180 GB of HBM per GPU every basis of BASELINE.json fits on ONE device many times
// over, so for operators k_gather applies to, the ranks can trade the reference's record exchange (24 bytes per
// off-diagonal term over NVLink, DMV:313-436) for one all-gather of x (E bytes per STATE): every rank keeps the
// whole sorted basis (a single-rank twin context), gathers x from all ranks into slots of equal size, and computes
// ITS rows by the atomics-free row traversal.  The hash partition of x, y and the representatives -- the layout the
// callers see (SE:129-156) -- is unchanged.  Local part of the set-up; no communication here.
void setup_replicated(dmv_context *ctx) {
  require_states(ctx);
  const int P = ctx->num_ranks;
  if (P > 32) throw std::runtime_error("replicated-x product supports at most 32 ranks");
  if (!ctx->global) {
    dmv_basis_desc b{};
    b.number_sites = ctx->n_sites; b.hamming_weight = ctx->hamming_weight; b.spin_inversion = ctx->spin_inversion;
    if (ctx->proj == PROJ_GROUP) {
      b.has_permutations = 1; b.group_order = ctx->k_group_order;
      b.perms = ctx->k_perms.data(); b.flips = ctx->k_flips.data(); b.characters = ctx->k_chars.data();
    }
    dmv_operator_desc o{};
    o.n_off = (int64_t)ctx->k_off_m.size(); o.off_v = ctx->k_off_v.data();
    o.off_m = ctx->k_off_m.data(); o.off_r = ctx->k_off_r.data(); o.off_x = ctx->k_off_x.data(); o.off_s = ctx->k_off_s.data();
    o.n_diag = (int64_t)ctx->k_diag_m.size(); o.diag_v = ctx->k_diag_v.data();
    o.diag_m = ctx->k_diag_m.data(); o.diag_r = ctx->k_diag_r.data(); o.diag_s = ctx->k_diag_s.data();
    // rough size check before enumerating: reps + directory + positions + gathered x
    double states = 1.0;
    if (ctx->hamming_weight >= 0) states = (double)binom().c[ctx->n_sites][ctx->hamming_weight];
    else states = std::ldexp(1.0, ctx->n_sites);
    if (ctx->spin_inversion != 0 && ctx->proj != PROJ_GROUP) states *= 0.5;
    if (ctx->proj == PROJ_GROUP) states = 1.5 * states / (double)std::max<int64_t>(1, ctx->k_group_order) + 1e4;
    size_t free_b = 0, total_b = 0;
    CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    if (states * 48.0 > 0.5 * (double)free_b) throw std::runtime_error("replicated-x product: the whole basis does not fit");
    dmv_context *g = nullptr;
    if (dmv_context_create(&b, &o, ctx->device, 0, 1, &g) != 0) throw std::runtime_error(g_last_error);
    ctx->global = g;
    g->opt_rows = ctx->opt_rows;
    g->opt_gather_walk = ctx->opt_gather_walk;
    g->opt_rows_index = ctx->opt_rows_index;
    g->opt_rows_ctas = ctx->opt_rows_ctas;
    g->opt_table_per_state = ctx->opt_table_per_state;
    if (ctx->opt_canon != g->opt_canon && g->proj == PROJ_GROUP) { g->opt_canon = ctx->opt_canon; upload_orbit(g); }
    if (dmv_basis_build(g) != 0) throw std::runtime_error(g_last_error);
  }
  dmv_context *g = ctx->global;
  CUDA_CHECK(cudaStreamSynchronize(g->stream));
  const int64_t n = g->n_states;
  // ---- slot of every global state: owner r = hash % P (SE:129-136), index inside r's ascending block
  const int64_t chunk = 256, n_chunks = (n + chunk - 1) / chunk;
  DevBuf<unsigned long long> d_counts, d_base;
  d_counts.alloc((size_t)n_chunks * P);
  d_base.alloc((size_t)n_chunks * P);
  ctx->d_pos.alloc((size_t)n);
  launch_owner_positions(g->d_reps.ptr, nullptr, n, P, chunk, false, d_counts.ptr, nullptr, 0, nullptr, ctx->stream);
  std::vector<unsigned long long> counts((size_t)n_chunks * P), base((size_t)n_chunks * P);
  CUDA_CHECK(cudaMemcpyAsync(counts.data(), d_counts.ptr, counts.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  std::vector<unsigned long long> total(P, 0);
  for (int64_t c = 0; c < n_chunks; ++c)
    for (int r = 0; r < P; ++r) { base[(size_t)c * P + r] = total[r]; total[r] += counts[(size_t)c * P + r]; }
  if ((int64_t)total[ctx->rank] != ctx->n_states)
    throw std::runtime_error("replicated-x product: this rank's block is not the hash partition of the full basis");
  int64_t block = 0;
  for (int r = 0; r < P; ++r) block = std::max<int64_t>(block, (int64_t)total[r]);
  block = (block + 1) / 2 * 2;
  if ((double)block * P >= 4294967295.0) throw std::runtime_error("replicated-x product: more than 2^32 slots");
  d_base.upload(base, ctx->stream);
  launch_owner_positions(g->d_reps.ptr, nullptr, n, P, chunk, true, d_counts.ptr, d_base.ptr, block, ctx->d_pos.ptr, ctx->stream);
  ctx->repl_block = block;
  ctx->d_xcat.alloc((size_t)block * P * 2 * 2);   // two buffers of P slots (alternating products), 16 bytes per element
  CUDA_CHECK(cudaMemsetAsync(ctx->d_xcat.ptr, 0, (size_t)block * P * 2 * 2 * sizeof(double), ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

// y (this rank's block) <- rows of H applied to the gathered x (slot r * repl_block holds rank r's block)
void replicated_rows(dmv_context *ctx, int elt, const void *x_cat, void *y_dev) {
  dmv_context *g = ctx->global;
  KernelParams p = base_params(g);
  p.x = x_cat;
  p.y = y_dev;
  p.status = ctx->d_status.ptr;
  p.row_states = ctx->d_reps.ptr;
  p.row_begin = 0;
  p.row_end = ctx->n_states;
  p.pos = ctx->d_pos.ptr;
  p.x_row_offset = (int64_t)ctx->rank * ctx->repl_block;
  if (use_gather(g)) {
    select_tables(g, p, true, g->complex_coefficients);
    p.row_split = choose_row_split(ctx->n_states, (int)g->h_pull.groups.size());
    p.uni_re = g->gather_uni[0]; p.uni_im = g->gather_uni[1];
    launch_gather(p, g->proj == PROJ_INVERSION, g->complex_coefficients, elt == DMV_C128, g->gather_narrow,
                  g->index_mode == INDEX_LIN, g->gather_uniform, ctx->stream);
    return;
  }
  p.row_norms = ctx->d_norms.ptr;
  if (use_rows(g)) {   // bases with permutation symmetries: hash table over the whole basis, filled from the gathered x
    rows_product(g, p, elt, x_cat, ctx->d_pos.ptr, ctx->stream, true, ctx);
    return;
  }
  // operators outside the bit-parallel test / non-trivial characters: the queued row traversal
  if (p.index.mode == INDEX_RANK) p.index.mode = INDEX_DIRECTORY;   // the incremental rank needs row index == rank
  p.row_split = 1;
  select_tables(g, p, true, complex_values(g, elt));
  launch_pull(p, g->proj, complex_values(g, elt), elt == DMV_C128, ctx->stream);
}

// Collective set-up of the overlapped record exchange: per-round counting passes, exchange of the counts, incoming
// buffers laid out round-major, CUDA IPC mapping of buffers and flags.  Leaves rounds.ready false when it does not apply
// (one round, IPC impossible): the caller then uses the one-shot exchange.
void setup_rounds(dmv_context *ctx) {
  dmv_context::Rounds &Q = ctx->rounds;
  NcclApi &N = nccl();
  const int P = ctx->num_ranks;
  Q.tried = true;
  Q.ready = false;
  int R = ctx->opt_rounds;
  if (R < 0) R = ctx->n_states >= (1 << 18) ? 4 : 1;
  // every rank must use the same number of rounds
  ctx->d_barrier.alloc(1);
  CUDA_CHECK(cudaMemcpyAsync(ctx->d_barrier.ptr, &R, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  NCCL_CHECK(N.AllReduce(ctx->d_barrier.ptr, ctx->d_barrier.ptr, 1, ncclInt32, ncclMin, ctx->comm, ctx->stream));
  CUDA_CHECK(cudaMemcpyAsync(&R, ctx->d_barrier.ptr, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (R <= 1 || P > 32 || ctx->opt_exchange == 0) return;
  Q.R = R;
  Q.row_split = 1;
  Q.row_begin.assign(R + 1, 0);
  for (int r = 0; r <= R; ++r) Q.row_begin[r] = std::min<int64_t>(ctx->n_states, (ctx->n_states * r / R + 31) / 32 * 32);
  Q.row_begin[R] = ctx->n_states;
  Q.grid = planned_grid((ctx->n_states + R - 1) / R, 1);
  const size_t n_warps = (size_t)Q.grid * kWarpsPerCta;
  // ---- counting pass per round: exact share of every warp for every destination
  std::vector<int64_t> offsets((size_t)R * n_warps * P, 0), counts((size_t)R * P, 0);
  ctx->d_warp_counts.alloc(n_warps * P);
  ctx->d_out_count.alloc(P);
  std::vector<unsigned long long> wc(n_warps * P);
  Q.terms = 0;
  for (int r = 0; r < R; ++r) {
    CUDA_CHECK(cudaMemsetAsync(ctx->d_warp_counts.ptr, 0, sizeof(unsigned long long) * n_warps * P, ctx->stream));
    KernelParams p = base_params(ctx);
    p.grid_blocks = Q.grid;
    p.row_split = 1;
    p.row_begin = Q.row_begin[r];
    p.row_end = Q.row_begin[r + 1];
    p.warp_counts = ctx->d_warp_counts.ptr;
    select_tables(ctx, p, false, ctx->complex_coefficients);
    launch_generate(p, ctx->proj, ctx->complex_coefficients, false, /*count_only=*/true, ctx->stream);
    CUDA_CHECK(cudaMemcpyAsync(wc.data(), ctx->d_warp_counts.ptr, sizeof(unsigned long long) * wc.size(),
                               cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    for (int d = 0; d < P; ++d)
      for (size_t w = 0; w < n_warps; ++w) {
        offsets[((size_t)r * n_warps + w) * P + d] = counts[(size_t)r * P + d];
        counts[(size_t)r * P + d] += (int64_t)wc[w * P + d];
      }
    for (int d = 0; d < P; ++d) Q.terms += counts[(size_t)r * P + d];
  }
  Q.d_warp_offsets.upload(offsets, ctx->stream);
  if (!ctx->planned) ctx->number_terms = Q.terms;
  std::vector<int64_t> capacity((size_t)R * P);
  for (int r = 0; r < R; ++r)
    for (int d = 0; d < P; ++d) capacity[(size_t)r * P + d] = d == ctx->rank ? 0 : counts[(size_t)r * P + d];
  Q.d_capacity.upload(capacity, ctx->stream);
  // ---- everybody's counts: all[s][r][d]
  DevBuf<int64_t> d_send, d_all;
  d_send.upload(counts, ctx->stream);
  d_all.alloc((size_t)P * R * P);
  NCCL_CHECK(N.AllGather(d_send.ptr, d_all.ptr, (size_t)R * P, ncclInt64, ctx->comm, ctx->stream));
  std::vector<int64_t> all((size_t)P * R * P);
  CUDA_CHECK(cudaMemcpyAsync(all.data(), d_all.ptr, all.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  auto cnt = [&](int s, int r, int d) { return all[((size_t)s * R + r) * P + d]; };
  // incoming buffer of rank q, round-major: [round 0: sources 0 .. P-1 (without q)] [round 1: ...] ...
  auto region = [&](int q, int r, int src) {   // first record of (round r, source src) inside q's buffer
    int64_t off = 0;
    for (int rr = 0; rr < r; ++rr)
      for (int s = 0; s < P; ++s) if (s != q) off += cnt(s, rr, q);
    for (int s = 0; s < src; ++s) if (s != q) off += cnt(s, r, q);
    return off;
  };
  Q.in_slice.assign(R + 1, 0);
  for (int r = 0; r <= R; ++r) Q.in_slice[r] = region(ctx->rank, r, 0);
  Q.in_total = Q.in_slice[R];
  Q.peer_total.assign(P, 0);
  for (int q = 0; q < P; ++q) Q.peer_total[q] = region(q, R, 0);
  Q.my_off.assign((size_t)R * P, 0);
  for (int r = 0; r < R; ++r)
    for (int q = 0; q < P; ++q) if (q != ctx->rank) Q.my_off[(size_t)r * P + q] = region(q, r, ctx->rank);
  Q.d_in_betas.alloc((size_t)std::max<int64_t>(1, 2 * Q.in_total));
  Q.d_in_coeffs.alloc((size_t)std::max<int64_t>(1, 4 * Q.in_total));
  Q.d_flags.alloc(P);
  CUDA_CHECK(cudaMemsetAsync(Q.d_flags.ptr, 0, sizeof(unsigned) * P, ctx->stream));
  Q.seq = 0;
  // ---- map the peers' buffers and flags
  for (auto *v : {&Q.peer_betas, &Q.peer_coeffs, &Q.peer_flags})
    for (auto &q : *v) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
  struct Handles { cudaIpcMemHandle_t betas, coeffs, flags; int ok; int pad[15]; };
  static_assert(sizeof(Handles) % 8 == 0, "handle block");
  Handles mine{};
  mine.ok = (cudaIpcGetMemHandle(&mine.betas, Q.d_in_betas.ptr) == cudaSuccess &&
             cudaIpcGetMemHandle(&mine.coeffs, Q.d_in_coeffs.ptr) == cudaSuccess &&
             cudaIpcGetMemHandle(&mine.flags, Q.d_flags.ptr) == cudaSuccess) ? 1 : 0;
  cudaGetLastError();
  DevBuf<char> d_mine, d_handles;
  d_mine.alloc(sizeof(Handles));
  d_handles.alloc(sizeof(Handles) * P);
  CUDA_CHECK(cudaMemcpyAsync(d_mine.ptr, &mine, sizeof(Handles), cudaMemcpyHostToDevice, ctx->stream));
  NCCL_CHECK(N.AllGather(d_mine.ptr, d_handles.ptr, sizeof(Handles), ncclChar, ctx->comm, ctx->stream));
  std::vector<Handles> handles(P);
  CUDA_CHECK(cudaMemcpyAsync(handles.data(), d_handles.ptr, sizeof(Handles) * P, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  int ok = 1;
  for (int q = 0; q < P; ++q) ok &= handles[q].ok;
  Q.peer_betas.assign(P, nullptr); Q.peer_coeffs.assign(P, nullptr); Q.peer_flags.assign(P, nullptr);
  for (int q = 0; q < P && ok; ++q) {
    if (q == ctx->rank) continue;
    if (cudaIpcOpenMemHandle(&Q.peer_betas[q], handles[q].betas, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
        cudaIpcOpenMemHandle(&Q.peer_coeffs[q], handles[q].coeffs, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
        cudaIpcOpenMemHandle(&Q.peer_flags[q], handles[q].flags, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      ok = 0;
      cudaGetLastError();
    }
  }
  int agree = ok;
  CUDA_CHECK(cudaMemcpyAsync(ctx->d_barrier.ptr, &agree, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  NCCL_CHECK(N.AllReduce(ctx->d_barrier.ptr, ctx->d_barrier.ptr, 1, ncclInt32, ncclMin, ctx->comm, ctx->stream));
  CUDA_CHECK(cudaMemcpyAsync(&agree, ctx->d_barrier.ptr, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (!agree) {
    for (auto *v : {&Q.peer_betas, &Q.peer_coeffs, &Q.peer_flags})
      for (auto &q : *v) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
    return;
  }
  std::vector<unsigned *> flags(P);
  for (int q = 0; q < P; ++q) flags[q] = q == ctx->rank ? Q.d_flags.ptr : reinterpret_cast<unsigned *>(Q.peer_flags[q]);
  Q.d_peer_flags.upload(flags, ctx->stream);
  if (!Q.acc_stream) CUDA_CHECK(cudaStreamCreateWithFlags(&Q.acc_stream, cudaStreamNonBlocking));
  if (!Q.ev_begin) CUDA_CHECK(cudaEventCreateWithFlags(&Q.ev_begin, cudaEventDisableTiming));
  if (!Q.ev_done) CUDA_CHECK(cudaEventCreateWithFlags(&Q.ev_done, cudaEventDisableTiming));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  Q.ptr_width = 0;
  Q.ready = true;
}

// where my records of (buffer, round, destination) go: [2][R][P] pointers into the peers' incoming buffers
void upload_round_pointers(dmv_context *ctx, int width) {
  dmv_context::Rounds &Q = ctx->rounds;
  const int P = ctx->num_ranks, R = Q.R;
  std::vector<uint64_t *> bp((size_t)2 * R * P, nullptr);
  std::vector<double *> cp((size_t)2 * R * P, nullptr);
  for (int b = 0; b < 2; ++b)
    for (int r = 0; r < R; ++r)
      for (int q = 0; q < P; ++q) {
        if (q == ctx->rank) continue;
        const int64_t first = (int64_t)b * Q.peer_total[q] + Q.my_off[(size_t)r * P + q];
        bp[((size_t)b * R + r) * P + q] = reinterpret_cast<uint64_t *>(Q.peer_betas[q]) + first;
        cp[((size_t)b * R + r) * P + q] = reinterpret_cast<double *>(Q.peer_coeffs[q]) + first * width;
      }
  Q.d_bptr.upload(bp, ctx->stream);
  Q.d_cptr.upload(cp, ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  Q.ptr_width = width;
}

// One product through the overlapped rounds (x, y device pointers).  Main stream: generate round 0, raise flags,
// generate round 1, ...; second stream: wait for every sender's flag of round r, accumulate its slice.  Returns with the
// main stream waiting for the last accumulate.
void rounds_product(dmv_context *ctx, int elt, const void *x_dev, void *y_dev) {
  dmv_context::Rounds &Q = ctx->rounds;
  const int P = ctx->num_ranks, R = Q.R;
  const bool cv = complex_values(ctx, elt);
  const int width = cv ? 2 : 1;
  if (Q.ptr_width != width) upload_round_pointers(ctx, width);
  ctx->record_width = width;
  zero_y_if_diag(ctx, elt, y_dev);
  CUDA_CHECK(cudaEventRecord(Q.ev_begin, ctx->stream));
  CUDA_CHECK(cudaStreamWaitEvent(Q.acc_stream, Q.ev_begin, 0));
  const int b = (int)(Q.seq & 1u);
  const size_t n_warps = (size_t)Q.grid * kWarpsPerCta;
  for (int r = 0; r < R; ++r) {
    KernelParams p = base_params(ctx);
    p.x = x_dev;
    p.y = y_dev;
    p.grid_blocks = Q.grid;
    p.row_split = 1;
    p.row_begin = Q.row_begin[r];
    p.row_end = Q.row_begin[r + 1];
    p.warp_offsets = Q.d_warp_offsets.ptr + (size_t)r * n_warps * P;
    p.out_capacity = Q.d_capacity.ptr + (size_t)r * P;
    p.out_betas_ptr = Q.d_bptr.ptr + ((size_t)b * R + r) * P;
    p.out_coeffs_ptr = Q.d_cptr.ptr + ((size_t)b * R + r) * P;
    select_tables(ctx, p, false, cv);
    launch_generate(p, ctx->proj, cv, elt == DMV_C128, false, ctx->stream);
    const unsigned value = Q.seq * (unsigned)R + (unsigned)r + 1u;
    launch_raise_flags(Q.d_peer_flags.ptr, P, ctx->rank, value, ctx->stream);
    // owner side, second stream: every sender has delivered round r -> search + accumulate its slice
    launch_wait_flags(Q.d_flags.ptr, P, value, ctx->d_status.ptr, Q.acc_stream);
    const int64_t first = (int64_t)b * Q.in_total + Q.in_slice[r], count = Q.in_slice[r + 1] - Q.in_slice[r];
    if (count > 0) {
      KernelParams pa = base_params(ctx);
      pa.y = y_dev;
      launch_accumulate(pa, ctx->proj, cv, elt == DMV_C128, count, Q.d_in_betas.ptr + first,
                        Q.d_in_coeffs.ptr + first * width, Q.acc_stream);
    }
  }
  ++Q.seq;
  CUDA_CHECK(cudaEventRecord(ctx->ev[2], ctx->stream));   // end of generation
  CUDA_CHECK(cudaEventRecord(ctx->ev[3], ctx->stream));
  CUDA_CHECK(cudaEventRecord(Q.ev_done, Q.acc_stream));
  CUDA_CHECK(cudaStreamWaitEvent(ctx->stream, Q.ev_done, 0));   // what is left of the accumulate is the exposed part
}

// Collective: map every rank's gathered-x buffers and flag words into every other rank (CUDA IPC over NVLink) so that
// the all-gather of x becomes one kernel of peer stores + flags (launch_push_block).  Falls back to the NCCL all-gather
// when any rank cannot map.
void setup_peer_gather(dmv_context *ctx) {
  NcclApi &N = nccl();
  const int P = ctx->num_ranks;
  ctx->peer_gather = false;
  ctx->d_flags.alloc(P);
  ctx->d_push_done.alloc(1);
  CUDA_CHECK(cudaMemsetAsync(ctx->d_flags.ptr, 0, sizeof(unsigned) * P, ctx->stream));
  CUDA_CHECK(cudaMemsetAsync(ctx->d_push_done.ptr, 0, sizeof(unsigned), ctx->stream));
  ctx->gather_epoch = 0;
  struct Handles { cudaIpcMemHandle_t xcat, flags; int ok; int pad[15]; };
  static_assert(sizeof(Handles) % 8 == 0, "handle block");
  Handles mine{};
  mine.ok = (ctx->opt_peer_gather != 0 && cudaIpcGetMemHandle(&mine.xcat, ctx->d_xcat.ptr) == cudaSuccess &&
             cudaIpcGetMemHandle(&mine.flags, ctx->d_flags.ptr) == cudaSuccess) ? 1 : 0;
  cudaGetLastError();
  DevBuf<char> d_mine, d_handles;
  d_mine.alloc(sizeof(Handles));
  d_handles.alloc(sizeof(Handles) * P);
  CUDA_CHECK(cudaMemcpyAsync(d_mine.ptr, &mine, sizeof(Handles), cudaMemcpyHostToDevice, ctx->stream));
  NCCL_CHECK(N.AllGather(d_mine.ptr, d_handles.ptr, sizeof(Handles), ncclChar, ctx->comm, ctx->stream));
  std::vector<Handles> handles(P);
  CUDA_CHECK(cudaMemcpyAsync(handles.data(), d_handles.ptr, sizeof(Handles) * P, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  int ok = 1;
  for (int q = 0; q < P; ++q) ok &= handles[q].ok;
  for (auto &q : ctx->peer_xcat) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
  for (auto &q : ctx->peer_flagmem) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
  ctx->peer_xcat.assign(P, nullptr);
  ctx->peer_flagmem.assign(P, nullptr);
  if (ok) {
    for (int q = 0; q < P && ok; ++q) {
      if (q == ctx->rank) continue;
      if (cudaIpcOpenMemHandle(&ctx->peer_xcat[q], handles[q].xcat, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
          cudaIpcOpenMemHandle(&ctx->peer_flagmem[q], handles[q].flags, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        ok = 0;
        cudaGetLastError();
      }
    }
  }
  int agree = ok;   // everybody must agree; the all-reduce is also the barrier after which flags may be raised
  ctx->d_barrier.alloc(1);
  CUDA_CHECK(cudaMemcpyAsync(ctx->d_barrier.ptr, &agree, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  NCCL_CHECK(N.AllReduce(ctx->d_barrier.ptr, ctx->d_barrier.ptr, 1, ncclInt32, ncclMin, ctx->comm, ctx->stream));
  CUDA_CHECK(cudaMemcpyAsync(&agree, ctx->d_barrier.ptr, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (!agree) {
    for (auto &q : ctx->peer_xcat) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
    for (auto &q : ctx->peer_flagmem) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
    return;
  }
  std::vector<unsigned *> flags(P);
  for (int q = 0; q < P; ++q)
    flags[q] = q == ctx->rank ? ctx->d_flags.ptr : reinterpret_cast<unsigned *>(ctx->peer_flagmem[q]);
  ctx->d_peer_flags.upload(flags, ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  ctx->peer_slot_elt = 0;
  ctx->peer_gather = true;
}

// slot `rank` of buffer b of every rank's gathered vector, for elements of `elt` doubles
void upload_peer_slots(dmv_context *ctx, int elt) {
  const int P = ctx->num_ranks;
  const size_t buffer_doubles = (size_t)ctx->repl_block * P * 2;   // buffers are sized for 16-byte elements
  for (int b = 0; b < 2; ++b) {
    std::vector<void *> slots(P);
    for (int q = 0; q < P; ++q) {
      double *base = q == ctx->rank ? ctx->d_xcat.ptr : reinterpret_cast<double *>(ctx->peer_xcat[q]);
      slots[q] = base + b * buffer_doubles + (size_t)ctx->rank * ctx->repl_block * elt;
    }
    ctx->d_peer_slot[b].upload(slots, ctx->stream);
  }
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  ctx->peer_slot_elt = elt;
}

// Collective: which exchange the distributed product uses.  exchange = -1 (auto) prefers the replicated-x product
// when k_gather applies and the whole basis fits, else the record exchange (peer-direct / NCCL, see setup_exchange).
void decide_exchange(dmv_context *ctx) {
  NcclApi &N = nccl();
  int ok = 0;
  std::string why;
  const bool want = (ctx->opt_exchange == 2 || ctx->opt_exchange == -1) && ctx->opt_mode != 0;
  if (want && ctx->num_ranks <= 32) {
    try { setup_replicated(ctx); ok = 1; } catch (const std::exception &e) { why = e.what(); ok = 0; }
  } else {
    why = "switched off (exchange / mode options) or more than 32 ranks";
  }
  ctx->d_barrier.alloc(1);
  CUDA_CHECK(cudaMemcpyAsync(ctx->d_barrier.ptr, &ok, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  NCCL_CHECK(N.AllReduce(ctx->d_barrier.ptr, ctx->d_barrier.ptr, 1, ncclInt32, ncclMin, ctx->comm, ctx->stream));
  int agree = 0;
  CUDA_CHECK(cudaMemcpyAsync(&agree, ctx->d_barrier.ptr, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  ctx->replicated = agree != 0;
  ctx->exchange_decided = true;
  if (ctx->replicated) setup_peer_gather(ctx);
  if (!ctx->replicated) {
    delete ctx->global; ctx->global = nullptr;
    ctx->d_pos.release(); ctx->d_xcat.release();
    if (ctx->opt_exchange == 2)
      throw std::runtime_error("replicated-x exchange requested but not possible on every rank: " + why);
  }
}

// -------------------------------------------------------------------------------------------------
// Block <-> hashed redistribution of vectors (arrFromBlockToHashed, reference src/BlockToHashed.chpl:87-208;
// arrFromHashedToBlock, src/HashedToBlock.chpl:67-153).  "Block" = the global array in sorted-state order cut into
// contiguous chunks, one per rank; "hashed" = every rank holds the elements of the states it owns, ascending.
// positions: slot of element i of a chunk in the ordering "grouped by owner, stable": offsets[mask[i]] + #{j < i :
// mask[j] == mask[i]}; counts[r] = elements owned by r.  One counting pass, host prefix sums, one writing pass.
void hashed_positions(dmv_context *ctx, int64_t count, const uint8_t *d_masks, int P, std::vector<int64_t> &counts,
                      uint32_t *d_pos) {
  if (P > 32) throw std::runtime_error("block <-> hashed redistribution supports at most 32 ranks");
  counts.assign(P, 0);
  if (count <= 0) return;
  if (count >= (1ll << 32)) throw std::runtime_error("chunks of more than 2^32 elements are not supported");
  const int64_t chunk = 256, n_chunks = (count + chunk - 1) / chunk;
  DevBuf<unsigned long long> d_counts, d_base;
  d_counts.alloc((size_t)n_chunks * P);
  launch_owner_positions(nullptr, d_masks, count, P, chunk, false, d_counts.ptr, nullptr, 0, nullptr, ctx->stream);
  std::vector<unsigned long long> c((size_t)n_chunks * P), base((size_t)n_chunks * P);
  CUDA_CHECK(cudaMemcpyAsync(c.data(), d_counts.ptr, c.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  for (int64_t k = 0; k < n_chunks; ++k)
    for (int r = 0; r < P; ++r) counts[r] += (int64_t)c[(size_t)k * P + r];
  std::vector<unsigned long long> run(P, 0);
  unsigned long long off = 0;
  for (int r = 0; r < P; ++r) { run[r] = off; off += (unsigned long long)counts[r]; }
  for (int64_t k = 0; k < n_chunks; ++k)
    for (int r = 0; r < P; ++r) { base[(size_t)k * P + r] = run[r]; run[r] += c[(size_t)k * P + r]; }
  d_base.upload(base, ctx->stream);
  launch_owner_positions(nullptr, d_masks, count, P, chunk, true, d_counts.ptr, d_base.ptr, 0, d_pos, ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));   // d_base is released on return
}

// all[r * P + q] = what rank r reported for q (collective)
std::vector<int64_t> all_gather_counts(dmv_context *ctx, const std::vector<int64_t> &mine) {
  NcclApi &N = nccl();
  const int P = ctx->num_ranks;
  DevBuf<int64_t> d_mine, d_all;
  d_mine.upload(mine, ctx->stream);
  d_all.alloc((size_t)P * P);
  NCCL_CHECK(N.AllGather(d_mine.ptr, d_all.ptr, (size_t)P, ncclInt64, ctx->comm, ctx->stream));
  std::vector<int64_t> all((size_t)P * P);
  CUDA_CHECK(cudaMemcpyAsync(all.data(), d_all.ptr, all.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  return all;
}

} }  // namespace dmv::host

extern "C" {


int dmv_comm_unique_id(void *id128) {
  API_BEGIN
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  NCCL_CHECK(nccl().GetUniqueId(&id));
  memcpy(id128, &id, sizeof(id));
  API_END
}

int dmv_comm_init(dmv_context *ctx, const void *id128) {
  API_BEGIN
  use_device(ctx);
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  NCCL_CHECK(nccl().CommInitRank(&ctx->comm, ctx->num_ranks, id, ctx->rank));
  API_END
}

int dmv_matvec(dmv_context *ctx, int elt, const void *x, void *y) {
  API_BEGIN
  use_device(ctx);
  require_states(ctx);
  if (elt != DMV_F64 && elt != DMV_C128) throw std::runtime_error("elt must be DMV_F64 or DMV_C128");
  const int P = ctx->num_ranks;
  if (P == 1) {
    const int rc = dmv_local_matvec(ctx, elt, x, y);
    if (rc) throw std::runtime_error(g_last_error);
    return 0;
  }
  if (!ctx->comm) throw std::runtime_error("dmv_matvec on several ranks needs dmv_comm_init");
  NcclApi &N = nccl();
  if (!ctx->exchange_decided) decide_exchange(ctx);
  if (ctx->replicated) {
    // ---- replicated-x product: all-gather x into equal slots, then this rank's rows by the row traversal
    if (x == y) throw std::runtime_error("x and y must not alias");
    const size_t esz = (size_t)8 * elt, bytes = (size_t)ctx->n_states * esz;
    CUDA_CHECK(cudaEventRecord(ctx->ev[0], ctx->stream));
    void *y_dev = y;
    const bool y_host = !is_device_pointer(y);
    if (y_host) {
      ctx->d_y.alloc((size_t)ctx->n_states * elt);
      y_dev = ctx->d_y.ptr;
      if (ctx->h_diag_kept == 0) CUDA_CHECK(cudaMemcpyAsync(y_dev, y, bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    const double *x_cat = ctx->d_xcat.ptr;
    if (ctx->peer_gather) {
      // ---- peer-direct: my block goes straight into slot `rank` of every rank's buffer (epoch parity picks the buffer:
      // a rank raises its flag for epoch e + 1 only after it has consumed buffer e, see DESIGN.md)
      const void *x_dev = x;
      if (!is_device_pointer(x)) {
        ctx->d_x.alloc((size_t)ctx->n_states * elt);
        CUDA_CHECK(cudaMemcpyAsync(ctx->d_x.ptr, x, bytes, cudaMemcpyHostToDevice, ctx->stream));
        x_dev = ctx->d_x.ptr;
      }
      CUDA_CHECK(cudaEventRecord(ctx->ev[1], ctx->stream));
      if (ctx->peer_slot_elt != elt) upload_peer_slots(ctx, elt);
      const unsigned epoch = ++ctx->gather_epoch;
      const int b = (int)(epoch & 1u);
      const int64_t n_doubles = ctx->n_states * elt;
      const bool wide = (n_doubles % 2 == 0) && (reinterpret_cast<uintptr_t>(x_dev) % 16 == 0) &&
                        ((size_t)ctx->repl_block * elt) % 2 == 0;
      launch_push_block(x_dev, n_doubles, P, ctx->d_peer_slot[b].ptr, ctx->d_push_done.ptr, ctx->d_peer_flags.ptr,
                        ctx->rank, epoch, wide, ctx->stream);
      launch_wait_flags(ctx->d_flags.ptr, P, epoch, ctx->d_status.ptr, ctx->stream);
      x_cat = ctx->d_xcat.ptr + (size_t)b * ctx->repl_block * P * 2;
    } else {
      char *slot = reinterpret_cast<char *>(ctx->d_xcat.ptr) + (size_t)ctx->rank * ctx->repl_block * esz;
      CUDA_CHECK(cudaMemcpyAsync(slot, x, bytes, cudaMemcpyDefault, ctx->stream));   // host or device x
      CUDA_CHECK(cudaEventRecord(ctx->ev[1], ctx->stream));
      NCCL_CHECK(N.AllGather(slot, ctx->d_xcat.ptr, (size_t)ctx->repl_block * elt, ncclDouble, ctx->comm, ctx->stream));
    }
    CUDA_CHECK(cudaEventRecord(ctx->ev[6], ctx->stream));
    replicated_rows(ctx, elt, x_cat, y_dev);
    CUDA_CHECK(cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_CHECK(cudaEventRecord(ctx->ev[3], ctx->stream));
    CUDA_CHECK(cudaEventRecord(ctx->ev[4], ctx->stream));
    if (y_host) CUDA_CHECK(cudaMemcpyAsync(y, y_dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_CHECK(cudaEventRecord(ctx->ev[5], ctx->stream));
    ctx->timeline_replicated = true;
    if (y_host || !is_device_pointer(x)) {
      check_status(ctx);
      collect_timings(ctx);
    }
    return 0;
  }
  ctx->timeline_replicated = false;
  if (!ctx->rounds.tried) setup_rounds(ctx);
  if (ctx->rounds.ready) {
    // ---- record exchange in overlapped rounds (peer-direct NVLink stores + per-round flags)
    VecStage v = stage_vectors(ctx, elt, x, y);
    if (v.x_host_pending) {   // (single-rank pipelining of the upload does not apply here)
      CUDA_CHECK(cudaMemcpyAsync(ctx->d_x.ptr, v.x_host_pending, v.bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    rounds_product(ctx, elt, v.x_dev, v.y_dev);
    finish_vectors(ctx, v);
    if (v.y_host || !is_device_pointer(x)) {
      check_status(ctx);
      collect_timings(ctx);
    }
    return 0;
  }
  if (!ctx->planned) do_plan(ctx);
  if (ctx->recv_counts[0] < 0) setup_exchange(ctx);
  auto barrier = [&]() {
    NCCL_CHECK(N.AllReduce(ctx->d_barrier.ptr, ctx->d_barrier.ptr, 1, ncclInt32, ncclMax, ctx->comm, ctx->stream));
  };
  // peer-direct: nobody may overwrite my incoming buffer before I have consumed the previous product
  if (ctx->peer_direct) barrier();
  VecStage v = stage_vectors(ctx, elt, x, y);
  do_generate(ctx, elt, v.x_dev, v.y_dev, v.x_host_pending);
  CUDA_CHECK(cudaEventRecord(ctx->ev[2], ctx->stream));
  const int width = ctx->record_width;
  int64_t total_in = 0;
  if (ctx->peer_direct) {
    // the records are already in the peers' incoming buffers (NVLink stores issued by k_generate, overlapped
    // with generation); the all-reduce is the "every sender has finished" fence
    barrier();
    for (int q = 0; q < P; ++q) total_in += ctx->recv_counts[q];
  } else {
  NCCL_CHECK(N.GroupStart());
  {
    int64_t in_off = 0;
    for (int q = 0; q < P; ++q) {
      if (q == ctx->rank) continue;
      const int64_t off = ctx->h_out_offset[q], cnt = ctx->h_out_offset[q + 1] - off;
      if (cnt > 0) {
        NCCL_CHECK(N.Send(ctx->d_out_betas.ptr + off, (size_t)cnt, ncclUint64, q, ctx->comm, ctx->stream));
        NCCL_CHECK(N.Send(ctx->d_out_coeffs.ptr + off * width, (size_t)cnt * width, ncclDouble, q, ctx->comm, ctx->stream));
      }
      const int64_t rc = ctx->recv_counts[q];
      if (rc > 0) {
        NCCL_CHECK(N.Recv(ctx->d_in_betas.ptr + in_off, (size_t)rc, ncclUint64, q, ctx->comm, ctx->stream));
        NCCL_CHECK(N.Recv(ctx->d_in_coeffs.ptr + in_off * width, (size_t)rc * width, ncclDouble, q, ctx->comm, ctx->stream));
      }
      in_off += rc;
    }
    total_in = in_off;
  }
  NCCL_CHECK(N.GroupEnd());
  }
  CUDA_CHECK(cudaEventRecord(ctx->ev[3], ctx->stream));
  do_accumulate(ctx, elt, total_in, ctx->d_in_betas.ptr, ctx->d_in_coeffs.ptr, v.y_dev);
  finish_vectors(ctx, v);
  if (v.y_host || !is_device_pointer(x)) {
    check_status(ctx);
    collect_timings(ctx);
  }
  API_END
}

// ---- block <-> hashed redistribution ("next" row f2)
int dmv_hashed_positions(dmv_context *ctx, int64_t count, const uint8_t *masks, int num_ranks, int64_t *counts,
                         uint32_t *positions) {
  API_BEGIN
  use_device(ctx);
  if (count < 0 || num_ranks < 1) throw std::runtime_error("bad arguments");
  InArg<uint8_t> m(masks, (size_t)count, ctx->stream);
  OutArg<uint32_t> out(positions, (size_t)count);
  std::vector<int64_t> c;
  hashed_positions(ctx, count, m.ptr, num_ranks, c, out.ptr);
  if (counts) std::copy(c.begin(), c.end(), counts);
  out.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_permute(dmv_context *ctx, int elt, int64_t count, const uint32_t *positions, const void *in, void *out,
                int gather) {
  API_BEGIN
  use_device(ctx);
  if (elt != 1 && elt != 2) throw std::runtime_error("elt must be 1 (8-byte) or 2 (16-byte elements)");
  if (in == out) throw std::runtime_error("in and out must not alias");
  InArg<uint32_t> p(positions, (size_t)count, ctx->stream);
  InArg<double> i(reinterpret_cast<const double *>(in), (size_t)count * elt, ctx->stream);
  OutArg<double> o(reinterpret_cast<double *>(out), (size_t)count * elt);
  launch_permute(count, elt, p.ptr, i.ptr, o.ptr, gather != 0, ctx->stream);
  o.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_block_to_hashed(dmv_context *ctx, int elt, int64_t chunk_count, const uint8_t *masks_chunk,
                        const void *block_chunk, void *hashed, int64_t hashed_count) {
  API_BEGIN
  use_device(ctx);
  if (elt != 1 && elt != 2) throw std::runtime_error("elt must be 1 (8-byte) or 2 (16-byte elements)");
  const int P = ctx->num_ranks;
  InArg<uint8_t> m(masks_chunk, (size_t)chunk_count, ctx->stream);
  InArg<double> in(reinterpret_cast<const double *>(block_chunk), (size_t)chunk_count * elt, ctx->stream);
  OutArg<double> out(reinterpret_cast<double *>(hashed), (size_t)hashed_count * elt);
  DevBuf<uint32_t> d_pos;
  DevBuf<double> d_grouped;
  d_pos.alloc((size_t)chunk_count);
  d_grouped.alloc((size_t)chunk_count * elt);
  std::vector<int64_t> counts;
  hashed_positions(ctx, chunk_count, m.ptr, P, counts, d_pos.ptr);
  launch_permute(chunk_count, elt, d_pos.ptr, in.ptr, d_grouped.ptr, false, ctx->stream);
  if (P == 1) {
    if (hashed_count != chunk_count) throw std::runtime_error("hashed block size does not match the masks");
    CUDA_CHECK(cudaMemcpyAsync(out.ptr, d_grouped.ptr, (size_t)chunk_count * elt * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  } else {
    if (!ctx->comm) throw std::runtime_error("dmv_block_to_hashed on several ranks needs dmv_comm_init");
    NcclApi &N = nccl();
    const std::vector<int64_t> all = all_gather_counts(ctx, counts);   // all[r * P + q]: chunk r holds for owner q
    int64_t incoming = 0;
    for (int r = 0; r < P; ++r) incoming += all[(size_t)r * P + ctx->rank];
    if (incoming != hashed_count) throw std::runtime_error("hashed block size does not match the masks");
    NCCL_CHECK(N.GroupStart());
    int64_t send_off = 0, recv_off = 0;
    for (int q = 0; q < P; ++q) {
      const int64_t sc = counts[q], rc = all[(size_t)q * P + ctx->rank];
      if (q == ctx->rank) {
        if (sc > 0) CUDA_CHECK(cudaMemcpyAsync(out.ptr + recv_off * elt, d_grouped.ptr + send_off * elt, (size_t)sc * elt * 8,
                                               cudaMemcpyDeviceToDevice, ctx->stream));
      } else {
        if (sc > 0) NCCL_CHECK(N.Send(d_grouped.ptr + send_off * elt, (size_t)sc * elt, ncclDouble, q, ctx->comm, ctx->stream));
        if (rc > 0) NCCL_CHECK(N.Recv(out.ptr + recv_off * elt, (size_t)rc * elt, ncclDouble, q, ctx->comm, ctx->stream));
      }
      send_off += sc;
      recv_off += rc;
    }
    NCCL_CHECK(N.GroupEnd());
  }
  out.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

int dmv_hashed_to_block(dmv_context *ctx, int elt, int64_t chunk_count, const uint8_t *masks_chunk,
                        const void *hashed, int64_t hashed_count, void *block_chunk) {
  API_BEGIN
  use_device(ctx);
  if (elt != 1 && elt != 2) throw std::runtime_error("elt must be 1 (8-byte) or 2 (16-byte elements)");
  const int P = ctx->num_ranks;
  InArg<uint8_t> m(masks_chunk, (size_t)chunk_count, ctx->stream);
  InArg<double> in(reinterpret_cast<const double *>(hashed), (size_t)hashed_count * elt, ctx->stream);
  OutArg<double> out(reinterpret_cast<double *>(block_chunk), (size_t)chunk_count * elt);
  DevBuf<uint32_t> d_pos;
  DevBuf<double> d_grouped;
  d_pos.alloc((size_t)chunk_count);
  d_grouped.alloc((size_t)chunk_count * elt);
  std::vector<int64_t> counts;   // counts[q]: positions of MY chunk owned by q = what q sends me
  hashed_positions(ctx, chunk_count, m.ptr, P, counts, d_pos.ptr);
  if (P == 1) {
    if (hashed_count != chunk_count) throw std::runtime_error("hashed block size does not match the masks");
    CUDA_CHECK(cudaMemcpyAsync(d_grouped.ptr, in.ptr, (size_t)chunk_count * elt * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  } else {
    if (!ctx->comm) throw std::runtime_error("dmv_hashed_to_block on several ranks needs dmv_comm_init");
    NcclApi &N = nccl();
    const std::vector<int64_t> all = all_gather_counts(ctx, counts);   // all[r * P + q]: chunk r needs from owner q
    int64_t outgoing = 0;
    for (int r = 0; r < P; ++r) outgoing += all[(size_t)r * P + ctx->rank];
    if (outgoing != hashed_count) throw std::runtime_error("hashed block size does not match the masks");
    NCCL_CHECK(N.GroupStart());
    int64_t send_off = 0, recv_off = 0;
    for (int q = 0; q < P; ++q) {
      // my hashed block is ascending in global position: the part for chunk q follows the parts for chunks < q
      const int64_t sc = all[(size_t)q * P + ctx->rank], rc = counts[q];
      if (q == ctx->rank) {
        if (sc > 0) CUDA_CHECK(cudaMemcpyAsync(d_grouped.ptr + recv_off * elt, in.ptr + send_off * elt, (size_t)sc * elt * 8,
                                               cudaMemcpyDeviceToDevice, ctx->stream));
      } else {
        if (sc > 0) NCCL_CHECK(N.Send(in.ptr + send_off * elt, (size_t)sc * elt, ncclDouble, q, ctx->comm, ctx->stream));
        if (rc > 0) NCCL_CHECK(N.Recv(d_grouped.ptr + recv_off * elt, (size_t)rc * elt, ncclDouble, q, ctx->comm, ctx->stream));
      }
      send_off += sc;
      recv_off += rc;
    }
    NCCL_CHECK(N.GroupEnd());
  }
  launch_permute(chunk_count, elt, d_pos.ptr, d_grouped.ptr, out.ptr, true, ctx->stream);
  out.finish(ctx->stream);
  CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  API_END
}

// Replicated-x product without a communicator (the host owns the all-gather): set-up, then rows of H applied to
// a caller-assembled x_cat (rank r's block at r * dmv_get_info("replicated_block") elements).  Device pointers.
int dmv_replicated_setup(dmv_context *ctx) {
  API_BEGIN
  use_device(ctx);
  setup_replicated(ctx);
  API_END
}

int dmv_replicated_product(dmv_context *ctx, int elt, const void *x_cat, void *y) {
  API_BEGIN
  use_device(ctx);
  require_states(ctx);
  if (!ctx->global || ctx->repl_block <= 0) throw std::runtime_error("dmv_replicated_setup has not run");
  if (elt != DMV_F64 && elt != DMV_C128) throw std::runtime_error("elt must be DMV_F64 or DMV_C128");
  if (!is_device_pointer(x_cat) || !is_device_vector(y, ctx->n_states)) throw std::runtime_error("dmv_replicated_product needs device pointers");
  replicated_rows(ctx, elt, x_cat, y);
  check_status(ctx);
  API_END
}

}  // extern "C"
