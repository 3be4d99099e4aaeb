// dmv_context.h -- internal declarations shared by the translation units of the C ABI: the per-GPU context, its helpers,
// error / NCCL plumbing.  Not installed: the public interface is include/dmv_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types only; the library itself is resolved with dlopen at dmv_comm_init

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/dmv_b200.h"
#include "dmv_host.h"

using namespace dmv;


namespace dmv { namespace host {


extern thread_local std::string g_last_error;   // defined in dmv_api.cu

#define CUDA_CHECK(expr)                                                                        \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      throw std::runtime_error(std::string(#expr) + ": " + cudaGetErrorString(_e));            \
  } while (0)

#define API_BEGIN try {
#define API_END                                         \
  return 0;                                             \
  }                                                     \
  catch (const std::exception &e) {                     \
    g_last_error = e.what();                            \
    return 1;                                           \
  }                                                     \
  catch (...) {                                         \
    g_last_error = "unknown error";                     \
    return 1;                                           \
  }

template <typename T>
struct DevBuf {
  T *ptr = nullptr;
  size_t count = 0;
  void alloc(size_t n) {
    if (n <= count && ptr) return;
    release();
    if (n == 0) n = 1;
    CUDA_CHECK(cudaMalloc(&ptr, n * sizeof(T)));
    count = n;
  }
  void release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    count = 0;
  }
  void upload(const std::vector<T> &h, cudaStream_t s) {
    alloc(h.size());
    if (!h.empty()) CUDA_CHECK(cudaMemcpyAsync(ptr, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  }
  ~DevBuf() { release(); }
};

inline bool is_device_pointer(const void *p) {
  if (!p) return false;
  cudaPointerAttributes attr;
  cudaError_t e = cudaPointerGetAttributes(&attr, p);
  if (e != cudaSuccess) { cudaGetLastError(); return false; }
  return attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged;
}
// a vector of a context that owns no states (a rank of a small basis) has no elements: a tensor of zero elements may
// carry a null pointer, and nothing is read from or written to it
inline bool is_device_vector(const void *p, int64_t n_states) { return n_states == 0 ? true : is_device_pointer(p); }

// ---- NCCL through dlopen ------------------------------------------------------------------------
struct NcclApi {
  void *handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
inline NcclApi &nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
      api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (api.handle) break;
    }
    if (!api.handle) return;
#define LOAD(sym) api.sym = reinterpret_cast<decltype(api.sym)>(dlsym(api.handle, "nccl" #sym))
    LOAD(GetUniqueId); LOAD(CommInitRank); LOAD(CommDestroy); LOAD(GroupStart); LOAD(GroupEnd);
    LOAD(Send); LOAD(Recv); LOAD(AllGather); LOAD(AllReduce); LOAD(GetErrorString);
#undef LOAD
  });
  if (!api.handle || !api.Send) throw std::runtime_error("NCCL (libnccl.so.2) is not available");
  return api;
}
#define NCCL_CHECK(expr)                                                                       \
  do {                                                                                         \
    ncclResult_t _r = (expr);                                                                  \
    if (_r != ncclSuccess)                                                                     \
      throw std::runtime_error(std::string(#expr) + ": " + nccl().GetErrorString(_r));        \
  } while (0)

// stages of one product (the coarse part of the reference's timing tree, DMV:1028-1052; the split of the fused kernels
// into the reference's inner timers -- applyOffDiag / stateInfo / indexing / accessing -- comes from tools/ncu_tree.py)
enum Timing { T_H2D = 0, T_GENERATE, T_EXCHANGE, T_ACCUMULATE, T_D2H, T_TOTAL, T_TABLE_FILL, T_COUNT };
inline const char *const kTimingNames[T_COUNT] = {"h2d", "generate(diag+offdiag+local accumulate)", "exchange(all-to-all)",
                                     "accumulate(remote records)", "d2h", "total",
                                     "table refill (k_rows; part of generate)"};

// Flip-mask groups of an operator in look-up-table form (see LutGroup in dmv_device.cuh).
struct HostTables {
  std::vector<LutGroup> groups;
  std::vector<double> lut_re, lut_c;   // real parts only / interleaved complex
  std::vector<OffTerm> terms;
  std::vector<BpWord> bp;               // non-empty: bit-parallel emit test (see BpWord)
  bool any_generic = false, any_s_out = false;
};
struct DevTables {
  DevBuf<LutGroup> groups;
  DevBuf<double> lut_re, lut_c;
  DevBuf<OffTerm> terms;
  DevBuf<BpWord> bp;
  void upload(const HostTables &h, cudaStream_t s) {
    groups.upload(h.groups, s); lut_re.upload(h.lut_re, s); lut_c.upload(h.lut_c, s); terms.upload(h.terms, s);
    bp.upload(h.bp, s);
  }
};

} }  // namespace dmv::host
using namespace dmv::host;

struct dmv_context {
  int device = 0, rank = 0, num_ranks = 1;
  // basis
  int n_sites = 0, hamming_weight = -1, spin_inversion = 0;
  bool has_permutations = false;
  Projection proj = PROJ_NONE;
  bool identity_index = false;
  uint64_t site_mask = 0;
  bool complex_coefficients = false;  // operator or characters are complex
  HostOrbitProgram host_orbit;
  DevBuf<uint64_t> d_orbit64;
  DevBuf<int32_t> d_orbit32;
  DevBuf<double> d_chars;
  DevBuf<uint16_t> d_canon_lut;
  DevBuf<uint64_t> d_canon_masks, d_cc_mask;
  DevBuf<uint32_t> d_canon_lut2;
  DevBuf<int32_t> d_cc_begin, d_cc_delta;
  DevBuf<uint16_t> d_tor_lutm;
  DevBuf<uint8_t> d_tor_frow;
  DevBuf<uint32_t> d_tor_luts;
  DevBuf<uint64_t> d_tor_net_mask;
  DevBuf<int32_t> d_tor_net_delta;
  int opt_canon = -1;    // -1 auto (block-rotation canonical form when the chain subgroup allows it), 0 walk the chain
  OrbitProgram orbit{};  // device view
  // operator
  std::vector<DiagTerm> h_diag;
  HostTables h_push, h_pull;          // column-traversal (scatter) / row-traversal (gather) tables
  DevTables d_push, d_pull;
  DevBuf<DiagTerm> d_diag;
  std::vector<DiagClass> h_diag_classes;  // bit-parallel part of the diagonal; h_diag is reordered: rest first
  DevBuf<DiagClass> d_diag_classes;
  int n_diag_rest = 0;
  size_t h_diag_kept = 0;   // number of diagonal terms of the operator (h_diag itself only keeps the non-class rest)
  // options
  int opt_mode = -1;    // -1 auto (pull when one rank owns the basis), 0 push (scatter), 1 pull (gather)
  int opt_index = -1;   // -1 auto, 0 directory search, 2 combinadic rank
  int opt_bitparallel = 1;  // 0: walk the groups one by one even when the bit-parallel test applies
  int opt_gather = -1;      // row traversal kernel: -1 auto (k_gather when it applies), 0 always the queued k_pull
  // k_gather applicability (set at context creation from the row-traversal tables)
  bool gather_ok = false, gather_narrow = false, gather_uniform = false;
  // k_rows applicability (bases with permutation symmetries, trivial characters, real bit-parallel operator) and its
  // hash table over this context's representatives (see table_slot in dmv_device.cuh)
  bool rows_ok = false;
  int opt_rows = -1;        // -1 auto (k_rows when it applies), 0 the queued k_pull
  int opt_rows_ctas = 3;    // k_rows: resident CTAs per SM: 3 (80 registers, default) | 2 (122 registers) | 4 (64 registers)
  int rows_kernel = 0;      // instantiation of the last k_rows launch: 100 CTAS + 10 TK + MPH (0: none yet)
  int rows_batch_kernel = 0;   // the same for k_rows_batch: 100 CTAS + 10 TK
  int opt_table_per_state = 0;   // buckets per state of the complex128 and k_rows_batch tables: 0 auto | 2 | 4 | 8
  int opt_gather_walk = 0;  // k_gather: 0 per-lane walk from the top bit (default), 1 group-major warp-uniform walk
                            // (measured slower), 2 per-lane walk from the bottom bit (round 1)
  DevBuf<unsigned char> d_table;
  DevBuf<unsigned char> d_mph_blocks, d_dense;   // dense index: perfect-hash blocks, dense table of (key, value) slots
  PerfectHash mph{};
  bool dense_index = false;
  int opt_rows_index = -1;   // -1 auto / 0 open-addressing table; 1 dense index through a perfect hash (measured slower:
                             // profiles/r02_rows_pipelines.md)
  DevBuf<uint32_t> d_slot_of;
  uint32_t table_slots = 0;
  int table_elt = 0;        // element type the slots are laid out for (0: not built)
  // k_rows_batch: 64-byte buckets { key, six doubles, spare }, eight per state (fewer when memory is short); built on the first
  // batched product
  DevBuf<unsigned char> d_table_batch;
  DevBuf<uint32_t> d_slot_of_batch;
  uint32_t table_batch_slots = 0;
  int opt_rows_batch_min = 2;   // doubles per state (vectors x element width) from which a batch goes through k_rows_batch
  int opt_rows_batch = -1;  // -1 / 1: batched products of symmetric bases go through k_rows_batch | 0: vector by vector
  double gather_uni[2] = {0.0, 0.0};
  int index_mode = INDEX_DIRECTORY;
  DevBuf<uint32_t> d_binom, d_lin_a, d_lin_b;
  int lin_bits = 0;
  int binom_stride = 0;
  uint64_t rank_total = 0;
  // representatives of this rank
  int64_t n_states = -1;
  DevBuf<uint64_t> d_reps;
  DevBuf<double> d_norms;
  DevBuf<uint32_t> d_dir;
  uint64_t n_buckets = 0;
  int dir_shift = 0;
  // vectors staged for host callers
  DevBuf<double> d_x, d_y;
  // outgoing / incoming records
  bool planned = false;
  std::vector<int64_t> send_counts;        // [num_ranks]
  std::vector<int64_t> recv_counts;        // [num_ranks] (filled by dmv_comm plan exchange)
  std::vector<int64_t> h_out_offset;       // [num_ranks + 1]
  DevBuf<int64_t> d_out_offset;
  DevBuf<unsigned long long> d_out_count;
  DevBuf<uint64_t> d_out_betas, d_in_betas;
  DevBuf<double> d_out_coeffs, d_in_coeffs;
  int record_width = 2;                    // doubles per coefficient of the current buckets
  int plan_grid = 0;                       // CTAs of the planned launches (exact warp-private regions)
  int row_split = 1;                       // lanes per source state (chosen at plan time from the block size)
  bool peer_direct = false;                // records are stored straight into the peers' incoming buffers
  int ptr_width = 0;                       // record width the destination pointer table was built for
  int opt_exchange = -1;                   // -1 auto (peer-direct when possible), 0 NCCL send/recv, 1 peer-direct
  std::vector<void *> peer_betas, peer_coeffs;   // IPC-mapped incoming buffers of the peers
  std::vector<int64_t> my_offset_in_peer;         // first slot of MY region in every peer's incoming buffer
  DevBuf<int> d_barrier;
  DevBuf<unsigned long long> d_warp_counts;
  DevBuf<int64_t> d_warp_offsets, d_out_capacity;
  DevBuf<uint64_t *> d_out_betas_ptr;
  DevBuf<double *> d_out_coeffs_ptr;
  std::vector<uint64_t *> h_out_betas_ptr;   // where the records for every destination go (local bucket or peer)
  std::vector<double *> h_out_coeffs_ptr;
  int64_t number_terms = 0;
  DevBuf<unsigned long long> d_status;
  // streams
  cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
  static constexpr int kCopyChunks = 8;
  cudaEvent_t ev_chunk[kCopyChunks] = {};
  cudaEvent_t ev[T_COUNT + 2] = {};
  cudaEvent_t ev_fill[2] = {};
  bool fill_timed = false;
  double timings[T_COUNT] = {};
  // communicator
  ncclComm_t comm = nullptr;
  // replicated-x product (exchange = 2, see setup_replicated): a single-rank twin context holding the WHOLE basis,
  // the slot of every global state in the all-gathered x, and the gathered x itself
  std::vector<double> k_off_v, k_diag_v;                      // copies of the creation arguments
  std::vector<uint64_t> k_off_m, k_off_r, k_off_x, k_off_s, k_diag_m, k_diag_r, k_diag_s;
  std::vector<int32_t> k_perms;
  std::vector<uint8_t> k_flips;
  std::vector<double> k_chars;
  int64_t k_group_order = 0;
  dmv_context *global = nullptr;
  DevBuf<uint32_t> d_pos;
  int64_t repl_block = 0;        // slot size per rank in the gathered x (the largest block)
  DevBuf<double> d_xcat;
  bool replicated = false, exchange_decided = false, timeline_replicated = false;
  // peer-direct all-gather of x (launch_push_block): the peers' gathered vectors (two buffers, alternating by epoch) and
  // flag words mapped with CUDA IPC
  bool peer_gather = false;
  int opt_peer_gather = -1;                 // -1 auto, 0 NCCL all-gather
  std::vector<void *> peer_xcat, peer_flagmem;
  DevBuf<unsigned> d_flags, d_push_done;    // [num_ranks] epochs raised by the peers; CTA counter of k_push_block
  DevBuf<void *> d_peer_slot[2];            // [num_ranks] slot `rank` of every rank's buffer b
  DevBuf<unsigned *> d_peer_flags;          // [num_ranks]
  int peer_slot_elt = 0;                    // element width the slot pointers were computed for
  unsigned gather_epoch = 0;
  // record exchange in overlapped ROUNDS (peer-direct records; reference DMV:638-661, 818-852, 957-1011): the rows are cut
  // into R rounds; round r's records land in the owners' buffers while round r + 1 is being generated, and the owner
  // accumulates round r on a second stream as soon as every sender has raised its flag for it
  struct Rounds {
    bool ready = false, tried = false;
    int R = 0, grid = 0, row_split = 1;
    std::vector<int64_t> row_begin;           // [R + 1]
    DevBuf<int64_t> d_warp_offsets;           // [R][warps][P]: first slot of every warp inside MY region of (round, dest)
    DevBuf<int64_t> d_capacity;               // [R][P]
    std::vector<int64_t> in_slice;            // [R + 1]: rounds inside my incoming buffer (records)
    std::vector<int64_t> my_off;              // [R][P]: my region of round r inside rank q's incoming buffer
    int64_t in_total = 0;
    std::vector<int64_t> peer_total;          // [P]: in_total of every rank (start of its second buffer)
    DevBuf<uint64_t> d_in_betas;              // two buffers (alternating products) of in_total records
    DevBuf<double> d_in_coeffs;               // two doubles per record
    std::vector<void *> peer_betas, peer_coeffs, peer_flags;
    DevBuf<unsigned> d_flags;                 // [P] raised by the senders: product * R + round + 1
    DevBuf<unsigned *> d_peer_flags;
    DevBuf<uint64_t *> d_bptr;                // [2][R][P]
    DevBuf<double *> d_cptr;
    int ptr_width = 0;
    unsigned seq = 0;
    cudaStream_t acc_stream = nullptr;
    cudaEvent_t ev_begin = nullptr, ev_done = nullptr;
    int64_t terms = 0;
  } rounds;
  int opt_rounds = -1;                        // -1 auto, 0 / 1 off (generate everything, fence, accumulate), R > 1

  // Lanczos work space (dmv_lanczos)
  DevBuf<double> lz_v[4];
  DevBuf<double> lz_scal;

  ~dmv_context() {
    delete global;
    for (void *q : peer_betas) if (q) cudaIpcCloseMemHandle(q);
    for (void *q : peer_coeffs) if (q) cudaIpcCloseMemHandle(q);
    for (void *q : peer_xcat) if (q) cudaIpcCloseMemHandle(q);
    for (void *q : rounds.peer_betas) if (q) cudaIpcCloseMemHandle(q);
    for (void *q : rounds.peer_coeffs) if (q) cudaIpcCloseMemHandle(q);
    for (void *q : rounds.peer_flags) if (q) cudaIpcCloseMemHandle(q);
    if (rounds.acc_stream) cudaStreamDestroy(rounds.acc_stream);
    if (rounds.ev_begin) cudaEventDestroy(rounds.ev_begin);
    if (rounds.ev_done) cudaEventDestroy(rounds.ev_done);
    for (void *q : peer_flagmem) if (q) cudaIpcCloseMemHandle(q);
    if (comm) nccl().CommDestroy(comm);
    for (auto &e : ev) if (e) cudaEventDestroy(e);
    for (auto &e : ev_fill) if (e) cudaEventDestroy(e);
    for (auto &e : ev_chunk) if (e) cudaEventDestroy(e);
    if (copy_stream) cudaStreamDestroy(copy_stream);
    if (own_stream) cudaStreamDestroy(own_stream);
  }
};


namespace dmv { namespace host {

bool use_gather(const dmv_context *ctx);
bool use_rows(const dmv_context *ctx);
bool use_pull(const dmv_context *ctx);
void use_device(const dmv_context *ctx);
bool complex_values(const dmv_context *ctx, int elt);
KernelParams base_params(dmv_context *ctx);
void build_diag_classes(dmv_context *ctx);
void select_tables(dmv_context *ctx, KernelParams &p, bool pull, bool complex_vals);
void require_states(const dmv_context *ctx);
void check_status(dmv_context *ctx);

// binomial table for the combinadic ranking of fixed-Hamming-weight states
struct Binomials {
  uint64_t c[65][65];
  Binomials() {
    for (int n = 0; n <= 64; ++n)
      for (int k = 0; k <= 64; ++k) {
        if (k == 0 || k == n) c[n][k] = (k <= n) ? 1 : 0;
        else if (k > n) c[n][k] = 0;
        else {
          const unsigned __int128 v = (unsigned __int128)c[n - 1][k - 1] + c[n - 1][k];
          c[n][k] = v > (unsigned __int128)~0ull ? ~0ull : (uint64_t)v;
        }
      }
  }
};
const Binomials &binom();
void select_index_mode(dmv_context *ctx);
void install_directory(dmv_context *ctx);
void upload_orbit(dmv_context *ctx);
uint64_t fixed_hamming_rank(uint64_t s);
uint64_t fixed_hamming_unrank(uint64_t r, int weight);
void zero_y_if_diag(dmv_context *ctx, int elt, void *y);

struct VecStage {  // x / y either used in place (device pointers) or staged through context buffers
  const void *x_dev; void *y_dev; bool y_host; void *y_user; size_t bytes;
  const void *x_host_pending;   // host x whose upload is pipelined with generation (push traversal)
};
VecStage stage_vectors(dmv_context *ctx, int elt, const void *x, void *y);
void finish_vectors(dmv_context *ctx, const VecStage &v);
void upload_out_pointers(dmv_context *ctx);
void do_plan(dmv_context *ctx);
void ensure_table(dmv_context *ctx, int elt);
void rows_product_batch(dmv_context *ctx, int elt, int nv, const void *x, void *y, int64_t stride);
void rows_product(dmv_context *basis, KernelParams &p, int elt, const void *x_all, const uint32_t *pos, cudaStream_t stream, bool fill = true, dmv_context *timer = nullptr);
void do_generate(dmv_context *ctx, int elt, const void *x_dev, void *y_dev, const void *x_host_pending = nullptr, int64_t row_begin = 0, int64_t row_end = 0);
void do_accumulate(dmv_context *ctx, int elt, int64_t count, const uint64_t *betas, const double *coeffs, void *y_dev);
void collect_timings(dmv_context *ctx);
extern std::mutex g_bind_mutex;
extern std::map<const void *, dmv_context *> g_bindings;

template <typename T>
struct InArg {  // device view of an input array
  DevBuf<T> buf; const T *ptr;
  InArg(const T *p, size_t n, cudaStream_t s) {
    if (is_device_pointer(p)) ptr = p;
    else { buf.alloc(n); if (n) CUDA_CHECK(cudaMemcpyAsync(buf.ptr, p, n * sizeof(T), cudaMemcpyHostToDevice, s)); ptr = buf.ptr; }
  }
};
template <typename T>
struct OutArg {  // device view of an output array, copied back by finish()
  DevBuf<T> buf; T *ptr; T *user; size_t n; bool host;
  OutArg(T *p, size_t n_) : user(p), n(n_) {
    host = !is_device_pointer(p);
    if (host) { buf.alloc(n); ptr = buf.ptr; } else ptr = p;
  }
  void finish(cudaStream_t s, size_t used = (size_t)-1) {
    if (host && user) { const size_t m = used == (size_t)-1 ? n : used; if (m) CUDA_CHECK(cudaMemcpyAsync(user, ptr, m * sizeof(T), cudaMemcpyDeviceToHost, s)); }
  }
};
void setup_exchange(dmv_context *ctx);
void setup_replicated(dmv_context *ctx);
void replicated_rows(dmv_context *ctx, int elt, const void *x_cat, void *y_dev);
void setup_rounds(dmv_context *ctx);
void upload_round_pointers(dmv_context *ctx, int width);
void rounds_product(dmv_context *ctx, int elt, const void *x_dev, void *y_dev);
void setup_peer_gather(dmv_context *ctx);
void upload_peer_slots(dmv_context *ctx, int elt);
void decide_exchange(dmv_context *ctx);
void hashed_positions(dmv_context *ctx, int64_t count, const uint8_t *d_masks, int P, std::vector<int64_t> &counts, uint32_t *d_pos);
std::vector<int64_t> all_gather_counts(dmv_context *ctx, const std::vector<int64_t> &mine);
double tridiagonal_lowest(const std::vector<double> &a, const std::vector<double> &b, std::vector<double> &vec);

} }  // namespace dmv::host
