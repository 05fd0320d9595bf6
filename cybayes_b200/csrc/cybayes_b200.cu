// cybayes_b200 -- host scheduler and C ABI (see include/cybayes_b200.h).
//
// One context drives one B200: leaf state codes, a pool of P matrices and a pool of
// partial-likelihood buffers live in HBM; an evaluation is turned into a handful of kernel
// launches (one per tree level, or ONE for a dirty path / a batch of candidate paths) on a
// single stream, followed by an optional scalar NCCL all-reduce and an 8-byte read-back.
// Snapshots are immutable node -> buffer tables with reference-counted buffers: the
// copy-on-write equivalent of the reference's aliased cache dicts (ML_gamma.pyx:114).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <limits.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <time.h>

#include <algorithm>
#include <exception>
#include <new>
#include <string>
#include <vector>

#include "cb_types.cuh"
#include "kernels_dmma.cuh"
#include "kernels_dmma_rc.cuh"
#include "kernels_general.cuh"
#include "kernels_pmat.cuh"
#include "kernels_s2.cuh"
#include "kernels_s2t.cuh"

using namespace cb;

// ------------------------------------------------------------------------------ errors
static thread_local std::string g_err;
static int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}
#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) return fail("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
  } while (0)
#define REQUIRE(cond, ...)            \
  do {                                \
    if (!(cond)) return fail(__VA_ARGS__); \
  } while (0)


static inline double now_us() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}

// No C++ exception may cross the C ABI: every entry point that allocates runs under this guard.
template <typename F>
static int guarded(F&& f) {
  try {
    return f();
  } catch (const std::bad_alloc&) {
    return fail("out of host memory");
  } catch (const std::exception& e) {
    return fail("internal error: %s", e.what());
  } catch (...) {
    return fail("internal error: unknown exception");
  }
}

// ------------------------------------------------------------------------------- NCCL (dlopen)
struct NcclId { char internal[128]; };
typedef struct ncclComm* ncclComm_t;
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, NcclId, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static int load_nccl() {
  if (g_nccl.lib) return 0;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  REQUIRE(g_nccl.lib, "cannot dlopen libnccl.so.2: %s", dlerror());
  g_nccl.GetUniqueId = (int (*)(NcclId*))dlsym(g_nccl.lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (int (*)(ncclComm_t*, int, NcclId, int))dlsym(g_nccl.lib, "ncclCommInitRank");
  g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(g_nccl.lib, "ncclAllReduce");
  g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t))dlsym(g_nccl.lib, "ncclAllGather");
  g_nccl.CommDestroy = (int (*)(ncclComm_t))dlsym(g_nccl.lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
  REQUIRE(g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.AllReduce && g_nccl.CommDestroy,
          "libnccl is missing expected symbols");
  return 0;
}
enum { NCCL_DOUBLE = 8, NCCL_SUM = 0, NCCL_INT8 = 0 };  // ncclFloat64 / ncclSum / ncclInt8 in nccl.h

// ------------------------------------------------------------------------------ context
constexpr int DMMA_RC_MIN_STATES = 9;   // measured: 1.65x (S = 23, 2304 patterns) .. 3.1x (S = 30, 16384) over the plain FP64 kernel
constexpr int64_t DMMA_RC_MIN_SITES = 1024;  // measured crossover against the 64-site tile kernel + level schedule (S = 47, 64)
constexpr int64_t S2_TILED_MIN_SITES = 64 * 2 * 148 * 4;  // 75 776: from here a 2-state alignment fills the GPU with 256-site blocks

struct Buffer {
  double* data = nullptr;
  int32_t* scale = nullptr;
  int refs = 0;
};
struct Snapshot {
  std::vector<int32_t> buf_of_node;     // index by node id; -1 = absent
  std::vector<int32_t> cherry_of_node;  // 2-state family: record of a folded cherry (never materialised), or -1
  int refs = 0;
};
// A small subtree kept by a snapshot as a RECORD instead of a stored partial: its two children and, in the library's own
// P pool at slots [rec * 2C, (rec + 1) * 2C), copies of the P matrices of its two child edges (child 0: C slots, child 1:
// C slots).  A cherry (both children tips) is folded into its parent's lookup table; a node whose children are tips or
// cherries (3 or 4 tips below it; tiled kernel only) is recomputed on the fly when a later dirty path needs it as a
// sibling -- two table look-ups and a product per site instead of 68 bytes of HBM per site.  child[k] <= n_taxa: a tip;
// otherwise the node id of a cherry that the same snapshot holds as a record.
struct CherryRec {
  int32_t tip[2] = {0, 0};   // (children; named tip for the common case)
  int refs = 0;
};

// ---- evaluation plans (see build_plan)
struct PlanChild {
  int32_t kind;  // SrcKind
  int32_t ref;   // SRC_TIP: tip id.  SRC_BUFFER: position of the producing op, or ~node (< 0) when the input snapshot
                 // holds it.  SRC_CHERRY: caller's op index of the folded cherry, or ~node for a record of the input
                 // snapshot.  SRC_STACK: tile buffer.  SRC_CARRIED: unused.
  int32_t edge;  // 2 * (caller's op index) + child: where this edge's P slots sit in the caller's arrays; < 0: the edge
                 // belongs to a record of the input snapshot, its P copies start at library slot ~edge
};
struct PlanOp {
  int32_t node;
  PlanChild ch[2];
  int32_t out_buf;               // tiled kernel: shared-memory tile buffer of the result, or -1
  int32_t pf_buf;                // tiled kernel: tile buffer a stored child is prefetched into, or -1
  uint8_t is_root, keep, stream, spill, pushed;
  uint8_t make_rec;              // not stored: the returned snapshot keeps the node as a record (small subtree)
  uint8_t synthetic;             // not in the caller's list: a record of the input snapshot recomputed as a sibling
};
struct PlanLaunch { int r_begin, r_end, max_ops, n_bufs; };
struct EvalPlan {
  // key (full evaluations only)
  int flags = 0, n_lists = 0, split_env = 0;
  std::vector<int32_t> key_offsets, key_nodes, key_children;
  // compiled form
  std::vector<PlanOp> ops;
  std::vector<RangeDesc> ranges;
  std::vector<PlanLaunch> launches;
  int64_t bytes_written = 0, bytes_read = 0;
  int n_stored = 0, n_buffer_reads = 0, n_stack = 0, n_spills = 0, n_cherries = 0, n_small_recs = 0;
  int n_inlined = 0;   // ops computed inside their parent's op (SRC_SMALL): in `ops` for their descriptor, in no range
  uint64_t stamp = 0;
};
constexpr int PLAN_FLAG_MASK = CB_EVAL_WANT_SNAPSHOT | CB_EVAL_STORE_ROOT | CB_EVAL_FORCE_LEVELS | CB_EVAL_FORCE_WALK | CB_EVAL_NO_FOLD;
constexpr int PLAN_CACHE_SIZE = 6;

struct cb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_stage = nullptr, ev_mark[2] = {nullptr, nullptr};
  int sm_count = 148;
  // alignment
  int n_taxa = 0, n_states = 0, n_cats = 0, code_bytes = 1, n_amb = 0;
  int64_t n_sites = 0, P = 0;  // real and padded pattern counts
  bool family_s2 = false;
  bool use_dmma = false;  // general family, 32 <= S <= 64: FP64 tensor-core kernel (below that the plain kernel wins)
  bool dmma_rc = false;   // ... its register-carried variant (128-site blocks): large alignments, compile-time S
  int rc_stagger = 1;     // anti-lockstep barriers between the warps of one SM sub-partition, see kernels_dmma_rc.cuh
  double* d_staged = nullptr;  // P matrices of the current evaluation in stage layout and consumption order
  size_t staged_bytes = 0;
  bool s2_tiled = false;  // 2-state family on a large alignment: tile-interleaved partials + prune_s2t_kernel
  int s2t_slots = 3;      // its shared-memory stack slots per tile
  int s2t_minb = 3;       // resident blocks per SM it is launched for (2: 4-stage image ring, up to 4 slots; 3: 3-stage ring,
                          // 3 slots).  Measured on C4 (profiles/README.md): V = 2 with 3 blocks 6.17 ms, V = 1 with 3 blocks
                          // 6.56 ms, V = 1 with 2 blocks and 4 slots 7.10 ms, V = 2 with 2 blocks 7.84 ms, 4 blocks 7.0 ms
  int s2t_v = 2;          // tiles per warp (2: 4 warps per block, each handling two 32-site tiles; 1: 8 warps, one tile each)
  bool s2t_bulk = false;  // stored partials leave through staging tiles + bulk-async copies instead of plain stores
  bool s2t_prefetch = true;  // stored siblings of a carried child arrive through cp.async two ops ahead (dirty paths)
  bool s2t_small_recs = true;  // nodes whose children are tips / cherries are kept as records, not stored
  S2TImage* d_images = nullptr;  // op images of the current evaluation (s2t_image_kernel)
  int s2_vec = 1;  // sites per thread of the 2-state kernel on large alignments
  int s2_minb = 3; // its __launch_bounds__ min blocks per SM (experiment knob)
  bool s2_stream_stores = true;  // st.global.cs for partials the walk never reads back (10.67 vs 11.0 ms on C4)
  void* d_codes = nullptr;
  double* d_weights = nullptr;
  double* d_amb = nullptr;
  double* d_pi = nullptr;
  // P matrices
  double* d_pmats = nullptr;
  int pmat_cap = 0;
  // partial buffers
  std::vector<Buffer> buffers;
  std::vector<int> free_buffers;
  size_t buffer_bytes = 0;
  std::vector<Snapshot> snaps;
  std::vector<int> free_snaps;
  std::vector<CherryRec> recs;
  std::vector<int> free_recs;
  double* d_pmats_lib = nullptr;
  int lib_cap = 0;  // records the library pool can hold
  // staging
  // one pinned block + its device mirror per evaluation: [ops][ranges][pi], uploaded with ONE copy
  unsigned char* h_stage = nullptr;
  unsigned char* d_stage = nullptr;
  size_t stage_cap = 0;
  int images_cap = 0;  // op images (tiled 2-state kernel), in ops
  cudaEvent_t ev_scratch = nullptr;  // the last host -> device copy out of h_scratch has finished
  bool timing = true;                // record the per-evaluation timing events (the native chain switches them off)
  bool results_mapped = false;       // h_results is mapped: the root kernel writes lnL straight into host memory
  double* d_block_sums = nullptr;
  unsigned* d_tickets = nullptr;
  double* d_results = nullptr;
  double* h_results = nullptr;
  double* d_root_dot = nullptr;
  int32_t* d_root_exp = nullptr;
  int out_cap = 0, max_blocks = 0;
  int last_n_out = 0;
  // scratch for pmat builds
  void* d_scratch = nullptr;
  void* h_scratch = nullptr;
  size_t scratch_cap = 0;
  // L2 flush
  void* d_flush = nullptr;
  size_t flush_bytes = 0;
  // NCCL (set-up, and the all-reduce of batches with more than CB_MB_OUTS results) + the fused all-reduce's mailboxes
  ncclComm_t comm = nullptr;
  int n_ranks = 1, rank = 0;
  bool fused_allreduce = false;
  Mail* d_mailbox = nullptr;           // [2][CB_MB_OUTS][n_ranks], written by the peers
  Mail** d_peer_mailbox = nullptr;     // device array of every rank's mailbox
  std::vector<void*> peer_opened;      // IPC mappings to close
  int32_t* d_comm_error = nullptr;
  unsigned long long epoch = 0;
  // plans of full evaluations, cached per topology; scratch plan of dirty-path evaluations
  std::vector<EvalPlan> plans;
  EvalPlan scratch_plan;
  uint64_t plan_clock = 0, plan_builds = 0;
  bool no_plan_cache = false;
  std::vector<int> work_new_bufs, work_new_nodes, work_cherry_nodes;
  cudaEvent_t ev_main0 = nullptr, ev_main1 = nullptr;  // around the pruning launches proper (without pre-passes)
  double host_us[6] = {0, 0, 0, 0, 0, 0};  // accumulated per-evaluation host time: plan, fill, upload+launch, sync, bookkeeping, calls
  int64_t last_bytes_written = 0, last_bytes_read = 0;
  int32_t last_counts[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  // stats
  int64_t launches = 0, h2d = 0, d2h = 0, dev_bytes = 0, max_dev_bytes = 0;
  bool timing_valid = false;
};

static void dev_account(int device, int64_t delta);
static int dev_alloc(cb_ctx* c, void** p, size_t bytes) {
  // CYBAYES_MAX_DEVICE_BYTES caps what one context may hold (a share of a GPU; also how the tests reach this path)
  cudaError_t e = (c->max_dev_bytes > 0 && c->dev_bytes + (int64_t)bytes > c->max_dev_bytes) ? cudaErrorMemoryAllocation
                                                                                              : cudaMalloc(p, bytes);
  if (e == cudaErrorMemoryAllocation) {
    cudaGetLastError();  // not sticky: clear it
    size_t fr = 0, tot = 0;
    cudaMemGetInfo(&fr, &tot);
    return fail("out of device memory: %.2f GB requested with %.2f GB in use by this context (%.2f GB free on the GPU%s). "
                "The partial cache of this alignment needs about %.1f GB: shard the patterns over more GPUs (CYBAYES_SHARD=1 "
                "under torchrun) or evaluate without keeping the cache",
                bytes / 1e9, c->dev_bytes / 1e9, fr / 1e9, c->max_dev_bytes > 0 ? ", context capped by CYBAYES_MAX_DEVICE_BYTES" : "",
                (double)c->buffer_bytes * std::max(0, c->n_taxa - 2) / 1e9);
  }
  if (e != cudaSuccess) return fail("%s:%d cudaMalloc: %s", __FILE__, __LINE__, cudaGetErrorString(e));
  c->dev_bytes += (int64_t)bytes;
  dev_account(c->device, (int64_t)bytes);
  return 0;
}
static void dev_free(cb_ctx* c, void* p, size_t bytes) {
  if (p) {
    cudaFree(p);
    c->dev_bytes -= (int64_t)bytes;
    dev_account(c->device, -(int64_t)bytes);
  }
}

extern "C" const char* cb_last_error(void) { return g_err.c_str(); }
extern "C" int cb_version(void) { return 100; }
extern "C" int cb_device_count(int* out) {
  REQUIRE(out, "null argument");
  CU(cudaGetDeviceCount(out));
  return 0;
}

static int create_impl(int device, cb_ctx** out);
extern "C" int cb_create(int device, cb_ctx** out) {
  return guarded([&] { return create_impl(device, out); });
}
static int create_impl(int device, cb_ctx** out) {
  REQUIRE(out, "null argument");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail("no CUDA device available (%s); cybayes_b200 has no CPU fallback", cudaGetErrorString(e));
  REQUIRE(device >= 0 && device < n, "device %d out of range (have %d)", device, n);
  CU(cudaSetDevice(device));
  cb_ctx* c = new cb_ctx();
  c->device = device;
  CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CU(cudaEventCreate(&c->ev0));
  CU(cudaEventCreate(&c->ev1));
  CU(cudaEventCreateWithFlags(&c->ev_stage, cudaEventDisableTiming));
  CU(cudaEventCreate(&c->ev_mark[0]));
  CU(cudaEventCreate(&c->ev_mark[1]));
  CU(cudaEventCreateWithFlags(&c->ev_scratch, cudaEventDisableTiming));
  CU(cudaEventCreate(&c->ev_main0));
  CU(cudaEventCreate(&c->ev_main1));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  if (const char* v = getenv("CYBAYES_S2_V")) c->s2_vec = (atoi(v) == 2) ? 2 : 1;
  if (const char* v = getenv("CYBAYES_S2_MINB")) c->s2_minb = (atoi(v) == 4) ? 4 : 3;
  if (getenv("CYBAYES_S2_NO_CS")) c->s2_stream_stores = false;
  if (const char* v = getenv("CYBAYES_S2T_MINB")) c->s2t_minb = std::max(2, std::min(4, atoi(v)));
  if (const char* v = getenv("CYBAYES_S2T_V")) c->s2t_v = atoi(v) == 2 ? 2 : 1;
  if (c->s2t_minb == 4) c->s2t_v = 1;
  if (getenv("CYBAYES_S2T_BULK")) c->s2t_bulk = atoi(getenv("CYBAYES_S2T_BULK")) != 0;
  if (getenv("CYBAYES_S2T_PREFETCH")) c->s2t_prefetch = atoi(getenv("CYBAYES_S2T_PREFETCH")) != 0;
  if (getenv("CYBAYES_S2T_SMALL_RECS")) c->s2t_small_recs = atoi(getenv("CYBAYES_S2T_SMALL_RECS")) != 0;
  c->s2t_slots = c->s2t_minb == 4 ? 2 : c->s2t_minb == 3 ? 3 : 4;
  if (const char* v = getenv("CYBAYES_S2T_SLOTS")) c->s2t_slots = std::max(0, std::min(8, atoi(v)));
  if (getenv("CYBAYES_NO_PLAN_CACHE")) c->no_plan_cache = true;
  if (const char* v = getenv("CYBAYES_MAX_DEVICE_BYTES")) c->max_dev_bytes = atoll(v);
#define CB_S2T_ATTR(CC, MB, VV) CU(cudaFuncSetAttribute(prune_s2t_kernel<CC, MB, VV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024))
  CB_S2T_ATTR(4, 2, 1); CB_S2T_ATTR(4, 3, 1); CB_S2T_ATTR(1, 2, 1); CB_S2T_ATTR(1, 3, 1);   // + 384 B static each
  CB_S2T_ATTR(4, 2, 2); CB_S2T_ATTR(1, 2, 2); CB_S2T_ATTR(4, 3, 2); CB_S2T_ATTR(1, 3, 2); CB_S2T_ATTR(4, 4, 1); CB_S2T_ATTR(1, 4, 1);
#undef CB_S2T_ATTR
  CU(cudaFuncSetAttribute(prune_general_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
#define CB_DMMA_ATTR(SS) CU(cudaFuncSetAttribute(prune_dmma_kernel<SS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024))
  CB_DMMA_ATTR(0); CB_DMMA_ATTR(32); CB_DMMA_ATTR(40); CB_DMMA_ATTR(47); CB_DMMA_ATTR(48); CB_DMMA_ATTR(56); CB_DMMA_ATTR(64);
#undef CB_DMMA_ATTR
#define CB_RC_ATTR(SS)                                                                                                          \
  CU(cudaFuncSetAttribute(prune_dmma_rc_kernel<SS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RcCfg<SS>::SMEM)); \
  CU(cudaFuncSetAttribute(prune_dmma_rc_kernel<SS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RcCfg<SS>::SMEM))
  CB_RC_ATTR(16); CB_RC_ATTR(24); CB_RC_ATTR(32); CB_RC_ATTR(40); CB_RC_ATTR(48); CB_RC_ATTR(56); CB_RC_ATTR(64);
#undef CB_RC_ATTR
  if (const char* v = getenv("CYBAYES_RC_STAGGER")) c->rc_stagger = atoi(v) != 0;
  *out = c;
  return 0;
}

static void free_alignment(cb_ctx* c) {
  c->plans.clear();
  if (c->d_images) dev_free(c, c->d_images, (size_t)c->images_cap * sizeof(S2TImage));
  c->d_images = nullptr;
  c->images_cap = 0;
  for (auto& b : c->buffers) dev_free(c, b.data, c->buffer_bytes);
  c->buffers.clear();
  c->free_buffers.clear();
  c->snaps.clear();
  c->free_snaps.clear();
  c->recs.clear();
  c->free_recs.clear();
  if (c->d_pmats_lib) dev_free(c, c->d_pmats_lib, (size_t)c->lib_cap * 2 * c->n_cats * c->n_states * c->n_states * 8);
  c->d_pmats_lib = nullptr;
  c->lib_cap = 0;
  if (c->d_codes) dev_free(c, c->d_codes, (size_t)c->n_taxa * c->P * c->code_bytes);
  if (c->d_weights) dev_free(c, c->d_weights, (size_t)c->P * 8);
  if (c->d_amb) dev_free(c, c->d_amb, (size_t)std::max(1, c->n_amb) * c->n_states * 8);
  if (c->d_pi) dev_free(c, c->d_pi, (size_t)c->n_states * 8);
  if (c->d_pmats) dev_free(c, c->d_pmats, (size_t)c->pmat_cap * c->n_states * c->n_states * 8);
  if (c->d_staged) dev_free(c, c->d_staged, c->staged_bytes);
  c->d_staged = nullptr;
  c->staged_bytes = 0;
  c->d_codes = nullptr;
  c->d_weights = c->d_amb = c->d_pi = c->d_pmats = nullptr;
  c->pmat_cap = 0;
  if (c->d_block_sums) dev_free(c, c->d_block_sums, (size_t)c->out_cap * c->max_blocks * 8);
  if (c->d_tickets) dev_free(c, c->d_tickets, (size_t)c->out_cap * 4);
  if (c->d_results) dev_free(c, c->d_results, (size_t)c->out_cap * 8);
  if (c->d_root_dot) dev_free(c, c->d_root_dot, (size_t)c->out_cap * c->n_cats * c->P * 8);
  if (c->d_root_exp) dev_free(c, c->d_root_exp, (size_t)c->out_cap * c->n_cats * c->P * 4);
  if (c->h_results) cudaFreeHost(c->h_results);
  c->d_block_sums = c->d_results = c->d_root_dot = nullptr;
  c->d_tickets = nullptr;
  c->d_root_exp = nullptr;
  c->h_results = nullptr;
  c->out_cap = 0;
}

extern "C" int cb_destroy(cb_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (void* ptr : c->peer_opened) cudaIpcCloseMemHandle(ptr);
  if (c->d_mailbox) cudaFree(c->d_mailbox);
  if (c->d_peer_mailbox) cudaFree(c->d_peer_mailbox);
  if (c->d_comm_error) cudaFree(c->d_comm_error);
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  free_alignment(c);
  if (c->d_stage) dev_free(c, c->d_stage, c->stage_cap);
  if (c->h_stage) cudaFreeHost(c->h_stage);
  if (c->ev_scratch) cudaEventDestroy(c->ev_scratch);
  if (c->d_scratch) dev_free(c, c->d_scratch, c->scratch_cap);
  if (c->h_scratch) cudaFreeHost(c->h_scratch);
  if (c->d_flush) dev_free(c, c->d_flush, c->flush_bytes);
  cudaEventDestroy(c->ev0);
  cudaEventDestroy(c->ev1);
  cudaEventDestroy(c->ev_stage);
  cudaEventDestroy(c->ev_mark[0]);
  cudaEventDestroy(c->ev_mark[1]);
  cudaEventDestroy(c->ev_main0);
  cudaEventDestroy(c->ev_main1);
  cudaStreamDestroy(c->stream);
  delete c;
  return 0;
}

// --------------------------------------------------------------------------------- NCCL
extern "C" int cb_nccl_unique_id(void* id128_out) {
  REQUIRE(id128_out, "null argument");
  if (load_nccl()) return 1;
  NcclId id;
  int r = g_nccl.GetUniqueId(&id);
  REQUIRE(r == 0, "ncclGetUniqueId: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error");
  memcpy(id128_out, &id, sizeof id);
  return 0;
}
extern "C" int cb_comm_init(cb_ctx* c, const void* id128, int rank, int n_ranks) {
  REQUIRE(c && id128, "null argument");
  REQUIRE(n_ranks >= 1 && rank >= 0 && rank < n_ranks, "bad rank %d of %d", rank, n_ranks);
  if (load_nccl()) return 1;
  CU(cudaSetDevice(c->device));
  NcclId id;
  memcpy(&id, id128, sizeof id);
  int r = g_nccl.CommInitRank(&c->comm, n_ranks, id, rank);
  REQUIRE(r == 0, "ncclCommInitRank: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error");
  c->n_ranks = n_ranks;
  c->rank = rank;
  // Fused scalar all-reduce over NVLink peer memory: every rank owns a mailbox, opens the others' through CUDA IPC
  // (handles exchanged once with ncclAllGather) and from then on the root kernel delivers and collects the shard sums
  // itself.  Any failure here just leaves the NCCL all-reduce in place.
  if (n_ranks > 1 && n_ranks <= 32 && g_nccl.AllGather && !getenv("CYBAYES_NO_FUSED_ALLREDUCE")) {
    const size_t mb_bytes = (size_t)2 * CB_MB_OUTS * n_ranks * sizeof(Mail);
    cudaIpcMemHandle_t* d_handles = nullptr;
    std::vector<cudaIpcMemHandle_t> handles(n_ranks);
    bool ok = cudaMalloc((void**)&c->d_mailbox, mb_bytes) == cudaSuccess && cudaMemset(c->d_mailbox, 0, mb_bytes) == cudaSuccess &&
              cudaMalloc((void**)&d_handles, sizeof(cudaIpcMemHandle_t) * n_ranks) == cudaSuccess &&
              cudaMalloc((void**)&c->d_peer_mailbox, sizeof(Mail*) * n_ranks) == cudaSuccess &&
              cudaMalloc((void**)&c->d_comm_error, 4) == cudaSuccess && cudaMemset(c->d_comm_error, 0, 4) == cudaSuccess;
    if (ok) ok = cudaIpcGetMemHandle(&handles[rank], c->d_mailbox) == cudaSuccess &&
                 cudaMemcpy(d_handles + rank, &handles[rank], sizeof(cudaIpcMemHandle_t), cudaMemcpyHostToDevice) == cudaSuccess;
    // every rank must take part in the collective, whatever happened locally
    const int gr = g_nccl.AllGather(ok ? (const void*)(d_handles + rank) : (const void*)d_handles, d_handles, sizeof(cudaIpcMemHandle_t),
                                    NCCL_INT8, c->comm, c->stream);
    ok = ok && gr == 0 && cudaStreamSynchronize(c->stream) == cudaSuccess &&
         cudaMemcpy(handles.data(), d_handles, sizeof(cudaIpcMemHandle_t) * n_ranks, cudaMemcpyDeviceToHost) == cudaSuccess;
    std::vector<Mail*> peers(n_ranks, nullptr);
    for (int q = 0; ok && q < n_ranks; ++q) {
      if (q == rank) { peers[q] = c->d_mailbox; continue; }
      void* ptr = nullptr;
      ok = cudaIpcOpenMemHandle(&ptr, handles[q], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
      if (ok) { peers[q] = (Mail*)ptr; c->peer_opened.push_back(ptr); }
    }
    if (ok) ok = cudaMemcpy(c->d_peer_mailbox, peers.data(), sizeof(Mail*) * n_ranks, cudaMemcpyHostToDevice) == cudaSuccess;
    if (d_handles) cudaFree(d_handles);
    // all ranks agree on the outcome (one rank without peer access must not leave the others waiting in a kernel)
    double* d_flag = nullptr;
    double flag = ok ? 0.0 : 1.0;
    if (cudaMalloc((void**)&d_flag, 8) == cudaSuccess) {
      cudaMemcpy(d_flag, &flag, 8, cudaMemcpyHostToDevice);
      g_nccl.AllReduce(d_flag, d_flag, 1, NCCL_DOUBLE, NCCL_SUM, c->comm, c->stream);
      cudaStreamSynchronize(c->stream);
      cudaMemcpy(&flag, d_flag, 8, cudaMemcpyDeviceToHost);
      cudaFree(d_flag);
    } else {
      flag = 1.0;
    }
    cudaGetLastError();
    c->fused_allreduce = (flag == 0.0);
  }
  return 0;
}

// ---------------------------------------------------------------------------- alignment
static int ensure_scratch(cb_ctx* c, size_t bytes) {
  if (bytes <= c->scratch_cap) return 0;
  size_t cap = std::max(bytes, c->scratch_cap * 2);
  cap = (cap + 4095) & ~(size_t)4095;
  CU(cudaStreamSynchronize(c->stream));
  if (c->d_scratch) dev_free(c, c->d_scratch, c->scratch_cap);
  if (c->h_scratch) cudaFreeHost(c->h_scratch);
  c->d_scratch = c->h_scratch = nullptr;
  c->scratch_cap = 0;
  if (dev_alloc(c, &c->d_scratch, cap)) return 1;
  CU(cudaMallocHost(&c->h_scratch, cap));
  c->scratch_cap = cap;
  return 0;
}

static int set_tips_impl(cb_ctx* c, int n_taxa, int64_t n_sites, int n_states, int n_cats, const void* codes,
                         int code_bytes, const double* amb_sets, int n_amb, const double* weights);
extern "C" int cb_set_tips(cb_ctx* c, int n_taxa, int64_t n_sites, int n_states, int n_cats,
                           const void* codes, int code_bytes, const double* amb_sets, int n_amb,
                           const double* weights) {
  return guarded([&] { return set_tips_impl(c, n_taxa, n_sites, n_states, n_cats, codes, code_bytes, amb_sets, n_amb, weights); });
}
static int set_tips_impl(cb_ctx* c, int n_taxa, int64_t n_sites, int n_states, int n_cats, const void* codes,
                         int code_bytes, const double* amb_sets, int n_amb, const double* weights) {
  REQUIRE(c && codes, "null argument");
  REQUIRE(n_taxa >= 2 && n_sites >= 1 && n_states >= 2, "bad alignment shape %d x %lld x %d", n_taxa,
          (long long)n_sites, n_states);
  REQUIRE(n_cats >= 1 && n_cats <= CB_MAX_CATS, "n_cats must be 1..%d", CB_MAX_CATS);
  REQUIRE(code_bytes == 1 || code_bytes == 2, "code_bytes must be 1 or 2");
  REQUIRE(n_amb >= 1 && amb_sets, "amb_sets must at least hold the all-ones set");
  REQUIRE(n_states + n_amb <= (code_bytes == 1 ? 256 : 65536), "codes do not fit code_bytes");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  free_alignment(c);
  c->n_taxa = n_taxa;
  c->n_sites = n_sites;
  c->n_states = n_states;
  c->n_cats = n_cats;
  c->code_bytes = code_bytes;
  c->n_amb = n_amb;
  c->P = (n_sites + 63) / 64 * 64;
  c->family_s2 = (n_states == 2 && (n_cats == 4 || n_cats == 1));
  {
    // large binary alignments use the tiled kernel (kernels_s2t.cuh); CYBAYES_S2_TILED=1/0 forces it on / off (tests)
    const char* v = getenv("CYBAYES_S2_TILED");
    c->s2_tiled = c->family_s2 && code_bytes == 1 && (v ? atoi(v) != 0 : c->P >= S2_TILED_MIN_SITES);
  }
  c->use_dmma = !c->family_s2 && n_states >= 32 && n_states <= 64 && !getenv("CYBAYES_NO_DMMA");
  {
    // The kernel is fixed per alignment (never per schedule), so every evaluation of an alignment sums in one order.
    // The register-carried variant (always with the walk schedule, cut into parallel subtrees when there are few site
    // tiles) wins from ~1k patterns up: 0.37 vs 0.54 ms at 2048 x 94 taxa, 10.0 vs 18.5 ms at 16384 x 512 taxa (S = 64).
    // CYBAYES_DMMA_RC=1/0 forces it on / off, CYBAYES_RC_MIN_SITES moves the threshold.
    const char* v = getenv("CYBAYES_DMMA_RC");
    const char* m = getenv("CYBAYES_RC_MIN_SITES");
    const char* ms = getenv("CYBAYES_RC_MIN_STATES");
    const bool states_ok = !c->family_s2 && n_states >= (ms ? std::max(9, atoi(ms)) : DMMA_RC_MIN_STATES) && n_states <= 64 &&
                           !getenv("CYBAYES_NO_DMMA");
    c->dmma_rc = states_ok && (v ? atoi(v) != 0 : c->P >= (m ? atoll(m) : DMMA_RC_MIN_SITES));
  }
  const int64_t P = c->P;
  if (dev_alloc(c, &c->d_codes, (size_t)n_taxa * P * code_bytes)) return 1;
  // padding sites carry the all-ones code (a no-op factor) and weight 0
  if (code_bytes == 1) {
    CU(cudaMemsetAsync(c->d_codes, n_states, (size_t)n_taxa * P, c->stream));
  } else {
    std::vector<uint16_t> fill((size_t)P, (uint16_t)n_states);
    for (int t = 0; t < n_taxa; ++t)
      CU(cudaMemcpyAsync((char*)c->d_codes + (size_t)t * P * 2, fill.data(), (size_t)P * 2, cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  CU(cudaMemcpy2DAsync(c->d_codes, (size_t)P * code_bytes, codes, (size_t)n_sites * code_bytes,
                       (size_t)n_sites * code_bytes, n_taxa, cudaMemcpyHostToDevice, c->stream));
  c->h2d += (int64_t)n_taxa * n_sites * code_bytes;
  if (dev_alloc(c, (void**)&c->d_weights, (size_t)P * 8)) return 1;
  CU(cudaMemsetAsync(c->d_weights, 0, (size_t)P * 8, c->stream));
  {
    std::vector<double> w((size_t)n_sites, 1.0);
    if (weights) memcpy(w.data(), weights, (size_t)n_sites * 8);
    CU(cudaMemcpyAsync(c->d_weights, w.data(), (size_t)n_sites * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->h2d += n_sites * 8;
  }
  if (dev_alloc(c, (void**)&c->d_amb, (size_t)n_amb * n_states * 8)) return 1;
  CU(cudaMemcpyAsync(c->d_amb, amb_sets, (size_t)n_amb * n_states * 8, cudaMemcpyHostToDevice, c->stream));
  if (dev_alloc(c, (void**)&c->d_pi, (size_t)n_states * 8)) return 1;
  CU(cudaStreamSynchronize(c->stream));
  const size_t scale_ints = c->family_s2 ? (size_t)P : (size_t)n_cats * P;
  c->buffer_bytes = (size_t)n_cats * n_states * P * 8 + scale_ints * 4;
  return 0;
}

// ------------------------------------------------------------------------ P matrices
extern "C" int cb_pmat_reserve(cb_ctx* c, int n_slots) {
  REQUIRE(c && c->n_states > 0, "cb_set_tips must come first");
  if (n_slots <= c->pmat_cap) return 0;
  CU(cudaSetDevice(c->device));
  int cap = std::max(n_slots, std::max(1024, c->pmat_cap * 2));
  const size_t mat = (size_t)c->n_states * c->n_states * 8;
  double* nd = nullptr;
  if (dev_alloc(c, (void**)&nd, (size_t)cap * mat)) return 1;
  if (c->d_pmats) {
    CU(cudaMemcpyAsync(nd, c->d_pmats, (size_t)c->pmat_cap * mat, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    dev_free(c, c->d_pmats, (size_t)c->pmat_cap * mat);
  }
  c->d_pmats = nd;
  c->pmat_cap = cap;
  return 0;
}

static int check_slots(cb_ctx* c, int count, const int32_t* slots) {
  REQUIRE(c && slots && count >= 0, "bad argument");
  for (int i = 0; i < count; ++i)
    REQUIRE(slots[i] >= 0 && slots[i] < c->pmat_cap, "P slot %d out of range (reserved %d)", slots[i], c->pmat_cap);
  return 0;
}

extern "C" int cb_pmat_upload(cb_ctx* c, int count, const int32_t* slots, const double* mats) {
  if (check_slots(c, count, slots)) return 1;
  REQUIRE(mats, "null argument");
  CU(cudaSetDevice(c->device));
  const size_t mat = (size_t)c->n_states * c->n_states * 8;
  if (ensure_scratch(c, (size_t)count * mat)) return 1;
  CU(cudaEventSynchronize(c->ev_scratch));  // the previous copy out of the pinned scratch has finished
  memcpy(c->h_scratch, mats, (size_t)count * mat);
  int i = 0;
  while (i < count) {  // coalesce runs of consecutive slots into one copy
    int j = i + 1;
    while (j < count && slots[j] == slots[j - 1] + 1) ++j;
    CU(cudaMemcpyAsync(c->d_pmats + (size_t)slots[i] * c->n_states * c->n_states, (char*)c->h_scratch + (size_t)i * mat,
                       (size_t)(j - i) * mat, cudaMemcpyHostToDevice, c->stream));
    i = j;
  }
  CU(cudaEventRecord(c->ev_scratch, c->stream));
  c->h2d += (int64_t)count * mat;
  return 0;
}

extern "C" int cb_pmat_download(cb_ctx* c, int count, const int32_t* slots, double* out) {
  if (check_slots(c, count, slots)) return 1;
  REQUIRE(out, "null argument");
  CU(cudaSetDevice(c->device));
  const size_t mat = (size_t)c->n_states * c->n_states * 8;
  for (int i = 0; i < count; ++i)
    CU(cudaMemcpyAsync((char*)out + (size_t)i * mat, c->d_pmats + (size_t)slots[i] * c->n_states * c->n_states, mat,
                       cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  c->d2h += (int64_t)count * mat;
  return 0;
}

extern "C" int cb_pmat_build(cb_ctx* c, int model, const double* pi, double beta, const double* gtr,
                             int count, const int32_t* slots, const double* d, const double* x) {
  if (check_slots(c, count, slots)) return 1;
  REQUIRE(d, "null argument");
  REQUIRE(model >= CB_MODEL_JC && model <= CB_MODEL_GTR_EIG, "unknown model %d", model);
  REQUIRE(model == CB_MODEL_JC || pi, "pi required");
  REQUIRE(model != CB_MODEL_GTR_EIG || gtr, "GTR eigensystem required");
  REQUIRE(model != CB_MODEL_F81_BINARY || c->n_states == 2, "binary F81 needs 2 states");
  if (count == 0) return 0;
  CU(cudaSetDevice(c->device));
  const int S = c->n_states;
  const size_t n_gtr = (model == CB_MODEL_GTR_EIG) ? (size_t)S + 2 * (size_t)S * S : 0;
  // scratch layout: pi[S] | gtr[n_gtr] | d[count] | x[count] | slots[count] (int32)
  const size_t doubles = (size_t)S + n_gtr + 2 * (size_t)count;
  const size_t bytes = doubles * 8 + (size_t)count * 4;
  if (ensure_scratch(c, bytes)) return 1;
  CU(cudaEventSynchronize(c->ev_scratch));  // the previous copy out of the pinned scratch has finished
  double* h = (double*)c->h_scratch;
  if (pi) memcpy(h, pi, (size_t)S * 8); else memset(h, 0, (size_t)S * 8);
  if (n_gtr) memcpy(h + S, gtr, n_gtr * 8);
  memcpy(h + S + n_gtr, d, (size_t)count * 8);
  if (x) memcpy(h + S + n_gtr + count, x, (size_t)count * 8);
  memcpy(h + doubles, slots, (size_t)count * 4);
  CU(cudaMemcpyAsync(c->d_scratch, c->h_scratch, bytes, cudaMemcpyHostToDevice, c->stream));
  CU(cudaEventRecord(c->ev_scratch, c->stream));
  c->h2d += (int64_t)bytes;
  const double* dd = (const double*)c->d_scratch;
  const int threads = (S * S >= 256) ? 256 : ((S * S + 31) / 32 * 32);
  pmat_build_kernel<<<count, threads, (size_t)S * 8, c->stream>>>(
      model, S, dd, beta, n_gtr ? dd + S : nullptr, count, (const int32_t*)(dd + doubles), dd + S + n_gtr,
      x ? dd + S + n_gtr + count : nullptr, c->d_pmats);
  CU(cudaGetLastError());
  c->launches += 1;
  return 0;
}

// ------------------------------------------------------------------------ buffers/snapshots
static int buffer_acquire(cb_ctx* c, int* out) {
  if (!c->free_buffers.empty()) {
    *out = c->free_buffers.back();
    c->free_buffers.pop_back();
  } else {
    Buffer b;
    void* p = nullptr;
    if (dev_alloc(c, &p, c->buffer_bytes)) return 1;
    b.data = (double*)p;
    b.scale = (int32_t*)(b.data + (size_t)c->n_cats * c->n_states * c->P);
    c->buffers.push_back(b);
    *out = (int)c->buffers.size() - 1;
  }
  c->buffers[*out].refs = 1;
  return 0;
}
static void buffer_release(cb_ctx* c, int b) {
  if (b < 0) return;
  if (--c->buffers[b].refs == 0) c->free_buffers.push_back(b);
}
static int rec_acquire(cb_ctx* c, int tip0, int tip1, int* out) {
  if (!c->free_recs.empty()) {
    *out = c->free_recs.back();
    c->free_recs.pop_back();
  } else {
    c->recs.emplace_back();
    *out = (int)c->recs.size() - 1;
  }
  c->recs[*out].tip[0] = tip0;
  c->recs[*out].tip[1] = tip1;
  c->recs[*out].refs = 1;
  return 0;
}
static void rec_release(cb_ctx* c, int r) {
  if (r < 0) return;
  if (--c->recs[r].refs == 0) c->free_recs.push_back(r);
}
// the library's P pool must hold every record that exists (old contents are kept when it grows)
static int ensure_lib_pool(cb_ctx* c) {
  const int need = (int)c->recs.size();
  if (need <= c->lib_cap) return 0;
  const int cap = std::max(need, std::max(1024, c->lib_cap * 2));
  const size_t per = (size_t)2 * c->n_cats * c->n_states * c->n_states * 8;
  double* nd = nullptr;
  if (dev_alloc(c, (void**)&nd, (size_t)cap * per)) return 1;
  if (c->d_pmats_lib) {
    CU(cudaMemcpyAsync(nd, c->d_pmats_lib, (size_t)c->lib_cap * per, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    dev_free(c, c->d_pmats_lib, (size_t)c->lib_cap * per);
  }
  c->d_pmats_lib = nd;
  c->lib_cap = cap;
  return 0;
}
static bool snapshot_valid(cb_ctx* c, int s) {
  return s >= 0 && s < (int)c->snaps.size() && c->snaps[s].refs > 0;
}
extern "C" int cb_snapshot_retain(cb_ctx* c, int s) {
  REQUIRE(c && snapshot_valid(c, s), "invalid snapshot %d", s);
  c->snaps[s].refs++;
  return 0;
}
extern "C" int cb_snapshot_release(cb_ctx* c, int s) {
  REQUIRE(c && snapshot_valid(c, s), "invalid snapshot %d", s);
  if (--c->snaps[s].refs == 0) {
    for (int32_t b : c->snaps[s].buf_of_node) buffer_release(c, b);
    for (int32_t r : c->snaps[s].cherry_of_node) rec_release(c, r);
    c->snaps[s].buf_of_node.clear();
    c->snaps[s].cherry_of_node.clear();
    c->free_snaps.push_back(s);
  }
  return 0;
}

static int snapshot_read_impl(cb_ctx* c, int s, int node, double* out, int32_t* scale_out);
extern "C" int cb_snapshot_read(cb_ctx* c, int s, int node, double* out, int32_t* scale_out) {
  return guarded([&] { return snapshot_read_impl(c, s, node, out, scale_out); });
}
static int materialize_cherry(cb_ctx* c, const Snapshot& sn, int rec, int* buf_out);
static int snapshot_read_impl(cb_ctx* c, int s, int node, double* out, int32_t* scale_out) {
  REQUIRE(c && out && snapshot_valid(c, s), "invalid snapshot %d", s);
  const Snapshot& sn = c->snaps[s];
  REQUIRE(node >= 0 && node < (int)sn.buf_of_node.size(), "node %d is not in snapshot %d", node, s);
  CU(cudaSetDevice(c->device));
  int bidx = sn.buf_of_node[node], tmp_buf = -1;
  if (bidx < 0 && node < (int)sn.cherry_of_node.size() && sn.cherry_of_node[node] >= 0) {
    // a folded cherry has no stored partial: compute it now, from the P copies the snapshot keeps
    if (materialize_cherry(c, sn, sn.cherry_of_node[node], &tmp_buf)) return 1;
    bidx = tmp_buf;
  }
  REQUIRE(bidx >= 0, "node %d is not in snapshot %d", node, s);
  const Buffer& b = c->buffers[bidx];
  const int C = c->n_cats, S = c->n_states;
  const int64_t P = c->P, n = c->n_sites;
  std::vector<double> tmp((size_t)C * S * P);
  const size_t n_scale = c->family_s2 ? (size_t)P : (size_t)C * P;
  std::vector<int32_t> sc(n_scale);
  if (c->s2_tiled) {
    // tile-interleaved layout (kernels_s2t.cuh): per 32 sites, 2C rows of 32 doubles then 32 exponents
    std::vector<unsigned char> raw(c->buffer_bytes);
    CU(cudaMemcpyAsync(raw.data(), b.data, raw.size(), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    const size_t TB = (size_t)s2t_tile_bytes(C);
    for (int64_t t = 0; t < P / S2T_W; ++t) {
      const double* rows = reinterpret_cast<const double*>(raw.data() + (size_t)t * TB);
      const int32_t* ex = reinterpret_cast<const int32_t*>(rows + (size_t)2 * C * S2T_W);
      for (int r = 0; r < 2 * C; ++r)
        for (int l = 0; l < S2T_W; ++l) tmp[(size_t)r * P + t * S2T_W + l] = rows[(size_t)r * S2T_W + l];
      for (int l = 0; l < S2T_W; ++l) sc[(size_t)t * S2T_W + l] = ex[l];
    }
  } else {
    CU(cudaMemcpyAsync(tmp.data(), b.data, tmp.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(sc.data(), b.scale, n_scale * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  c->d2h += (int64_t)tmp.size() * 8 + (int64_t)n_scale * 4;
  for (int k = 0; k < C; ++k)
    for (int i = 0; i < S; ++i)
      for (int64_t p = 0; p < n; ++p) {
        const int e = c->family_s2 ? sc[p] : sc[(size_t)k * P + p];
        double v = tmp[((size_t)k * S + i) * P + p];
        if (!scale_out) v = ldexp(v, e);
        out[((size_t)k * S + i) * n + p] = v;
      }
  if (scale_out) {
    // one exponent per site: categories of the general family are brought to their max
    for (int64_t p = 0; p < n; ++p) {
      if (c->family_s2) {
        scale_out[p] = sc[p];
      } else {
        int emax = INT_MIN;
        for (int k = 0; k < C; ++k) emax = std::max(emax, sc[(size_t)k * P + p]);
        scale_out[p] = emax;
        for (int k = 0; k < C; ++k)
          for (int i = 0; i < S; ++i) {
            double& v = out[((size_t)k * S + i) * n + p];
            v = ldexp(v, sc[(size_t)k * P + p] - emax);
          }
      }
    }
  }
  if (tmp_buf >= 0) buffer_release(c, tmp_buf);
  return 0;
}

// ---------------------------------------------------------------------------- evaluation
static int ensure_staging(cb_ctx* c, int n_ops, int n_ranges, int n_out) {
  const size_t need = (size_t)n_ops * sizeof(OpDesc) + (size_t)n_ranges * sizeof(RangeDesc) + (size_t)c->n_states * 8;
  if (need > c->stage_cap) {
    const size_t cap = std::max(need, std::max((size_t)64 << 10, c->stage_cap * 2));
    CU(cudaStreamSynchronize(c->stream));
    if (c->d_stage) dev_free(c, c->d_stage, c->stage_cap);
    if (c->h_stage) cudaFreeHost(c->h_stage);
    c->d_stage = nullptr; c->h_stage = nullptr; c->stage_cap = 0;
    if (dev_alloc(c, (void**)&c->d_stage, cap)) return 1;
    CU(cudaMallocHost(&c->h_stage, cap));
    c->stage_cap = cap;
  }
  if (c->s2_tiled && n_ops > c->images_cap) {
    const int cap = std::max(n_ops, std::max(256, c->images_cap * 2));
    CU(cudaStreamSynchronize(c->stream));
    if (c->d_images) dev_free(c, c->d_images, (size_t)c->images_cap * sizeof(S2TImage));
    c->d_images = nullptr; c->images_cap = 0;
    if (dev_alloc(c, (void**)&c->d_images, (size_t)cap * sizeof(S2TImage))) return 1;
    c->images_cap = cap;
  }
  if (n_out > c->out_cap) {
    int cap = std::max(n_out, std::max(1, c->out_cap * 2));
    CU(cudaStreamSynchronize(c->stream));
    if (c->d_block_sums) dev_free(c, c->d_block_sums, (size_t)c->out_cap * c->max_blocks * 8);
    if (c->d_tickets) dev_free(c, c->d_tickets, (size_t)c->out_cap * 4);
    if (c->d_results) dev_free(c, c->d_results, (size_t)c->out_cap * 8);
    if (c->d_root_dot) dev_free(c, c->d_root_dot, (size_t)c->out_cap * c->n_cats * c->P * 8);
    if (c->d_root_exp) dev_free(c, c->d_root_exp, (size_t)c->out_cap * c->n_cats * c->P * 4);
    if (c->h_results) cudaFreeHost(c->h_results);
    c->d_block_sums = c->d_results = c->d_root_dot = nullptr;
    c->d_tickets = nullptr; c->d_root_exp = nullptr; c->h_results = nullptr; c->out_cap = 0;
    c->max_blocks = (int)(c->P / 32) + 1;
    if (dev_alloc(c, (void**)&c->d_block_sums, (size_t)cap * c->max_blocks * 8)) return 1;
    if (dev_alloc(c, (void**)&c->d_tickets, (size_t)cap * 4)) return 1;
    CU(cudaMemsetAsync(c->d_tickets, 0, (size_t)cap * 4, c->stream));
    if (dev_alloc(c, (void**)&c->d_results, (size_t)cap * 8)) return 1;
    if (!c->family_s2) {
      if (dev_alloc(c, (void**)&c->d_root_dot, (size_t)cap * c->n_cats * c->P * 8)) return 1;
      if (dev_alloc(c, (void**)&c->d_root_exp, (size_t)cap * c->n_cats * c->P * 4)) return 1;
    }
    CU(cudaHostAlloc(&c->h_results, (size_t)cap * 8, cudaHostAllocMapped));
    c->out_cap = cap;
  }
  return 0;
}

static LaunchConst make_const(cb_ctx* c) {
  LaunchConst k;
  k.ops = reinterpret_cast<const OpDesc*>(c->d_stage);
  k.ranges = nullptr;  // set per evaluation: the ranges and pi follow the ops in the staging block
  k.pmats = c->d_pmats;
  k.pmats_lib = c->d_pmats_lib;
  k.staged = c->d_staged;
  k.weights = c->d_weights;
  k.pi = c->d_pi;   // (overridden per evaluation, see above)
  k.amb = c->d_amb;
  k.block_sums = c->d_block_sums;
  k.tickets = c->d_tickets;
  k.results = c->d_results;
  k.root_dot = c->d_root_dot;
  k.root_exp = c->d_root_exp;
  k.n_sites = c->P;
  k.n_states = c->n_states;
  k.n_cats = c->n_cats;
  k.code_bytes = c->code_bytes;
  k.max_blocks = c->max_blocks;
  k.cats = (double)c->n_cats;
  k.rc_stagger = c->rc_stagger;
  k.n_amb = c->n_amb;
  k.codes = c->d_codes;
  k.s2t_bulk = c->s2t_bulk ? 1 : 0;
  k.n_ranks = 1;
  k.my_rank = 0;
  k.epoch = 0;
  k.mailbox = nullptr;
  k.peer_mailbox = nullptr;
  k.comm_error = nullptr;
  return k;
}

constexpr int MAX_CHAIN_OPS = 4096;          // longer dirty paths fall back to the level schedule
constexpr int64_t WALK_MIN_SITES_S2 = 32768; // below this a site tile cannot fill the GPU: use levels
constexpr int64_t WALK_MIN_SITES_GENERAL = 32768;

static int general_rows_per_chunk(int S) {
  // rows of the two P matrices staged per pass (multiple of 4, <= 64).  Prefer a footprint
  // <= 100 KB (two blocks per SM) as long as that keeps >= 16 rows; else use up to 226 KB.
  const int rmax = std::min((S + 3) / 4 * 4, 64);
  for (int R = rmax; R >= std::min(16, rmax); R -= 4)
    if (gen_smem_bytes(S, R) <= (size_t)100 * 1024) return R;
  for (int R = rmax; R >= 4; R -= 4)
    if (gen_smem_bytes(S, R) <= (size_t)226 * 1024) return R;
  return 0;
}

// Launch the ranges [r_begin, r_end) (all independent) as one kernel.  n_bufs: shared-memory tile buffers per
// warp the ops of these ranges name (tiled 2-state kernel only).
static int launch_ranges(cb_ctx* c, const LaunchConst& k, int r_begin, int r_end, int max_ops_in_range, int n_bufs) {
  const int n_r = r_end - r_begin;
  LaunchConst kk = k;
  kk.ranges = k.ranges + r_begin;
  if (c->s2_tiled) {
    // large binary alignments: tile-interleaved partials, shared-memory stack, bulk-async stores (kernels_s2t.cuh)
    const size_t smem = s2t_smem_bytes(n_bufs, c->n_cats, c->s2t_minb);
    REQUIRE(smem <= (size_t)226 * 1024, "internal error: %d tile buffers do not fit shared memory", n_bufs);
    const int64_t n_tiles = c->P / S2T_W;
    dim3 grid((unsigned)((n_tiles + S2T_WARPS - 1) / S2T_WARPS), (unsigned)n_r);
    // V tiles per warp (8 / V warps per block): fixed per context, so every evaluation of an alignment sums in one order
#define CB_S2T_LAUNCH(MB, VV)                                                                                              \
  do {                                                                                                                     \
    if (c->n_cats == 4) prune_s2t_kernel<4, MB, VV><<<grid, S2T_THREADS / VV, smem, c->stream>>>(kk, c->d_images, n_bufs); \
    else prune_s2t_kernel<1, MB, VV><<<grid, S2T_THREADS / VV, smem, c->stream>>>(kk, c->d_images, n_bufs);                \
  } while (0)
    if (c->s2t_v == 2 && c->s2t_minb >= 3) CB_S2T_LAUNCH(3, 2);
    else if (c->s2t_v == 2) CB_S2T_LAUNCH(2, 2);
    else if (c->s2t_minb == 4) CB_S2T_LAUNCH(4, 1);
    else if (c->s2t_minb == 3) CB_S2T_LAUNCH(3, 1);
    else CB_S2T_LAUNCH(2, 1);
#undef CB_S2T_LAUNCH
  } else if (c->family_s2) {
    // Fixed per alignment (independent of the schedule) so the reduction order never changes:
    // 64-thread blocks, one site per thread, to spread a small alignment over the SMs (the tiled kernel above
    // takes over from 75 776 patterns); CYBAYES_S2_TILED=0 keeps this kernel on large alignments too (256 threads).
    const size_t smem = s2_smem_bytes(max_ops_in_range, c->n_cats);
    const bool small = c->P < S2_TILED_MIN_SITES;
    const int V = small ? 1 : c->s2_vec;
    const int threads = small ? 64 : 256;
    dim3 grid((unsigned)((c->P + (int64_t)threads * V - 1) / ((int64_t)threads * V)), (unsigned)n_r);
#define CB_LAUNCH_S2(CC, VV, TT, MB) prune_s2_kernel<CC, VV, TT, MB><<<grid, TT, smem, c->stream>>>(kk)
    if (c->n_cats == 4) {
      if (small) CB_LAUNCH_S2(4, 1, 64, 8);
      else if (V == 1 && c->s2_minb == 4) CB_LAUNCH_S2(4, 1, 256, 4);
      else if (V == 1) CB_LAUNCH_S2(4, 1, 256, 3);
      else CB_LAUNCH_S2(4, 2, 256, 2);
    } else {
      if (small) CB_LAUNCH_S2(1, 1, 64, 8); else if (V == 1) CB_LAUNCH_S2(1, 1, 256, 4); else CB_LAUNCH_S2(1, 2, 256, 4);
    }
#undef CB_LAUNCH_S2
  } else if (c->dmma_rc) {
    dim3 grid((unsigned)((c->P + RC_T - 1) / RC_T), (unsigned)n_r, (unsigned)c->n_cats);
    switch ((c->n_states + 7) / 8 * 8) {  // compiled per padded state count; the real one is a run-time value
#define CB_RC_CASE(SS)                                                                                          \
  case SS:                                                                                                      \
    if (c->n_states == SS) prune_dmma_rc_kernel<SS, true><<<grid, RC_THREADS, RcCfg<SS>::SMEM, c->stream>>>(kk); \
    else prune_dmma_rc_kernel<SS, false><<<grid, RC_THREADS, RcCfg<SS>::SMEM, c->stream>>>(kk);                  \
    break
      CB_RC_CASE(16); CB_RC_CASE(24); CB_RC_CASE(32); CB_RC_CASE(40); CB_RC_CASE(48); CB_RC_CASE(56); CB_RC_CASE(64);
#undef CB_RC_CASE
      default: return fail("internal error: no register-carried DMMA kernel for %d states", c->n_states);
    }
  } else if (c->use_dmma) {
    dim3 grid((unsigned)(c->P / DM_T), (unsigned)n_r, (unsigned)c->n_cats);
    const size_t smem = dm_smem_bytes(c->n_states);
    switch (c->n_states) {  // compile-time state counts for the common sizes, run-time S otherwise
#define CB_DMMA_CASE(SS) case SS: prune_dmma_kernel<SS><<<grid, DM_THREADS, smem, c->stream>>>(kk); break
      CB_DMMA_CASE(32); CB_DMMA_CASE(40); CB_DMMA_CASE(47); CB_DMMA_CASE(48); CB_DMMA_CASE(56); CB_DMMA_CASE(64);
#undef CB_DMMA_CASE
      default: prune_dmma_kernel<0><<<grid, DM_THREADS, smem, c->stream>>>(kk);
    }
  } else {
    const int R = general_rows_per_chunk(c->n_states);
    REQUIRE(R > 0, "n_states = %d does not fit the shared-memory tiling", c->n_states);
    dim3 grid((unsigned)(c->P / GEN_T), (unsigned)n_r, (unsigned)c->n_cats);
    prune_general_kernel<<<grid, GEN_THREADS, gen_smem_bytes(c->n_states, R), c->stream>>>(kk, R);
  }
  CU(cudaGetLastError());
  c->launches += 1;
  return 0;
}

// tiled 2-state kernel: build the op images of ops [0, n_ops) (one launch per evaluation)
static int launch_images(cb_ctx* c, const LaunchConst& k, int n_ops) {
  if (!c->s2_tiled) return 0;
  if (c->n_cats == 4) s2t_image_kernel<4><<<n_ops, 32, 0, c->stream>>>(k, n_ops, c->d_images);
  else s2t_image_kernel<1><<<n_ops, 32, 0, c->stream>>>(k, n_ops, c->d_images);
  CU(cudaGetLastError());
  c->launches += 1;
  return 0;
}

// Compute the partial of a node that a snapshot keeps as a record (a folded cherry or a small subtree) into a fresh
// buffer (debug / read-back path): one ordinary op whose P matrices come from the library's pool; a child that is itself
// a cherry record of the same snapshot is looked up in its table, as in a normal evaluation.
static int materialize_cherry(cb_ctx* c, const Snapshot& sn, int rec, int* buf_out) {
  REQUIRE(c->family_s2 && rec >= 0 && rec < (int)c->recs.size(), "bad record %d", rec);
  if (ensure_staging(c, 1, 1, 1)) return 1;
  CU(cudaStreamSynchronize(c->stream));
  int bi;
  if (buffer_acquire(c, &bi)) return 1;
  OpDesc& op = *reinterpret_cast<OpDesc*>(c->h_stage);
  memset(&op, 0, sizeof op);
  op.dst = c->buffers[bi].data;
  op.dst_scale = c->buffers[bi].scale;
  op.out_buf = op.pf_buf = op.frec_out = -1;
  const int C = c->n_cats, N = c->n_taxa;
  const size_t row_bytes = (size_t)c->P * c->code_bytes;
  int order[2] = {0, 1};
  if (c->s2_tiled && c->recs[rec].tip[0] > N && c->recs[rec].tip[1] <= N) { order[0] = 1; order[1] = 0; }  // canonical: tip first
  for (int w = 0; w < 2; ++w) {
    const int kx = order[w], ch = c->recs[rec].tip[kx];
    for (int q = 0; q < C; ++q) op.pslot[w][q] = CB_LIB_SLOT | (rec * 2 * C + kx * C + q);
    op.crec_out[w] = -1;
    if (ch <= N) {
      op.kind[w] = SRC_TIP;
      op.src[w] = (const char*)c->d_codes + (size_t)(ch - 1) * row_bytes;
    } else {
      const int yrec = ch < (int)sn.cherry_of_node.size() ? sn.cherry_of_node[ch] : -1;
      if (yrec < 0) { buffer_release(c, bi); return fail("internal error: cherry %d of record %d is not in the snapshot", ch, rec); }
      op.kind[w] = SRC_CHERRY;
      for (int t = 0; t < 2; ++t) {
        op.ctip[w][t] = (const char*)c->d_codes + (size_t)(c->recs[yrec].tip[t] - 1) * row_bytes;
        for (int q = 0; q < CB_S2_MAX_CATS; ++q) op.cslot[w][t][q] = q < C ? (CB_LIB_SLOT | (yrec * 2 * C + t * C + q)) : 0;
      }
    }
  }
  *reinterpret_cast<RangeDesc*>(c->h_stage + sizeof(OpDesc)) = RangeDesc{0, 1, -1, 0};
  CU(cudaMemcpyAsync(c->d_stage, c->h_stage, sizeof(OpDesc) + sizeof(RangeDesc), cudaMemcpyHostToDevice, c->stream));
  LaunchConst k = make_const(c);
  k.ranges = reinterpret_cast<const RangeDesc*>(c->d_stage + sizeof(OpDesc));
  if (launch_images(c, k, 1)) { buffer_release(c, bi); return 1; }
  if (launch_ranges(c, k, 0, 1, 1, 0)) { buffer_release(c, bi); return 1; }
  CU(cudaStreamSynchronize(c->stream));
  *buf_out = bi;
  return 0;
}

// ---- plans --------------------------------------------------------------------------------------------------
// An evaluation is compiled into a PLAN: which ops run (cherries folded away), in which order, in which ranges
// and launches, where every child comes from, which results are stored.  The plan of a FULL evaluation depends only
// on the op list and the flags, so it is cached per topology (a handful of trees are alive at a time in an MCMC
// run: the current one and the proposals); executing a cached plan only refills buffer pointers and P slots.
//
// Schedules (all run the same per-node arithmetic, so results are bit-identical):
//   CHAIN  a dirty path: one launch, one block range walks the ops, the on-path partial is
//          carried in registers / shared memory                        (ML_gamma.pyx:99-114)
//   WALK   a whole (sub)tree in ONE launch; every block walks all ops for its site tile depth-first.  The child
//          finished last is carried on chip; the other child of a node with two internal children is pushed on a
//          stack in shared memory (tiled 2-state kernel: K tile buffers per warp) or, when the stack is full or the
//          kernel has none, written to its buffer and read back.  The visiting order minimises those read-backs
//          (dynamic programme over the tree; ties: heavier subtree first, so a read-back finds its line in L2).
//   LEVELS one launch per tree level, grid.y = nodes of the level: the latency schedule for
//          small alignments where a site tile alone cannot fill the GPU.
enum Schedule { SCHED_CHAIN = 0, SCHED_WALK = 1, SCHED_LEVELS = 2 };


static int build_plan(cb_ctx* c, const Snapshot* sin, int n_lists, const int32_t* offsets_in, const int32_t* nodes_in,
                      const int32_t* children_in, int flags, EvalPlan& plan) {
  const int N = c->n_taxa, n_nodes = 2 * N;  // ids 1 .. 2N-1
  const bool fold = c->family_s2 && !(flags & CB_EVAL_NO_FOLD);
  const bool want_snap = (flags & CB_EVAL_WANT_SNAPSHOT) != 0;
  const bool store_root = (flags & CB_EVAL_STORE_ROOT) != 0;
  const int C = c->n_cats;
  const int K = c->s2_tiled ? c->s2t_slots : 0;  // stack slots of the kernel
  const int slot_base = c->s2t_bulk ? S2T_STAGING : 0;  // tile buffers below it are the staging buffers of the bulk-store path
  plan.ops.clear(); plan.ranges.clear(); plan.launches.clear();
  plan.bytes_written = plan.bytes_read = 0;
  plan.n_stored = plan.n_buffer_reads = plan.n_stack = plan.n_spills = plan.n_cherries = plan.n_small_recs = 0;
  plan.n_inlined = 0;
  const int64_t tip_row_bytes = c->P * c->code_bytes;
  // small subtrees (children: tips / cherries) of a cache-kept pass are kept as records instead of being stored
  const bool small_recs = c->s2_tiled && c->s2t_small_recs && want_snap;
  auto snap_cherry = [&](int nd) {   // the input snapshot holds node nd as a record (a folded cherry or a small subtree)
    return fold && sin && nd < (int)sin->cherry_of_node.size() && sin->cherry_of_node[nd] >= 0;
  };

  struct LOp { int32_t node, caller; int32_t child[2], folded[2]; };
  std::vector<LOp> L;
  std::vector<int32_t> parent_op(n_nodes), folded_at(n_nodes), op_of_node(n_nodes, -1);
  std::vector<int> kid[2], n_sub, order, pos_of, range_id, push_slot, first_kid, level_of, by_level;
  std::vector<std::pair<int, int>> segs;
  std::vector<int> seg_of;     // op -> segment (0 = top / whole list, s + 1 = cut subtree s)
  std::vector<int> f;          // DP table [op][k]
  std::vector<char> read_back;
  std::vector<int> small_of;   // op -> its child (0 / 1) that it computes itself (SRC_SMALL), or -1
  std::vector<char> inlined;   // op -> computed inside its parent's op
  bool single_launch = true;

  for (int li = 0; li < n_lists; ++li) {
    const int b_in = offsets_in[li], e_in = offsets_in[li + 1];
    REQUIRE(e_in > b_in, "empty op list %d", li);
    // ---- cherry folding (2-state family): an op whose two children are tips is not run: its parent (always in the
    // list) takes it as a SRC_CHERRY child and looks the cherry's 3 x 3 possible partials up
    L.clear();
    std::fill(parent_op.begin(), parent_op.end(), -1);
    std::fill(folded_at.begin(), folded_at.end(), -1);
    for (int i = b_in; i < e_in; ++i)
      for (int kx = 0; kx < 2; ++kx) {
        const int ch = children_in[2 * i + kx];
        REQUIRE((ch >= 1 && ch <= N) || (ch > N && ch < n_nodes), "op %d: bad child id %d", i, ch);
        if (ch > N) parent_op[ch] = i;
      }
    for (int i = b_in; i < e_in; ++i) {
      const int node = nodes_in[i], c0 = children_in[2 * i], c1 = children_in[2 * i + 1];
      REQUIRE(node > N && node < n_nodes, "op %d: node %d is not an internal node", i, node);
      const bool cherry = fold && c0 <= N && c1 <= N && i != e_in - 1 && parent_op[node] > i;
      if (cherry) {
        folded_at[node] = i;
        plan.n_cherries++;
        continue;
      }
      LOp o;
      o.node = node;
      o.caller = i;
      for (int kx = 0; kx < 2; ++kx) {
        const int ch = children_in[2 * i + kx];
        o.child[kx] = ch;
        o.folded[kx] = ch > N ? folded_at[ch] : -1;
      }
      L.push_back(o);
    }
    // Children that the input snapshot holds as records of small subtrees (not cherries) are recomputed here: one
    // synthetic op each, placed before the caller's ops; the walk pushes / carries its result like any other child.
    if (sin && c->s2_tiled) {
      std::vector<LOp> syn;
      auto is_rec = [&](int nd) { return nd > N && nd < (int)sin->cherry_of_node.size() && sin->cherry_of_node[nd] >= 0; };
      for (const LOp& o : L)
        for (int kx = 0; kx < 2; ++kx) {
          const int ch = o.child[kx];
          if (ch <= N || o.folded[kx] >= 0 || !is_rec(ch)) continue;
          const CherryRec& r = c->recs[sin->cherry_of_node[ch]];
          if (r.tip[0] <= N && r.tip[1] <= N) continue;   // a cherry: folded into the parent's table
          bool in_list = false;
          for (const LOp& q : L) in_list = in_list || q.node == ch;
          if (in_list) continue;
          LOp so;
          so.node = ch;
          so.caller = ~sin->cherry_of_node[ch];            // < 0: synthetic, names the record
          so.child[0] = r.tip[0]; so.child[1] = r.tip[1];
          so.folded[0] = so.folded[1] = -1;
          syn.push_back(so);
        }
      if (!syn.empty()) L.insert(L.begin(), syn.begin(), syn.end());
    }
    const int n = (int)L.size();
    // producers of the children inside this list (-1: tip, folded cherry or snapshot)
    for (int j = 0; j < n; ++j) {
      REQUIRE(op_of_node[L[j].node] < 0, "op %d: node %d is computed twice", L[j].caller, L[j].node);
      op_of_node[L[j].node] = j;
    }
    auto cleanup = [&] { for (int j = 0; j < n; ++j) op_of_node[L[j].node] = -1; };
    kid[0].assign(n, -1);
    kid[1].assign(n, -1);
    for (int j = 0; j < n; ++j)
      for (int kx = 0; kx < 2; ++kx) {
        const int ch = L[j].child[kx];
        if (ch > N && L[j].folded[kx] < 0 && op_of_node[ch] >= 0) {
          if (op_of_node[ch] >= j) { cleanup(); return fail("op %d: child %d is computed after its parent", L[j].caller, ch); }
          kid[kx][j] = op_of_node[ch];
        } else if (ch > N && L[j].folded[kx] < 0) {
          const bool in_snap = sin && ch < (int)sin->buf_of_node.size() &&
                               (sin->buf_of_node[ch] >= 0 || (ch < (int)sin->cherry_of_node.size() && sin->cherry_of_node[ch] >= 0));
          if (!in_snap) { cleanup(); return fail("op %d: child %d is neither recomputed nor in the input snapshot", L[j].caller, ch); }
        }
      }
    cleanup();
    // chain: every op after the first consumes exactly the previous op and nothing else of the list
    bool chain = !(flags & CB_EVAL_FORCE_LEVELS) && n <= MAX_CHAIN_OPS;
    for (int j = 0; j < n && chain; ++j) {
      const int a0 = kid[0][j], a1 = kid[1][j];
      if (j == 0) chain = (a0 < 0 && a1 < 0);
      else chain = (a0 == j - 1) != (a1 == j - 1) && (a0 < 0 || a0 == j - 1) && (a1 < 0 || a1 == j - 1);
    }
    Schedule sched = SCHED_CHAIN;
    if (!chain) {
      // the register-carried kernel only pays off when the partial is carried: its alignments always walk;
      // candidates of a batch always walk (one range per candidate)
      const bool big = c->dmma_rc || c->P >= (c->family_s2 ? WALK_MIN_SITES_S2 : WALK_MIN_SITES_GENERAL);
      sched = ((big || n_lists > 1 || (flags & CB_EVAL_FORCE_WALK)) && !(flags & CB_EVAL_FORCE_LEVELS)) ? SCHED_WALK : SCHED_LEVELS;
      if (n_lists > 1 && sched == SCHED_LEVELS) return fail("cb_eval_batch: candidate %d is not a chain (level schedule forced)", li);
    }

    // Tiled kernel: a (tip, cherry) subtree that is not stored is computed inside its parent's op (SRC_SMALL) when the
    // parent runs in the same range and its other child is a tip or the op carried into it -- the same arithmetic
    // without an op of its own (image, dispatch, rescale, loop iteration) and without a stack slot.
    small_of.assign(n, -1);
    inlined.assign(n, 0);
    int n_inl = 0;
    auto is_cherry = [&](int j, int kx) {   // the child resolves to SRC_CHERRY (below)
      const int ch = L[j].child[kx];
      return ch > N && (L[j].folded[kx] >= 0 || (kid[kx][j] < 0 && snap_cherry(ch)));
    };
    auto pick_small = [&] {
      if (!c->s2_tiled) return;
      for (int j = 0; j < n; ++j)
        for (int kx = 1; kx >= 0 && small_of[j] < 0; --kx) {
          const int s = kid[kx][j], o = kid[1 - kx][j];
          if (s < 0 || seg_of[s] != seg_of[j]) continue;
          const bool tip_cherry = (L[s].child[0] <= N && is_cherry(s, 1)) || (L[s].child[1] <= N && is_cherry(s, 0));
          // not stored: likelihood-only pass, a recomputed record, or kept as a record (make_rec below; checked there)
          const bool unstored = !want_snap || L[s].caller < 0 || small_recs;
          const bool sibling_ok = L[j].child[1 - kx] <= N || (o >= 0 && seg_of[o] == seg_of[j]);
          if (tip_cherry && unstored && sibling_ok) {
            small_of[j] = kx;
            inlined[s] = 1;
            n_inl++;
          }
        }
    };
    order.resize(n);
    for (int j = 0; j < n; ++j) order[j] = j;
    seg_of.assign(n, 0);
    push_slot.assign(n, -1);
    segs.clear();
    if (sched == SCHED_WALK) {
      // subtree sizes in ops (children precede parents in the caller's order)
      n_sub.assign(n, 1);
      for (int j = 0; j < n; ++j)
        for (int kx = 0; kx < 2; ++kx)
          if (kid[kx][j] >= 0) n_sub[j] += n_sub[kid[kx][j]];
      bool rooted = (n_sub[n - 1] == n);  // every op under the last one
      if (!rooted) {
        REQUIRE(n_lists == 1, "cb_eval_batch: candidate %d has ops that are not under its root", li);
        sched = SCHED_LEVELS;
      } else {
        // When the alignment gives too few site tiles to fill the GPU for a whole sequential walk (small shards), the
        // tree is cut into independent subtrees of at most `limit` ops that run as parallel ranges of a first launch;
        // the ops above the cut follow in a second launch.
        int limit = n + 1;
        if (n_lists == 1) {
          const int64_t tile_sites = c->s2_tiled ? S2T_THREADS : (c->family_s2 ? (int64_t)256 * c->s2_vec : (c->dmma_rc ? RC_T : (c->use_dmma ? DM_T : GEN_T)));
          const int64_t blocks = (c->P + tile_sites - 1) / tile_sites * (c->family_s2 ? 1 : c->n_cats);
          const int64_t slots = (int64_t)c->sm_count * (c->s2_tiled ? c->s2t_minb : (c->family_s2 ? (c->s2_vec == 1 ? 3 : 2) : (c->dmma_rc ? 1 : 2)));
          // Every block walks the whole list (0.7 ms on C4, 3 ms on a C5 shard), so a ragged last wave is expensive even
          // at many waves: 2-3 % at 8.8 waves, 12 % at 4.4 and 5.3.  Measured: C4 6.07 -> 5.91 ms on 1 GPU and 3.28 ->
          // 2.98 ms per GPU on 2; the C5 shard of an 8-GPU run (25 000 patterns x 64 states) 17.7 -> 15.9 ms.
          // Under one wave the cut is there for parallelism (about 8 waves of ranges); from one wave up it only has to
          // even out the tail, and a small limit costs more in the launch of the ops above the cut (16 ops at limit 93
          // on a 125 000-pattern shard: 65 us of 800) than it gains: a third of the tree per range measured best there
          // (0.794 -> 0.77 ms).
          if (blocks < 16 * slots && n >= 64 && !(flags & CB_EVAL_FORCE_WALK)) {
            int lim = (int)(n * blocks / (8 * slots)) + 1;
            if (blocks >= slots) lim = std::max(lim, n / 3);
            limit = std::max(16, std::min(256, lim));
          }
          if (plan.split_env > 0) limit = std::max(2, plan.split_env);
          if (limit >= n) limit = n + 1;  // nothing to cut
        }
        std::vector<int> cut, top, stack;
        if (limit <= n) {
          // walk down from the root: ops with a subtree above the limit stay in the top segment
          stack.push_back(n - 1);
          while (!stack.empty()) {
            const int j = stack.back();
            stack.pop_back();
            if (n_sub[j] <= limit) { cut.push_back(j); continue; }
            for (int kx = 0; kx < 2; ++kx)
              if (kid[kx][j] >= 0) stack.push_back(kid[kx][j]);
          }
          std::stable_sort(cut.begin(), cut.end(), [&](int x, int y) { return n_sub[x] > n_sub[y]; });  // big first
          // segment membership: everything under a cut root belongs to that root's segment
          for (size_t s = 0; s < cut.size(); ++s) {
            stack.push_back(cut[s]);
            while (!stack.empty()) {
              const int j = stack.back();
              stack.pop_back();
              seg_of[j] = (int)s + 1;
              for (int kx = 0; kx < 2; ++kx)
                if (kid[kx][j] >= 0) stack.push_back(kid[kx][j]);
            }
          }
        }
        pick_small();
        // children the walk visits: a cut root lives in another launch and is read from its buffer; an inlined subtree
        // is computed by its parent, like a tip
        auto walk_kid = [&](int kx, int j) {
          const int a = kid[kx][j];
          return a >= 0 && seg_of[a] == seg_of[j] && !inlined[a] ? a : -1;
        };
        // visiting order per segment: f[j][k] = fewest read-backs in j's subtree (inside its segment) with k free stack
        // slots; of two internal children the first visited is pushed (or read back when k == 0), the second carried
        f.assign((size_t)n * (K + 1), 0);
        first_kid.assign((size_t)n * (K + 1), 0);
        for (int j = 0; j < n; ++j) {
          const int a = walk_kid(0, j), b2 = walk_kid(1, j);
          for (int kk = 0; kk <= K; ++kk) {
            int& fj = f[(size_t)j * (K + 1) + kk];
            if (a >= 0 && b2 >= 0) {
              const int k1 = kk > 0 ? kk - 1 : 0, miss = kk == 0 ? 1 : 0;
              const int ca = f[(size_t)a * (K + 1) + kk] + miss + f[(size_t)b2 * (K + 1) + k1];
              const int cb2 = f[(size_t)b2 * (K + 1) + kk] + miss + f[(size_t)a * (K + 1) + k1];
              const bool a_first = ca < cb2 || (ca == cb2 && n_sub[a] >= n_sub[b2]);
              fj = a_first ? ca : cb2;
              first_kid[(size_t)j * (K + 1) + kk] = a_first ? 0 : 1;
              // third choice: read the first child back although a slot is free, so that the second keeps all kk slots
              // (one read-back here instead of one at every fork of a subtree left with too few slots)
              const int cs = f[(size_t)a * (K + 1) + kk] + 1 + f[(size_t)b2 * (K + 1) + kk];
              if (kk > 0 && cs < fj) {
                fj = cs;
                first_kid[(size_t)j * (K + 1) + kk] = (n_sub[a] >= n_sub[b2] ? 0 : 1) | 2;
              }
            } else if (a >= 0) {
              fj = f[(size_t)a * (K + 1) + kk];
            } else if (b2 >= 0) {
              fj = f[(size_t)b2 * (K + 1) + kk];
            }
          }
        }
        std::vector<int> out;
        out.reserve(n);
        struct Frame { int j, k, phase; };
        std::vector<Frame> fr;
        auto emit = [&](int root_op) {
          fr.push_back({root_op, K, 0});
          while (!fr.empty()) {
            Frame& t = fr.back();
            const int j = t.j, kk = t.k;
            const int a = walk_kid(0, j), b2 = walk_kid(1, j);
            if (a >= 0 && b2 >= 0) {
              const int fk = first_kid[(size_t)j * (K + 1) + kk];
              const bool push = kk > 0 && !(fk & 2);
              const int x = (fk & 1) == 0 ? a : b2, y = (fk & 1) == 0 ? b2 : a;
              if (t.phase == 0) { t.phase = 1; fr.push_back({x, kk, 0}); continue; }
              if (t.phase == 1) {
                push_slot[x] = push ? slot_base + (K - kk) : -1;
                t.phase = 2;
                fr.push_back({y, push ? kk - 1 : kk, 0});
                continue;
              }
            } else if (a >= 0 || b2 >= 0) {
              if (t.phase == 0) { t.phase = 2; fr.push_back({a >= 0 ? a : b2, kk, 0}); continue; }
            }
            out.push_back(j);
            fr.pop_back();
          }
        };
        if (limit > n) {
          emit(n - 1);
        } else {
          for (int r : cut) {
            const int b0 = (int)out.size();
            emit(r);
            segs.push_back({b0, (int)out.size()});
          }
          emit(n - 1);
        }
        REQUIRE((int)out.size() == n - n_inl, "internal error: walk order covers %d of %d ops", (int)out.size(), n - n_inl);
        for (int j = 0; j < n; ++j)
          if (inlined[j]) out.push_back(j);   // descriptors only: after the ops the ranges run
        order = out;
      }
    } else if (sched == SCHED_CHAIN) {
      pick_small();   // only the first op of a chain can be such a subtree; its parent takes it beside a tip
      if (n_inl > 0) {
        std::stable_partition(order.begin(), order.end(), [&](int j) { return !inlined[j]; });
      }
    }
    const int n_exec = n - n_inl;   // positions [n_exec, n): inlined ops
    plan.n_inlined += n_inl;
    pos_of.assign(n, 0);
    for (int p = 0; p < n; ++p) pos_of[order[p]] = p;
    range_id.assign(n, 0);   // by position
    for (size_t si = 0; si < segs.size(); ++si)
      for (int p = segs[si].first; p < segs[si].second; ++p) range_id[p] = (int)si + 1;
    // launch of a position: split walk = cut segments first (0), top second (1); levels: see below
    auto same_range = [&](int p0, int p1) { return sched != SCHED_LEVELS && range_id[p0] == range_id[p1]; };

    // where does each child come from; which ops are read back from memory by a later op?
    read_back.assign(n, 0);
    const int base = (int)plan.ops.size();
    plan.ops.resize(base + n);
    int staging_rr = 0;
    for (int p = 0; p < n; ++p) {
      const int j = order[p];
      PlanOp& po = plan.ops[base + p];
      po.node = L[j].node;
      po.is_root = (j == n - 1);
      REQUIRE(!po.is_root || p == n_exec - 1, "internal error: root is not last");
      po.keep = po.stream = po.spill = po.pushed = po.make_rec = 0;
      po.synthetic = L[j].caller < 0 ? 1 : 0;
      po.out_buf = po.pf_buf = -1;
      for (int kx = 0; kx < 2; ++kx) {
        PlanChild& pc = po.ch[kx];
        const int ch = L[j].child[kx];
        pc.edge = L[j].caller >= 0 ? 2 * L[j].caller + kx : ~((~L[j].caller) * 2 * C + kx * C);
        if (ch <= N) {
          pc.kind = SRC_TIP;
          pc.ref = ch;
          plan.bytes_read += tip_row_bytes;
        } else if (L[j].folded[kx] >= 0) {
          pc.kind = SRC_CHERRY;
          pc.ref = L[j].folded[kx];
          plan.bytes_read += 2 * tip_row_bytes;
        } else if (small_of[j] == kx) {
          pc.kind = SRC_SMALL;
          pc.ref = base + pos_of[kid[kx][j]];   // its descriptor
        } else if (kid[kx][j] >= 0) {
          const int jj = kid[kx][j], pp = pos_of[jj];
          if (same_range(pp, p) && pp == p - 1) {
            pc.kind = SRC_CARRIED;
            pc.ref = 0;
          } else if (same_range(pp, p) && push_slot[jj] >= 0) {
            pc.kind = SRC_STACK;
            pc.ref = push_slot[jj];
            plan.n_stack++;
          } else {
            REQUIRE(pp < p, "internal error: producer of node %d runs after its consumer", ch);
            pc.kind = SRC_BUFFER;
            pc.ref = base + pp;
            read_back[jj] = same_range(pp, p) ? 2 : 1;   // 2: inside one launch (a spill)
            plan.bytes_read += (int64_t)c->buffer_bytes;
            plan.n_buffer_reads++;
          }
        } else {
          const bool rec = snap_cherry(ch);
          pc.kind = rec ? SRC_CHERRY : SRC_BUFFER;
          pc.ref = ~ch;
          plan.bytes_read += rec ? 2 * tip_row_bytes : (int64_t)c->buffer_bytes;
          if (!rec) plan.n_buffer_reads++;
        }
      }
    }
    plan.bytes_read += c->P * 8;  // pattern weights at the root
    if (c->s2_tiled)  // the tiled kernel wants the children in canonical order (products and exponent sums commute exactly)
      for (int p = 0; p < n; ++p) {
        PlanOp& po = plan.ops[base + p];
        if (s2t_rank(po.ch[1].kind) < s2t_rank(po.ch[0].kind)) std::swap(po.ch[0], po.ch[1]);
        REQUIRE(s2t_combo(po.ch[0].kind, po.ch[1].kind) >= 0, "internal error: op of node %d has children of kinds %d, %d", po.node,
                po.ch[0].kind, po.ch[1].kind);
      }
    for (int p = 0; p < n; ++p) {
      const int j = order[p];
      PlanOp& po = plan.ops[base + p];
      po.keep = po.is_root ? (want_snap && store_root) : ((want_snap && !po.synthetic) || read_back[j] != 0);
      po.stream = (po.keep && read_back[j] == 0 && c->s2_stream_stores) ? 1 : 0;
      po.spill = (read_back[j] == 2) ? 1 : 0;
      if (po.keep) {
        plan.bytes_written += (int64_t)c->buffer_bytes;
        plan.n_stored++;
        if (po.spill) plan.n_spills++;
      }
      // small subtrees (children: tips / cherries) are not stored: the returned snapshot keeps a record
      if (small_recs && po.keep && !po.is_root && !po.synthetic && read_back[j] == 0 &&
          (po.ch[0].kind == SRC_TIP || po.ch[0].kind == SRC_CHERRY) && po.ch[1].kind == SRC_CHERRY) {
        po.keep = 0;
        po.stream = 0;
        po.make_rec = 1;
        plan.bytes_written -= (int64_t)c->buffer_bytes;
        plan.n_stored--;
        plan.n_small_recs++;
      }
      // an inlined op has no store of its own: a buffer given to it would enter the snapshot unwritten
      REQUIRE(!inlined[j] || !po.keep, "internal error: inlined node %d would be stored", po.node);
      if (c->s2_tiled) {
        if (push_slot[j] >= 0 && !po.is_root) { po.out_buf = push_slot[j]; po.pushed = 1; }
        else if (c->s2t_bulk && po.keep && !po.spill) { po.out_buf = staging_rr; staging_rr ^= 1; }
      }
    }
    int max_slot = -1;
    for (int j = 0; j < n; ++j) max_slot = std::max(max_slot, push_slot[j]);
    if (c->s2_tiled && c->s2t_prefetch && max_slot < 2 && !c->s2t_bulk) {
      // Dirty paths and other lists with a shallow stack: a stored partial that comes from the input snapshot (or an
      // earlier launch) and is read beside a carried child is prefetched into a tile buffer two ops ahead (three rotating
      // buffers above the stack slots in use) and then read like a stack slot: the path keeps three sibling tiles per
      // warp in flight instead of exposing one DRAM latency per op.
      const int pf_base = max_slot + 1;
      int rr = 0;
      for (int p = 0; p < n; ++p) {
        PlanOp& po = plan.ops[base + p];
        if (po.ch[0].kind != SRC_CARRIED || po.ch[1].kind != SRC_BUFFER) continue;
        const int ref = po.ch[1].ref;
        const bool other_launch = ref < 0 || !same_range(ref - base, p);
        if (!other_launch) continue;
        po.ch[1].kind = SRC_STACK;     // read from the tile buffer; po.ch[1].ref keeps naming the stored partial
        po.pf_buf = pf_base + rr;
        rr = (rr + 1) % 3;
      }
    }

    // ranges and launches
    auto bufs_of = [&](int p0, int p1) {
      int nb = 0;
      for (int p = p0; p < p1; ++p) {
        const PlanOp& po = plan.ops[base + p];
        nb = std::max(nb, std::max(po.out_buf, po.pf_buf) + 1);
        for (int kx = 0; kx < 2; ++kx)
          if (po.ch[kx].kind == SRC_STACK && po.pf_buf < 0) nb = std::max(nb, po.ch[kx].ref + 1);
      }
      return nb;
    };
    if (sched == SCHED_WALK && !segs.empty()) {
      single_launch = false;
      const int start = (int)plan.ranges.size();
      int mx = 1, nb = 0;
      for (auto& sg : segs) {
        plan.ranges.push_back(RangeDesc{base + sg.first, base + sg.second, -1, 0});
        mx = std::max(mx, sg.second - sg.first);
        nb = std::max(nb, bufs_of(sg.first, sg.second));
      }
      plan.launches.push_back({start, (int)plan.ranges.size(), mx, nb});
      const int tb = segs.back().second;
      plan.ranges.push_back(RangeDesc{base + tb, base + n_exec, li, 0});
      plan.launches.push_back({(int)plan.ranges.size() - 1, (int)plan.ranges.size(), n_exec - tb, bufs_of(tb, n_exec)});
    } else if (sched != SCHED_LEVELS) {
      plan.ranges.push_back(RangeDesc{base, base + n_exec, li, 0});
    } else {
      single_launch = false;
      level_of.assign(n, 1);
      int max_level = 1;
      for (int j = 0; j < n; ++j) {
        int lv = 1;
        for (int kx = 0; kx < 2; ++kx)
          if (kid[kx][j] >= 0) lv = std::max(lv, level_of[kid[kx][j]] + 1);
        level_of[j] = lv;
        max_level = std::max(max_level, lv);
      }
      by_level.resize(n);
      for (int j = 0; j < n; ++j) by_level[j] = j;
      std::stable_sort(by_level.begin(), by_level.end(), [&](int x, int y) { return level_of[x] < level_of[y]; });
      int pos = 0;
      for (int lv = 1; lv <= max_level; ++lv) {
        const int start = (int)plan.ranges.size();
        int nb = 0;
        while (pos < n && level_of[by_level[pos]] == lv) {
          const int j = by_level[pos++];   // order is the identity for this schedule
          plan.ranges.push_back(RangeDesc{base + j, base + j + 1, (j == n - 1) ? li : -1, 0});
          nb = std::max(nb, bufs_of(j, j + 1));
        }
        if ((int)plan.ranges.size() > start) plan.launches.push_back({start, (int)plan.ranges.size(), 1, nb});
      }
    }
  }
  if (single_launch) {
    int mx = 0, nb = 0;
    for (const RangeDesc& r : plan.ranges) mx = std::max(mx, r.end - r.begin);
    for (const PlanOp& po : plan.ops) {
      nb = std::max(nb, std::max(po.out_buf, po.pf_buf) + 1);
      for (int kx = 0; kx < 2; ++kx)
        if (po.ch[kx].kind == SRC_STACK && po.pf_buf < 0) nb = std::max(nb, po.ch[kx].ref + 1);
    }
    plan.launches.push_back({0, (int)plan.ranges.size(), mx, nb});
  }
  return 0;
}

// Releases what an evaluation acquired when it fails part-way (buffers and cherry records go back to their pools).
struct EvalGuard {
  cb_ctx* c;
  std::vector<int> bufs, recs;
  bool armed = true;
  ~EvalGuard() {
    if (!armed) return;
    for (int b : bufs) buffer_release(c, b);
    for (int r : recs) rec_release(c, r);
  }
};

// Shared implementation of cb_eval (n_lists = 1) and cb_eval_batch.
static int eval_impl(cb_ctx* c, int snapshot_in, int n_lists, const int32_t* offsets_in, const int32_t* nodes_in,
                     const int32_t* children_in, const int32_t* pslots_in, const double* pi, int flags,
                     int* snapshot_out, double* lnl_out) {
  REQUIRE(c && c->n_states > 0, "cb_set_tips must come first");
  REQUIRE(offsets_in && nodes_in && children_in && pslots_in && pi, "null argument");
  REQUIRE(snapshot_in < 0 || snapshot_valid(c, snapshot_in), "invalid snapshot %d", snapshot_in);
  const int C = c->n_cats, N = c->n_taxa, n_nodes = 2 * N;
  REQUIRE(n_lists >= 1 && offsets_in[0] == 0 && offsets_in[n_lists] > 0, "empty op list");
  const int total_in = offsets_in[n_lists];
  const bool want_snap = (flags & CB_EVAL_WANT_SNAPSHOT) != 0;
  REQUIRE(!(want_snap && n_lists != 1), "snapshots are only kept for single evaluations");
  CU(cudaSetDevice(c->device));

  const double t_begin = now_us();
  // ---- the plan: cached per (op list, flags) for full evaluations, built on the spot for dirty paths
  const int split_env = getenv("CYBAYES_WALK_SPLIT") ? atoi(getenv("CYBAYES_WALK_SPLIT")) : 0;
  EvalPlan* plan = nullptr;
  if (snapshot_in < 0 && !c->no_plan_cache) {
    for (auto& p : c->plans)
      if (p.n_lists == n_lists && p.flags == (flags & PLAN_FLAG_MASK) && p.split_env == split_env &&
          (int)p.key_nodes.size() == total_in && memcmp(p.key_offsets.data(), offsets_in, (size_t)(n_lists + 1) * 4) == 0 &&
          memcmp(p.key_nodes.data(), nodes_in, (size_t)total_in * 4) == 0 &&
          memcmp(p.key_children.data(), children_in, (size_t)total_in * 8) == 0) {
        plan = &p;
        break;
      }
    if (!plan) {
      if ((int)c->plans.size() < PLAN_CACHE_SIZE) {
        c->plans.emplace_back();
        plan = &c->plans.back();
      } else {  // evict the least recently used
        plan = &c->plans[0];
        for (auto& p : c->plans)
          if (p.stamp < plan->stamp) plan = &p;
      }
      plan->n_lists = 0;  // invalid while it is rebuilt
      plan->split_env = split_env;
      if (build_plan(c, nullptr, n_lists, offsets_in, nodes_in, children_in, flags, *plan)) { plan->key_nodes.clear(); return 1; }
      plan->n_lists = n_lists;
      plan->flags = flags & PLAN_FLAG_MASK;
      plan->key_offsets.assign(offsets_in, offsets_in + n_lists + 1);
      plan->key_nodes.assign(nodes_in, nodes_in + total_in);
      plan->key_children.assign(children_in, children_in + 2 * (size_t)total_in);
      c->plan_builds++;
    }
    plan->stamp = ++c->plan_clock;
  } else {
    plan = &c->scratch_plan;
    plan->split_env = split_env;
    if (build_plan(c, snapshot_in >= 0 ? &c->snaps[snapshot_in] : nullptr, n_lists, offsets_in, nodes_in, children_in, flags, *plan))
      return 1;
    c->plan_builds++;
  }
  const int total_ops = (int)plan->ops.size();
  const int n_ranges = (int)plan->ranges.size();

  // every P slot the ops name, before anything is acquired
  for (size_t i = 0; i < (size_t)total_in * 2 * C; ++i)
    REQUIRE(pslots_in[i] >= 0 && pslots_in[i] < c->pmat_cap, "P slot %d out of range (reserved %d)", pslots_in[i], c->pmat_cap);

  if (ensure_staging(c, total_ops, n_ranges, n_lists)) return 1;
  CU(cudaEventSynchronize(c->ev_stage));  // previous H2D of the staging area finished
  const double t_planned = now_us();

  // ---- fill the descriptors: buffers, pointers, P slots
  const Snapshot* sin = snapshot_in >= 0 ? &c->snaps[snapshot_in] : nullptr;
  EvalGuard guard{c};
  std::vector<int>& new_bufs = c->work_new_bufs;
  std::vector<int>& new_nodes = c->work_new_nodes;
  std::vector<int>& new_cherry_nodes = c->work_cherry_nodes;
  new_bufs.clear(); new_nodes.clear(); new_cherry_nodes.clear();
  const char* codes = (const char*)c->d_codes;
  const size_t row_bytes = (size_t)c->P * c->code_bytes;
  OpDesc* const h_ops = reinterpret_cast<OpDesc*>(c->h_stage);
  const size_t off_ranges = (size_t)total_ops * sizeof(OpDesc), off_pi = off_ranges + (size_t)n_ranges * sizeof(RangeDesc);
  for (int p = 0; p < total_ops; ++p) {
    const PlanOp& po = plan->ops[p];
    OpDesc& op = h_ops[p];
    op.is_root = po.is_root;
    op.pad_ = po.stream;
    op.spill = (po.spill ? 1 : 0) | (po.pushed ? 2 : 0);
    op.frec_out = -1;
    op.pf_buf = po.pf_buf;
    op.out_buf = po.out_buf;
    op.dst = nullptr;
    op.dst_scale = nullptr;
    if (po.keep) {
      int bi;
      if (buffer_acquire(c, &bi)) return 1;
      guard.bufs.push_back(bi);
      op.dst = c->buffers[bi].data;
      op.dst_scale = c->buffers[bi].scale;
      if (want_snap) {
        new_bufs.push_back(bi);
        new_nodes.push_back(po.node);
      }
    }
    for (int kx = 0; kx < 2; ++kx) {
      const PlanChild& pc = po.ch[kx];
      op.kind[kx] = pc.kind;
      op.src[kx] = nullptr;
      op.src_scale[kx] = nullptr;
      op.ctip[kx][0] = op.ctip[kx][1] = nullptr;
      op.crec_out[kx] = -1;
      op.in_buf[kx] = -1;
      if (pc.edge >= 0) {
        const int32_t* ps = pslots_in + (size_t)pc.edge * C;
        for (int q = 0; q < C; ++q) op.pslot[kx][q] = ps[q];
      } else {  // an edge of a record of the input snapshot: its P copies live in the library's pool
        for (int q = 0; q < C; ++q) op.pslot[kx][q] = CB_LIB_SLOT | (~pc.edge + q);
      }
      for (int q = C; q < CB_MAX_CATS; ++q) op.pslot[kx][q] = 0;
      switch (pc.kind) {
        case SRC_TIP:
          op.src[kx] = codes + (size_t)(pc.ref - 1) * row_bytes;
          break;
        case SRC_BUFFER:
          if (pc.ref >= 0) {
            op.src[kx] = h_ops[pc.ref].dst;
            op.src_scale[kx] = h_ops[pc.ref].dst_scale;
          } else {
            const Buffer& bf = c->buffers[sin->buf_of_node[~pc.ref]];
            op.src[kx] = bf.data;
            op.src_scale[kx] = bf.scale;
          }
          break;
        case SRC_SMALL:
          op.in_buf[kx] = pc.ref;
          break;
        case SRC_STACK:
          if (po.pf_buf >= 0 && kx == 1) {   // a prefetched stored partial: the source is a buffer, the op reads the tile buffer
            op.in_buf[kx] = po.pf_buf;
            op.src[kx] = pc.ref >= 0 ? (const void*)h_ops[pc.ref].dst : (const void*)c->buffers[sin->buf_of_node[~pc.ref]].data;
          } else {
            op.in_buf[kx] = pc.ref;
          }
          break;
        case SRC_CHERRY:
          if (pc.ref >= 0) {  // folded out of the caller's list: its P matrices are the caller's slots
            const int fo = pc.ref;
            for (int t = 0; t < 2; ++t) {
              const int tip = children_in[2 * fo + t];
              op.ctip[kx][t] = codes + (size_t)(tip - 1) * row_bytes;
              const int32_t* cs = pslots_in + (size_t)(2 * fo + t) * C;
              for (int q = 0; q < CB_S2_MAX_CATS; ++q) op.cslot[kx][t][q] = q < C ? cs[q] : 0;
            }
            if (want_snap) {
              int r;
              if (rec_acquire(c, children_in[2 * fo], children_in[2 * fo + 1], &r)) return 1;
              guard.recs.push_back(r);
              op.crec_out[kx] = r;
              new_cherry_nodes.push_back(nodes_in[fo]);
            }
          } else {            // kept by the input snapshot: its P matrices live in the library's pool
            const int rec = sin->cherry_of_node[~pc.ref];
            for (int t = 0; t < 2; ++t) {
              op.ctip[kx][t] = codes + (size_t)(c->recs[rec].tip[t] - 1) * row_bytes;
              for (int q = 0; q < CB_S2_MAX_CATS; ++q) op.cslot[kx][t][q] = q < C ? (CB_LIB_SLOT | (rec * 2 * C + t * C + q)) : 0;
            }
          }
          break;
        default: break;
      }
    }
    if (po.make_rec) {  // the node stays in the returned snapshot as a record: children (tip ids / cherry node ids) + P copies
      int ids[2];
      for (int kx = 0; kx < 2; ++kx) {
        const PlanChild& pc = po.ch[kx];
        ids[kx] = pc.kind == SRC_TIP ? pc.ref : (pc.ref >= 0 ? nodes_in[pc.ref] : ~pc.ref);
      }
      int r;
      if (rec_acquire(c, ids[0], ids[1], &r)) return 1;
      guard.recs.push_back(r);
      op.frec_out = r;
      new_cherry_nodes.push_back(po.node);
    }
  }
  memcpy(c->h_stage + off_ranges, plan->ranges.data(), (size_t)n_ranges * sizeof(RangeDesc));
  memcpy(c->h_stage + off_pi, pi, (size_t)c->n_states * 8);

  const double t_filled = now_us();
  if (ensure_lib_pool(c)) return 1;
  // upload descriptors + ranges + pi with one copy, launch
  const size_t stage_bytes = off_pi + (size_t)c->n_states * 8;
  CU(cudaMemcpyAsync(c->d_stage, c->h_stage, stage_bytes, cudaMemcpyHostToDevice, c->stream));
  CU(cudaEventRecord(c->ev_stage, c->stream));
  c->h2d += (int64_t)stage_bytes;

  if (c->dmma_rc) {
    // every P matrix the ops use, re-laid out into the shared-memory stage image, in consumption order
    const int S8 = (c->n_states + 7) / 8 * 8;
    const size_t need = (size_t)total_ops * 2 * C * (S8 + RC_EXTRA_ROWS) * S8 * 8;
    if (need > c->staged_bytes) {
      CU(cudaStreamSynchronize(c->stream));
      if (c->d_staged) dev_free(c, c->d_staged, c->staged_bytes);
      c->d_staged = nullptr;
      c->staged_bytes = 0;
      const size_t cap = std::max(need, (size_t)64 << 20);
      if (dev_alloc(c, (void**)&c->d_staged, cap)) return 1;
      c->staged_bytes = cap;
    }
  }
  LaunchConst k = make_const(c);
  k.ranges = reinterpret_cast<const RangeDesc*>(c->d_stage + off_ranges);
  k.pi = reinterpret_cast<const double*>(c->d_stage + off_pi);
  // Sharded over GPUs: the root kernel all-reduces the shard sums itself over peer memory (batches beyond CB_MB_OUTS
  // results: ncclAllReduce).  Either way without NCCL in the step the kernel writes lnL straight into mapped host
  // memory: no device -> host copy.
  const bool fused = c->comm != nullptr && c->fused_allreduce && n_lists <= CB_MB_OUTS;
  if (fused) {
    k.n_ranks = c->n_ranks;
    k.my_rank = c->rank;
    k.epoch = ++c->epoch;
    k.mailbox = c->d_mailbox;
    k.peer_mailbox = c->d_peer_mailbox;
    k.comm_error = c->d_comm_error;
  }
  const bool mapped = c->comm == nullptr || fused;
  if (mapped) {
    double* dev_view = nullptr;
    CU(cudaHostGetDevicePointer((void**)&dev_view, c->h_results, 0));
    k.results = dev_view;
  }
  if (c->timing) CU(cudaEventRecord(c->ev0, c->stream));
  if (c->dmma_rc) {
    const unsigned jobs = (unsigned)(total_ops * 2 * C);
    switch ((c->n_states + 7) / 8 * 8) {
#define CB_RS_CASE(SS) case SS: rc_restage_kernel<SS><<<jobs, 256, 0, c->stream>>>(k, total_ops, c->d_staged); break
      CB_RS_CASE(16); CB_RS_CASE(24); CB_RS_CASE(32); CB_RS_CASE(40); CB_RS_CASE(48); CB_RS_CASE(56); CB_RS_CASE(64);
#undef CB_RS_CASE
      default: return fail("internal error: no register-carried DMMA kernel for %d states", c->n_states);
    }
    CU(cudaGetLastError());
    c->launches += 1;
  }
  if (launch_images(c, k, total_ops)) return 1;
  if (c->timing) CU(cudaEventRecord(c->ev_main0, c->stream));
  for (const PlanLaunch& pl : plan->launches)
    if (launch_ranges(c, k, pl.r_begin, pl.r_end, pl.max_ops, pl.n_bufs)) return 1;
  if (c->timing) CU(cudaEventRecord(c->ev_main1, c->stream));
  if (!c->family_s2) {
    dim3 grid((unsigned)((c->P + 255) / 256), (unsigned)n_lists);
    root_combine_kernel<<<grid, 256, 0, c->stream>>>(k);
    CU(cudaGetLastError());
    c->launches += 1;
  }
  if (c->timing) CU(cudaEventRecord(c->ev1, c->stream));
  c->timing_valid = c->timing;
  c->last_bytes_written = plan->bytes_written;
  c->last_bytes_read = plan->bytes_read;
  c->last_counts[0] = total_ops - plan->n_inlined; c->last_counts[1] = plan->n_stored; c->last_counts[2] = plan->n_buffer_reads;
  c->last_counts[3] = plan->n_stack; c->last_counts[4] = plan->n_spills; c->last_counts[5] = plan->n_cherries;
  c->last_counts[6] = (int)plan->launches.size(); c->last_counts[7] = plan->n_small_recs;

  if (c->comm && !fused) {
    int r = g_nccl.AllReduce(c->d_results, c->d_results, (size_t)n_lists, NCCL_DOUBLE, NCCL_SUM, c->comm, c->stream);
    REQUIRE(r == 0, "ncclAllReduce: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error");
  }
  if (!mapped) CU(cudaMemcpyAsync(c->h_results, c->d_results, (size_t)n_lists * 8, cudaMemcpyDeviceToHost, c->stream));
  c->d2h += (int64_t)n_lists * 8;
  c->last_n_out = n_lists;

  const double t_launched = now_us();
  // bookkeeping (stream-ordered: temporaries may be recycled by later launches on this stream)
  guard.armed = false;
  if (want_snap) {
    int sid;
    if (!c->free_snaps.empty()) {
      sid = c->free_snaps.back();
      c->free_snaps.pop_back();
    } else {
      c->snaps.emplace_back();
      sid = (int)c->snaps.size() - 1;
    }
    Snapshot& sn = c->snaps[sid];
    sin = snapshot_in >= 0 ? &c->snaps[snapshot_in] : nullptr;  // vector may have moved
    if (sin) sn.buf_of_node = sin->buf_of_node; else sn.buf_of_node.assign(n_nodes, -1);
    if (sin) sn.cherry_of_node = sin->cherry_of_node; else sn.cherry_of_node.assign(n_nodes, -1);
    sn.buf_of_node.resize(n_nodes, -1);
    sn.cherry_of_node.resize(n_nodes, -1);
    sn.refs = 1;
    // a recomputed node replaces whatever the input snapshot held for it (buffer or folded cherry)
    for (size_t i = 0; i < new_nodes.size(); ++i) {
      sn.buf_of_node[new_nodes[i]] = -2 - (int)i;
      sn.cherry_of_node[new_nodes[i]] = -1;
    }
    for (size_t i = 0; i < new_cherry_nodes.size(); ++i) {
      sn.buf_of_node[new_cherry_nodes[i]] = -1;
      sn.cherry_of_node[new_cherry_nodes[i]] = -2 - (int)i;
    }
    for (int nd = 0; nd < n_nodes; ++nd) {
      int32_t& bi = sn.buf_of_node[nd];
      if (bi >= 0) c->buffers[bi].refs++;
      else if (bi <= -2) bi = new_bufs[-2 - bi];  // ownership moves from this evaluation to the snapshot
      int32_t& ri = sn.cherry_of_node[nd];
      if (ri >= 0) c->recs[ri].refs++;
      else if (ri <= -2) ri = guard.recs[-2 - ri];
    }
    if (snapshot_out) *snapshot_out = sid;
  } else {
    for (int bi : guard.bufs) buffer_release(c, bi);   // temporaries of an evaluation that keeps no snapshot
    if (snapshot_out) *snapshot_out = -1;
  }

  const double t_booked = now_us();
  c->host_us[0] += t_planned - t_begin;
  c->host_us[1] += t_filled - t_planned;
  c->host_us[2] += t_launched - t_filled;
  c->host_us[4] += t_booked - t_launched;
  c->host_us[5] += 1.0;
  if (!(flags & CB_EVAL_NO_SYNC)) {
    CU(cudaStreamSynchronize(c->stream));
    c->host_us[3] += now_us() - t_booked;
    if (fused && c->h_results[0] != c->h_results[0]) {  // NaN: did a peer fail to deliver its shard sum?
      int32_t err = 0;
      CU(cudaMemcpy(&err, c->d_comm_error, 4, cudaMemcpyDeviceToHost));
      REQUIRE(err == 0, "fused all-reduce: a peer GPU never delivered its shard sum (rank %d of %d waited 10 s)", c->rank, c->n_ranks);
    }
    if (lnl_out) memcpy(lnl_out, c->h_results, (size_t)n_lists * 8);
  }
  return 0;
}

extern "C" int cb_eval(cb_ctx* c, int snapshot_in, int n_ops, const int32_t* nodes, const int32_t* children,
                       const int32_t* pslots, const double* pi, int flags, int* snapshot_out, double* lnl_out) {
  const int32_t offsets[2] = {0, n_ops};
  return guarded([&] { return eval_impl(c, snapshot_in, 1, offsets, nodes, children, pslots, pi, flags, snapshot_out, lnl_out); });
}

extern "C" int cb_eval_batch(cb_ctx* c, int snapshot_in, int n_batch, const int32_t* op_offsets, const int32_t* nodes,
                             const int32_t* children, const int32_t* pslots, const double* pi, double* lnl_out) {
  REQUIRE(n_batch >= 1, "empty batch");
  return guarded([&] { return eval_impl(c, snapshot_in, n_batch, op_offsets, nodes, children, pslots, pi, 0, nullptr, lnl_out); });
}

extern "C" int cb_result_wait(cb_ctx* c, double* lnl_out) {
  REQUIRE(c, "null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  if (lnl_out && c->h_results) memcpy(lnl_out, c->h_results, (size_t)c->last_n_out * 8);
  return 0;
}

// --------------------------------------------------------------------------- introspection
extern "C" int cb_stats(cb_ctx* c, int64_t* launches, int64_t* h2d, int64_t* d2h, int64_t* dev_bytes) {
  REQUIRE(c, "null argument");
  if (launches) *launches = c->launches;
  if (h2d) *h2d = c->h2d;
  if (d2h) *d2h = c->d2h;
  if (dev_bytes) *dev_bytes = c->dev_bytes;
  return 0;
}
// cudaMemGetInfo costs 0.5 - 20 ms once tens of GB are allocated, far too much to ask per evaluation: the driver is asked
// once per device; after that free memory is tracked from the library's own allocations (all contexts of the process).
static int64_t g_dev_bytes[64] = {0};     // bytes this process holds per device through dev_alloc
static void dev_account(int device, int64_t delta) { g_dev_bytes[device & 63] += delta; }
static int64_t g_free_at_query[64], g_held_at_query[64], g_total[64];
static bool g_queried[64] = {false};
extern "C" int cb_mem_info(cb_ctx* c, int64_t* free_bytes, int64_t* total_bytes, int64_t* pooled_bytes, int64_t* partial_bytes) {
  REQUIRE(c, "null argument");
  const int d = c->device & 63;
  if (!g_queried[d]) {
    CU(cudaSetDevice(c->device));
    size_t fr = 0, tot = 0;
    CU(cudaMemGetInfo(&fr, &tot));
    g_free_at_query[d] = (int64_t)fr;
    g_total[d] = (int64_t)tot;
    g_held_at_query[d] = g_dev_bytes[d];
    g_queried[d] = true;
  }
  int64_t fr = g_free_at_query[d] - (g_dev_bytes[d] - g_held_at_query[d]), tot = g_total[d];
  if (c->max_dev_bytes > 0) {  // a capped context sees its cap
    tot = c->max_dev_bytes;
    fr = std::max<int64_t>(0, std::min<int64_t>(fr, c->max_dev_bytes - c->dev_bytes));
  }
  if (free_bytes) *free_bytes = std::max<int64_t>(0, fr);
  if (total_bytes) *total_bytes = tot;
  if (pooled_bytes) *pooled_bytes = (int64_t)c->free_buffers.size() * (int64_t)c->buffer_bytes;
  if (partial_bytes) *partial_bytes = (int64_t)c->buffer_bytes;
  return 0;
}
extern "C" int cb_last_eval_ms(cb_ctx* c, float* ms) {
  REQUIRE(c && ms && c->timing_valid, "no evaluation has been timed");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(c->ev1));
  CU(cudaEventElapsedTime(ms, c->ev0, c->ev1));
  return 0;
}
extern "C" int cb_last_eval_main_ms(cb_ctx* c, float* ms) {
  REQUIRE(c && ms && c->timing_valid, "no evaluation has been timed");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(c->ev_main1));
  CU(cudaEventElapsedTime(ms, c->ev_main0, c->ev_main1));
  return 0;
}
extern "C" int cb_host_profile(cb_ctx* c, double* us6, int reset) {
  REQUIRE(c && us6, "null argument");
  memcpy(us6, c->host_us, sizeof c->host_us);
  if (reset) memset(c->host_us, 0, sizeof c->host_us);
  return 0;
}
extern "C" int cb_last_eval_info(cb_ctx* c, int64_t* bytes_written, int64_t* bytes_read, int32_t* counts8) {
  REQUIRE(c && c->timing_valid, "no evaluation has run");
  if (bytes_written) *bytes_written = c->last_bytes_written;
  if (bytes_read) *bytes_read = c->last_bytes_read;
  if (counts8) memcpy(counts8, c->last_counts, sizeof c->last_counts);
  return 0;
}
extern "C" int cb_mark(cb_ctx* c, int which) {
  REQUIRE(c && (which == 0 || which == 1), "bad argument");
  CU(cudaSetDevice(c->device));
  CU(cudaEventRecord(c->ev_mark[which], c->stream));
  return 0;
}
extern "C" int cb_mark_elapsed_ms(cb_ctx* c, float* ms) {
  REQUIRE(c && ms, "null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(c->ev_mark[1]));
  CU(cudaEventElapsedTime(ms, c->ev_mark[0], c->ev_mark[1]));
  return 0;
}
extern "C" int cb_sync(cb_ctx* c) {
  REQUIRE(c, "null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}
// FP64 tensor peak of this GPU, measured from registers: every warp keeps 4 independent DMMA m8n8k4 accumulator
// chains going (16 warps per SM).  The denominator of the S = 64 roofline in bench.py (MEASURED_PEAKS.json has no
// FP64 figure).
__global__ void __launch_bounds__(512) fp64_peak_kernel(double* out, int iters) {
  const double a = 1.0 + 1e-9 * threadIdx.x, b = 1.0 - 1e-9 * threadIdx.x;
  double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0, c4 = 0.0, c5 = 0.0, c6 = 0.0, c7 = 0.0;
#pragma unroll 1
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      rc_dmma(c0, c1, a, b);
      rc_dmma(c2, c3, a, b);
      rc_dmma(c4, c5, a, b);
      rc_dmma(c6, c7, a, b);
    }
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = c0 + c1 + c2 + c3 + c4 + c5 + c6 + c7;
}
extern "C" int cb_fp64_peak(cb_ctx* c, double* tflops_out) {
  REQUIRE(c && tflops_out, "null argument");
  CU(cudaSetDevice(c->device));
  const int blocks = c->sm_count, threads = 512, iters = 20000;
  double* d = nullptr;
  CU(cudaMalloc(&d, (size_t)blocks * threads * 8));
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {  // first repetition warms up
    CU(cudaEventRecord(c->ev_mark[0], c->stream));
    fp64_peak_kernel<<<blocks, threads, 0, c->stream>>>(d, iters);
    CU(cudaEventRecord(c->ev_mark[1], c->stream));
    CU(cudaEventSynchronize(c->ev_mark[1]));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, c->ev_mark[0], c->ev_mark[1]));
    if (rep > 0 && ms < best) best = ms;
  }
  CU(cudaGetLastError());
  cudaFree(d);
  const double flops = (double)blocks * (threads / 32) * (double)iters * 32.0 * 512.0;  // 32 DMMAs per iteration, 2*8*8*4 flop each
  *tflops_out = flops / (best * 1e-3) / 1e12;
  return 0;
}
extern "C" int cb_flush_l2(cb_ctx* c) {
  REQUIRE(c, "null argument");
  CU(cudaSetDevice(c->device));
  if (!c->d_flush) {
    c->flush_bytes = (size_t)256 << 20;  // 2x the 126 MB L2
    if (dev_alloc(c, &c->d_flush, c->flush_bytes)) return 1;
  }
  CU(cudaMemsetAsync(c->d_flush, 0x5a, c->flush_bytes, c->stream));
  return 0;
}


// --------------------------------------------------------------------------- pattern compression at scale
// Site-pattern compression (SURVEY 8f rank 2; the reference has none, utils.pyx:94-120 keeps every column): unique
// alignment columns in order of first appearance, with multiplicities.  For alignments of 10^5 .. 10^7 columns the
// column comparison is done on the GPU: one thread per column folds its n_taxa codes into a 128-bit hash (coalesced
// reads, HBM-bound), the host groups equal hashes (sort of n_sites 16-byte keys), and a second kernel verifies
// column by column that every site really equals the representative of its group -- so the result is exact, not
// probabilistic (a hash collision is reported, the caller then takes the exact host route).
template <typename T>
__global__ void __launch_bounds__(256) column_hash_kernel(const T* __restrict__ codes, int n_taxa, int64_t n_sites,
                                                           unsigned long long* __restrict__ out) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_sites) return;
  unsigned long long h1 = 0xcbf29ce484222325ull, h2 = 0x9e3779b97f4a7c15ull;
  for (int t = 0; t < n_taxa; ++t) {
    const unsigned long long v = (unsigned long long)codes[(int64_t)t * n_sites + s] + 1ull;
    h1 = (h1 ^ v) * 0x100000001b3ull;                                    // FNV-1a
    h2 = (h2 + v * 0xff51afd7ed558ccdull + (unsigned long long)t) * 0xc4ceb9fe1a85ec53ull;
    h2 ^= h2 >> 29;
  }
  out[2 * s] = h1;
  out[2 * s + 1] = h2;
}
template <typename T>
__global__ void __launch_bounds__(256) column_verify_kernel(const T* __restrict__ codes, int n_taxa, int64_t n_sites,
                                                             const int64_t* __restrict__ rep_of_site, unsigned long long* n_bad) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_sites) return;
  const int64_t r = rep_of_site[s];
  if (r == s) return;
  bool same = true;
  for (int t = 0; t < n_taxa && same; ++t) same = codes[(int64_t)t * n_sites + s] == codes[(int64_t)t * n_sites + r];
  if (!same) atomicAdd(n_bad, 1ull);
}
static int compress_impl(int device, const void* codes, int n_taxa, int64_t n_sites, int code_bytes, int64_t* site_to_pattern,
                         int64_t* first_site, double* weights, int64_t* n_patterns_out) {
  REQUIRE(codes && site_to_pattern && first_site && weights && n_patterns_out, "null argument");
  REQUIRE(n_taxa >= 1 && n_sites >= 1 && (code_bytes == 1 || code_bytes == 2), "bad alignment shape");
  int n_dev = 0;
  cudaError_t e0 = cudaGetDeviceCount(&n_dev);
  if (e0 != cudaSuccess || n_dev == 0) return fail("no CUDA device available (%s); cybayes_b200 has no CPU fallback", cudaGetErrorString(e0));
  REQUIRE(device >= 0 && device < n_dev, "device %d out of range (have %d)", device, n_dev);
  CU(cudaSetDevice(device));
  void* d_codes = nullptr;
  unsigned long long *d_hash = nullptr, *d_bad = nullptr;
  int64_t* d_rep = nullptr;
  const size_t code_total = (size_t)n_taxa * n_sites * code_bytes;
  auto cleanup = [&] { cudaFree(d_codes); cudaFree(d_hash); cudaFree(d_bad); cudaFree(d_rep); };
#define CUC(call)                                                                                              \
  do {                                                                                                         \
    cudaError_t e_ = (call);                                                                                   \
    if (e_ != cudaSuccess) { cleanup(); return fail("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); } \
  } while (0)
  CUC(cudaMalloc(&d_codes, code_total));
  CUC(cudaMalloc(&d_hash, (size_t)n_sites * 16));
  CUC(cudaMalloc(&d_rep, (size_t)n_sites * 8));
  CUC(cudaMalloc(&d_bad, 8));
  CUC(cudaMemcpy(d_codes, codes, code_total, cudaMemcpyHostToDevice));
  const unsigned blocks = (unsigned)((n_sites + 255) / 256);
  if (code_bytes == 1) column_hash_kernel<uint8_t><<<blocks, 256>>>((const uint8_t*)d_codes, n_taxa, n_sites, d_hash);
  else column_hash_kernel<uint16_t><<<blocks, 256>>>((const uint16_t*)d_codes, n_taxa, n_sites, d_hash);
  CUC(cudaGetLastError());
  std::vector<unsigned long long> h((size_t)n_sites * 2);
  CUC(cudaMemcpy(h.data(), d_hash, (size_t)n_sites * 16, cudaMemcpyDeviceToHost));
  // group equal hashes; the representative of a group is its first site
  std::vector<int64_t> idx((size_t)n_sites);
  for (int64_t i = 0; i < n_sites; ++i) idx[i] = i;
  std::sort(idx.begin(), idx.end(), [&](int64_t a, int64_t b) {
    if (h[2 * a] != h[2 * b]) return h[2 * a] < h[2 * b];
    if (h[2 * a + 1] != h[2 * b + 1]) return h[2 * a + 1] < h[2 * b + 1];
    return a < b;
  });
  std::vector<int64_t> rep((size_t)n_sites);
  for (int64_t i = 0; i < n_sites;) {
    int64_t j = i;
    while (j < n_sites && h[2 * idx[j]] == h[2 * idx[i]] && h[2 * idx[j] + 1] == h[2 * idx[i] + 1]) rep[idx[j++]] = idx[i];
    i = j;
  }
  CUC(cudaMemcpy(d_rep, rep.data(), (size_t)n_sites * 8, cudaMemcpyHostToDevice));
  CUC(cudaMemset(d_bad, 0, 8));
  if (code_bytes == 1) column_verify_kernel<uint8_t><<<blocks, 256>>>((const uint8_t*)d_codes, n_taxa, n_sites, d_rep, d_bad);
  else column_verify_kernel<uint16_t><<<blocks, 256>>>((const uint16_t*)d_codes, n_taxa, n_sites, d_rep, d_bad);
  CUC(cudaGetLastError());
  unsigned long long bad = 0;
  CUC(cudaMemcpy(&bad, d_bad, 8, cudaMemcpyDeviceToHost));
#undef CUC
  cleanup();
  REQUIRE(bad == 0, "128-bit column hashes collided for %llu sites: use the exact host route", bad);
  // patterns in order of first appearance (the representative is the smallest site of its group)
  int64_t n_pat = 0;
  std::vector<int64_t> pat_of_rep((size_t)n_sites, -1);
  for (int64_t s = 0; s < n_sites; ++s) {
    const int64_t r = rep[s];
    if (r == s) {
      pat_of_rep[s] = n_pat;
      first_site[n_pat] = s;
      weights[n_pat] = 0.0;
      ++n_pat;
    }
    site_to_pattern[s] = pat_of_rep[r];   // r <= s: already numbered
    weights[pat_of_rep[r]] += 1.0;
  }
  *n_patterns_out = n_pat;
  return 0;
}
extern "C" int cb_compress_patterns(int device, const void* codes, int n_taxa, int64_t n_sites, int code_bytes,
                                    int64_t* site_to_pattern, int64_t* first_site, double* weights, int64_t* n_patterns_out) {
  return guarded([&] { return compress_impl(device, codes, n_taxa, n_sites, code_bytes, site_to_pattern, first_site, weights, n_patterns_out); });
}

// ------------------------------------------------------------------------------- native generation loop
#include "mcmc_native.cuh"

struct cb_chain {
  cbm::Chain ch;
};
static int chain_err(cb_chain* c, int rc) {
  if (rc && !c->ch.err.empty()) {
    g_err = c->ch.err;
    c->ch.err.clear();
  }
  return rc;
}
extern "C" int cb_chain_create(cb_ctx* ctx, const cb_chain_backend* be, int n_taxa, int n_states, int n_cats, int model, int binary,
                               int root, int slot_base, int slot_count, int host_exp_max, int n_params, const int32_t* param_ids,
                               const double* params_cdf, const double* tree_cdf, const double* bl_cdf, cb_chain** out) {
  return guarded([&] {
    REQUIRE(be && out && param_ids && params_cdf && tree_cdf && bl_cdf, "null argument");
    REQUIRE(ctx || (be->pmat_build && be->eval && be->snapshot_release), "a chain needs a context or a full backend");
    REQUIRE(be->site_rates && be->f81_beta && be->gtr_eig, "host callbacks are required");
    REQUIRE(n_taxa >= 2 && n_states >= 2 && n_cats >= 1 && n_cats <= CB_MAX_CATS && model >= 0 && model <= 2, "bad chain shape");
    REQUIRE(root == 2 * n_taxa - 1, "root must be node 2 * n_taxa - 1 (mcmc_gamma.pyx:270-287)");
    REQUIRE(slot_count >= 2 * (2 * n_taxa - 2) * n_cats + 8 * n_cats, "slot range too small for the chain");
    cb_chain* c = new cb_chain();
    cbm::Chain& ch = c->ch;
    ch.ctx = ctx;
    ch.be = *be;
    ch.n_taxa = n_taxa; ch.S = n_states; ch.C = n_cats; ch.model = model; ch.binary = binary != 0; ch.root = root;
    ch.host_exp_max = host_exp_max;
    if (const char* e = getenv("CYBAYES_CHAIN_LNL_FIRST")) ch.lnl_first = atoi(e) != 0 ? 1 : 0;   // default: automatic
    ch.param_ids.assign(param_ids, param_ids + n_params);
    ch.params_cdf.assign(params_cdf, params_cdf + n_params);
    ch.tree_cdf.assign(tree_cdf, tree_cdf + 2);
    ch.bl_cdf.assign(bl_cdf, bl_cdf + 2);
    for (int i = slot_count - 1; i >= 0; --i) ch.free_slots.push_back(slot_base + i);
    for (auto& w : ch.py.mt) w = 0;
    for (auto& w : ch.np_.mt) w = 0;
    *out = c;
    return 0;
  });
}
extern "C" int cb_chain_set_state(cb_chain* c, int n_edges, const int32_t* parents, const int32_t* children, const double* lengths,
                                  const double* pi, int n_rates, const double* rates, double alpha, const double* site_rates, double beta,
                                  const double* gtr_eig, double* lnl_out) {
  return guarded([&] {
    REQUIRE(c && parents && children && lengths && pi && rates && site_rates, "null argument");
    cbm::Chain& ch = c->ch;
    REQUIRE(n_edges == 2 * ch.n_taxa - 2, "a rooted binary tree on %d taxa has %d edges", ch.n_taxa, 2 * ch.n_taxa - 2);
    REQUIRE(ch.model != 2 || gtr_eig, "GTR needs the eigensystem of the start state");
    for (const cbm::Edge& e : ch.tree) cbm::free_slots(&ch, e.slot, ch.C);
    cbm::be_release(&ch, ch.snap);
    ch.snap = -1;
    ch.tree.clear();
    for (int i = 0; i < n_edges; ++i) {
      REQUIRE(parents[i] > ch.n_taxa && parents[i] < 2 * ch.n_taxa && children[i] >= 1 && children[i] < 2 * ch.n_taxa, "bad edge %d", i);
      ch.tree.push_back(cbm::Edge{parents[i], children[i], lengths[i], {0}});
    }
    ch.pi.assign(pi, pi + ch.S);
    ch.rates.assign(rates, rates + n_rates);
    ch.site_rates.assign(site_rates, site_rates + ch.C);
    ch.alpha = alpha;
    ch.beta = beta;
    ch.gtr.clear();
    if (gtr_eig) ch.gtr.assign(gtr_eig, gtr_eig + ch.S + 2 * (size_t)ch.S * ch.S);
    if (chain_err(c, cbm::build_all(&ch, ch.tree, ch.pi.data(), ch.beta, ch.gtr.data(), ch.site_rates.data()))) return 1;
    std::vector<int32_t> k0, k1, par;
    cbm::build_kids(&ch, ch.tree, k0, k1, par);
    for (int nd = ch.n_taxa + 1; nd < 2 * ch.n_taxa; ++nd) REQUIRE(k0[nd] >= 0 && k1[nd] >= 0, "node %d does not have two children", nd);
    cbm::plan_nodes(&ch, k0, k1);
    REQUIRE((int)ch.order_nodes.size() == ch.n_taxa - 1, "the edges do not form a tree rooted at %d", ch.root);
    if (chain_err(c, cbm::evaluate(&ch, ch.tree, k0, k1, ch.order_nodes, -1, ch.pi.data(), &ch.snap, &ch.lnl))) return 1;
    if (lnl_out) *lnl_out = ch.lnl;
    return 0;
  });
}
extern "C" int cb_chain_set_rng(cb_chain* c, const uint32_t* py_mt, int py_pos, const uint32_t* np_mt, int np_pos) {
  REQUIRE(c && py_mt && np_mt && py_pos >= 0 && py_pos <= 624 && np_pos >= 0 && np_pos <= 624, "bad generator state");
  memcpy(c->ch.py.mt, py_mt, sizeof c->ch.py.mt);
  memcpy(c->ch.np_.mt, np_mt, sizeof c->ch.np_.mt);
  c->ch.py.pos = py_pos;
  c->ch.np_.pos = np_pos;
  return 0;
}
extern "C" int cb_chain_get_rng(cb_chain* c, uint32_t* py_mt, int* py_pos, uint32_t* np_mt, int* np_pos) {
  REQUIRE(c && py_mt && np_mt && py_pos && np_pos, "null argument");
  memcpy(py_mt, c->ch.py.mt, sizeof c->ch.py.mt);
  memcpy(np_mt, c->ch.np_.mt, sizeof c->ch.np_.mt);
  *py_pos = c->ch.py.pos;
  *np_pos = c->ch.np_.pos;
  return 0;
}
extern "C" int cb_chain_run(cb_chain* c, int64_t n_gens, int8_t* move, int8_t* accepted, double* current_ll, double* proposed_ll,
                            double* ll_ratio, double* log_u) {
  return guarded([&] {
    REQUIRE(c && n_gens >= 0 && c->ch.snap >= 0, "cb_chain_set_state must come first");
    cb_ctx* ctx = c->ch.ctx;
    const bool timing = ctx ? ctx->timing : false;
    if (ctx) ctx->timing = false;   // no per-evaluation timing events inside the loop
    const int rc = chain_err(c, cbm::run(&c->ch, n_gens, move, accepted, current_ll, proposed_ll, ll_ratio, log_u));
    if (ctx) ctx->timing = timing;
    return rc;
  });
}
extern "C" int cb_chain_get_state(cb_chain* c, int32_t* parents, int32_t* children, double* lengths, double* pi, double* rates,
                                  double* alpha, double* site_rates, double* lnl) {
  REQUIRE(c, "null argument");
  const cbm::Chain& ch = c->ch;
  for (size_t i = 0; i < ch.tree.size(); ++i) {
    if (parents) parents[i] = ch.tree[i].p;
    if (children) children[i] = ch.tree[i].c;
    if (lengths) lengths[i] = ch.tree[i].t;
  }
  if (pi) memcpy(pi, ch.pi.data(), ch.pi.size() * 8);
  if (rates) memcpy(rates, ch.rates.data(), ch.rates.size() * 8);
  if (alpha) *alpha = ch.alpha;
  if (site_rates) memcpy(site_rates, ch.site_rates.data(), ch.site_rates.size() * 8);
  if (lnl) *lnl = ch.lnl;
  return 0;
}
extern "C" int cb_chain_counters(cb_chain* c, int64_t* moves7, int64_t* accepts7) {
  REQUIRE(c && moves7 && accepts7, "null argument");
  memcpy(moves7, c->ch.n_moves, sizeof c->ch.n_moves);
  memcpy(accepts7, c->ch.n_accepts, sizeof c->ch.n_accepts);
  return 0;
}
extern "C" int cb_chain_destroy(cb_chain* c) {
  if (!c) return 0;
  cbm::be_release(&c->ch, c->ch.snap);
  delete c;
  return 0;
}
