// common.cuh — shared types of the CUDA Z-set library (sm_100a).
//
// Device layout of a batch (DESIGN.md §3): column-major, one contiguous u64
// array per lane + one i64 weight array; rows sorted lexicographically over
// (key lanes, val lanes), consolidated.  i64 lanes are compared through the
// order-preserving map x -> x ^ 0x8000000000000000 ("flip").
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <functional>
#include <map>
#include <mutex>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/dbsp_b200.h"

typedef uint64_t u64;
typedef int64_t i64;
typedef uint32_t u32;
#define MAXL DBSP_MAX_LANES

struct Ctx;
struct Comm;
// A producer kernel may publish its small result (row count, census words) to the host mailbox itself, which
// saves the separate publish launch of read_back(): the host passes a Mail, the designated last tile / last block of
// the kernel calls mail_publish, the host collects the words with mail_finish.
struct Mail {
  volatile uint64_t* p;   // device alias of the mapped host mailbox (nullptr: do not publish)
  uint64_t seq;
};

void set_error(const std::string& s);
#define CUDA_TRY(expr)                                                                    \
  do {                                                                                    \
    cudaError_t e__ = (expr);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      set_error(std::string(#expr) + ": " + cudaGetErrorString(e__) + " @" + __FILE__ + ":" + std::to_string(__LINE__)); \
      return DBSP_ERR_CUDA;                                                               \
    }                                                                                     \
  } while (0)
#define TRY(expr)                 \
  do {                            \
    int32_t rc__ = (expr);        \
    if (rc__ != DBSP_OK) return rc__; \
  } while (0)

// Column pointers + per-lane sign flips, passed to kernels by value.
struct Cols {
  const u64* c[MAXL];
};
struct MCols {
  u64* c[MAXL];
};
struct Flips {
  u64 f[MAXL];
};

// Stream-ordered device buffer (cudaMallocAsync on the context's stream).
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;   // requested
  size_t cls = 0;     // size class actually reserved
  Ctx* ctx = nullptr;
  ~DevBuf();
};
typedef std::shared_ptr<DevBuf> BufP;

struct Batch {
  dbsp_schema s;
  u64 n = 0;
  const u64* col[MAXL] = {nullptr};   // device pointers of the lanes
  const i64* w = nullptr;
  std::vector<BufP> bufs;             // storage kept alive (shared between views)
  // lazily built CSR view: row index of each key's first tuple
  u64 nkeys = ~0ull;
  BufP keystart;                      // u64[nkeys+1]
  std::atomic<int> refs{1};
  Ctx* ctx = nullptr;
  int nl() const { return s.n_key_lanes + s.n_val_lanes; }
  Cols cols() const {
    Cols c;
    for (int l = 0; l < MAXL; l++) c.c[l] = col[l];
    return c;
  }
  Flips flips() const {
    Flips f;
    for (int l = 0; l < MAXL; l++) f.f[l] = (l < nl() && s.lane_types[l] == DBSP_I64) ? 0x8000000000000000ull : 0ull;
    return f;
  }
};

// Spine (trace/spine_fueled.rs:107-119): the LSM of batches behind a trace.  `merging[i]` is the reference's
// MergeState of layer i (batches of at most 2^i rows); `batches` is the cursor view — every batch a CursorList
// would see (spine_fueled.rs:179-216), rebuilt after each mutation, borrowed pointers, largest layer first.
struct SpineLevel {
  enum Kind { VACANT, SINGLE, IN_PROGRESS, COMPLETE } kind = VACANT;
  Batch* a = nullptr;   // SINGLE: the batch (nullptr = structurally empty); IN_PROGRESS: batch1; COMPLETE: the result (or nullptr)
  Batch* b = nullptr;   // IN_PROGRESS: batch2
  i64 remaining = 0;    // IN_PROGRESS: fuel still to be paid before the merge is due (rows of batch1 + batch2)
};
struct Spine {
  dbsp_schema s;
  std::vector<SpineLevel> merging;
  std::vector<Batch*> batches;   // cursor view (no references held)
  u64 effort = 1;
  bool has_bound = false;
  u64 bound[MAXL];
  bool has_vbound = false;   // lower_val_bound (spine_fueled.rs:118)
  u64 vbound[MAXL];
  Ctx* ctx = nullptr;
};

// Kernel ids for the optional per-kernel timing (CUDA events on the lane's
// stream; bench.py's roofline figures come from here).
enum KernelId {
  KID_MERGE = 0, KID_MERGE_PARTITION, KID_PROBE_RANGES, KID_PROBE_FILL, KID_PROJECT, KID_RADIX_SORT, KID_PACK,
  KID_HEADS, KID_EMIT, KID_MINMAX, KID_SEG_REDUCE, KID_LOOKUP, KID_COMPACT, KID_SCAN, KID_AGG_PICK, KID_MISC, KID_SHARD, KID_CHUNK_SORT, KID_COUNT
};
struct ProfRec {
  cudaEvent_t a, b;
  int id;
  u64 bytes;
};

// An execution lane: a compute stream with its own scratch words, mailbox slot and timing records.  Lane 0 is the
// context's main stream; lane 1 runs the independent half of a grouped call (dbsp_join_step,
// dbsp_batches_from_tables) on a worker thread between a fork and a join.  The host thread that drives a lane reads
// it through lane(ctx), so the operator code is the same on both.
struct Lane {
  cudaStream_t stream = nullptr;
  u64* d_scratch = nullptr;         // 256 u64
  volatile u64* h_mail = nullptr;   // zero-copy mailbox: [0] = sequence flag, [8..] = payload (mapped pinned, 320 u64)
  u64* d_mail = nullptr;            // its device alias
  u64 mail_seq = 0;
  cudaEvent_t ev = nullptr;         // fork (lane 0) / join (lane 1) point
  u64 n_sync = 0;
  double t_sync_us = 0;
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
};
constexpr int N_LANES = 2;
struct LaneWorker;

struct Ctx {
  // lifetime: device buffers may outlive dbsp_ctx_destroy (host handles are
  // freed by a garbage collector); the struct is deleted with the last buffer.
  std::atomic<long> live_bufs{0};
  bool destroyed = false;
  bool prof_on = false;
  int device = 0;
  Lane lanes[N_LANES];
  cudaStream_t copy_stream = nullptr;   // pipelined H2D uploads (dbsp_upload_begin)
  cudaStream_t read_stream = nullptr;   // asynchronous D2H reads (dbsp_batch_download_begin): PCIe is full duplex
  // pinned scratch for small D2H readbacks (counts, min/max); lane 0 only
  u64* h_scratch = nullptr;   // 256 u64
  std::atomic<u64> kernel_launches{0}, h2d_bytes{0}, d2h_bytes{0};
  // Device memory: best-fit allocator with coalescing over large cudaMalloc
  // slabs.  Outside a fork everything runs on lane 0's stream, so a block freed
  // by the host can be handed out again at once: later work is ordered after the
  // work that last touched it.  Inside a fork the two lanes are not ordered
  // against each other: blocks freed then wait in `pending_free` until the join
  // has made lane 0 wait for lane 1.  (The stream-ordered cudaMallocAsync pool
  // cost ~25 ms/step in pool growth on q4; a cudaMalloc per slab costs ~10 ms,
  // so slabs are big.)
  std::mutex pool_mu;                          // guards everything below up to n_alloc
  bool fork_open = false;
  std::vector<std::pair<char*, size_t>> pending_free;
  std::map<char*, size_t> free_by_addr;        // free blocks, for coalescing
  std::multimap<size_t, char*> free_by_size;   // the same blocks, for best fit
  std::map<char*, size_t> slabs;               // slab start -> bytes
  size_t pool_reserved = 0, pool_free = 0;
  // host-side overhead counters (printed at destroy when DBSP_HOST_STATS is set)
  double t_alloc_us = 0;
  u64 n_alloc = 0;
  int sm_count = 148;
  Comm* comm = nullptr;   // exchange state (comm.cu), owned by the context
  LaneWorker* worker = nullptr;   // drives lane 1; created on the first fork
};

// The lane the calling thread drives: lane 1 on a context's worker thread, lane 0 everywhere else.
extern thread_local int t_lane;
inline Lane& lane(Ctx* c) { return c->lanes[t_lane]; }

// Run `a` on lane 0 (this thread) and `b` on lane 1 (the worker thread) after the work queued so far on lane 0;
// returns once both have been queued and lane 0 waits for lane 1.  The status is a's if it failed, else b's
// (with b's error message).
int32_t run_forked(Ctx* ctx, const std::function<int32_t()>& a, const std::function<int32_t()>& b);
void lanes_shutdown(Ctx* ctx);

#define LAUNCH_COUNT(ctx) ((ctx)->kernel_launches++)

// RAII timing scope: records events around the kernels launched inside it.
struct ProfScope {
  Lane* l;
  long idx = -1;
  ProfScope(Ctx* ctx, int id, u64 bytes);
  ~ProfScope();
  void set_bytes(u64 b) { if (idx >= 0) l->prof[idx].bytes = b; }
};
const char* kernel_name(int id);

// ---- host helpers (ctx.cu) ---------------------------------------------
int32_t dev_alloc(Ctx* ctx, size_t bytes, BufP* out);
// Allocate storage for an (L lanes + weights) batch of capacity n rows.
int32_t batch_alloc(Ctx* ctx, const dbsp_schema& s, u64 n, Batch** out, MCols* cols, i64** w);
Batch* batch_new_empty(Ctx* ctx, const dbsp_schema& s);
void batch_unref(Batch* b);
inline void batch_ref(Batch* b) { b->refs.fetch_add(1); }
// Copy `count` u64 from device to pinned host scratch and wait.
int32_t read_back(Ctx* ctx, const void* dsrc, size_t count_u64, u64* hdst);
int32_t read_back32(Ctx* ctx, const void* dsrc, u32* hdst);
int32_t exclusive_scan_u32(Ctx* ctx, const u32* in, u32* out, u64 n, const Mail* total_mail = nullptr);   // out[n] = total (n+1 entries); total_mail: the kernel publishes it
int32_t inclusive_scan_i64(Ctx* ctx, const i64* in, i64* out, u64 n);

int32_t mail_wait(Ctx* ctx, u64 seq);   // spin on the host mailbox until `seq` is published
Mail mail_begin(Ctx* ctx);
int32_t mail_finish(Ctx* ctx, const Mail& m, u64* out, int count);

// ---- comm.cu ---------------------------------------------------------------
int32_t comm_create(Ctx* ctx, int rank, int world, u64 slot_bytes, unsigned char* blob_out);
int32_t comm_connect(Ctx* ctx, const unsigned char* blobs);
void comm_free(Ctx* ctx);
int32_t comm_exchange(Ctx* ctx, const Batch* const* in, int ns, int fixed_dest, Batch** out);
int32_t comm_allreduce_max(Ctx* ctx, u64* x);
void comm_info(Ctx* ctx, int* rank, int* world, u64* bytes_sent);

// ---- consolidate.cu ------------------------------------------------------
// Sort (lanes, weights) rows, sum equal rows, drop zero weights -> batch.
// `cols`/`w` are device arrays of n rows; w == nullptr means all +1.
// `adopt` (optional): the buffer that owns cols/w; when the rows turn out to be
// canonical already (ordered, duplicate- and zero-free) it becomes the batch.
// `d_n` (optional): the exact row count lives on the device and `n` is only an
// upper bound; the census returns it (saves the producer a read-back).
int32_t consolidate_rows(Ctx* ctx, const dbsp_schema& s, const Cols& cols, const i64* w, u64 n, const BufP* adopt,
                         Batch** out, const u32* d_n = nullptr);

int32_t reduce_sorted_rows(Ctx* ctx, const dbsp_schema& s, const Cols& cols, const i64* w, u64 n, Batch** out);

// ---- merge.cu --------------------------------------------------------------
int32_t merge_batches(Ctx* ctx, const Batch* a, const Batch* b, Batch** out);
int32_t merge_path_split(Ctx* ctx, const Batch* a, const Batch* b, u64 d, u64* na, u64* nb);

// ---- device helpers ----------------------------------------------------------
#ifdef __CUDACC__
// called by ONE thread after the values it publishes are final
__device__ __forceinline__ void mail_publish(const Mail& m, const u64* vals, int count) {
  if (!m.p) return;
  for (int i = 0; i < count; i++) m.p[8 + i] = vals[i];
  __threadfence_system();
  m.p[0] = m.seq;
}
// ---- decoupled look-back over ticket-ordered tiles ----------------------------------------------------------
// Status word = 2-bit state (0 empty, 1 aggregate, 2 inclusive prefix) | 62-bit value; the status array is zeroed
// before the launch and tiles take their index from an atomic ticket, so every predecessor a tile waits on is
// resident or finished.  Relaxed device-scope accesses: flag and value share one word.
constexpr u64 LB_AGG = 1ull << 62, LB_PREFIX = 2ull << 62, LB_MASK = (1ull << 62) - 1;
__device__ __forceinline__ u64 lb_ld(const u64* p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void lb_st(u64* p, u64 v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Called by all 32 lanes of ONE warp of tile t with the tile's total: publishes the aggregate, sums the
// predecessors (32 status words per round trip), publishes the inclusive prefix and returns the exclusive prefix
// (the same value in every lane).
__device__ __forceinline__ u64 lb_exclusive_prefix(u64* status, u32 t, u64 tile_total) {
  const int lane = threadIdx.x & 31;
  if (t == 0) {
    if (lane == 0) lb_st(&status[0], LB_PREFIX | tile_total);
    return 0;
  }
  if (lane == 0) lb_st(&status[t], LB_AGG | tile_total);
  u64 base = 0;
  long long p = (long long)t - 1;
  while (true) {
    const long long q = p - lane;
    u64 x = LB_PREFIX;   // tiles before 0 contribute an empty prefix
    if (q >= 0) {
      do { x = lb_ld(&status[q]); } while ((x >> 62) == 0);
    }
    const unsigned isp = __ballot_sync(0xffffffffu, (x >> 62) == 2);
    const int first = isp ? (__ffs(isp) - 1) : 32;
    u64 c = (lane <= first) ? (x & LB_MASK) : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    base += c;
    if (isp) break;
    p -= 32;
  }
  if (lane == 0) lb_st(&status[t], LB_PREFIX | (base + tile_total));
  return base;
}
// lexicographic compare of row i of A against row j of B over lanes [0,nl)
__device__ __forceinline__ int cmp_rows_g(const Cols& A, u64 i, const Cols& B, u64 j, int nl, const Flips& f) {
  for (int l = 0; l < nl; l++) {
    u64 a = A.c[l][i] ^ f.f[l], b = B.c[l][j] ^ f.f[l];
    if (a != b) return a < b ? -1 : 1;
  }
  return 0;
}
// compare row i of A against a query tuple q (already flipped)
__device__ __forceinline__ int cmp_row_q(const Cols& A, u64 i, const u64* q, int nl, const Flips& f) {
  for (int l = 0; l < nl; l++) {
    u64 a = A.c[l][i] ^ f.f[l];
    if (a != q[l]) return a < q[l] ? -1 : 1;
  }
  return 0;
}
// first row in [lo,hi) whose first nl lanes are >= q  (q flipped)
__device__ __forceinline__ u64 lower_bound_q(const Cols& A, u64 lo, u64 hi, const u64* q, int nl, const Flips& f) {
  while (lo < hi) {
    u64 mid = lo + ((hi - lo) >> 1);
    if (cmp_row_q(A, mid, q, nl, f) < 0) lo = mid + 1; else hi = mid;
  }
  return lo;
}
// first row in [lo,hi) whose first nl lanes are > q
__device__ __forceinline__ u64 upper_bound_q(const Cols& A, u64 lo, u64 hi, const u64* q, int nl, const Flips& f) {
  while (lo < hi) {
    u64 mid = lo + ((hi - lo) >> 1);
    if (cmp_row_q(A, mid, q, nl, f) <= 0) lo = mid + 1; else hi = mid;
  }
  return lo;
}
#endif
