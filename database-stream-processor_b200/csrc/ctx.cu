// ctx.cu — context, stream-ordered memory, small host<->device plumbing.
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <iterator>
#include <cstdio>
#include <cstdlib>

#include "common.cuh"

static inline double now_us() {
  return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static thread_local std::string g_err;
thread_local int t_lane = 0;
void set_error(const std::string& s) { g_err = s; }
void print_host_stats(Ctx* c) {
  if (getenv("DBSP_HOST_STATS"))
    fprintf(stderr, "[dbsp host] allocs %llu in %.1f ms (pool %.2f GiB in %zu slabs); read-back syncs %llu + %llu waited %.1f + %.1f ms (lane 0 + 1); launches %llu\n",
            (unsigned long long)c->n_alloc, c->t_alloc_us / 1e3, c->pool_reserved / 1073741824.0, c->slabs.size(),
            (unsigned long long)c->lanes[0].n_sync, (unsigned long long)c->lanes[1].n_sync, c->lanes[0].t_sync_us / 1e3,
            c->lanes[1].t_sync_us / 1e3, (unsigned long long)c->kernel_launches.load());
}
const char* get_error() { return g_err.c_str(); }

static const char* KNAMES[KID_COUNT] = {
    "merge_tiles", "merge_partition", "probe_ranges", "probe_fill", "project_rows", "radix_sort", "pack_keys",
    "heads", "emit", "minmax", "seg_reduce", "lookup", "compact", "scan", "agg_pick", "misc", "shard_scatter", "chunk_sort"};
const char* kernel_name(int id) { return (id >= 0 && id < KID_COUNT) ? KNAMES[id] : "?"; }

ProfScope::ProfScope(Ctx* ctx, int id, u64 bytes) : l(&lane(ctx)) {
  if (!ctx->prof_on) return;
  ProfRec r;
  r.id = id;
  r.bytes = bytes;
  for (cudaEvent_t* e : {&r.a, &r.b}) {
    if (!l->ev_pool.empty()) { *e = l->ev_pool.back(); l->ev_pool.pop_back(); }
    else cudaEventCreate(e);
  }
  cudaEventRecord(r.a, l->stream);
  idx = (long)l->prof.size();
  l->prof.push_back(r);
}
ProfScope::~ProfScope() {
  if (idx >= 0) cudaEventRecord(l->prof[idx].b, l->stream);
}

static const size_t SLAB_BYTES = (size_t)8 << 30;   // 8 GiB per cudaMalloc
static const size_t ALIGN = 512;

void pool_release_all(Ctx* ctx) {
  for (auto& kv : ctx->slabs) cudaFree(kv.first);
  ctx->slabs.clear();
  ctx->free_by_addr.clear();
  ctx->free_by_size.clear();
  ctx->pool_reserved = ctx->pool_free = 0;
}

static void pool_insert_free(Ctx* ctx, char* p, size_t sz) {
  // coalesce with the free neighbours (never across a slab boundary)
  auto nxt = ctx->free_by_addr.lower_bound(p);
  if (nxt != ctx->free_by_addr.end() && nxt->first == p + sz && !ctx->slabs.count(nxt->first)) {
    auto range = ctx->free_by_size.equal_range(nxt->second);
    for (auto it = range.first; it != range.second; ++it)
      if (it->second == nxt->first) { ctx->free_by_size.erase(it); break; }
    sz += nxt->second;
    nxt = ctx->free_by_addr.erase(nxt);
  }
  if (nxt != ctx->free_by_addr.begin() && !ctx->slabs.count(p)) {
    auto prv = std::prev(nxt);
    if (prv->first + prv->second == p) {
      auto range = ctx->free_by_size.equal_range(prv->second);
      for (auto it = range.first; it != range.second; ++it)
        if (it->second == prv->first) { ctx->free_by_size.erase(it); break; }
      p = prv->first;
      sz += prv->second;
      ctx->free_by_addr.erase(prv);
    }
  }
  ctx->free_by_addr[p] = sz;
  ctx->free_by_size.insert({sz, p});
}

DevBuf::~DevBuf() {
  if (!ctx) return;
  if (p && !ctx->destroyed) {   // after ctx_destroy the slabs are already gone
    std::lock_guard<std::mutex> g(ctx->pool_mu);
    if (ctx->fork_open) {   // the other lane may still use the block: free it at the join
      ctx->pending_free.push_back({(char*)p, cls});
    } else {
      pool_insert_free(ctx, (char*)p, cls);
      ctx->pool_free += cls;
    }
  }
  if (ctx->live_bufs.fetch_sub(1) == 1 && ctx->destroyed) delete ctx;
}

int32_t dev_alloc(Ctx* ctx, size_t bytes, BufP* out) {
  auto b = std::make_shared<DevBuf>();
  b->ctx = ctx;
  ctx->live_bufs.fetch_add(1);
  b->bytes = bytes;
  if (bytes == 0) bytes = 16;
  size_t need = (bytes + ALIGN - 1) & ~(ALIGN - 1);
  std::lock_guard<std::mutex> g(ctx->pool_mu);
  double t0 = now_us();
  auto it = ctx->free_by_size.lower_bound(need);
  if (it == ctx->free_by_size.end()) {
    size_t slab = need > SLAB_BYTES ? need : SLAB_BYTES;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, slab);
    while (e != cudaSuccess && slab > need) {   // not enough room for a full slab: shrink towards the request
      cudaGetLastError();
      slab = std::max(need, slab / 2);
      e = cudaMalloc(&p, slab);
    }
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_error(std::string("cudaMalloc(") + std::to_string(slab) + "): " + cudaGetErrorString(e) + " (pool reserved " +
                std::to_string(ctx->pool_reserved) + " B, free " + std::to_string(ctx->pool_free) + " B)");
      return DBSP_ERR_CUDA;
    }
    ctx->slabs[(char*)p] = slab;
    ctx->pool_reserved += slab;
    ctx->pool_free += slab;
    pool_insert_free(ctx, (char*)p, slab);
    it = ctx->free_by_size.lower_bound(need);
  }
  char* p = it->second;
  size_t sz = it->first;
  ctx->free_by_size.erase(it);
  ctx->free_by_addr.erase(p);
  if (sz - need >= ALIGN) {   // split
    ctx->free_by_addr[p + need] = sz - need;
    ctx->free_by_size.insert({sz - need, p + need});
  } else {
    need = sz;
  }
  b->p = p;
  b->cls = need;
  ctx->pool_free -= need;
  ctx->t_alloc_us += now_us() - t0;
  ctx->n_alloc++;
  *out = b;
  return DBSP_OK;
}

int32_t batch_alloc(Ctx* ctx, const dbsp_schema& s, u64 n, Batch** out, MCols* cols, i64** w) {
  int L = s.n_key_lanes + s.n_val_lanes;
  u64 cap = (n + 32) & ~31ull;   // >= n+1 rows (TMA tiles may over-read one row), lanes 256-byte aligned
  if (cap == 0) cap = 32;
  BufP buf;
  TRY(dev_alloc(ctx, (size_t)cap * 8 * (L + 1), &buf));
  Batch* b = new Batch();
  b->s = s;
  b->n = n;
  b->ctx = ctx;
  b->bufs.push_back(buf);
  u64* base = (u64*)buf->p;
  for (int l = 0; l < L; l++) {
    b->col[l] = base + (size_t)l * cap;
    if (cols) cols->c[l] = base + (size_t)l * cap;
  }
  b->w = (const i64*)(base + (size_t)L * cap);
  if (w) *w = (i64*)(base + (size_t)L * cap);
  *out = b;
  return DBSP_OK;
}

Batch* batch_new_empty(Ctx* ctx, const dbsp_schema& s) {
  Batch* b = new Batch();
  b->s = s;
  b->n = 0;
  b->ctx = ctx;
  b->nkeys = 0;
  return b;
}

void batch_unref(Batch* b) {
  if (!b) return;
  if (b->refs.fetch_sub(1) == 1) delete b;
}

// ---- lane 1: a worker thread owned by the context ------------------------------------------------------------------
// The worker spins while it expects a fork (the forks of one circuit step follow each other within a fraction of a
// millisecond, and waking a parked thread costs about as much as one of the kernels the fork hides) and parks on a
// condition variable once it has been idle for LANE_SPIN_US.
static const double LANE_SPIN_US = 1000.0;
enum { W_IDLE = 0, W_POSTED, W_DONE, W_EXIT };
struct LaneWorker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::atomic<int> state{W_IDLE};
  const std::function<int32_t()>* job = nullptr;
  int32_t rc = DBSP_OK;
  std::string err;
};

static inline void cpu_relax() {
#if defined(__x86_64__) || defined(__i386__)
  __builtin_ia32_pause();
#else
  std::this_thread::yield();
#endif
}

static void lane_worker_main(Ctx* ctx, LaneWorker* w) {
  t_lane = 1;
  cudaSetDevice(ctx->device);
  while (true) {
    int st;
    double t0 = now_us();
    while ((st = w->state.load(std::memory_order_acquire)) != W_POSTED && st != W_EXIT) {
      if (now_us() - t0 < LANE_SPIN_US) { cpu_relax(); continue; }
      std::unique_lock<std::mutex> lk(w->m);
      w->cv.wait(lk, [w] { int x = w->state.load(); return x == W_POSTED || x == W_EXIT; });
    }
    if (st == W_EXIT) return;
    w->rc = (*w->job)();
    w->err = w->rc != DBSP_OK ? std::string(get_error()) : std::string();
    w->state.store(W_DONE, std::memory_order_release);
  }
}

void lanes_shutdown(Ctx* ctx) {
  LaneWorker* w = ctx->worker;
  if (!w) return;
  {
    std::lock_guard<std::mutex> g(w->m);
    w->state.store(W_EXIT);
  }
  w->cv.notify_one();
  w->th.join();
  delete w;
  ctx->worker = nullptr;
}

int32_t run_forked(Ctx* ctx, const std::function<int32_t()>& a, const std::function<int32_t()>& b) {
  if (t_lane != 0 || ctx->fork_open) { set_error("fork: already inside a fork"); return DBSP_ERR_INVALID; }
  Lane& l0 = ctx->lanes[0];
  Lane& l1 = ctx->lanes[1];
  if (!ctx->worker) {
    ctx->worker = new LaneWorker();
    ctx->worker->th = std::thread(lane_worker_main, ctx, ctx->worker);
  }
  LaneWorker* w = ctx->worker;
  // fork: lane 1 starts after everything queued on lane 0 so far
  CUDA_TRY(cudaEventRecord(l0.ev, l0.stream));
  CUDA_TRY(cudaStreamWaitEvent(l1.stream, l0.ev, 0));
  {
    std::lock_guard<std::mutex> g(ctx->pool_mu);
    ctx->fork_open = true;
  }
  w->job = &b;
  {
    std::lock_guard<std::mutex> g(w->m);
    w->state.store(W_POSTED, std::memory_order_release);
  }
  w->cv.notify_one();
  const int32_t ra = a();
  const std::string ea = ra != DBSP_OK ? std::string(get_error()) : std::string();
  while (w->state.load(std::memory_order_acquire) != W_DONE) cpu_relax();
  w->state.store(W_IDLE, std::memory_order_relaxed);
  // join: lane 0 continues after everything lane 1 queued; only then may the blocks freed inside the fork be reused
  cudaError_t e = cudaEventRecord(l1.ev, l1.stream);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(l0.stream, l1.ev, 0);
  {
    std::lock_guard<std::mutex> g(ctx->pool_mu);
    ctx->fork_open = false;
    if (e == cudaSuccess) {
      for (auto& f : ctx->pending_free) {
        pool_insert_free(ctx, f.first, f.second);
        ctx->pool_free += f.second;
      }
      ctx->pending_free.clear();
    }
  }
  if (e != cudaSuccess) { set_error(std::string("join of the lanes: ") + cudaGetErrorString(e)); return DBSP_ERR_CUDA; }
  if (ra != DBSP_OK) { set_error(ea); return ra; }
  if (w->rc != DBSP_OK) { set_error(w->err); return w->rc; }
  return DBSP_OK;
}

// Small device->host read-backs (row counts, lane ranges).  A one-warp kernel
// copies the words into mapped pinned host memory and then publishes a sequence
// number; the host spins on that word.  This costs a few microseconds instead of
// the ~20 us of cudaMemcpyAsync + cudaStreamSynchronize, and a step needs 20-40
// of them.
__global__ void k_publish(volatile u64* mail, const u64* src, int count, int words32, u64 seq) {
  int t = threadIdx.x;
  if (words32) {   // a single 32-bit word
    if (t == 0) mail[8] = (u64) * (const u32*)src;
  } else {
    for (int i = t; i < count; i += 32) mail[8 + i] = src[i];
  }
  __threadfence_system();
  __syncwarp();
  if (t == 0) {
    __threadfence_system();
    mail[0] = seq;
  }
}

int32_t mail_wait(Ctx* ctx, u64 seq) {
  Lane& ln = lane(ctx);
  u64 spins = 0;
  while (ln.h_mail[0] != seq) {
    if ((++spins & 0xffff) == 0) {   // the stream may have faulted: do not spin forever
      cudaError_t e = cudaStreamQuery(ln.stream);
      if (e != cudaSuccess && e != cudaErrorNotReady) {
        set_error(std::string("read_back: ") + cudaGetErrorString(e));
        return DBSP_ERR_CUDA;
      }
      if (e == cudaSuccess && ln.h_mail[0] != seq) {   // kernel done but the flag is not visible yet
        CUDA_TRY(cudaStreamSynchronize(ln.stream));
      }
    }
  }
  return DBSP_OK;
}

Mail mail_begin(Ctx* ctx) {
  Lane& ln = lane(ctx);
  Mail m;
  m.p = (volatile u64*)ln.d_mail;
  m.seq = ++ln.mail_seq;
  return m;
}
int32_t mail_finish(Ctx* ctx, const Mail& m, u64* out, int count) {
  Lane& ln = lane(ctx);
  double t0 = now_us();
  TRY(mail_wait(ctx, m.seq));
  ln.t_sync_us += now_us() - t0;
  ln.n_sync++;
  for (int i = 0; i < count; i++) out[i] = ln.h_mail[8 + i];
  ctx->d2h_bytes += (u64)count * 8;
  return DBSP_OK;
}

int32_t read_back(Ctx* ctx, const void* dsrc, size_t count_u64, u64* hdst) {
  if (count_u64 > 256) { set_error("read_back: too large"); return DBSP_ERR_INVALID; }
  Lane& ln = lane(ctx);
  double t0 = now_us();
  const u64 seq = ++ln.mail_seq;
  k_publish<<<1, 32, 0, ln.stream>>>((volatile u64*)ln.d_mail, (const u64*)dsrc, (int)count_u64, 0, seq);
  TRY(mail_wait(ctx, seq));
  ln.t_sync_us += now_us() - t0;
  ln.n_sync++;
  for (size_t i = 0; i < count_u64; i++) hdst[i] = ln.h_mail[8 + i];
  ctx->d2h_bytes += count_u64 * 8;
  return DBSP_OK;
}

int32_t read_back32(Ctx* ctx, const void* dsrc, u32* hdst) {
  Lane& ln = lane(ctx);
  double t0 = now_us();
  const u64 seq = ++ln.mail_seq;
  k_publish<<<1, 32, 0, ln.stream>>>((volatile u64*)ln.d_mail, (const u64*)dsrc, 1, 1, seq);
  TRY(mail_wait(ctx, seq));
  ln.t_sync_us += now_us() - t0;
  ln.n_sync++;
  *hdst = (u32)ln.h_mail[8];
  ctx->d2h_bytes += 4;
  return DBSP_OK;
}

// Device-wide exclusive prefix sum of u32 counts: one pass over HBM with a
// decoupled look-back across tiles (same protocol as the merge kernel: status
// word = 2-bit state | 62-bit value, tiles ordered by an atomic ticket, warp 0
// inspects 32 predecessors per round trip).
constexpr int SCAN_THREADS = 256, SCAN_IPT = 8, SCAN_TILE = SCAN_THREADS * SCAN_IPT;
constexpr u64 SC_AGG = 1ull << 62, SC_PREFIX = 2ull << 62, SC_MASK = (1ull << 62) - 1;

__device__ __forceinline__ u64 sc_ld(const u64* p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void sc_st(u64* p, u64 v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(SCAN_THREADS) k_exscan_u32(const u32* __restrict__ in, u32* __restrict__ out, u64 m,
                                                            u32* ticket, u64* status, Mail mail) {
  __shared__ u32 s_tile, s_warp[SCAN_THREADS / 32];
  __shared__ u64 s_base;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const u32 t = s_tile;
  const u64 base_i = (u64)t * SCAN_TILE + (u64)tid * SCAN_IPT;
  u32 v[SCAN_IPT];
  u32 sum = 0;
#pragma unroll
  for (int k = 0; k < SCAN_IPT; k++) {
    v[k] = (base_i + k < m) ? in[base_i + k] : 0u;
    sum += v[k];
  }
  u32 incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    u32 x = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += x;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  u32 woff = 0, tile_total = 0;
#pragma unroll
  for (int k = 0; k < SCAN_THREADS / 32; k++) {
    u32 x = s_warp[k];
    if (k < wid) woff += x;
    tile_total += x;
  }
  if (wid == 0) {
    u64 base = 0;
    if (t == 0) {
      if (lane == 0) sc_st(&status[0], SC_PREFIX | (u64)tile_total);
    } else {
      if (lane == 0) sc_st(&status[t], SC_AGG | (u64)tile_total);
      long long p = (long long)t - 1;
      while (true) {
        const long long q = p - lane;
        u64 x = SC_PREFIX;
        if (q >= 0) {
          do { x = sc_ld(&status[q]); } while ((x >> 62) == 0);
        }
        const unsigned isp = __ballot_sync(0xffffffffu, (x >> 62) == 2);
        const int first = isp ? (__ffs(isp) - 1) : 32;
        u64 c = (lane <= first) ? (x & SC_MASK) : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        base += c;
        if (isp) break;
        p -= 32;
      }
      if (lane == 0) sc_st(&status[t], SC_PREFIX | (base + tile_total));
    }
    if (lane == 0) s_base = base;
  }
  __syncthreads();
  u32 run = (u32)s_base + woff + incl - sum;
#pragma unroll
  for (int k = 0; k < SCAN_IPT; k++) {
    if (base_i + k < m) out[base_i + k] = run;
    if (base_i + k == m - 1) {   // the last entry is the total: publish it to the host if asked to
      const u64 tot = run;
      mail_publish(mail, &tot, 1);
    }
    run += v[k];
  }
}

int32_t exclusive_scan_u32(Ctx* ctx, const u32* in, u32* out, u64 n, const Mail* total_mail) {
  // out has n+1 entries: out[n] = total.  Scans the n+1 inputs (callers keep
  // in[n] == 0).
  const u64 m = n + 1;
  const u32 ntiles = (u32)((m + SCAN_TILE - 1) / SCAN_TILE);
  BufP aux;
  TRY(dev_alloc(ctx, (size_t)(ntiles + 1) * 8, &aux));
  CUDA_TRY(cudaMemsetAsync(aux->p, 0, (size_t)(ntiles + 1) * 8, lane(ctx).stream));
  u64* status = (u64*)aux->p;
  u32* ticket = (u32*)(status + ntiles);
  {
    ProfScope ps(ctx, KID_SCAN, m * 8);
    Mail mm;
    mm.p = nullptr;
    mm.seq = 0;
    if (total_mail) mm = *total_mail;
    k_exscan_u32<<<ntiles, SCAN_THREADS, 0, lane(ctx).stream>>>(in, out, m, ticket, status, mm);
  }
  LAUNCH_COUNT(ctx);
  return DBSP_OK;
}

// i64 running sums are only needed by the Fold-sum aggregator (rare path): the
// one library prefix sum left.
int32_t inclusive_scan_i64(Ctx* ctx, const i64* in, i64* out, u64 n) {
  size_t tmp_bytes = 0;
  CUDA_TRY(cub::DeviceScan::InclusiveSum(nullptr, tmp_bytes, in, out, (size_t)n, lane(ctx).stream));
  BufP tmp;
  TRY(dev_alloc(ctx, tmp_bytes, &tmp));
  CUDA_TRY(cub::DeviceScan::InclusiveSum(tmp->p, tmp_bytes, in, out, (size_t)n, lane(ctx).stream));
  LAUNCH_COUNT(ctx);
  return DBSP_OK;
}
