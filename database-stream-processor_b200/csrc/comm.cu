// comm.cu — K10: the exchange of delta batches between the circuit replicas (one replica = one context = one GPU).
//
// Replaces shard_batch + Exchange + the receiver's merge (operator/communication/shard.rs:106-199,
// exchange.rs:128-200), gather (gather.rs:41-103) and the watermark exchange (time_series/watermark.rs:53-70).
//
// B200-first design: no collective library on the data path and no host in the middle.  Every context owns one
// device region; at connect time each rank maps every peer's region (CUDA IPC between processes, plain peer access
// between the contexts of one process) so that NVLink stores reach it directly.
//   * One partition pass (hash -> per-tile histograms), one scan, one scatter kernel whose stores land straight in
//     the destination GPU's receive slot [parity][source rank] — the all-to-all IS the scatter, column-major so that
//     the receiver uses each segment in place as a sorted batch.
//   * Row counts travel the same way: after the scatter a one-warp kernel stores {counts, sequence number} into the
//     peer's flag slot (release, system scope).  The receiver's one-warp wait kernel polls its P flag slots and
//     publishes the P x streams counts to the host mailbox: ONE read-back per exchange round, none for counts going out.
//   * Slots and flags are double-buffered by the parity of the exchange sequence number.  A rank signals round s+1
//     only after the kernels that consume round s were queued before it on its stream, and a rank writes round s+2
//     only after it saw every peer's signal of round s+1 — so the flags themselves order slot reuse; no extra ack.
//   * All replicas issue the same sequence of exchange calls (SPMD, like the reference's workers).
#include <unistd.h>

#include "ops.cuh"

int32_t mail_wait(Ctx* ctx, u64 seq);

namespace {

constexpr int MAXP = DBSP_COMM_MAX_RANKS;   // 32: one warp polls all peers
constexpr int MAX_STREAMS = 2;              // the two inputs of a join share one round
constexpr u64 BLOB_MAGIC = 0x64627370636f6d6dull;
constexpr size_t CTRL_BYTES = 64 << 10;
constexpr int PT_THREADS = 256, PT_ROUNDS = 8, PT_TILE = PT_THREADS * PT_ROUNDS;

struct Blob {   // DBSP_COMM_BLOB_BYTES
  cudaIpcMemHandle_t ipc;
  u64 magic, pid, base, region_bytes, slot_bytes;
  int32_t device, rank, world, pad;
};
static_assert(sizeof(Blob) <= DBSP_COMM_BLOB_BYTES, "blob too large");

struct Flag {   // written by a source rank into the destination's control area
  u64 counts[MAX_STREAMS];
  u64 err;
  u64 seq;      // written last
};
struct RedSlot {
  u64 val, seq;
};
struct Ctrl {
  Flag flags[2][MAXP];
  RedSlot red[2][MAXP];
};
static_assert(sizeof(Ctrl) <= CTRL_BYTES, "control area too small");
static_assert(MAXP <= 32, "one warp polls all peers");

}  // namespace

struct Comm {
  int rank = 0, world = 1;
  size_t slot_bytes = 0, region_bytes = 0;
  char* region = nullptr;
  char* peer[MAXP] = {nullptr};
  bool ipc_open[MAXP] = {false};
  bool connected = false;
  u64 seq = 0, red_seq = 0;
  u64 bytes_sent = 0;
  char* slot(int dst, int parity, int src) const {
    return peer[dst] + CTRL_BYTES + ((size_t)parity * world + src) * slot_bytes;
  }
};

namespace {

__device__ __forceinline__ u64 mix64d(u64 x) {
  x += 0x9e3779b97f4a7c15ull;
  x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
  x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}
__device__ __forceinline__ u64 ld_acquire_sys(const u64* p) {
  u64 v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(u64* p, u64 v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ u64 globaltimer_ns() {
  u64 t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// shard_batch, pass 1 (shard.rs:165-199): destination of every row (hash of the key lanes — the same splitmix64 fold
// as the oracle; placement is unobservable, shard.rs:38-51) and one histogram per tile, stored [dest][tile] so that a
// single exclusive scan yields every (tile, dest) base.
__global__ void __launch_bounds__(PT_THREADS) k_shard_hist(Cols B, u64 n, int nk, u32 P, int fixed_dest, unsigned char* dest,
                                                           u32* hist, u32 ntiles) {
  __shared__ u32 s_h[MAXP];
  if (threadIdx.x < MAXP) s_h[threadIdx.x] = 0;
  __syncthreads();
  const u64 base = (u64)blockIdx.x * PT_TILE;
#pragma unroll
  for (int r = 0; r < PT_ROUNDS; r++) {
    const u64 i = base + (u64)r * PT_THREADS + threadIdx.x;
    if (i < n) {
      u32 d;
      if (fixed_dest >= 0) d = (u32)fixed_dest;
      else {
        u64 h = 0;
        for (int l = 0; l < nk; l++) h = mix64d(h ^ B.c[l][i]);
        d = (u32)(h % P);
      }
      dest[i] = (unsigned char)d;
      atomicAdd(&s_h[d], 1u);
    }
  }
  __syncthreads();
  if (threadIdx.x < P) hist[(u64)threadIdx.x * ntiles + blockIdx.x] = s_h[threadIdx.x];
  if (blockIdx.x == 0 && threadIdx.x == 0) hist[(u64)P * ntiles] = 0;   // terminator of the scan
}

struct SendArgs {
  char* slot[MAXP];     // destination slot [parity][my rank] of every peer
  u64 slot_bytes;
};

// per-destination totals of this stream and the byte offset of the stream inside every slot; flags capacity overflow
__global__ void k_shard_totals(const u32* pos, u32 ntiles, u32 P, int L, const u64* prev_end, u64 slot_bytes, u64* totals,
                               u64* stream_off, u64* stream_end, u64* err) {
  const u32 p = threadIdx.x;
  if (p >= P) return;
  const u64 cnt = (u64)pos[(u64)(p + 1) * ntiles] - (u64)pos[(u64)p * ntiles];
  totals[p] = cnt;
  const u64 off = prev_end ? prev_end[p] : 0;
  const u64 stride = (cnt + 32) & ~31ull;           // same padding rule as batch_alloc (TMA may over-read one row)
  const u64 end = off + (cnt ? stride * 8 * (u64)(L + 1) : 0);
  stream_off[p] = off;
  stream_end[p] = (end + 255) & ~255ull;
  if (end > slot_bytes) atomicExch((unsigned long long*)err, 1ull);
}

// pass 2: stable scatter straight into the destination GPUs' receive slots (NVLink stores).  Rows of one
// destination keep their order (tile base from the scan + rank inside the tile), so every segment stays sorted.
__global__ void __launch_bounds__(PT_THREADS) k_shard_scatter2(Cols B, const i64* w, u64 n, int L, u32 P, const unsigned char* dest,
                                                               const u32* pos, u32 ntiles, const u64* totals, const u64* stream_off,
                                                               const u64* err, SendArgs sa) {
  __shared__ u32 s_run[MAXP];
  __shared__ u32 s_wc[PT_THREADS / 32][MAXP];
  if (*err) return;   // a slot would overflow: nothing is written, the flag carries the error
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid < (int)P) s_run[tid] = pos[(u64)tid * ntiles + blockIdx.x] - pos[(u64)tid * ntiles];
  const u64 base = (u64)blockIdx.x * PT_TILE;
  for (int r = 0; r < PT_ROUNDS; r++) {
    for (int k = tid; k < (PT_THREADS / 32) * MAXP; k += PT_THREADS) (&s_wc[0][0])[k] = 0;
    __syncthreads();
    const u64 i = base + (u64)r * PT_THREADS + tid;
    const bool valid = i < n;
    const u32 d = valid ? dest[i] : 0xffu;
    const unsigned m = __match_any_sync(0xffffffffu, d);
    const u32 rank_w = __popc(m & ((1u << lane) - 1));
    if (valid && rank_w == 0) s_wc[wid][d] = __popc(m);
    __syncthreads();
    if (valid) {
      u32 o = s_run[d] + rank_w;
      for (int ww = 0; ww < wid; ww++) o += s_wc[ww][d];
      const u64 cnt = totals[d];
      const u64 stride = (cnt + 32) & ~31ull;
      u64* seg = (u64*)(sa.slot[d] + stream_off[d]);
      for (int l = 0; l < L; l++) seg[(u64)l * stride + o] = B.c[l][i];
      seg[(u64)L * stride + o] = (u64)w[i];
    }
    __syncthreads();
    if (tid < (int)P) {
      u32 add = 0;
      for (int ww = 0; ww < PT_THREADS / 32; ww++) add += s_wc[ww][tid];
      s_run[tid] += add;
    }
    __syncthreads();
  }
}

struct SignalArgs {
  Flag* flag[MAXP];   // my flag slot in every peer's control area (this round's parity)
};
// after the scatter kernels of this round (stream order): publish {counts, seq} to every destination
__global__ void k_comm_signal(SignalArgs sg, u32 P, int nstreams, const u64* totals0, const u64* totals1, const u64* err, u64 seq) {
  const u32 p = threadIdx.x;
  if (p >= P) return;
  __threadfence_system();
  Flag* f = sg.flag[p];
  f->counts[0] = totals0 ? totals0[p] : 0;
  f->counts[1] = (nstreams > 1 && totals1) ? totals1[p] : 0;
  f->err = *err;
  __threadfence_system();
  st_release_sys(&f->seq, seq);
}

// wait for the P flags of this round, then publish counts (and my own outgoing totals) to the host mailbox:
// mail[8 + src*2 + s] = rows of stream s from rank src; mail[8 + 2P + dst*2 + s] = rows I sent; mail[8 + 4P] = error
__global__ void k_comm_wait(const Flag* my_flags, u32 P, u64 seq, const u64* totals0, const u64* totals1, volatile u64* mail,
                            u64 mail_seq, u64 timeout_ns) {
  const u32 p = threadIdx.x;
  u64 e = 0;
  if (p < P) {
    const u64 t0 = globaltimer_ns();
    while (ld_acquire_sys(&my_flags[p].seq) != seq) {
      if (globaltimer_ns() - t0 > timeout_ns) { e = 2; break; }
      __nanosleep(200);
    }
    if (!e) {
      mail[8 + p * 2 + 0] = ld_acquire_sys(&my_flags[p].counts[0]);
      mail[8 + p * 2 + 1] = ld_acquire_sys(&my_flags[p].counts[1]);
      e = ld_acquire_sys(&my_flags[p].err);
    }
    mail[8 + 2 * P + p * 2 + 0] = totals0 ? totals0[p] : 0;
    mail[8 + 2 * P + p * 2 + 1] = totals1 ? totals1[p] : 0;
  }
  const unsigned any = __ballot_sync(0xffffffffu, e != 0);
  const unsigned tmo = __ballot_sync(0xffffffffu, e == 2);
  if (p == 0) mail[8 + 4 * P] = tmo ? 2 : (any ? 1 : 0);
  __threadfence_system();
  __syncwarp();
  if (p == 0) {
    __threadfence_system();
    mail[0] = mail_seq;
  }
}

struct RedArgs {
  RedSlot* slot[MAXP];   // my slot in every peer's control area
};
// allreduce(max) of one u64 per rank: store into every peer, poll my P slots, reduce, publish to the host mailbox
__global__ void k_comm_allreduce_max(RedArgs ra, const RedSlot* mine, u32 P, u64 x, u64 seq, volatile u64* mail, u64 mail_seq,
                                     u64 timeout_ns) {
  const u32 p = threadIdx.x;
  u64 v = 0, e = 0;
  if (p < P) {
    ra.slot[p]->val = x;
    __threadfence_system();
    st_release_sys(&ra.slot[p]->seq, seq);
    const u64 t0 = globaltimer_ns();
    while (ld_acquire_sys(&mine[p].seq) != seq) {
      if (globaltimer_ns() - t0 > timeout_ns) { e = 2; break; }
      __nanosleep(200);
    }
    if (!e) v = ld_acquire_sys(&mine[p].val);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const u64 y = __shfl_xor_sync(0xffffffffu, v, o);
    v = v > y ? v : y;
  }
  const unsigned tmo = __ballot_sync(0xffffffffu, e != 0);
  if (p == 0) {
    mail[8] = v;
    mail[9] = tmo ? 2 : 0;
    __threadfence_system();
    mail[0] = mail_seq;
  }
}

u64 comm_timeout_ns() {
  static const u64 t = [] {
    const char* e = getenv("DBSP_COMM_TIMEOUT_S");
    double s = e ? atof(e) : 30.0;
    return (u64)(s * 1e9);
  }();
  return t;
}

}  // namespace

void comm_free(Ctx* ctx) {
  Comm* c = ctx->comm;
  if (!c) return;
  for (int p = 0; p < c->world; p++)
    if (c->ipc_open[p] && c->peer[p]) cudaIpcCloseMemHandle(c->peer[p]);
  if (c->region) cudaFree(c->region);
  delete c;
  ctx->comm = nullptr;
}

int32_t comm_create(Ctx* ctx, int rank, int world, u64 slot_bytes, unsigned char* blob_out) {
  if (world < 1 || world > MAXP || rank < 0 || rank >= world) { set_error("comm_create: bad rank / world"); return DBSP_ERR_INVALID; }
  comm_free(ctx);
  Comm* c = new Comm();
  c->rank = rank;
  c->world = world;
  if (slot_bytes == 0) {
    const char* e = getenv("DBSP_COMM_SLOT_MB");
    slot_bytes = (u64)(e ? atof(e) : 512.0) << 20;   // default 512 MiB per (source, destination) and parity
  }
  c->slot_bytes = (slot_bytes + 255) & ~255ull;
  c->region_bytes = CTRL_BYTES + (size_t)2 * world * c->slot_bytes;
  cudaError_t e = cudaMalloc(&c->region, c->region_bytes);
  if (e != cudaSuccess) {
    delete c;
    set_error(std::string("comm_create: cudaMalloc of the receive region (") + std::to_string(c->region_bytes) + " B): " + cudaGetErrorString(e));
    return DBSP_ERR_CUDA;
  }
  ctx->comm = c;
  CUDA_TRY(cudaMemset(c->region, 0, CTRL_BYTES));
  Blob b;
  memset(&b, 0, sizeof(b));
  if (world > 1) CUDA_TRY(cudaIpcGetMemHandle(&b.ipc, c->region));
  b.magic = BLOB_MAGIC;
  b.pid = (u64)getpid();
  b.base = (u64)(size_t)c->region;
  b.region_bytes = c->region_bytes;
  b.slot_bytes = c->slot_bytes;
  b.device = ctx->device;
  b.rank = rank;
  b.world = world;
  memset(blob_out, 0, DBSP_COMM_BLOB_BYTES);
  memcpy(blob_out, &b, sizeof(b));
  return DBSP_OK;
}

int32_t comm_connect(Ctx* ctx, const unsigned char* blobs) {
  Comm* c = ctx->comm;
  if (!c) { set_error("comm_connect: dbsp_comm_create first"); return DBSP_ERR_INVALID; }
  for (int p = 0; p < c->world; p++) {
    Blob b;
    memcpy(&b, blobs + (size_t)p * DBSP_COMM_BLOB_BYTES, sizeof(b));
    if (b.magic != BLOB_MAGIC || b.rank != p || b.world != c->world || b.slot_bytes != c->slot_bytes) {
      set_error("comm_connect: blob " + std::to_string(p) + " does not describe rank " + std::to_string(p) + " of this group");
      return DBSP_ERR_INVALID;
    }
    if (p == c->rank) { c->peer[p] = c->region; continue; }
    if (b.pid == (u64)getpid()) {
      // a context of this very process (the reference's model: worker threads): plain peer access
      if (b.device != ctx->device) {
        cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
          set_error(std::string("comm_connect: cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
          return DBSP_ERR_CUDA;
        }
        cudaGetLastError();
      }
      c->peer[p] = (char*)(size_t)b.base;
    } else {
      void* ptr = nullptr;
      cudaError_t e = cudaIpcOpenMemHandle(&ptr, b.ipc, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        set_error(std::string("comm_connect: cudaIpcOpenMemHandle(rank ") + std::to_string(p) + "): " + cudaGetErrorString(e));
        return DBSP_ERR_CUDA;
      }
      c->peer[p] = (char*)ptr;
      c->ipc_open[p] = true;
    }
  }
  c->connected = true;
  return DBSP_OK;
}

// Segment of stream `s` received from `src` this round, viewed in place as a sorted batch.
static Batch* segment_view(Ctx* ctx, const dbsp_schema& sc, char* seg, u64 cnt) {
  Batch* v = new Batch();
  v->s = sc;
  v->ctx = ctx;
  v->n = cnt;
  const int L = sc.n_key_lanes + sc.n_val_lanes;
  const u64 stride = (cnt + 32) & ~31ull;
  for (int l = 0; l < L; l++) v->col[l] = (const u64*)seg + (size_t)l * stride;
  v->w = (const i64*)((const u64*)seg + (size_t)L * stride);
  if (cnt == 0) v->nkeys = 0;
  return v;   // no bufs: the region outlives the round's consumers (double buffering, see the header)
}

struct SegList {
  const u64* base[MAXP];   // lane 0 of the segment; lanes are `stride` rows apart, weights follow the last lane
  u64 cnt[MAXP], stride[MAXP], off[MAXP];
  int nseg;
};
// P-way merge of small deltas by rank: every row finds its place in the union by bisecting the other segments
// (rows of earlier segments sort before equal rows of later ones), so the P sorted segments land merged in one
// launch; equal rows from different sources end up adjacent and are summed by the epilogue (reduce_sorted_rows).
__global__ void k_pway_rank(SegList sl, int L, Flips f, u64 total, u64 out_stride, u64* out) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int sgm = 0;
  while (sgm + 1 < sl.nseg && i >= sl.off[sgm + 1]) sgm++;
  const u64 r = i - sl.off[sgm];
  u64 raw[MAXL + 1], q[MAXL];
  for (int l = 0; l <= L; l++) raw[l] = sl.base[sgm][(u64)l * sl.stride[sgm] + r];
  for (int l = 0; l < L; l++) q[l] = raw[l] ^ f.f[l];
  u64 pos = r;
  for (int t = 0; t < sl.nseg; t++) {
    if (t == sgm) continue;
    const u64* tb = sl.base[t];
    const u64 ts = sl.stride[t];
    u64 lo = 0, hi = sl.cnt[t];
    while (lo < hi) {   // rows of segment t that sort before this row (t < sgm: ties count too)
      const u64 mid = lo + ((hi - lo) >> 1);
      int c = 0;
      for (int l = 0; l < L && c == 0; l++) {
        const u64 a = tb[(u64)l * ts + mid] ^ f.f[l];
        if (a != q[l]) c = a < q[l] ? -1 : 1;
      }
      const bool before = c < 0 || (c == 0 && t < sgm);
      if (before) lo = mid + 1; else hi = mid;
    }
    pos += lo;
  }
  for (int l = 0; l <= L; l++) out[(u64)l * out_stride + pos] = raw[l];
}
constexpr u64 CONCAT_SORT_MAX_ROWS = 1ull << 20;

static int32_t merge_views(Ctx* ctx, std::vector<Batch*>& parts, const dbsp_schema& s, Batch** out) {
  // receiver side of shard() (shard.rs:136-144): a balanced merge tree of the P sorted segments, or — for small
  // deltas from more than two sources — ONE rank-merge launch + the reduce epilogue instead of P-1 merge launches
  std::vector<Batch*> live;
  for (Batch* p : parts) { if (p->n) live.push_back(p); else batch_unref(p); }
  parts.clear();
  int32_t rc = DBSP_OK;
  u64 total = 0;
  for (Batch* b : live) total += b->n;
  if (live.size() > 2 && total <= CONCAT_SORT_MAX_ROWS) {
    const int L = s.n_key_lanes + s.n_val_lanes;
    const u64 cap = (total + 32) & ~31ull;
    BufP buf;
    rc = dev_alloc(ctx, (size_t)cap * 8 * (L + 1), &buf);
    if (rc) { for (Batch* b : live) batch_unref(b); return rc; }
    SegList sl;
    sl.nseg = (int)live.size();
    u64 off = 0;
    for (size_t k = 0; k < live.size(); k++) {
      sl.base[k] = live[k]->col[0];
      sl.cnt[k] = live[k]->n;
      sl.stride[k] = (live[k]->n + 32) & ~31ull;   // the segment's lane stride (segment_view)
      sl.off[k] = off;
      off += live[k]->n;
    }
    Flips f;
    for (int l = 0; l < MAXL; l++) f.f[l] = (l < L && s.lane_types[l] == DBSP_I64) ? 0x8000000000000000ull : 0ull;
    {
      ProfScope ps(ctx, KID_SHARD, total * (u64)(L + 1) * 8 * 2);
      k_pway_rank<<<(unsigned)((total + 255) / 256), 256, 0, ctx->lanes[0].stream>>>(sl, L, f, total, cap, (u64*)buf->p);
    }
    LAUNCH_COUNT(ctx);
    for (Batch* b : live) batch_unref(b);
    Cols c;
    for (int l = 0; l < MAXL; l++) c.c[l] = l < L ? (const u64*)buf->p + (size_t)l * cap : nullptr;
    return reduce_sorted_rows(ctx, s, c, (const i64*)((const u64*)buf->p + (size_t)L * cap), total, out);
  }
  while (live.size() > 1 && rc == DBSP_OK) {
    std::vector<Batch*> nxt;
    size_t i = 0;
    for (; i + 1 < live.size(); i += 2) {
      Batch* m = nullptr;
      if (rc == DBSP_OK) rc = merge_batches(ctx, live[i], live[i + 1], &m);
      batch_unref(live[i]);
      batch_unref(live[i + 1]);
      if (m) nxt.push_back(m);
    }
    if (i < live.size()) nxt.push_back(live[i]);
    live.swap(nxt);
  }
  if (rc != DBSP_OK) { for (Batch* b : live) batch_unref(b); return rc; }
  if (live.empty()) { *out = batch_new_empty(ctx, s); return DBSP_OK; }
  Batch* r = live[0];
  if (r->bufs.empty() && r->n) {
    // still a view of the receive slot (a single non-empty segment): copy it out before the slot is reused
    Batch* o;
    MCols oc;
    i64* ow;
    rc = batch_alloc(ctx, s, r->n, &o, &oc, &ow);
    if (rc) { batch_unref(r); return rc; }
    const int L = s.n_key_lanes + s.n_val_lanes;
    for (int l = 0; l < L; l++) cudaMemcpyAsync(oc.c[l], r->col[l], r->n * 8, cudaMemcpyDeviceToDevice, ctx->lanes[0].stream);
    cudaMemcpyAsync(ow, r->w, r->n * 8, cudaMemcpyDeviceToDevice, ctx->lanes[0].stream);
    batch_unref(r);
    r = o;
  }
  *out = r;
  return DBSP_OK;
}

// One exchange round for `ns` (1 or 2) streams.  fixed_dest >= 0: every row goes to that rank (gather).
int32_t comm_exchange(Ctx* ctx, const Batch* const* in, int ns, int fixed_dest, Batch** out) {
  Comm* c = ctx->comm;
  // the exchange runs on lane 0 and its peers expect one round at a time
  if (t_lane != 0 || ctx->fork_open) { set_error("exchange: called inside a fork of the execution lanes"); return DBSP_ERR_INVALID; }
  if (!c || c->world == 1) {
    for (int i = 0; i < ns; i++) { batch_ref((Batch*)in[i]); out[i] = (Batch*)in[i]; }
    return DBSP_OK;
  }
  if (!c->connected) { set_error("exchange: dbsp_comm_connect has not been called"); return DBSP_ERR_INVALID; }
  if (ns < 1 || ns > MAX_STREAMS) { set_error("exchange: 1 or 2 streams per round"); return DBSP_ERR_INVALID; }
  cudaStream_t st = ctx->lanes[0].stream;
  const u32 P = (u32)c->world;
  const u64 seq = ++c->seq;
  const int par = (int)(seq & 1);
  // per-round scratch: totals / offsets / ends per stream, error word
  BufP sb;
  TRY(dev_alloc(ctx, (size_t)(MAX_STREAMS * 3 * MAXP + 8) * 8, &sb));
  u64* totals[MAX_STREAMS];
  u64* soff[MAX_STREAMS];
  u64* send[MAX_STREAMS];
  for (int i = 0; i < MAX_STREAMS; i++) {
    totals[i] = (u64*)sb->p + (size_t)(i * 3 + 0) * MAXP;
    soff[i] = (u64*)sb->p + (size_t)(i * 3 + 1) * MAXP;
    send[i] = (u64*)sb->p + (size_t)(i * 3 + 2) * MAXP;
  }
  u64* err = (u64*)sb->p + (size_t)MAX_STREAMS * 3 * MAXP;
  CUDA_TRY(cudaMemsetAsync(sb->p, 0, (size_t)(MAX_STREAMS * 3 * MAXP + 8) * 8, st));
  SendArgs sa;
  SignalArgs sg;
  for (u32 p = 0; p < P; p++) {
    sa.slot[p] = c->slot((int)p, par, c->rank);
    sg.flag[p] = &((Ctrl*)c->peer[p])->flags[par][c->rank];
  }
  sa.slot_bytes = c->slot_bytes;
  std::vector<BufP> hold;
  for (int i = 0; i < ns; i++) {
    const Batch* b = in[i];
    const u64 n = b->n;
    const int L = b->nl();
    if (n >= 0xffffffffull) { set_error("exchange: 2^32-1 or more rows in one batch"); return DBSP_ERR_UNSUPPORTED; }
    if (n == 0) {
      // totals stay zero; the stream's offsets still follow the previous stream's end
      if (i > 0) CUDA_TRY(cudaMemcpyAsync(send[i], send[i - 1], MAXP * 8, cudaMemcpyDeviceToDevice, st));
      continue;
    }
    const u32 ntiles = (u32)((n + PT_TILE - 1) / PT_TILE);
    BufP db, hb;
    TRY(dev_alloc(ctx, (size_t)n, &db));
    TRY(dev_alloc(ctx, ((size_t)P * ntiles + 1) * 4 * 2, &hb));
    hold.push_back(db);
    hold.push_back(hb);
    unsigned char* dest = (unsigned char*)db->p;
    u32* hist = (u32*)hb->p;
    u32* pos = hist + ((size_t)P * ntiles + 1);
    {
      ProfScope ps(ctx, KID_SHARD, n * (u64)(b->s.n_key_lanes * 8 + 1));
      k_shard_hist<<<ntiles, PT_THREADS, 0, st>>>(b->cols(), n, b->s.n_key_lanes, P, fixed_dest, dest, hist, ntiles);
    }
    TRY(exclusive_scan_u32(ctx, hist, pos, (u64)P * ntiles));
    k_shard_totals<<<1, MAXP, 0, st>>>(pos, ntiles, P, L, i > 0 ? send[i - 1] : nullptr, c->slot_bytes, totals[i], soff[i], send[i], err);
    {
      ProfScope ps(ctx, KID_SHARD, n * (u64)((L + 1) * 8 * 2 + 1));
      k_shard_scatter2<<<ntiles, PT_THREADS, 0, st>>>(b->cols(), b->w, n, L, P, dest, pos, ntiles, totals[i], soff[i], err, sa);
    }
    ctx->kernel_launches += 3;
  }
  k_comm_signal<<<1, MAXP, 0, st>>>(sg, P, ns, totals[0], ns > 1 ? totals[1] : nullptr, err, seq);
  const u64 mseq = ++ctx->lanes[0].mail_seq;
  k_comm_wait<<<1, 32, 0, st>>>(((Ctrl*)c->region)->flags[par], P, seq, totals[0], ns > 1 ? totals[1] : nullptr,
                                                   (volatile u64*)ctx->lanes[0].d_mail, mseq, comm_timeout_ns());
  ctx->kernel_launches += 2;
  TRY(mail_wait(ctx, mseq));
  ctx->lanes[0].n_sync++;
  u64 hc[4 * MAXP + 1];
  for (u32 k = 0; k < 4 * P + 1; k++) hc[k] = ctx->lanes[0].h_mail[8 + k];
  ctx->d2h_bytes += (4 * P + 1) * 8;
  if (hc[4 * P] == 2) { set_error("exchange: timed out waiting for a peer's flag (a replica did not reach this exchange)"); return DBSP_ERR_CUDA; }
  if (hc[4 * P] != 0) {
    set_error("exchange: a receive slot is too small for this round (raise slot_bytes of dbsp_comm_create / DBSP_COMM_SLOT_MB)");
    return DBSP_ERR_UNSUPPORTED;
  }
  for (u32 p = 0; p < P; p++)
    if ((int)p != c->rank)
      for (int i = 0; i < ns; i++) c->bytes_sent += hc[2 * P + p * 2 + i] * (u64)(in[i]->nl() + 1) * 8;
  // views over my receive slots, then the receiver's merge
  for (int i = 0; i < ns; i++) {
    std::vector<Batch*> parts;
    for (u32 src = 0; src < P; src++) {
      u64 off = 0;
      for (int j = 0; j < i; j++) {
        const u64 cj = hc[src * 2 + j];
        const u64 stride = (cj + 32) & ~31ull;
        off = ((off + (cj ? stride * 8 * (u64)(in[j]->nl() + 1) : 0)) + 255) & ~255ull;
      }
      parts.push_back(segment_view(ctx, in[i]->s, c->slot(c->rank, par, (int)src) + off, hc[src * 2 + i]));
    }
    Batch* o = nullptr;
    int32_t rc = merge_views(ctx, parts, in[i]->s, &o);
    if (rc) { for (int j = 0; j < i; j++) { batch_unref(out[j]); out[j] = nullptr; } return rc; }
    out[i] = o;
  }
  return DBSP_OK;
}

int32_t comm_allreduce_max(Ctx* ctx, u64* x) {
  Comm* c = ctx->comm;
  if (t_lane != 0 || ctx->fork_open) { set_error("allreduce: called inside a fork of the execution lanes"); return DBSP_ERR_INVALID; }
  if (!c || c->world == 1) return DBSP_OK;
  if (!c->connected) { set_error("allreduce: dbsp_comm_connect has not been called"); return DBSP_ERR_INVALID; }
  const u64 seq = ++c->red_seq;
  const int par = (int)(seq & 1);
  RedArgs ra;
  for (int p = 0; p < c->world; p++) ra.slot[p] = &((Ctrl*)c->peer[p])->red[par][c->rank];
  const u64 mseq = ++ctx->lanes[0].mail_seq;
  k_comm_allreduce_max<<<1, 32, 0, ctx->lanes[0].stream>>>(ra, ((Ctrl*)c->region)->red[par], (u32)c->world, *x, seq,
                                                                        (volatile u64*)ctx->lanes[0].d_mail, mseq, comm_timeout_ns());
  ctx->kernel_launches++;
  TRY(mail_wait(ctx, mseq));
  ctx->lanes[0].n_sync++;
  if (ctx->lanes[0].h_mail[9] != 0) { set_error("allreduce: timed out waiting for a peer"); return DBSP_ERR_CUDA; }
  *x = ctx->lanes[0].h_mail[8];
  return DBSP_OK;
}

void comm_info(Ctx* ctx, int* rank, int* world, u64* bytes_sent) {
  Comm* c = ctx->comm;
  if (rank) *rank = c ? c->rank : 0;
  if (world) *world = c ? c->world : 1;
  if (bytes_sent) *bytes_sent = c ? c->bytes_sent : 0;
}
