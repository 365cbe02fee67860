// capi.cu — the extern "C" boundary declared in include/dbsp_b200.h, plus the
// host-side Spine (trace) logic.  No CPU compute path lives here: every
// data-touching call launches kernels from consolidate.cu / merge.cu / ops.cu.
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "ops.cuh"

const char* get_error();
void print_host_stats(Ctx* c);
void pool_release_all(Ctx* ctx);

struct dbsp_ctx : Ctx {};
struct dbsp_batch : Batch {};
struct dbsp_spine : Spine {};
struct Merger;
struct dbsp_merger;
struct dbsp_batcher;

static inline Batch* B(const dbsp_batch* b) { return (Batch*)b; }
static inline dbsp_batch* H(Batch* b) { return (dbsp_batch*)b; }

// every entry point makes the context's device current: a host may drive several contexts (GPUs) from one
// process, one per worker thread (INTEGRATION.md §3)
#define ENTER(c) CUDA_TRY(cudaSetDevice((c)->device))
#define CHECK_ARG(c, msg)                 \
  do {                                    \
    if (!(c)) { set_error(msg); return DBSP_ERR_INVALID; } \
  } while (0)

// Stage host columns on the device (stream-ordered).  Host memory may be
// pageable; pinned memory makes the copy asynchronous.
static int32_t stage_columns(Ctx* ctx, const u64* const* cols, int ncols, const i64* w, u64 n, int on_device, BufP* hold,
                             Cols* dc, const i64** dw, unsigned col_mask = ~0u) {
  for (int l = 0; l < MAXL; l++) dc->c[l] = nullptr;
  *dw = nullptr;
  if (on_device || n == 0) {
    for (int l = 0; l < ncols; l++) dc->c[l] = cols[l];
    *dw = w;
    return DBSP_OK;
  }
  u64 cap = (n + 32) & ~31ull;
  TRY(dev_alloc(ctx, (size_t)cap * 8 * (ncols + 1), hold));
  u64* base = (u64*)(*hold)->p;
  for (int l = 0; l < ncols; l++) {
    if (!((col_mask >> l) & 1)) continue;   // column never read by the closure: not copied
    CUDA_TRY(cudaMemcpyAsync(base + (size_t)l * cap, cols[l], n * 8, cudaMemcpyHostToDevice, lane(ctx).stream));
    dc->c[l] = base + (size_t)l * cap;
    ctx->h2d_bytes += n * 8;
  }
  if (w) {
    i64* p = (i64*)(base + (size_t)ncols * cap);
    CUDA_TRY(cudaMemcpyAsync(p, w, n * 8, cudaMemcpyHostToDevice, lane(ctx).stream));
    ctx->h2d_bytes += n * 8;
    *dw = p;
  }
  return DBSP_OK;
}

// ---- Spine: the fuelled LSM of trace/spine_fueled.rs ---------------------------------------------------------------
// The layer structure and the schedule are the reference's, restated: insert -> introduce_batch (:728-812: apply
// fuel to the merges in progress, roll_up, insert_at, tidy_layers), roll_up (:819-846), apply_fuel (:856-882),
// insert_at (:889-908), tidy_layers (:916-974), exert (:561-581), consolidate (:583-600), reduced (:663-680),
// MergeState / MergeVariant (:1012-1188).  One deliberate difference in *how* a merge spends its fuel: the
// reference's Merger advances a few thousand rows per call; the GPU merges two whole batches in one launch, so a
// merge in progress is a fuel account — the two batches stay visible to cursors exactly as long as in the
// reference (until the fuel paid reaches their length) and the single merge launch happens when the account is
// settled.  The schedule (which batches meet, when a layer becomes complete) is therefore the reference's.
static int32_t merge_bounded(Ctx* ctx, const Batch* x, const Batch* y, const u64* vbound, Batch** out);

static u64 level_len(const SpineLevel& l) {   // MergeState::len (:1034-1041)
  switch (l.kind) {
    case SpineLevel::SINGLE: return l.a ? l.a->n : 0;
    case SpineLevel::IN_PROGRESS: return l.a->n + l.b->n;
    case SpineLevel::COMPLETE: return l.a ? l.a->n : 0;
    default: return 0;
  }
}
static inline bool level_is_double(const SpineLevel& l) { return l.kind == SpineLevel::IN_PROGRESS || l.kind == SpineLevel::COMPLETE; }

static void spine_refresh_view(Spine* s) {   // the batches a SpineCursor is built from (:179-216)
  s->batches.clear();
  for (size_t i = s->merging.size(); i-- > 0;) {
    const SpineLevel& l = s->merging[i];
    if (l.kind == SpineLevel::IN_PROGRESS) {
      if (l.a->n) s->batches.push_back(l.a);
      if (l.b->n) s->batches.push_back(l.b);
    } else if ((l.kind == SpineLevel::SINGLE || l.kind == SpineLevel::COMPLETE) && l.a && l.a->n) {
      s->batches.push_back(l.a);
    }
  }
}

// MergeState::begin_merge (:1106-1124); takes over the references of both batches
static SpineLevel level_begin_merge(Batch* b1, Batch* b2) {
  SpineLevel l;
  if (b1 && b2) {
    l.kind = SpineLevel::IN_PROGRESS;
    l.a = b1;
    l.b = b2;
    l.remaining = (i64)(b1->n + b2->n);
  } else {
    l.kind = SpineLevel::COMPLETE;
    l.a = b1 ? b1 : b2;
  }
  return l;
}

// MergeVariant::work (:1176-1188): pay `*fuel` into the account; when it is settled the merge runs (one launch)
// and the layer becomes Complete.  *fuel > 0 afterwards <=> the merge completed (trace/mod.rs:388-395).
static int32_t level_work(Ctx* ctx, Spine* s, SpineLevel& l, i64* fuel) {
  if (l.kind != SpineLevel::IN_PROGRESS) return DBSP_OK;
  if (*fuel < l.remaining) {
    l.remaining -= *fuel;
    *fuel = 0;
    return DBSP_OK;
  }
  *fuel = (*fuel == INT64_MAX) ? INT64_MAX : (*fuel - l.remaining > 0 ? *fuel - l.remaining : 1);
  Batch* merged = nullptr;
  TRY(merge_bounded(ctx, l.a, l.b, s->has_vbound ? s->vbound : nullptr, &merged));
  batch_unref(l.a);
  batch_unref(l.b);
  l.kind = SpineLevel::COMPLETE;
  l.a = merged;
  l.b = nullptr;
  l.remaining = 0;
  return DBSP_OK;
}

// MergeState::complete (:1060-1066): finish whatever the layer holds and take it out (nullptr = nothing)
static int32_t level_complete(Ctx* ctx, Spine* s, SpineLevel& l, Batch** out) {
  *out = nullptr;
  if (l.kind == SpineLevel::IN_PROGRESS) {
    i64 fuel = INT64_MAX;
    TRY(level_work(ctx, s, l, &fuel));
  }
  if (l.kind == SpineLevel::SINGLE || l.kind == SpineLevel::COMPLETE) *out = l.a;
  l = SpineLevel();
  return DBSP_OK;
}

// insert_at (:889-908)
static int32_t spine_insert_at(Spine* s, Batch* batch, size_t index) {
  while (s->merging.size() <= index) s->merging.push_back(SpineLevel());
  SpineLevel& l = s->merging[index];
  switch (l.kind) {
    case SpineLevel::VACANT:
      l.kind = SpineLevel::SINGLE;
      l.a = batch;
      return DBSP_OK;
    case SpineLevel::SINGLE: {
      Batch* old = l.a;
      l = level_begin_merge(old, batch);
      return DBSP_OK;
    }
    default:
      if (batch) batch_unref(batch);
      set_error("spine: attempted to insert a batch into an incomplete merge");   // panic! in the reference (:904)
      return DBSP_ERR_INVALID;
  }
}

// apply_fuel (:856-882): every layer receives the same fuel; a merge that completes moves up at once
static int32_t spine_apply_fuel(Ctx* ctx, Spine* s, i64 fuel_each) {
  for (size_t index = 0; index < s->merging.size(); index++) {
    i64 fuel = fuel_each;
    TRY(level_work(ctx, s, s->merging[index], &fuel));
    if (s->merging[index].kind == SpineLevel::COMPLETE) {
      Batch* done = nullptr;
      TRY(level_complete(ctx, s, s->merging[index], &done));
      TRY(spine_insert_at(s, done, index + 1));
    }
  }
  return DBSP_OK;
}

// roll_up (:819-846)
static int32_t spine_roll_up(Ctx* ctx, Spine* s, size_t index) {
  while (s->merging.size() <= index) s->merging.push_back(SpineLevel());
  bool any = false;
  for (size_t i = 0; i < index; i++) any = any || s->merging[i].kind != SpineLevel::VACANT;
  if (!any) return DBSP_OK;
  Batch* merged = nullptr;
  for (size_t i = 0; i < index; i++) {
    TRY(spine_insert_at(s, merged, i));
    TRY(level_complete(ctx, s, s->merging[i], &merged));
  }
  TRY(spine_insert_at(s, merged, index));
  if (level_is_double(s->merging[index])) {
    Batch* m2 = nullptr;
    TRY(level_complete(ctx, s, s->merging[index], &m2));
    TRY(spine_insert_at(s, m2, index + 1));
  }
  return DBSP_OK;
}

// tidy_layers (:916-974)
static int32_t spine_tidy_layers(Spine* s) {
  if (s->merging.empty()) return DBSP_OK;
  size_t length = s->merging.size();
  if (s->merging[length - 1].kind != SpineLevel::SINGLE) return DBSP_OK;
  const u64 len = level_len(s->merging[length - 1]);
  size_t appropriate = 0;   // len.next_power_of_two().trailing_zeros()
  while ((1ull << appropriate) < len) appropriate++;
  while (appropriate < length - 1) {
    SpineLevel& below = s->merging[length - 2];
    if (below.kind == SpineLevel::VACANT || (below.kind == SpineLevel::SINGLE && below.a == nullptr)) {
      s->merging.erase(s->merging.begin() + (length - 2));
      length = s->merging.size();
    } else if (below.kind == SpineLevel::SINGLE) {
      u64 smaller = 0;
      for (size_t i = 0; i + 2 < length; i++) {
        if (s->merging[i].kind == SpineLevel::SINGLE) smaller += 1ull << i;
        else if (level_is_double(s->merging[i])) smaller += 2ull << i;
      }
      if (smaller <= (1ull << length) / 8) {
        Batch* batch = below.a;
        s->merging.erase(s->merging.begin() + (length - 2));
        TRY(spine_insert_at(s, batch, length - 2));
      }
      return DBSP_OK;
    } else {
      return DBSP_OK;   // a merge is in progress: nothing to do
    }
  }
  return DBSP_OK;
}

// introduce_batch (:728-812)
static int32_t spine_introduce_batch(Ctx* ctx, Spine* s, Batch* batch, size_t batch_index) {
  i64 fuel = batch_index >= 59 ? INT64_MAX : (i64)((8ull << batch_index) * s->effort);
  int32_t rc = spine_apply_fuel(ctx, s, fuel);
  if (rc == DBSP_OK) rc = spine_roll_up(ctx, s, batch_index);
  if (rc != DBSP_OK) { if (batch) batch_unref(batch); return rc; }
  TRY(spine_insert_at(s, batch, batch_index));
  return spine_tidy_layers(s);
}

// reduced (:663-680)
static bool spine_reduced(const Spine* s) {
  int non_empty = 0;
  for (const SpineLevel& l : s->merging) {
    if (level_is_double(l)) return false;
    if (level_len(l) > 0) non_empty++;
    if (non_empty > 1) return false;
  }
  return true;
}

// exert (:561-581)
static int32_t spine_exert(Ctx* ctx, Spine* s, i64* effort) {
  TRY(spine_tidy_layers(s));
  if (!spine_reduced(s)) {
    bool any_double = false;
    for (const SpineLevel& l : s->merging) any_double = any_double || level_is_double(l);
    if (any_double) {
      TRY(spine_apply_fuel(ctx, s, *effort));
    } else {
      size_t level = 0;   // (*effort as usize).next_power_of_two().trailing_zeros()
      while ((1ull << level) < (u64)(*effort > 0 ? *effort : 1) && level < 62) level++;
      TRY(spine_introduce_batch(ctx, s, nullptr, level));
    }
  }
  spine_refresh_view(s);
  return DBSP_OK;
}

// truncate_keys_below (spine_fueled.rs:223-233; column_layer/mod.rs:316-319):
// a zero-copy suffix view of the batch.
static int32_t spine_truncate_batch(Ctx* ctx, Spine* s, Batch* b, Batch** out) {
  u64 pos;
  TRY(batch_lower_bound(ctx, b, s->bound, &pos));
  if (pos == 0) { batch_ref(b); *out = b; return DBSP_OK; }
  *out = batch_slice(ctx, b, pos, b->n);
  return DBSP_OK;
}

// Trace::insert (:605-634)
static int32_t spine_insert(Ctx* ctx, Spine* s, Batch* b) {
  if (b->n == 0) return DBSP_OK;   // empty batches are ignored (:609-611)
  Batch* nb = nullptr;
  if (s->has_bound) {
    TRY(spine_truncate_batch(ctx, s, b, &nb));
  } else {
    batch_ref(b);
    nb = b;
  }
  size_t index = 0;   // batch.len().next_power_of_two().trailing_zeros()
  while ((1ull << index) < nb->n) index++;
  int32_t rc = spine_introduce_batch(ctx, s, nb, index);
  spine_refresh_view(s);
  return rc;
}

// Merge of two batches with the spine's lower value bound applied to the
// result (Merger::work(.., lower_val_bound, ..), spine_fueled.rs:866,911,981).
static int32_t merge_bounded(Ctx* ctx, const Batch* x, const Batch* y, const u64* vbound, Batch** out) {
  Batch* merged = nullptr;
  TRY(merge_batches(ctx, x, y, &merged));
  if (!vbound || merged->s.n_val_lanes == 0) { *out = merged; return DBSP_OK; }
  int32_t rc = op_truncate_values(ctx, merged, vbound, out);
  batch_unref(merged);
  return rc;
}

// complete_merges (:977-985)
static int32_t spine_complete_merges(Ctx* ctx, Spine* s) {
  for (SpineLevel& l : s->merging) {
    i64 fuel = INT64_MAX;
    TRY(level_work(ctx, s, l, &fuel));
  }
  return DBSP_OK;
}

static void spine_release(Spine* s) {
  for (SpineLevel& l : s->merging) {
    if (l.a) batch_unref(l.a);
    if (l.b) batch_unref(l.b);
  }
  s->merging.clear();
  s->batches.clear();
}

// The fuelled Merger (trace/mod.rs:371-396).  On the device a unit of fuel is
// one input row: work() cuts the merge path `fuel` rows further along, merges
// the two row ranges in between with the tile kernel and keeps the chunk; the
// chunks are ordered and disjoint, done() concatenates them.
struct Merger {
  Ctx* ctx;
  Batch *a, *b;
  u64 ai = 0, bi = 0;
  bool has_vb = false;
  u64 vb[MAXL];
  std::vector<Batch*> chunks;
  bool complete() const { return ai == a->n && bi == b->n; }
};

extern "C" {

const char* dbsp_last_error(void) { return get_error(); }

int32_t dbsp_ctx_create(int32_t device, dbsp_ctx** out) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0 || device >= count) {
    set_error(std::string("no usable CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU fallback");
    return DBSP_ERR_NO_DEVICE;
  }
  CUDA_TRY(cudaSetDevice(device));
  dbsp_ctx* c = new dbsp_ctx();
  c->device = device;
  CUDA_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&c->read_stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaMallocHost(&c->h_scratch, 256 * 8));
  {
    // one mailbox slot (320 words) and 256 scratch words per lane
    void* hm = nullptr;
    CUDA_TRY(cudaHostAlloc(&hm, N_LANES * 320 * 8, cudaHostAllocMapped));
    memset(hm, 0, N_LANES * 320 * 8);
    void* dm = nullptr;
    CUDA_TRY(cudaHostGetDevicePointer(&dm, hm, 0));
    u64* ds = nullptr;
    CUDA_TRY(cudaMalloc(&ds, N_LANES * 256 * 8));
    CUDA_TRY(cudaMemset(ds, 0, N_LANES * 256 * 8));
    for (int i = 0; i < N_LANES; i++) {
      Lane& l = c->lanes[i];
      CUDA_TRY(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
      CUDA_TRY(cudaEventCreateWithFlags(&l.ev, cudaEventDisableTiming));
      l.h_mail = (volatile u64*)hm + i * 320;
      l.d_mail = (u64*)dm + i * 320;
      l.d_scratch = ds + i * 256;
    }
  }
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  // optional up-front pool reservation (GiB) so that slab growth never lands
  // inside a timed region: DBSP_POOL_RESERVE_GB
  if (const char* e = getenv("DBSP_POOL_RESERVE_GB")) {
    double gb = atof(e);
    if (gb > 0) {
      std::vector<BufP> hold;   // released together at the end of this scope: the slabs stay pooled
      size_t bytes = (size_t)(gb * 1073741824.0);
      for (size_t done = 0; done < bytes; done += ((size_t)8 << 30)) {
        BufP x;
        if (dev_alloc(c, std::min<size_t>((size_t)8 << 30, bytes - done), &x) != DBSP_OK) break;
        hold.push_back(x);
      }
    }
  }
  *out = c;
  return DBSP_OK;
}
int32_t dbsp_ctx_destroy(dbsp_ctx* c) {
  if (!c) return DBSP_OK;
  print_host_stats(c);
  cudaSetDevice(c->device);
  lanes_shutdown(c);
  for (Lane& l : c->lanes) cudaStreamSynchronize(l.stream);
  comm_free(c);
  cudaFreeHost(c->h_scratch);
  cudaFreeHost((void*)c->lanes[0].h_mail);
  cudaFree(c->lanes[0].d_scratch);
  pool_release_all(c);
  for (Lane& l : c->lanes) {
    for (auto& r : l.prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto& e : l.ev_pool) cudaEventDestroy(e);
    l.prof.clear();
    l.ev_pool.clear();
    cudaEventDestroy(l.ev);
    cudaStreamDestroy(l.stream);
    l.stream = nullptr;
  }
  cudaStreamDestroy(c->copy_stream);
  cudaStreamDestroy(c->read_stream);
  c->destroyed = true;
  if (c->live_bufs.load() == 0) delete c;   // else the last DevBuf deletes it
  return DBSP_OK;
}
int32_t dbsp_ctx_sync(dbsp_ctx* c) { ENTER(c);
  CUDA_TRY(cudaStreamSynchronize(c->lanes[0].stream));   // lane 0 waits for lane 1 at every join
  return DBSP_OK;
}
int32_t dbsp_ctx_stats(dbsp_ctx* c, uint64_t* k, uint64_t* h2d, uint64_t* d2h, int32_t reset) { ENTER(c);
  if (k) *k = c->kernel_launches;
  if (h2d) *h2d = c->h2d_bytes;
  if (d2h) *d2h = c->d2h_bytes;
  if (reset) { c->kernel_launches = 0; c->h2d_bytes = 0; c->d2h_bytes = 0; }
  return DBSP_OK;
}
int32_t dbsp_ctx_sync_stats(dbsp_ctx* c, uint64_t* n_waits, double* wait_us, int32_t reset) {
  // both lanes: waits on lane 1 overlap lane 0's work, so wait_us may exceed the wall time it covers
  if (n_waits) *n_waits = c->lanes[0].n_sync + c->lanes[1].n_sync;
  if (wait_us) *wait_us = c->lanes[0].t_sync_us + c->lanes[1].t_sync_us;
  if (reset) for (Lane& l : c->lanes) { l.n_sync = 0; l.t_sync_us = 0; }
  return DBSP_OK;
}
void* dbsp_ctx_stream(dbsp_ctx* c) { return (void*)c->lanes[0].stream; }

int32_t dbsp_ctx_profile(dbsp_ctx* c, int32_t enable) { ENTER(c);
  if (enable == 2) { c->prof_on = false; return DBSP_OK; }   // pause: keep what was collected, record nothing more
  CUDA_TRY(cudaStreamSynchronize(c->lanes[0].stream));
  for (Lane& l : c->lanes) {
    for (auto& r : l.prof) { l.ev_pool.push_back(r.a); l.ev_pool.push_back(r.b); }
    l.prof.clear();
  }
  c->prof_on = enable != 0;
  return DBSP_OK;
}
int32_t dbsp_ctx_profile_read(dbsp_ctx* c, int32_t id, char* name32, uint64_t* launches, double* ms, uint64_t* bytes) { ENTER(c);
  if (id < 0 || id >= KID_COUNT) return DBSP_ERR_INVALID;
  CUDA_TRY(cudaStreamSynchronize(c->lanes[0].stream));
  u64 n = 0, b = 0;
  double t = 0;
  for (Lane& l : c->lanes) {
    for (auto& r : l.prof) {
      if (r.id != id) continue;
      float e = 0;
      if (cudaEventElapsedTime(&e, r.a, r.b) == cudaSuccess) t += e;
      n++;
      b += r.bytes;
    }
  }
  if (name32) { strncpy(name32, kernel_name(id), 31); name32[31] = 0; }
  if (launches) *launches = n;
  if (ms) *ms = t;
  if (bytes) *bytes = b;
  return DBSP_OK;
}

int32_t dbsp_batch_from_tuples(dbsp_ctx* ctx, const dbsp_schema* s, const uint64_t* const* cols, const int64_t* w,
                               uint64_t n, int32_t on_device, dbsp_batch** out) { ENTER(ctx);
  int L = s->n_key_lanes + s->n_val_lanes;
  CHECK_ARG(L >= 1 && L <= MAXL, "schema must have 1..8 lanes");
  BufP hold;
  Cols dc;
  const i64* dw;
  TRY(stage_columns(ctx, cols, L, w, n, on_device, &hold, &dc, &dw));
  Batch* b = nullptr;
  TRY(consolidate_rows(ctx, *s, dc, dw, n, (hold && dw) ? &hold : nullptr, &b));
  *out = H(b);
  return DBSP_OK;
}

struct dbsp_upload {
  Ctx* ctx;
  BufP buf;
  Cols dc;
  const i64* dw;
  u64 n;
  int n_cols;
  cudaEvent_t done;
};

// flat_map_index of one raw table on the calling thread's lane
static int32_t table_to_batch(Ctx* ctx, const dbsp_table_job& j, Batch** out) {
  CHECK_ARG(j.proj != nullptr, "table: projection is NULL");
  if (j.upload) {
    CUDA_TRY(cudaStreamWaitEvent(lane(ctx).stream, j.upload->done, 0));   // the lane waits for the copy
    return project_and_consolidate(ctx, j.upload->dc, 0, j.upload->n_cols, j.upload->dw, j.upload->n, *j.proj, out);
  }
  CHECK_ARG(j.n_cols >= 1 && j.n_cols <= MAXL, "table must have 1..8 columns");
  BufP hold;
  Cols dc;
  const i64* dw;
  TRY(stage_columns(ctx, j.cols, (int)j.n_cols, j.weights, j.n, j.on_device, &hold, &dc, &dw, proj_used_mask(*j.proj, 0)));
  return project_and_consolidate(ctx, dc, 0, (int)j.n_cols, dw, j.n, *j.proj, out);
}

int32_t dbsp_batch_from_table(dbsp_ctx* ctx, const uint64_t* const* cols, uint32_t n_cols, const int64_t* w, uint64_t n,
                              int32_t on_device, const dbsp_proj* proj, dbsp_batch** out) { ENTER(ctx);
  dbsp_table_job j = {cols, w, n, nullptr, proj, n_cols, on_device};
  Batch* b = nullptr;
  TRY(table_to_batch(ctx, j, &b));
  *out = H(b);
  return DBSP_OK;
}

int32_t dbsp_batches_from_tables(dbsp_ctx* ctx, uint32_t k, const dbsp_table_job* jobs, dbsp_batch** outs) { ENTER(ctx);
  CHECK_ARG(k == 0 || (jobs && outs), "batches_from_tables: jobs / outs is NULL");
  // Largest table first, each onto the lane with fewer rows so far: lane 0 (this thread) starts on the largest one
  // while the worker picks up its share.
  std::vector<uint32_t> order(k);
  for (uint32_t i = 0; i < k; i++) order[i] = i;
  auto rows = [&](uint32_t i) { return jobs[i].upload ? jobs[i].upload->n : jobs[i].n; };
  std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return rows(a) > rows(b); });
  std::vector<uint32_t> on[N_LANES];
  u64 load[N_LANES] = {0, 0};
  for (uint32_t i : order) {
    const int l = load[1] < load[0] ? 1 : 0;
    on[l].push_back(i);
    load[l] += rows(i);
  }
  std::vector<Batch*> o(k, nullptr);
  auto run = [&](const std::vector<uint32_t>& js) -> int32_t {
    for (uint32_t i : js) TRY(table_to_batch(ctx, jobs[i], &o[i]));
    return DBSP_OK;
  };
  const int32_t rc = on[1].empty() ? run(on[0]) : run_forked(ctx, [&] { return run(on[0]); }, [&] { return run(on[1]); });
  if (rc != DBSP_OK) {
    for (Batch* b : o) batch_unref(b);
    return rc;
  }
  for (uint32_t i = 0; i < k; i++) outs[i] = H(o[i]);
  return DBSP_OK;
}

uint32_t dbsp_proj_table_mask(const dbsp_proj* proj) { return proj_used_mask(*proj, 0); }

int32_t dbsp_upload_begin(dbsp_ctx* ctx, const uint64_t* const* cols, uint32_t n_cols, uint32_t col_mask,
                          const int64_t* w, uint64_t n, dbsp_upload** out) { ENTER(ctx);
  CHECK_ARG(n_cols >= 1 && n_cols <= MAXL, "table must have 1..8 columns");
  dbsp_upload* u = new dbsp_upload();
  u->ctx = ctx;
  u->n = n;
  u->n_cols = (int)n_cols;
  u->dw = nullptr;
  for (int l = 0; l < MAXL; l++) u->dc.c[l] = nullptr;
  CUDA_TRY(cudaEventCreateWithFlags(&u->done, cudaEventDisableTiming));
  if (n) {
    u64 cap = (n + 32) & ~31ull;
    TRY(dev_alloc(ctx, (size_t)cap * 8 * (n_cols + 1), &u->buf));
    // the block may have been used by work still queued on the compute stream
    cudaEvent_t ev;
    CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(ev, lane(ctx).stream));
    CUDA_TRY(cudaStreamWaitEvent(ctx->copy_stream, ev, 0));
    CUDA_TRY(cudaEventDestroy(ev));
    u64* base = (u64*)u->buf->p;
    for (uint32_t l = 0; l < n_cols; l++) {
      if (!((col_mask >> l) & 1)) continue;
      CUDA_TRY(cudaMemcpyAsync(base + (size_t)l * cap, cols[l], n * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
      u->dc.c[l] = base + (size_t)l * cap;
      ctx->h2d_bytes += n * 8;
    }
    if (w) {
      i64* p = (i64*)(base + (size_t)n_cols * cap);
      CUDA_TRY(cudaMemcpyAsync(p, w, n * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
      ctx->h2d_bytes += n * 8;
      u->dw = p;
    }
  }
  CUDA_TRY(cudaEventRecord(u->done, ctx->copy_stream));
  *out = u;
  return DBSP_OK;
}

int32_t dbsp_batch_from_upload(dbsp_ctx* ctx, dbsp_upload* u, const dbsp_proj* proj, dbsp_batch** out) { ENTER(ctx);
  dbsp_table_job j = {nullptr, nullptr, 0, u, proj, 0, 0};
  Batch* b = nullptr;
  TRY(table_to_batch(ctx, j, &b));
  *out = H(b);
  return DBSP_OK;
}

int32_t dbsp_upload_free(dbsp_upload* u) {
  if (!u) return DBSP_OK;
  // a consumed upload's buffer is only reused by later work on the compute
  // stream (ordered after the consumer); an unconsumed one must drain first
  cudaEventSynchronize(u->done);
  cudaEventDestroy(u->done);
  delete u;
  return DBSP_OK;
}

int32_t dbsp_batch_from_sorted(dbsp_ctx* ctx, const dbsp_schema* s, const uint64_t* const* cols, const int64_t* w,
                               uint64_t n, int32_t on_device, dbsp_batch** out) { ENTER(ctx);
  int L = s->n_key_lanes + s->n_val_lanes;
  if (n == 0) { *out = H(batch_new_empty(ctx, *s)); return DBSP_OK; }
  Batch* b;
  MCols oc;
  i64* ow;
  TRY(batch_alloc(ctx, *s, n, &b, &oc, &ow));
  cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  for (int l = 0; l < L; l++) CUDA_TRY(cudaMemcpyAsync(oc.c[l], cols[l], n * 8, kind, lane(ctx).stream));
  CUDA_TRY(cudaMemcpyAsync(ow, w, n * 8, kind, lane(ctx).stream));
  if (!on_device) { ctx->h2d_bytes += n * 8 * (L + 1); CUDA_TRY(cudaStreamSynchronize(lane(ctx).stream)); }
  *out = H(b);
  return DBSP_OK;
}

// MergeBatcher (trace/ord/merge_batcher/mod.rs:155-260): queue of consolidated
// batches, newest last; the two newest are merged while the newer holds at least
// half the rows of the older (the reference compares chunk counts of 8 KiB
// buffers — the same geometric rule; the schedule is not observable in seal()).
struct Batcher {
  dbsp_schema s;
  std::vector<Batch*> queue;
};
static int32_t batcher_enqueue(Ctx* ctx, Batcher* q, Batch* b) {
  if (b->n == 0) { batch_unref(b); return DBSP_OK; }
  q->queue.push_back(b);
  while (q->queue.size() > 1 && q->queue[q->queue.size() - 1]->n >= q->queue[q->queue.size() - 2]->n / 2) {
    Batch* y = q->queue.back(); q->queue.pop_back();
    Batch* x = q->queue.back(); q->queue.pop_back();
    Batch* m = nullptr;
    int32_t rc = merge_batches(ctx, x, y, &m);
    batch_unref(x);
    batch_unref(y);
    if (rc) return rc;
    if (m->n) q->queue.push_back(m); else batch_unref(m);
  }
  return DBSP_OK;
}
int32_t dbsp_batcher_new(dbsp_ctx*, const dbsp_schema* s, dbsp_batcher** out) {
  int L = s->n_key_lanes + s->n_val_lanes;
  CHECK_ARG(L >= 1 && L <= MAXL, "schema must have 1..8 lanes");
  Batcher* q = new Batcher();
  q->s = *s;
  *out = (dbsp_batcher*)q;
  return DBSP_OK;
}
int32_t dbsp_batcher_push(dbsp_ctx* ctx, dbsp_batcher* bq, const uint64_t* const* cols, const int64_t* w, uint64_t n,
                          int32_t on_device) { ENTER(ctx);
  Batcher* q = (Batcher*)bq;
  if (n == 0) return DBSP_OK;
  dbsp_batch* b = nullptr;
  TRY(dbsp_batch_from_tuples(ctx, &q->s, cols, w, n, on_device, &b));
  return batcher_enqueue(ctx, q, B(b));
}
int32_t dbsp_batcher_push_consolidated(dbsp_ctx* ctx, dbsp_batcher* bq, const uint64_t* const* cols, const int64_t* w,
                                       uint64_t n, int32_t on_device) { ENTER(ctx);
  Batcher* q = (Batcher*)bq;
  if (n == 0) return DBSP_OK;
  CHECK_ARG(w != nullptr, "push_consolidated: weights required");
  dbsp_batch* b = nullptr;
  TRY(dbsp_batch_from_sorted(ctx, &q->s, cols, w, n, on_device, &b));
  return batcher_enqueue(ctx, q, B(b));
}
int32_t dbsp_batcher_tuples(const dbsp_batcher* bq, uint64_t* n) {
  u64 t = 0;
  for (Batch* b : ((const Batcher*)bq)->queue) t += b->n;
  *n = t;
  return DBSP_OK;
}
int32_t dbsp_batcher_free(dbsp_batcher* bq) {
  Batcher* q = (Batcher*)bq;
  if (!q) return DBSP_OK;
  for (Batch* b : q->queue) batch_unref(b);
  delete q;
  return DBSP_OK;
}
int32_t dbsp_batcher_seal(dbsp_ctx* ctx, dbsp_batcher* bq, dbsp_batch** out) { ENTER(ctx);   // finish_into (:251-265) + Builder
  Batcher* q = (Batcher*)bq;
  while (q->queue.size() >= 2) {
    Batch* y = q->queue.back(); q->queue.pop_back();
    Batch* x = q->queue.back(); q->queue.pop_back();
    Batch* m = nullptr;
    int32_t rc = merge_batches(ctx, x, y, &m);
    batch_unref(x);
    batch_unref(y);
    if (rc) return rc;
    if (m->n) q->queue.push_back(m); else batch_unref(m);
  }
  Batch* r = q->queue.empty() ? batch_new_empty(ctx, q->s) : q->queue.back();
  q->queue.clear();
  delete q;
  *out = H(r);
  return DBSP_OK;
}

int32_t dbsp_batch_empty(dbsp_ctx* ctx, const dbsp_schema* s, dbsp_batch** out) { ENTER(ctx);
  *out = H(batch_new_empty(ctx, *s));
  return DBSP_OK;
}

int32_t dbsp_batch_merge(dbsp_ctx* ctx, const dbsp_batch* a, const dbsp_batch* b, dbsp_batch** out) { ENTER(ctx);
  Batch* o = nullptr;
  TRY(merge_batches(ctx, B(a), B(b), &o));
  *out = H(o);
  return DBSP_OK;
}

int32_t dbsp_batch_merge_bounded(dbsp_ctx* ctx, const dbsp_batch* a, const dbsp_batch* b, const uint64_t* vb,
                                 dbsp_batch** out) { ENTER(ctx);
  Batch* o = nullptr;
  TRY(merge_bounded(ctx, B(a), B(b), vb, &o));
  *out = H(o);
  return DBSP_OK;
}

int32_t dbsp_batch_truncate_keys_below(dbsp_ctx* ctx, const dbsp_batch* b, const uint64_t* key, dbsp_batch** out) { ENTER(ctx);
  u64 pos;
  TRY(batch_lower_bound(ctx, B(b), key, &pos));
  if (pos == 0) { batch_ref(B(b)); *out = (dbsp_batch*)b; return DBSP_OK; }
  *out = H(batch_slice(ctx, B(b), pos, B(b)->n));
  return DBSP_OK;
}

int32_t dbsp_merger_new(dbsp_ctx* ctx, const dbsp_batch* a, const dbsp_batch* b, const uint64_t* vb, dbsp_merger** out) { ENTER(ctx);
  CHECK_ARG(memcmp(&B(a)->s, &B(b)->s, sizeof(dbsp_schema)) == 0, "merger_new: schema mismatch");
  Merger* m = new Merger();
  m->ctx = ctx;
  m->a = B(a);
  m->b = B(b);
  batch_ref(m->a);
  batch_ref(m->b);
  if (vb && B(a)->s.n_val_lanes) {
    m->has_vb = true;
    for (int l = 0; l < B(a)->s.n_val_lanes; l++) m->vb[l] = vb[l];
  }
  *out = (dbsp_merger*)m;
  return DBSP_OK;
}

int32_t dbsp_merger_work(dbsp_ctx* ctx, dbsp_merger* mm, int64_t* fuel) { ENTER(ctx);
  Merger* m = (Merger*)mm;
  if (!m->complete() && *fuel > 0) {
    u64 na, nb;
    TRY(merge_path_split(ctx, m->a, m->b, m->ai + m->bi + (u64)*fuel, &na, &nb));
    Batch* xa = batch_slice(ctx, m->a, m->ai, na);
    Batch* xb = batch_slice(ctx, m->b, m->bi, nb);
    Batch* chunk = nullptr;
    int32_t rc = merge_bounded(ctx, xa, xb, m->has_vb ? m->vb : nullptr, &chunk);
    batch_unref(xa);
    batch_unref(xb);
    if (rc) return rc;
    m->chunks.push_back(chunk);
    *fuel -= (int64_t)((na - m->ai) + (nb - m->bi));
    m->ai = na;
    m->bi = nb;
  }
  // fuel > 0 after the call <=> the merge is complete (trace/mod.rs:388-395)
  if (m->complete()) { if (*fuel < 1) *fuel = 1; } else if (*fuel > 0) *fuel = 0;
  return DBSP_OK;
}

int32_t dbsp_merger_free(dbsp_merger* mm) {
  Merger* m = (Merger*)mm;
  if (!m) return DBSP_OK;
  for (Batch* c : m->chunks) batch_unref(c);
  batch_unref(m->a);
  batch_unref(m->b);
  delete m;
  return DBSP_OK;
}

int32_t dbsp_merger_done(dbsp_ctx* ctx, dbsp_merger* mm, dbsp_batch** out) { ENTER(ctx);
  Merger* m = (Merger*)mm;
  CHECK_ARG(m->complete(), "merger_done: merge not complete");
  Batch* o = nullptr;
  TRY(batch_concat(ctx, m->a->s, m->chunks, &o));   // on failure the merger stays owned by the caller
  dbsp_merger_free(mm);
  *out = H(o);
  return DBSP_OK;
}

int32_t dbsp_batch_neg(dbsp_ctx* ctx, const dbsp_batch* a, dbsp_batch** out) { ENTER(ctx);
  Batch* o = nullptr;
  TRY(op_neg(ctx, B(a), &o));
  *out = H(o);
  return DBSP_OK;
}

int32_t dbsp_batch_reindex(dbsp_ctx* ctx, const dbsp_batch* a, uint32_t nk, dbsp_batch** out) { ENTER(ctx);
  const Batch* x = B(a);
  CHECK_ARG((int)nk <= x->nl(), "reindex: too many key lanes");
  Batch* v = new Batch();
  v->s = x->s;
  v->s.n_key_lanes = (uint8_t)nk;
  v->s.n_val_lanes = (uint8_t)(x->nl() - nk);
  v->ctx = ctx;
  v->n = x->n;
  for (int l = 0; l < MAXL; l++) v->col[l] = x->col[l];
  v->w = x->w;
  v->bufs = x->bufs;
  if (v->n == 0) v->nkeys = 0;
  *out = H(v);
  return DBSP_OK;
}

int32_t dbsp_batch_len(const dbsp_batch* b, uint64_t* n) { *n = B(b)->n; return DBSP_OK; }
int32_t dbsp_batch_key_count(dbsp_ctx* ctx, const dbsp_batch* b, uint64_t* n) { ENTER(ctx);
  Batch* x = B(b);
  if (x->s.n_val_lanes == 0) { *n = x->n; return DBSP_OK; }
  TRY(batch_build_csr(ctx, x));
  *n = x->nkeys;
  return DBSP_OK;
}
int32_t dbsp_batch_schema(const dbsp_batch* b, dbsp_schema* out) { *out = B(b)->s; return DBSP_OK; }

int32_t dbsp_batch_download_csr(dbsp_ctx* ctx, const dbsp_batch* bb, uint64_t* const* keys, uint64_t* offs,
                                uint64_t* const* vals, int64_t* diffs) { ENTER(ctx);
  Batch* b = B(bb);
  cudaStream_t st = lane(ctx).stream;
  int nk = b->s.n_key_lanes, nv = b->s.n_val_lanes;
  if (b->n == 0) { if (offs && nv) offs[0] = 0; return DBSP_OK; }
  if (nv == 0) {
    if (keys) for (int l = 0; l < nk; l++) if (keys[l]) { CUDA_TRY(cudaMemcpyAsync(keys[l], b->col[l], b->n * 8, cudaMemcpyDeviceToHost, st)); ctx->d2h_bytes += b->n * 8; }
  } else {
    TRY(batch_build_csr(ctx, b));
    u64 nkeys = b->nkeys;
    if (offs) { CUDA_TRY(cudaMemcpyAsync(offs, b->keystart->p, (nkeys + 1) * 8, cudaMemcpyDeviceToHost, st)); ctx->d2h_bytes += (nkeys + 1) * 8; }
    if (keys && nk) {
      // gather the key lanes at the key starts: download flat, compact on the host side of the ABI
      std::vector<u64> ks(nkeys + 1);
      CUDA_TRY(cudaMemcpyAsync(ks.data(), b->keystart->p, (nkeys + 1) * 8, cudaMemcpyDeviceToHost, st));
      std::vector<u64> flat(b->n);
      for (int l = 0; l < nk; l++) {
        if (!keys[l]) continue;
        CUDA_TRY(cudaMemcpyAsync(flat.data(), b->col[l], b->n * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        ctx->d2h_bytes += b->n * 8;
        for (u64 k = 0; k < nkeys; k++) keys[l][k] = flat[ks[k]];
      }
    }
    if (vals) for (int l = 0; l < nv; l++) if (vals[l]) { CUDA_TRY(cudaMemcpyAsync(vals[l], b->col[nk + l], b->n * 8, cudaMemcpyDeviceToHost, st)); ctx->d2h_bytes += b->n * 8; }
  }
  if (diffs) { CUDA_TRY(cudaMemcpyAsync(diffs, b->w, b->n * 8, cudaMemcpyDeviceToHost, st)); ctx->d2h_bytes += b->n * 8; }
  CUDA_TRY(cudaStreamSynchronize(st));
  return DBSP_OK;
}

struct dbsp_download {
  Ctx* ctx;
  Batch* b;
  cudaEvent_t done;
};
int32_t dbsp_batch_download_begin(dbsp_ctx* ctx, const dbsp_batch* bb, uint64_t* const* cols, int64_t* diffs,
                                  dbsp_download** out) { ENTER(ctx);
  Batch* b = B(bb);
  cudaEvent_t done;
  CUDA_TRY(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
  auto queue = [&]() -> int32_t {
    if (b->n) {
      // the read stream picks the batch up once the kernels that produce it have run
      cudaEvent_t ev;
      CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      cudaError_t e1 = cudaEventRecord(ev, lane(ctx).stream);
      cudaError_t e2 = cudaStreamWaitEvent(ctx->read_stream, ev, 0);
      cudaEventDestroy(ev);
      CUDA_TRY(e1);
      CUDA_TRY(e2);
      for (int l = 0; l < b->nl(); l++) {
        if (!cols || !cols[l]) continue;
        CUDA_TRY(cudaMemcpyAsync(cols[l], b->col[l], b->n * 8, cudaMemcpyDeviceToHost, ctx->read_stream));
        ctx->d2h_bytes += b->n * 8;
      }
      if (diffs) {
        CUDA_TRY(cudaMemcpyAsync(diffs, b->w, b->n * 8, cudaMemcpyDeviceToHost, ctx->read_stream));
        ctx->d2h_bytes += b->n * 8;
      }
    }
    CUDA_TRY(cudaEventRecord(done, ctx->read_stream));
    return DBSP_OK;
  };
  const int32_t rc = queue();
  if (rc != DBSP_OK) {   // whatever was queued must not outlive the caller's buffers
    cudaStreamSynchronize(ctx->read_stream);
    cudaEventDestroy(done);
    return rc;
  }
  dbsp_download* d = new dbsp_download();
  d->ctx = ctx;
  d->b = b;
  d->done = done;
  batch_ref(b);   // the rows must outlive the copy
  *out = d;
  return DBSP_OK;
}
int32_t dbsp_download_finish(dbsp_download* d) {
  if (!d) return DBSP_OK;
  cudaError_t e = cudaEventSynchronize(d->done);
  cudaEventDestroy(d->done);
  batch_unref(d->b);
  delete d;
  if (e != cudaSuccess) { set_error(std::string("download_finish: ") + cudaGetErrorString(e)); return DBSP_ERR_CUDA; }
  return DBSP_OK;
}

int32_t dbsp_batch_device_columns(const dbsp_batch* b, const uint64_t** cols, const int64_t** w) {
  const Batch* x = B(b);
  for (int l = 0; l < x->nl(); l++) cols[l] = x->col[l];
  if (w) *w = x->w;
  return DBSP_OK;
}

int32_t dbsp_batch_last_key(dbsp_ctx* ctx, const dbsp_batch* b, uint64_t* key, int32_t* valid) { ENTER(ctx);
  const Batch* x = B(b);
  *valid = x->n > 0;
  if (!x->n) return DBSP_OK;
  for (int l = 0; l < x->s.n_key_lanes; l++) {
    CUDA_TRY(cudaMemcpyAsync(ctx->h_scratch + l, x->col[l] + (x->n - 1), 8, cudaMemcpyDeviceToHost, lane(ctx).stream));
  }
  CUDA_TRY(cudaStreamSynchronize(lane(ctx).stream));
  for (int l = 0; l < x->s.n_key_lanes; l++) key[l] = ctx->h_scratch[l];
  ctx->d2h_bytes += 8 * x->s.n_key_lanes;
  return DBSP_OK;
}

int32_t dbsp_batch_clone(const dbsp_batch* b, dbsp_batch** out) { batch_ref(B(b)); *out = (dbsp_batch*)b; return DBSP_OK; }
int32_t dbsp_batch_free(dbsp_batch* b) { batch_unref(B(b)); return DBSP_OK; }

int32_t dbsp_spine_new(dbsp_ctx* ctx, const dbsp_schema* s, dbsp_spine** out) { ENTER(ctx);
  dbsp_spine* sp = new dbsp_spine();
  sp->s = *s;
  sp->ctx = ctx;
  *out = sp;
  return DBSP_OK;
}
int32_t dbsp_spine_insert(dbsp_ctx* ctx, dbsp_spine* s, const dbsp_batch* b) { ENTER(ctx);
  CHECK_ARG(memcmp(&s->s, &B(b)->s, sizeof(dbsp_schema)) == 0, "spine_insert: schema mismatch");
  return spine_insert(ctx, s, B(b));
}
int32_t dbsp_spine_consolidate(dbsp_ctx* ctx, dbsp_spine* s, dbsp_batch** out) { ENTER(ctx);
  // A consolidated read of the trace: the merge of everything a cursor sees, with the value bound applied.
  // Trace::consolidate (:583-600) consumes the trace; this leaves the layers (and their merge schedule) as they are.
  const u64* vb = s->has_vbound ? s->vbound : nullptr;
  Batch* acc = batch_new_empty(ctx, s->s);
  for (size_t i = s->batches.size(); i-- > 0;) {   // smallest first: the accumulator grows geometrically
    Batch* m = nullptr;
    int32_t rc = merge_bounded(ctx, acc, s->batches[i], vb, &m);
    batch_unref(acc);
    if (rc) return rc;
    acc = m;
  }
  *out = H(acc);
  return DBSP_OK;
}
int32_t dbsp_spine_truncate_keys_below(dbsp_ctx* ctx, dbsp_spine* s, const uint64_t* key) { ENTER(ctx);
  bool raise = !s->has_bound;
  if (!raise) {   // the bound only grows (spine_fueled.rs:223-233)
    for (int l = 0; l < s->s.n_key_lanes; l++) {
      u64 flip = s->s.lane_types[l] == DBSP_I64 ? 0x8000000000000000ull : 0ull;
      u64 x = key[l] ^ flip, y = s->bound[l] ^ flip;
      if (x != y) { raise = x > y; break; }
    }
  }
  if (!raise) return DBSP_OK;
  TRY(spine_complete_merges(ctx, s));   // :224
  s->has_bound = true;
  for (int l = 0; l < s->s.n_key_lanes; l++) s->bound[l] = key[l];
  for (SpineLevel& l : s->merging) {   // map_batches_mut (:988-1004)
    if ((l.kind == SpineLevel::SINGLE || l.kind == SpineLevel::COMPLETE) && l.a) {
      Batch* v = nullptr;
      TRY(spine_truncate_batch(ctx, s, l.a, &v));
      batch_unref(l.a);
      l.a = v;
    }
  }
  spine_refresh_view(s);
  return DBSP_OK;
}
int32_t dbsp_spine_truncate_values_below(dbsp_ctx*, dbsp_spine* s, const uint64_t* val) {
  int nk = s->s.n_key_lanes, nv = s->s.n_val_lanes;
  bool raise = !s->has_vbound;
  if (!raise) {   // the bound only grows (spine_fueled.rs:644-652)
    for (int l = 0; l < nv; l++) {
      u64 flip = s->s.lane_types[nk + l] == DBSP_I64 ? 0x8000000000000000ull : 0ull;
      u64 x = val[l] ^ flip, y = s->vbound[l] ^ flip;
      if (x != y) { raise = x > y; break; }
    }
  }
  if (raise) for (int l = 0; l < nv; l++) s->vbound[l] = val[l];
  s->has_vbound = true;
  return DBSP_OK;
}
int32_t dbsp_spine_exert(dbsp_ctx* ctx, dbsp_spine* s, int64_t* effort) { ENTER(ctx);
  i64 e = *effort;
  return spine_exert(ctx, s, &e);
}
int32_t dbsp_spine_len(const dbsp_spine* s, uint64_t* n, uint32_t* nb) {
  u64 t = 0;
  for (Batch* b : s->batches) t += b->n;
  if (n) *n = t;
  if (nb) *nb = (uint32_t)s->batches.size();
  return DBSP_OK;
}
int32_t dbsp_spine_free(dbsp_spine* s) {
  if (!s) return DBSP_OK;
  spine_release(s);
  delete s;
  return DBSP_OK;
}

// ---- checkpoint / resume (include/dbsp_b200.h "Checkpoint"; format shared with oracle/dbsp_oracle.cpp) -------------
static const char SPINE_MAGIC[8] = {'D', 'B', 'S', 'P', 'S', 'P', 'N', '1'};
static bool fwrite_all(FILE* f, const void* p, size_t n) { return n == 0 || fwrite(p, 1, n, f) == n; }
static bool fread_all(FILE* f, void* p, size_t n) { return n == 0 || fread(p, 1, n, f) == n; }

static int32_t save_batch(Ctx* ctx, FILE* f, const Batch* b, std::vector<u64>& stage) {
  const u64 n = b ? b->n : 0;
  const u64 present = b ? 1 : 0;
  if (!fwrite_all(f, &present, 8) || !fwrite_all(f, &n, 8)) { set_error("spine_save: write failed"); return DBSP_ERR_INVALID; }
  if (!n) return DBSP_OK;
  const int L = b->nl();
  for (int l = 0; l <= L; l++) {
    const void* src = l < L ? (const void*)b->col[l] : (const void*)b->w;
    for (u64 off = 0; off < n; off += stage.size()) {
      const u64 m = std::min<u64>(stage.size(), n - off);
      CUDA_TRY(cudaMemcpyAsync(stage.data(), (const u64*)src + off, m * 8, cudaMemcpyDeviceToHost, lane(ctx).stream));
      CUDA_TRY(cudaStreamSynchronize(lane(ctx).stream));
      ctx->d2h_bytes += m * 8;
      if (!fwrite_all(f, stage.data(), m * 8)) { set_error("spine_save: write failed"); return DBSP_ERR_INVALID; }
    }
  }
  return DBSP_OK;
}
static int32_t load_batch(Ctx* ctx, FILE* f, const dbsp_schema& sc, Batch** out, std::vector<u64>& stage) {
  u64 present = 0, n = 0;
  *out = nullptr;
  if (!fread_all(f, &present, 8) || !fread_all(f, &n, 8)) { set_error("spine_load: truncated file"); return DBSP_ERR_INVALID; }
  if (!present) return DBSP_OK;
  if (!n) { *out = batch_new_empty(ctx, sc); return DBSP_OK; }
  Batch* b;
  MCols oc;
  i64* ow;
  TRY(batch_alloc(ctx, sc, n, &b, &oc, &ow));
  const int L = sc.n_key_lanes + sc.n_val_lanes;
  for (int l = 0; l <= L; l++) {
    u64* dst = l < L ? oc.c[l] : (u64*)ow;
    for (u64 off = 0; off < n; off += stage.size()) {
      const u64 m = std::min<u64>(stage.size(), n - off);
      if (!fread_all(f, stage.data(), m * 8)) { batch_unref(b); set_error("spine_load: truncated file"); return DBSP_ERR_INVALID; }
      cudaError_t e = cudaMemcpyAsync(dst + off, stage.data(), m * 8, cudaMemcpyHostToDevice, lane(ctx).stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(lane(ctx).stream);
      if (e != cudaSuccess) { batch_unref(b); set_error(cudaGetErrorString(e)); return DBSP_ERR_CUDA; }
      ctx->h2d_bytes += m * 8;
    }
  }
  *out = b;
  return DBSP_OK;
}

int32_t dbsp_spine_save(dbsp_ctx* ctx, const dbsp_spine* s, const char* path) { ENTER(ctx);
  FILE* f = fopen(path, "wb");
  if (!f) { set_error(std::string("spine_save: cannot open ") + path); return DBSP_ERR_INVALID; }
  std::vector<u64> stage((size_t)8 << 20);   // 64 MiB staging
  u64 hdr[4] = {s->has_bound ? 1ull : 0ull, s->has_vbound ? 1ull : 0ull, s->effort, (u64)s->merging.size()};
  bool ok = fwrite_all(f, SPINE_MAGIC, 8) && fwrite_all(f, &s->s, sizeof(dbsp_schema)) && fwrite_all(f, hdr, sizeof(hdr)) &&
            fwrite_all(f, s->bound, sizeof(u64) * MAXL) && fwrite_all(f, s->vbound, sizeof(u64) * MAXL);
  int32_t rc = ok ? DBSP_OK : DBSP_ERR_INVALID;
  for (size_t i = 0; rc == DBSP_OK && i < s->merging.size(); i++) {
    const SpineLevel& l = s->merging[i];
    u64 lh[2] = {(u64)l.kind, (u64)l.remaining};
    if (!fwrite_all(f, lh, sizeof(lh))) { rc = DBSP_ERR_INVALID; break; }
    rc = save_batch(ctx, f, l.a, stage);
    if (rc == DBSP_OK) rc = save_batch(ctx, f, l.b, stage);
  }
  if (fclose(f) != 0 && rc == DBSP_OK) rc = DBSP_ERR_INVALID;
  if (rc == DBSP_ERR_INVALID && !ok) set_error("spine_save: write failed");
  return rc;
}
int32_t dbsp_spine_load(dbsp_ctx* ctx, const char* path, dbsp_spine** out) { ENTER(ctx);
  FILE* f = fopen(path, "rb");
  if (!f) { set_error(std::string("spine_load: cannot open ") + path); return DBSP_ERR_INVALID; }
  std::vector<u64> stage((size_t)8 << 20);
  char magic[8];
  u64 hdr[4];
  dbsp_spine* sp = new dbsp_spine();
  sp->ctx = ctx;
  int32_t rc = DBSP_OK;
  if (!fread_all(f, magic, 8) || memcmp(magic, SPINE_MAGIC, 8) != 0 || !fread_all(f, &sp->s, sizeof(dbsp_schema)) ||
      !fread_all(f, hdr, sizeof(hdr)) || !fread_all(f, sp->bound, sizeof(u64) * MAXL) || !fread_all(f, sp->vbound, sizeof(u64) * MAXL)) {
    set_error("spine_load: not a spine snapshot");
    rc = DBSP_ERR_INVALID;
  }
  if (rc == DBSP_OK) {
    sp->has_bound = hdr[0] != 0;
    sp->has_vbound = hdr[1] != 0;
    sp->effort = hdr[2] ? hdr[2] : 1;
    if (hdr[3] > 64) { set_error("spine_load: corrupt layer count"); rc = DBSP_ERR_INVALID; }
  }
  for (u64 i = 0; rc == DBSP_OK && i < hdr[3]; i++) {
    u64 lh[2];
    if (!fread_all(f, lh, sizeof(lh)) || lh[0] > (u64)SpineLevel::COMPLETE) { set_error("spine_load: truncated file"); rc = DBSP_ERR_INVALID; break; }
    SpineLevel l;
    l.kind = (SpineLevel::Kind)lh[0];
    l.remaining = (i64)lh[1];
    rc = load_batch(ctx, f, sp->s, &l.a, stage);
    if (rc == DBSP_OK) rc = load_batch(ctx, f, sp->s, &l.b, stage);
    if (rc == DBSP_OK && l.kind == SpineLevel::IN_PROGRESS && (!l.a || !l.b)) { set_error("spine_load: corrupt layer"); rc = DBSP_ERR_INVALID; }
    sp->merging.push_back(l);
  }
  fclose(f);
  if (rc != DBSP_OK) { spine_release(sp); delete sp; return rc; }
  spine_refresh_view(sp);
  *out = sp;
  return DBSP_OK;
}

#define OUT1(call)            \
  Batch* o__ = nullptr;       \
  TRY(call);                  \
  *out = H(o__);              \
  return DBSP_OK;

int32_t dbsp_join_delta_trace(dbsp_ctx* ctx, const dbsp_batch* d, const dbsp_spine* t, const dbsp_proj* p, int32_t dl,
                              dbsp_batch** out) { ENTER(ctx); OUT1(op_join_delta_trace(ctx, B(d), t, p, dl, &o__)) }
// The join operator (join.rs:180-292) over one step: lane 0 inserts δright into the right trace and joins δleft
// with it; lane 1 joins δright with the left trace as it was before this step (z^-1) and then inserts δleft.  The
// halves touch different traces, so each trace sees the same operations as in the sequential order.
int32_t dbsp_join_step(dbsp_ctx* ctx, const dbsp_batch* dl, const dbsp_batch* dr, dbsp_spine* lt, dbsp_spine* rt,
                       const dbsp_proj* p, dbsp_batch** out) { ENTER(ctx);
  CHECK_ARG(dl && dr && lt && rt && p && out, "join_step: NULL argument");
  CHECK_ARG(lt != rt, "join_step: the left and right traces must differ");
  CHECK_ARG(memcmp(&lt->s, &B(dl)->s, sizeof(dbsp_schema)) == 0, "join_step: left delta / trace schema mismatch");
  CHECK_ARG(memcmp(&rt->s, &B(dr)->s, sizeof(dbsp_schema)) == 0, "join_step: right delta / trace schema mismatch");
  Batch *o1 = nullptr, *o2 = nullptr;
  int32_t rc = run_forked(
      ctx,
      [&]() -> int32_t {
        TRY(spine_insert(ctx, rt, B(dr)));
        return op_join_delta_trace(ctx, B(dl), rt, p, 1, &o1);
      },
      [&]() -> int32_t {
        TRY(op_join_delta_trace(ctx, B(dr), lt, p, 0, &o2));
        return spine_insert(ctx, lt, B(dl));
      });
  Batch* o = nullptr;
  if (rc == DBSP_OK) rc = merge_batches(ctx, o1, o2, &o);
  batch_unref(o1);
  batch_unref(o2);
  if (rc != DBSP_OK) return rc;
  *out = H(o);
  return DBSP_OK;
}
int32_t dbsp_join_batches(dbsp_ctx* ctx, const dbsp_batch* l, const dbsp_batch* r, const dbsp_proj* p, dbsp_batch** out) { ENTER(ctx);
  OUT1(op_join_batches(ctx, B(l), B(r), p, &o__)) }
int32_t dbsp_semijoin(dbsp_ctx* ctx, const dbsp_batch* pairs, const dbsp_batch* keys, dbsp_batch** out) { ENTER(ctx);
  OUT1(op_semijoin(ctx, B(pairs), B(keys), &o__)) }
int32_t dbsp_aggregate_delta(dbsp_ctx* ctx, const dbsp_batch* d, const dbsp_spine* in_tr, const dbsp_spine* out_tr,
                             int32_t kind, dbsp_batch** out) { ENTER(ctx); OUT1(op_aggregate_delta(ctx, B(d), in_tr, out_tr, kind, &o__)) }
int32_t dbsp_weigh(dbsp_ctx* ctx, const dbsp_batch* b, const dbsp_expr* f, int32_t mode, dbsp_batch** out) { ENTER(ctx);
  OUT1(op_weigh(ctx, B(b), f, mode, &o__)) }
int32_t dbsp_distinct_delta(dbsp_ctx* ctx, const dbsp_batch* d, const dbsp_spine* i, dbsp_batch** out) { ENTER(ctx);
  OUT1(op_distinct_delta(ctx, B(d), i, &o__)) }
int32_t dbsp_stream_distinct(dbsp_ctx* ctx, const dbsp_batch* b, dbsp_batch** out) { ENTER(ctx); OUT1(op_stream_distinct(ctx, B(b), &o__)) }
int32_t dbsp_window_delta(dbsp_ctx* ctx, const dbsp_spine* t, const dbsp_batch* d, int32_t has_prev, const uint64_t* s0,
                          const uint64_t* e0, const uint64_t* s1, const uint64_t* e1, dbsp_batch** out) { ENTER(ctx);
  OUT1(op_window_delta(ctx, t, B(d), has_prev, s0, e0, s1, e1, &o__)) }
int32_t dbsp_map_index(dbsp_ctx* ctx, const dbsp_batch* b, const dbsp_proj* p, dbsp_batch** out) { ENTER(ctx);
  OUT1(op_map_index(ctx, B(b), p, &o__)) }
int32_t dbsp_shard_partition(dbsp_ctx* ctx, const dbsp_batch* b, uint32_t P, dbsp_batch** outs) { ENTER(ctx);
  std::vector<Batch*> o(P, nullptr);
  TRY(op_shard_partition(ctx, B(b), P, o.data()));
  for (uint32_t p = 0; p < P; p++) outs[p] = H(o[p]);
  return DBSP_OK;
}

int32_t dbsp_comm_create(dbsp_ctx* ctx, int32_t rank, int32_t world, uint64_t slot_bytes, uint8_t* blob_out) { ENTER(ctx);
  CHECK_ARG(blob_out != nullptr, "comm_create: blob_out is NULL");
  return comm_create(ctx, rank, world, slot_bytes, blob_out);
}
int32_t dbsp_comm_connect(dbsp_ctx* ctx, const uint8_t* blobs) { ENTER(ctx);
  CHECK_ARG(blobs != nullptr, "comm_connect: blobs is NULL");
  return comm_connect(ctx, blobs);
}
int32_t dbsp_comm_destroy(dbsp_ctx* ctx) { ENTER(ctx);
  CUDA_TRY(cudaStreamSynchronize(lane(ctx).stream));
  comm_free(ctx);
  return DBSP_OK;
}
int32_t dbsp_comm_info(dbsp_ctx* ctx, int32_t* rank, int32_t* world, uint64_t* bytes_sent) {
  int r, w;
  u64 b;
  comm_info(ctx, &r, &w, &b);
  if (rank) *rank = r;
  if (world) *world = w;
  if (bytes_sent) *bytes_sent = b;
  return DBSP_OK;
}
int32_t dbsp_shard(dbsp_ctx* ctx, const dbsp_batch* b, dbsp_batch** out) { ENTER(ctx);
  const Batch* in[1] = {B(b)};
  Batch* o[1] = {nullptr};
  TRY(comm_exchange(ctx, in, 1, -1, o));
  *out = H(o[0]);
  return DBSP_OK;
}
int32_t dbsp_shard2(dbsp_ctx* ctx, const dbsp_batch* a, const dbsp_batch* b, dbsp_batch** out_a, dbsp_batch** out_b) { ENTER(ctx);
  const Batch* in[2] = {B(a), B(b)};
  Batch* o[2] = {nullptr, nullptr};
  TRY(comm_exchange(ctx, in, 2, -1, o));
  *out_a = H(o[0]);
  *out_b = H(o[1]);
  return DBSP_OK;
}
int32_t dbsp_gather(dbsp_ctx* ctx, const dbsp_batch* b, int32_t root, dbsp_batch** out) { ENTER(ctx);
  int r, w;
  comm_info(ctx, &r, &w, nullptr);
  CHECK_ARG(root >= 0 && root < w, "gather: root out of range");
  const Batch* in[1] = {B(b)};
  Batch* o[1] = {nullptr};
  TRY(comm_exchange(ctx, in, 1, root, o));
  *out = H(o[0]);
  return DBSP_OK;
}
int32_t dbsp_allreduce_max_u64(dbsp_ctx* ctx, uint64_t* x) { ENTER(ctx);
  u64 v = *x;
  TRY(comm_allreduce_max(ctx, &v));
  *x = v;
  return DBSP_OK;
}

}  // extern "C"
