// ops.cu — operator kernels: projection/filter, delta-vs-trace probes (join,
// aggregate, distinct), window ranges, shard partition.  Each host entry
// cites the reference `eval` it replaces (paths under crates/dbsp/src/).
#include "ops.cuh"

namespace {

constexpr int TB = 256;

// up to MAX_REFS spine batches passed to a kernel by value
struct BatchRef {
  Cols c;
  const i64* w;
  u64 n;
};
constexpr int MAX_REFS = 16;
struct BatchRefs {
  BatchRef b[MAX_REFS];
  int nb;
};

// ---------------- declarative row expressions on the device ------------------
struct Env {
  const u64* key;
  const u64* lv;
  const u64* rv;
  __device__ __forceinline__ u64 k(int i) const { return key[i]; }
  __device__ __forceinline__ u64 l(int i) const { return lv[i]; }
  __device__ __forceinline__ u64 r(int i) const { return rv[i]; }
};
// one row of a column table / batch, read in place: only the lanes the closure names are ever loaded
struct ColEnv {
  const Cols& c;
  int nk;
  u64 row;
  __device__ __forceinline__ u64 k(int i) const { return c.c[i][row]; }
  __device__ __forceinline__ u64 l(int i) const { return c.c[nk + i][row]; }
  __device__ __forceinline__ u64 r(int i) const { return c.c[nk + i][row]; }
};
template <class E>
__device__ __forceinline__ u64 src_val(const dbsp_src& s, const E& e) {
  switch (s.kind) {
    case DBSP_SRC_KEY: return e.k(s.idx);
    case DBSP_SRC_LVAL: return e.l(s.idx);
    case DBSP_SRC_RVAL: return e.r(s.idx);
    default: return (u64)s.cst;
  }
}
template <class E>
__device__ __forceinline__ u64 expr_val(const dbsp_expr& x, const E& e) {
  u64 a = src_val(x.a, e);
  switch (x.op) {
    case DBSP_OP_COPY: return a;
    case DBSP_OP_NEG: return (u64)0 - a;
    case DBSP_OP_ADD: return a + src_val(x.b, e);
    case DBSP_OP_SUB: return a - src_val(x.b, e);
    case DBSP_OP_MUL: return a * src_val(x.b, e);
    case DBSP_OP_DIV: {
      i64 d = (i64)src_val(x.b, e);
      return d == 0 ? 0 : (u64)((i64)a / d);
    }
  }
  return a;
}
template <class E>
__device__ __forceinline__ bool pred_ok(const dbsp_pred& p, const E& e) {
  u64 a = src_val(p.a, e), b = src_val(p.b, e);
  if (p.cmp == DBSP_CMP_IN) return a < 64 && ((b >> a) & 1);
  int c = p.is_signed ? (((i64)a < (i64)b) ? -1 : ((i64)a > (i64)b)) : ((a < b) ? -1 : (a > b));
  switch (p.cmp) {
    case DBSP_CMP_EQ: return c == 0;
    case DBSP_CMP_NE: return c != 0;
    case DBSP_CMP_LT: return c < 0;
    case DBSP_CMP_LE: return c <= 0;
    case DBSP_CMP_GT: return c > 0;
    case DBSP_CMP_GE: return c >= 0;
  }
  return false;
}
// evaluates the output row unconditionally (a filtered row keeps its place in
// an ordered output with weight 0) and returns whether the predicates hold
__device__ __forceinline__ bool project(const dbsp_proj& p, const Env& e, u64* row) {
  bool ok = true;
  for (int i = 0; i < p.n_pred; i++) ok = ok && pred_ok(p.pred[i], e);
  int nl = p.out_schema.n_key_lanes + p.out_schema.n_val_lanes;
  for (int l = 0; l < nl; l++) row[l] = expr_val(p.out[l], e);
  return ok;
}

// flat_map_index over a raw table (filter_map.rs:700-724) / map_index over a
// batch, in one pass and order preserving: a CTA evaluates the predicates of its PROJ_ROWS rows, a decoupled
// look-back over the CTA totals gives it its output base, and the survivors' output rows are evaluated and written
// in input order — so inputs that are already ordered on the output key (id-ordered event tables, monotone
// projections) reach the sort-free path of consolidate_rows.  The surviving-row count stays on the device
// (*d_m): the census of consolidate_rows returns it.  identity != 0 (no predicates): output slot = input row.
constexpr int PROJ_IT = 4;
constexpr int PROJ_ROWS = TB * PROJ_IT;
__global__ void __launch_bounds__(TB)
k_project_rows(Cols in, int nk_in, const i64* w, u64 n, dbsp_proj proj, int identity, u32 ntiles, u32* ticket,
               u64* status, MCols out, i64* out_w, u32* d_m) {
  static_assert(PROJ_IT * (TB / 32) == 32, "one warp scans the per-(round, warp) counts");
  __shared__ u32 s_tile;
  __shared__ u32 s_cnt[32], s_off[32];
  __shared__ u64 s_base;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nl = proj.out_schema.n_key_lanes + proj.out_schema.n_val_lanes;
  if (identity) {
    const u64 base = (u64)blockIdx.x * PROJ_ROWS;
    for (int it = 0; it < PROJ_IT; it++) {
      const u64 i = base + (u64)it * TB + tid;
      if (i < n) {
        const ColEnv e{in, nk_in, i};
        for (int l = 0; l < nl; l++) out.c[l][i] = expr_val(proj.out[l], e);
        out_w[i] = w ? w[i] : 1;
      }
    }
    return;
  }
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const u32 t = s_tile;
  const u64 base_row = (u64)t * PROJ_ROWS;
  unsigned okbits = 0, rk = 0;   // rk: 8 bits per round = number of surviving rows before this lane in its warp
  for (int it = 0; it < PROJ_IT; it++) {
    const u64 i = base_row + (u64)it * TB + tid;
    bool ok = false;
    if (i < n) {
      const ColEnv e{in, nk_in, i};
      ok = true;
      for (int q = 0; q < proj.n_pred; q++) ok = ok && pred_ok(proj.pred[q], e);
    }
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) s_cnt[it * (TB / 32) + wid] = __popc(m);
    if (ok) {
      okbits |= 1u << it;
      rk |= (unsigned)__popc(m & ((1u << lane) - 1)) << (8 * it);
    }
  }
  __syncthreads();
  if (wid == 0) {
    const u32 c = s_cnt[lane];
    u32 incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const u32 v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    const u32 total = __shfl_sync(0xffffffffu, incl, 31);
    s_off[lane] = incl - c;
    const u64 base = lb_exclusive_prefix(status, t, (u64)total);
    if (lane == 0) {
      s_base = base;
      if (t == ntiles - 1) *d_m = (u32)(base + total);
    }
  }
  __syncthreads();
  const u64 base = s_base;
  for (int it = 0; it < PROJ_IT; it++) {
    if (!((okbits >> it) & 1)) continue;
    const u64 i = base_row + (u64)it * TB + tid;
    const u64 pos = base + s_off[it * (TB / 32) + wid] + ((rk >> (8 * it)) & 0xffu);
    const ColEnv e{in, nk_in, i};
    for (int l = 0; l < nl; l++) out.c[l][pos] = expr_val(proj.out[l], e);
    out_w[pos] = w ? w[i] : 1;
  }
}

// ---------------- delta x trace probes -----------------------------------------
// One pass per chunk of (up to MAX_REFS) trace batches over ticketed tiles of PR_TILE sorted delta rows.  A segment
// is a run of equal keys (first nk lanes) inside one tile: it starts at a key head or at the tile's first row, so a
// key whose rows span tiles is searched once per tile and no tile waits on another except in the match-count
// look-back.
//  1. segments: ki[i] = first row of row i's segment; the tile's segment heads are listed in shared memory.
//  2. windows: per batch, the rows [wl, wh) between the tile's first and last key, by 16-way half-warp searches
//     whose pivots include both ends of the range, so a tile whose keys all lie outside a batch settles it in one
//     round.  An empty window settles every segment of the tile for that batch without touching the batch again.
//  3. ranges: per batch, every segment searches only inside the window — in shared memory when the window's key
//     lanes fit PR_STAGE words, else in place: lower bound by bisection, upper bound by galloping (the `seek_key`
//     of cursor/mod.rs + advance.rs:25-72).  lo/cnt[first_row * nb + b].
//  4. counts: matches of a row = matches of its segment (saturated to u32, so a 64-bit total >= 2^32-1 still trips
//     the host's guard), block scan + decoupled look-back: ex[i] = output slot of row i's first match, ex[nd] =
//     total (32-bit, wraps on a rejected step); the last tile publishes the 64-bit total to the host mailbox.
constexpr int PR_IPT = 4, PR_TILE = TB * PR_IPT, PR_STAGE = 2048;

// bound of q in rows [lo,hi) of T — first row >= q, or > q when `upper` — searched by the 16 lanes of a half warp
// (each lane one pivot per round).  Both halves of the warp must call it together; their ranges may differ.
__device__ __forceinline__ u64 half_warp_bound(const Cols& T, u64 lo, u64 hi, const u64* q, int nk, const Flips& f,
                                               bool upper) {
  const int hl = threadIdx.x & 15, hs = threadIdx.x & 16;
  while (true) {
    const bool live = lo < hi;
    if (!__any_sync(0xffffffffu, live)) break;
    bool before = false;
    if (live) {
      const int c = cmp_row_q(T, lo + (u64)hl * (hi - lo - 1) / 15, q, nk, f);
      before = upper ? c <= 0 : c < 0;
    }
    const int c = __popc((__ballot_sync(0xffffffffu, before) >> hs) & 0xffffu);   // pivots before the bound
    if (live) {
      const u64 span = hi - lo - 1;
      if (c == 0) hi = lo;
      else {
        if (c < 16) hi = lo + (u64)c * span / 15;
        lo = lo + (u64)(c - 1) * span / 15 + 1;
      }
    }
  }
  return lo;
}

// first staged row in [lo,hi) whose key is >= q (upper: > q); lane l of row j at s[l * ws + j]
__device__ __forceinline__ u32 smem_bound(const u64* s, u32 ws, u32 lo, u32 hi, const u64* q, int nk, bool upper) {
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    int c = 0;
    for (int l = 0; l < nk && c == 0; l++) {
      const u64 a = s[l * ws + mid];
      if (a != q[l]) c = a < q[l] ? -1 : 1;
    }
    if (upper ? c <= 0 : c < 0) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(TB)
k_probe_ranges(Cols D, u64 nd, BatchRefs tr, int nk, Flips f, u32 ntiles, u32* ticket, u64* status, u32* ki, u32* lo_out,
               u32* cnt_out, u32* ex, Mail mail) {
  __shared__ u32 s_tile, s_wcnt[TB / 32], s_wl[MAX_REFS], s_wh[MAX_REFS];
  __shared__ u64 s_wsum[TB / 32], s_base;
  __shared__ u32 s_first[PR_TILE];   // first row (tile offset) of each segment
  __shared__ u64 s_tot[PR_TILE];     // matches of each segment over the chunk's batches
  __shared__ u64 s_stage[PR_STAGE];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const u32 t = s_tile;
  const u64 t0 = (u64)t * PR_TILE;
  const u64 tn = nd - t0 < (u64)PR_TILE ? nd - t0 : (u64)PR_TILE;   // rows of the tile
  const int nb = tr.nb;

  // 1. segments
  const u32 r0 = (u32)tid * PR_IPT;
  unsigned heads = 0;
#pragma unroll
  for (int k = 0; k < PR_IPT; k++) {
    const u64 i = t0 + r0 + k;
    if (r0 + k < tn) {
      bool head = r0 + k == 0;
      if (!head)
        for (int l = 0; l < nk; l++)
          if (D.c[l][i] != D.c[l][i - 1]) { head = true; break; }
      heads |= (head ? 1u : 0u) << k;
    }
  }
  const u32 hc = __popc(heads);
  u32 hincl = hc;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 v = __shfl_up_sync(0xffffffffu, hincl, o);
    if (lane >= o) hincl += v;
  }
  if (lane == 31) s_wcnt[wid] = hincl;
  // 2. windows: half warp h searches batch h / 2 (h even: lower bound of the first key, odd: upper bound of the
  // last); both halves of a warp take the same number of rounds
  {
    const int h = tid >> 4;
    const u64 qrow = (h & 1) ? t0 + tn - 1 : t0;
    u64 q[MAXL];
    for (int l = 0; l < nk; l++) q[l] = D.c[l][qrow] ^ f.f[l];
    for (int s = h; s < 2 * nb; s += TB / 16) {
      const int b = s >> 1;
      const u64 bound = half_warp_bound(tr.b[b].c, 0, tr.b[b].n, q, nk, f, h & 1);
      if ((tid & 15) == 0) {
        if (h & 1) s_wh[b] = (u32)bound; else s_wl[b] = (u32)bound;
      }
    }
  }
  __syncthreads();
  u32 nseg = 0, woff = 0;
#pragma unroll
  for (int k = 0; k < TB / 32; k++) {
    const u32 v = s_wcnt[k];
    if (k < wid) woff += v;
    nseg += v;
  }
  u32 seg[PR_IPT];   // segment of each of the thread's rows
  {
    u32 run = woff + hincl - hc;
#pragma unroll
    for (int k = 0; k < PR_IPT; k++) {
      if ((heads >> k) & 1) { s_first[run] = r0 + k; run++; }
      seg[k] = run - 1;
    }
  }
  __syncthreads();

  // 3. ranges: thread tid owns segments tid + j * TB for every batch
  u64 tot[PR_IPT] = {};
  for (int b = 0; b < nb; b++) {
    const Cols& T = tr.b[b].c;
    const u32 wl = s_wl[b], wh = s_wh[b], ws = wh - wl;
    const bool staged = ws > 0 && (u64)ws * nk <= (u64)PR_STAGE;   // uniform over the CTA
    if (staged) {
      for (u32 x = tid; x < ws * (u32)nk; x += TB) {
        const u32 l = x / ws, j = x - l * ws;
        s_stage[x] = T.c[l][wl + j] ^ f.f[l];
      }
      __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < PR_IPT; j++) {
      const u32 sg = (u32)tid + (u32)j * TB;
      if (sg >= nseg) break;
      const u64 row = t0 + s_first[sg];
      u64 lo = wl, hi = wl;
      if (ws > 0) {
        u64 q[MAXL];
        for (int l = 0; l < nk; l++) q[l] = D.c[l][row] ^ f.f[l];
        if (staged) {
          const u32 a = smem_bound(s_stage, ws, 0, ws, q, nk, false);
          lo = wl + a;
          hi = wl + smem_bound(s_stage, ws, a, ws, q, nk, true);
        } else {
          lo = lower_bound_q(T, wl, wh, q, nk, f);
          u64 step = 1;
          hi = lo;
          while (hi + step <= wh && cmp_row_q(T, hi + step - 1, q, nk, f) == 0) { hi += step; step <<= 1; }
          const u64 top = hi + step <= wh ? hi + step : wh;
          hi = upper_bound_q(T, hi, top, q, nk, f);
        }
      }
      lo_out[row * nb + b] = (u32)lo;
      cnt_out[row * nb + b] = (u32)(hi - lo);
      tot[j] += hi - lo;
    }
    if (staged) __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < PR_IPT; j++) {
    const u32 sg = (u32)tid + (u32)j * TB;
    if (sg < nseg) s_tot[sg] = tot[j];
  }
  __syncthreads();

  // 4. counts and their exclusive prefix
  u32 c[PR_IPT];
  u64 sum = 0;
#pragma unroll
  for (int k = 0; k < PR_IPT; k++) {
    c[k] = 0;
    if (r0 + k < tn) {
      const u64 m = s_tot[seg[k]];
      c[k] = m > 0xffffffffull ? 0xffffffffu : (u32)m;
      ki[t0 + r0 + k] = (u32)t0 + s_first[seg[k]];
    }
    sum += c[k];
  }
  u64 incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u64 v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_wsum[wid] = incl;
  __syncthreads();
  u64 soff = 0, tile_total = 0;
#pragma unroll
  for (int k = 0; k < TB / 32; k++) {
    const u64 v = s_wsum[k];
    if (k < wid) soff += v;
    tile_total += v;
  }
  if (wid == 0) {
    const u64 base = lb_exclusive_prefix(status, t, tile_total);
    if (lane == 0) {
      s_base = base;
      if (t == ntiles - 1) {
        const u64 total = base + tile_total;
        ex[nd] = (u32)total;
        mail_publish(mail, &total, 1);
      }
    }
  }
  __syncthreads();
  u64 run = s_base + soff + incl - sum;
#pragma unroll
  for (int k = 0; k < PR_IPT; k++) {
    if (r0 + k < tn) ex[t0 + r0 + k] = (u32)run;
    run += c[k];
  }
}

// Expand the matches: output slot o -> (delta row i, batch b, trace row).  Slots
// are ordered by (delta row, batch, trace row): for a monotone join_func and keys
// that live in a single batch that is already the output order, so consolidation
// needs no sort.  proj_mode 1: join_func(k, v1, v2) with filter
// (join.rs:751-787), weight w1*w2, rejected rows keep their slot with weight 0;
// proj_mode 0: copy the trace row (gather of a key group).
// Load balancing: a CTA owns ipt * 256 consecutive output slots whatever the fan-out of the keys behind them
// (skew-proof); the host picks ipt (1..PF_IPT) so that outputs of a few tens of thousands of slots still spread over
// the SMs.  Two threads bisect the scanned match counts for the delta rows of the tile's first and last
// slot; the counts in between are staged in shared memory, where every slot finds its delta row — one global
// bisection per tile instead of one per slot.  A slot's batch comes from its segment's nb counts, loaded side by
// side (no load waits on another) and walked in registers.  Consecutive slots read consecutive trace rows and the same / adjacent delta rows,
// and write consecutive output rows.
constexpr int PF_IPT = 4, PF_SMEM_ROWS = 3072;
__global__ void __launch_bounds__(256)
k_probe_fill(Cols D, const i64* wD, u64 nd, BatchRefs tr, int nk, int nvD, int nvT, const u32* lo, const u32* cnt,
             const u32* ki, const u32* exscan, u64 total, int ipt, int proj_mode, int delta_is_left, dbsp_proj proj,
             MCols out, i64* out_w) {
  __shared__ u32 s_ex[PF_SMEM_ROWS + 1];
  __shared__ u64 s_rows[2];
  const int tid = threadIdx.x;
  const u64 tile = (u64)ipt * 256;
  const u64 o0 = (u64)blockIdx.x * tile;
  if (o0 >= total) return;
  const u64 o1 = o0 + tile < total ? o0 + tile : total;
  if (tid < 2) {   // largest i with exscan[i] <= target
    const u64 target = tid == 0 ? o0 : o1 - 1;
    u64 a = 0, b = nd;
    while (b - a > 1) {
      const u64 mid = (a + b) >> 1;
      if (exscan[mid] <= target) a = mid; else b = mid;
    }
    s_rows[tid] = a;
  }
  __syncthreads();
  const u64 row_lo = s_rows[0], row_hi = s_rows[1];
  const u64 nr = row_hi - row_lo + 1;
  const bool staged = nr <= (u64)PF_SMEM_ROWS;
  if (staged)
    for (u64 k = tid; k <= nr; k += 256) s_ex[k] = exscan[row_lo + k];
  __syncthreads();
#pragma unroll 1
  for (int qq = 0; qq < ipt; qq++) {
    const u64 o = o0 + (u64)qq * 256 + tid;
    if (o >= o1) break;
    u64 i;
    u32 r;
    if (staged) {
      u32 a = 0, b = (u32)nr;
      while (b - a > 1) {
        const u32 mid = (a + b) >> 1;
        if (s_ex[mid] <= o) a = mid; else b = mid;
      }
      i = row_lo + a;
      r = (u32)(o - s_ex[a]);
    } else {
      u64 a = row_lo, b = row_hi + 1;
      while (b - a > 1) {
        const u64 mid = (a + b) >> 1;
        if (exscan[mid] <= o) a = mid; else b = mid;
      }
      i = a;
      r = (u32)(o - exscan[i]);
    }
    const u64 kbase = (u64)ki[i] * tr.nb;
    int bb = 0;
    u32 before = 0;   // matches in the batches before bb
#pragma unroll 4
    for (int b = 0; b < tr.nb - 1; b++) {   // load addresses do not depend on loaded counts: the loads overlap
      const u32 c = cnt[kbase + b];
      if (bb == b && r >= before + c) { before += c; bb = b + 1; }
    }
    r -= before;
    const Cols& T = tr.b[bb].c;
    const u64 t = (u64)lo[kbase + bb] + r;
    u64 row[MAXL];
    i64 wout;
    int nl_out;
    bool ok = true;
    if (proj_mode == 0) {
      nl_out = nk + nvT;
      for (int l = 0; l < nl_out; l++) row[l] = T.c[l][t];
      wout = tr.b[bb].w[t];
    } else {
      u64 key[MAXL], dv[MAXL], tv[MAXL];
      for (int l = 0; l < nk; l++) key[l] = D.c[l][i];
      for (int l = 0; l < nvD; l++) dv[l] = D.c[nk + l][i];
      for (int l = 0; l < nvT; l++) tv[l] = T.c[nk + l][t];
      Env e = delta_is_left ? Env{key, dv, tv} : Env{key, tv, dv};
      ok = project(proj, e, row);
      nl_out = proj.out_schema.n_key_lanes + proj.out_schema.n_val_lanes;
      wout = (i64)((u64)wD[i] * (u64)tr.b[bb].w[t]);
    }
    for (int l = 0; l < nl_out; l++) out.c[l][o] = row[l];
    out_w[o] = ok ? wout : 0;
  }
}

// Sum over one trace batch of the weight of the *exact* row (all L lanes).
__global__ void k_lookup_add(Cols D, u64 nd, Cols T, const i64* wT, u64 nt, int L, Flips f, i64* acc) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nd) return;
  u64 q[MAXL];
  for (int l = 0; l < L; l++) q[l] = D.c[l][i] ^ f.f[l];
  u64 lo = lower_bound_q(T, 0, nt, q, L, f);
  if (lo < nt && cmp_row_q(T, lo, q, L, f) == 0) acc[i] = (i64)((u64)acc[i] + (u64)wT[lo]);
}

// DistinctIncrementalTotal::eval decision (distinct.rs:196-254).
__global__ void k_distinct_decide(const i64* wD, const i64* oldw, u64 n, u32* keep, i64* neww) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { keep[n] = 0; return; }
  i64 o = oldw[i], nw = (i64)((u64)o + (u64)wD[i]);
  u32 k = 0;
  i64 w = 0;
  if (o <= 0) { if (nw > 0) { k = 1; w = 1; } }
  else if (nw <= 0) { k = 1; w = -1; }
  keep[i] = k;
  neww[i] = w;
}

// IndexedZSet::distinct (algebra/zset/mod.rs:14-38).
__global__ void k_positive(const i64* w, u64 n, u32* keep, i64* neww) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { keep[n] = 0; return; }
  keep[i] = w[i] > 0 ? 1u : 0u;
  neww[i] = 1;
}

// SemiJoinStream::eval (semijoin.rs:100-142): weight product with the key set.
__global__ void k_semijoin(Cols P, const i64* wP, u64 np, Cols K, const i64* wK, u64 nkeys, int nk, Flips f, u32* keep,
                           i64* neww) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > np) return;
  if (i == np) { keep[np] = 0; return; }
  u64 q[MAXL];
  for (int l = 0; l < nk; l++) q[l] = P.c[l][i] ^ f.f[l];
  u64 lo = lower_bound_q(K, 0, nkeys, q, nk, f);
  i64 w = 0;
  if (lo < nkeys && cmp_row_q(K, lo, q, nk, f) == 0) w = (i64)((u64)wP[i] * (u64)wK[lo]);
  keep[i] = w != 0;
  neww[i] = w;
}

// cursor.seek(val_bound) of the truncating merge (ordered/mod.rs:652-664,
// 729-734) on flat rows: keep the rows whose value lanes are >= the bound.
struct RowBound { u64 v[MAXL]; };   // value lanes, order-flipped
__global__ void k_vals_ge(Cols C, u64 n, int nk, int nv, RowBound b, Flips f, u32* keep) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { keep[n] = 0; return; }
  bool ge = true;
  for (int l = 0; l < nv; l++) {
    u64 x = C.c[nk + l][i] ^ f.f[nk + l];
    if (x != b.v[l]) { ge = x > b.v[l]; break; }
  }
  keep[i] = ge ? 1u : 0u;
}

// head flag over the first nk lanes (key boundaries of the flat rows).
__global__ void k_key_heads(Cols C, u64 n, int nk, u32* flags) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { flags[n] = 0; return; }
  bool head = i == 0;
  if (!head)
    for (int l = 0; l < nk; l++)
      if (C.c[l][i] != C.c[l][i - 1]) { head = true; break; }
  flags[i] = head ? 1u : 0u;
}

// ordered compaction: out[pos[i]] = row i for keep[i] != 0
__global__ void k_scatter(Cols in, int L, const i64* w, const u32* keep, const u32* pos, u64 n, MCols out, i64* out_w) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !keep[i]) return;
  u32 o = pos[i];
  for (int l = 0; l < L; l++) out.c[l][o] = in.c[l][i];
  if (out_w) out_w[o] = w[i];
}
__global__ void k_scatter_index(const u32* keep, const u32* pos, u64 n, u64* out, u64 nout) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && keep[i]) out[pos[i]] = i;
  if (i == 0) out[nout] = n;
}
__global__ void k_fill_i64(i64* out, u64 n, i64 v) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = v;
}

__global__ void k_neg(const i64* w, u64 n, i64* out) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (i64)((u64)0 - (u64)w[i]);
}

// Aggregator pick over a gathered, consolidated key group batch G (rows of the
// affected keys, weights summed over the spine's batches, zeros dropped):
// Max = last row of each key (max.rs:36-55), Min = first (min.rs:38-57),
// Fold count / sum (fold.rs:76-96), WeightedCount (aggregate/mod.rs:129-156).
__global__ void k_agg_pick(Cols G, const i64* wG, u64 n, int nk, int nv, int kind, const i64* psum, Flips f, u32* keep,
                           MCols out, int out_nv) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { keep[n] = 0; return; }
  bool first = i == 0, last = i == n - 1;
  if (!first)
    for (int l = 0; l < nk; l++)
      if (G.c[l][i] != G.c[l][i - 1]) { first = true; break; }
  if (!last)
    for (int l = 0; l < nk; l++)
      if (G.c[l][i] != G.c[l][i + 1]) { last = true; break; }
  u32 k = 0;
  u64 v[MAXL];
  if (kind == DBSP_AGG_MAX) {
    k = last;
    for (int l = 0; l < nv; l++) v[l] = G.c[nk + l][i];
  } else if (kind == DBSP_AGG_MIN) {
    k = first;
    for (int l = 0; l < nv; l++) v[l] = G.c[nk + l][i];
  } else if (kind == DBSP_AGG_FOLD_COUNT || kind == DBSP_AGG_FOLD_SUM) {
    k = last;
    if (last) {
      u64 q[MAXL];
      for (int l = 0; l < nk; l++) q[l] = G.c[l][i] ^ f.f[l];
      u64 start = lower_bound_q(G, 0, i + 1, q, nk, f);
      if (kind == DBSP_AGG_FOLD_COUNT) v[0] = i - start + 1;
      else v[0] = (u64)psum[i] - (start ? (u64)psum[start - 1] : 0ull);
    }
  } else if (kind == DBSP_AGG_WCOUNT) {
    k = 1;
    v[0] = (u64)wG[i];
  } else {   // WCOUNT2: rows (K.., which): sum at which == 0, count at which == 1
    k = first;
    if (first) {
      u64 which = G.c[nk][i];
      bool two = !last;   // a second row of the same key follows
      v[0] = which == 0 ? (u64)wG[i] : 0;
      v[1] = which == 1 ? (u64)wG[i] : (two ? (u64)wG[i + 1] : 0);
    }
  }
  keep[i] = k;
  if (k)
    for (int l = 0; l < out_nv; l++) out.c[l][i] = v[l];
}

// Max / Min.  Per key, a walk over the union of the spine batches' value lists from the extreme end — the
// CursorList walk of max.rs:36-55 (backwards from the end) / min.rs:38-57 (forwards): per batch a cursor into the
// key's value range; the candidate is the extreme value under the cursors, its weight the sum over the batches that
// hold it (cursor_list.rs:200-210); a zero sum (the value was retracted by another batch — e.g. a merge still in
// progress holds +1 and -1 in two batches) steps those cursors and tries the next value.  Keys that need more than
// AGG_WALK steps are flagged for the general gather path.
constexpr int AGG_WALK = 64;
__global__ void k_agg_extremum(Cols K, u64 nkeys, int nk, int nv, BatchRefs tr, Flips f, int is_max, u32* keep,
                               MCols outv, u64* slow_counter) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > nkeys) return;
  if (i == nkeys) { keep[nkeys] = 0; return; }
  u64 q[MAXL], best[MAXL];
  for (int l = 0; l < nk; l++) q[l] = K.c[l][i] ^ f.f[l];
  // the key's value range [lo, hi) in every batch; cur = next candidate position
  u32 lo[MAX_REFS], hi[MAX_REFS];
  for (int b = 0; b < tr.nb; b++) {
    const Cols& T = tr.b[b].c;
    const u64 nt = tr.b[b].n;
    const u64 l0 = lower_bound_q(T, 0, nt, q, nk, f);
    u64 h0 = l0;
    if (l0 < nt && cmp_row_q(T, l0, q, nk, f) == 0) {
      u64 step = 1;
      h0 = l0 + 1;
      while (h0 + step <= nt && cmp_row_q(T, h0 + step - 1, q, nk, f) == 0) { h0 += step; step <<= 1; }
      const u64 top = h0 + step <= nt ? h0 + step : nt;
      h0 = upper_bound_q(T, h0, top, q, nk, f);
    }
    lo[b] = (u32)l0;
    hi[b] = (u32)h0;
  }
  bool have = false, exhausted = false;
  i64 wsum = 0;
  for (int it = 0; it < AGG_WALK; it++) {
    have = false;
    for (int b = 0; b < tr.nb; b++) {
      if (lo[b] >= hi[b]) continue;
      const Cols& T = tr.b[b].c;
      const u64 r = is_max ? (u64)hi[b] - 1 : (u64)lo[b];
      int c = 0;   // cmp(candidate, best) over the value lanes
      u64 cand[MAXL];
      for (int l = 0; l < nv; l++) {
        cand[l] = T.c[nk + l][r] ^ f.f[nk + l];
        if (have && c == 0 && cand[l] != best[l]) c = cand[l] < best[l] ? -1 : 1;
      }
      if (!have || (is_max ? c > 0 : c < 0)) {
        for (int l = 0; l < nv; l++) best[l] = cand[l];
        have = true;
      }
    }
    if (!have) break;   // every cursor ran off its range: the key has no value left
    wsum = 0;
    for (int b = 0; b < tr.nb; b++) {
      if (lo[b] >= hi[b]) continue;
      const Cols& T = tr.b[b].c;
      const u64 r = is_max ? (u64)hi[b] - 1 : (u64)lo[b];
      bool eq = true;
      for (int l = 0; l < nv; l++) eq = eq && ((T.c[nk + l][r] ^ f.f[nk + l]) == best[l]);
      if (eq) {
        wsum = (i64)((u64)wsum + (u64)tr.b[b].w[r]);
        if (is_max) hi[b]--; else lo[b]++;   // step past the candidate
      }
    }
    if (wsum != 0) break;
    if (it == AGG_WALK - 1) exhausted = true;
  }
  u32 k = 0;
  if (exhausted) {
    atomicAdd((unsigned long long*)slow_counter, 1ull);
  } else if (have && wsum != 0) {
    k = 1;
    for (int l = 0; l < nv; l++) outv.c[l][i] = best[l] ^ f.f[nk + l];
  }
  keep[i] = k;
}

// weigh (aggregate/mod.rs:297-323): per row f(k,v)*w; AVG mode emits the
// (sum, count) pair weight as two rows (K,0) / (K,1).
__global__ void k_weigh(Cols B, const i64* w, u64 n, int nk, int nv, dbsp_expr fx, int mode, MCols out, i64* out_w) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 lanes[MAXL];
  for (int l = 0; l < nk + nv; l++) lanes[l] = B.c[l][i];
  Env e{lanes, lanes + nk, lanes + nk};
  u64 fv = expr_val(fx, e);
  if (mode == DBSP_WEIGH_AVG) {
    for (int l = 0; l < nk; l++) { out.c[l][2 * i] = lanes[l]; out.c[l][2 * i + 1] = lanes[l]; }
    out.c[nk][2 * i] = 0;
    out.c[nk][2 * i + 1] = 1;
    out_w[2 * i] = (i64)(fv * (u64)w[i]);
    out_w[2 * i + 1] = w[i];
  } else {
    for (int l = 0; l < nk; l++) out.c[l][i] = lanes[l];
    out_w[i] = (i64)(fv * (u64)w[i]);
  }
}

// lower bounds of several key tuples in one batch (window ranges, truncation)
__global__ void k_lower_bounds(Cols T, u64 nt, int nk, Flips f, const u64* queries, int nq, u64* out) {
  int qi = blockIdx.x * blockDim.x + threadIdx.x;
  if (qi >= nq) return;
  u64 q[MAXL];
  for (int l = 0; l < nk; l++) q[l] = queries[qi * MAXL + l] ^ f.f[l];
  out[qi] = lower_bound_q(T, 0, nt, q, nk, f);
}

__device__ __forceinline__ u64 mix64(u64 x) {
  x += 0x9e3779b97f4a7c15ull;
  x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
  x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}
// shard_batch (communication/shard.rs:165-199): flags[p*(n+1) + i] = (hash(key) % P == p).
// One exclusive scan over the concatenated flag arrays is a *stable* P-way
// partition: shard p's rows follow shard p-1's, each shard keeps its order.
__global__ void k_shard_flags(Cols B, u64 n, int nk, u32 P, u32* flags) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  u32 dest = P;   // i == n: terminator slot of every shard
  if (i < n) {
    u64 h = 0;
    for (int l = 0; l < nk; l++) h = mix64(h ^ B.c[l][i]);
    dest = (u32)(h % P);
  }
  for (u32 p = 0; p < P; p++) flags[(u64)p * (n + 1) + i] = (p == dest) ? 1u : 0u;
}
__global__ void k_shard_scatter(Cols in, int L, const i64* w, const u32* flags, const u32* pos, u64 n, u32 P, MCols out,
                                i64* out_w, u64* bounds) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P) bounds[i] = pos[i * (n + 1)];           // first output slot of shard i
  if (i == P) bounds[P] = pos[(u64)P * (n + 1) - 1]; // total (= n)
  if (i >= n) return;
  for (u32 p = 0; p < P; p++) {
    u64 j = (u64)p * (n + 1) + i;
    if (flags[j]) {
      u32 o = pos[j];
      for (int l = 0; l < L; l++) out.c[l][o] = in.c[l][i];
      out_w[o] = w[i];
    }
  }
}

inline unsigned blocks(u64 n) { return (unsigned)((n + TB - 1) / TB); }
// Row indices, offsets and scans of the operator kernels are 32-bit: reject (never wrap) anything larger.
#define ROWS32(n, what)                                                                        \
  do {                                                                                         \
    if ((u64)(n) >= 0xffffffffull) {                                                           \
      set_error(std::string(what) + ": 2^32-1 or more rows in one batch; split the batch");   \
      return DBSP_ERR_UNSUPPORTED;                                                             \
    }                                                                                          \
  } while (0)
#define CHECK_P(c, msg)                                   \
  do {                                                    \
    if (!(c)) { set_error(msg); return DBSP_ERR_INVALID; } \
  } while (0)

}  // namespace

// ============================ host side =======================================

// Temporary unsorted row store (L lanes + weights) of capacity cap.
struct TmpRows {
  BufP buf;
  MCols c;
  i64* w = nullptr;
  Cols cc() const {
    Cols r;
    for (int l = 0; l < MAXL; l++) r.c[l] = c.c[l];
    return r;
  }
};
static int32_t tmp_alloc(Ctx* ctx, int L, u64 cap, TmpRows* t) {
  u64 c = (cap + 32) & ~31ull;
  if (c == 0) c = 32;
  TRY(dev_alloc(ctx, (size_t)c * 8 * (L + 1), &t->buf));
  u64* base = (u64*)t->buf->p;
  for (int l = 0; l < MAXL; l++) t->c.c[l] = l < L ? base + (size_t)l * c : nullptr;
  t->w = (i64*)(base + (size_t)L * c);
  return DBSP_OK;
}

int32_t compact_ordered(Ctx* ctx, const dbsp_schema& s, const Cols& in, const i64* w, const u32* keep, u64 n, Batch** out) {
  // keep has n+1 entries (keep[n] == 0)
  ROWS32(n, "compact");
  int L = s.n_key_lanes + s.n_val_lanes;
  BufP pbuf;
  TRY(dev_alloc(ctx, (size_t)(n + 1) * 4, &pbuf));
  u32* pos = (u32*)pbuf->p;
  const Mail mail = mail_begin(ctx);
  TRY(exclusive_scan_u32(ctx, keep, pos, n, &mail));
  u64 nout64;
  TRY(mail_finish(ctx, mail, &nout64, 1));
  const u32 nout = (u32)nout64;
  if (nout == 0) { *out = batch_new_empty(ctx, s); return DBSP_OK; }
  Batch* b;
  MCols oc;
  i64* ow;
  TRY(batch_alloc(ctx, s, nout, &b, &oc, &ow));
  k_scatter<<<blocks(n), TB, 0, lane(ctx).stream>>>(in, L, w, keep, pos, n, oc, ow);
  LAUNCH_COUNT(ctx);
  *out = b;
  return DBSP_OK;
}

// Drop the rows whose value is below `val_bound` (n_val_lanes u64).  Keys left
// without values vanish with their rows.  Shares the batch when nothing is cut.
int32_t op_truncate_values(Ctx* ctx, const Batch* b, const u64* val_bound, Batch** out) {
  int nk = b->s.n_key_lanes, nv = b->s.n_val_lanes;
  if (b->n == 0 || nv == 0) { batch_ref((Batch*)b); *out = (Batch*)b; return DBSP_OK; }
  Flips f = b->flips();
  RowBound rb;
  for (int l = 0; l < nv; l++) rb.v[l] = val_bound[l] ^ f.f[nk + l];
  u64 n = b->n;
  ROWS32(n, "truncate_values");
  BufP kb;
  TRY(dev_alloc(ctx, (size_t)(n + 1) * 4 * 2, &kb));
  u32* keep = (u32*)kb->p;
  u32* pos = keep + (n + 1);
  {
    ProfScope ps(ctx, KID_COMPACT, n * (u64)nv * 8);
    k_vals_ge<<<blocks(n + 1), TB, 0, lane(ctx).stream>>>(b->cols(), n, nk, nv, rb, f, keep);
  }
  LAUNCH_COUNT(ctx);
  const Mail mail = mail_begin(ctx);
  TRY(exclusive_scan_u32(ctx, keep, pos, n, &mail));
  u64 nout64;
  TRY(mail_finish(ctx, mail, &nout64, 1));
  const u32 nout = (u32)nout64;
  if (nout == n) { batch_ref((Batch*)b); *out = (Batch*)b; return DBSP_OK; }
  if (nout == 0) { *out = batch_new_empty(ctx, b->s); return DBSP_OK; }
  Batch* o;
  MCols oc;
  i64* ow;
  TRY(batch_alloc(ctx, b->s, nout, &o, &oc, &ow));
  {
    ProfScope ps(ctx, KID_COMPACT, (n + nout) * (u64)(b->nl() + 1) * 8);
    k_scatter<<<blocks(n), TB, 0, lane(ctx).stream>>>(b->cols(), b->nl(), b->w, keep, pos, n, oc, ow);
  }
  LAUNCH_COUNT(ctx);
  *out = o;
  return DBSP_OK;
}

// Zero-copy view of rows [lo, hi) of a batch (shares its storage).
Batch* batch_slice(Ctx* ctx, const Batch* b, u64 lo, u64 hi) {
  Batch* v = new Batch();
  v->s = b->s;
  v->ctx = ctx;
  v->n = hi - lo;
  for (int l = 0; l < b->nl(); l++) v->col[l] = b->col[l] + lo;
  v->w = b->w + lo;
  v->bufs = b->bufs;
  if (v->n == 0) v->nkeys = 0;
  return v;
}

// Concatenation of consolidated batches whose row ranges are already ordered
// and disjoint (the chunks of a fuelled merge): device-to-device copies only.
// Consumes one reference of each part.
int32_t batch_concat(Ctx* ctx, const dbsp_schema& s, std::vector<Batch*>& parts, Batch** out) {
  std::vector<Batch*> live;
  u64 total = 0;
  for (Batch* p : parts) {
    if (p->n) { live.push_back(p); total += p->n; } else batch_unref(p);
  }
  parts.clear();
  if (live.empty()) { *out = batch_new_empty(ctx, s); return DBSP_OK; }
  if (live.size() == 1) { *out = live[0]; return DBSP_OK; }
  Batch* o;
  MCols oc;
  i64* ow;
  int32_t rc = batch_alloc(ctx, s, total, &o, &oc, &ow);
  if (rc) { for (Batch* p : live) batch_unref(p); return rc; }
  int L = s.n_key_lanes + s.n_val_lanes;
  u64 off = 0;
  for (Batch* p : live) {
    for (int l = 0; l < L; l++)
      cudaMemcpyAsync(oc.c[l] + off, p->col[l], p->n * 8, cudaMemcpyDeviceToDevice, lane(ctx).stream);
    cudaMemcpyAsync(ow + off, p->w, p->n * 8, cudaMemcpyDeviceToDevice, lane(ctx).stream);
    off += p->n;
    batch_unref(p);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { batch_unref(o); set_error(cudaGetErrorString(e)); return DBSP_ERR_CUDA; }
  *out = o;
  return DBSP_OK;
}

// input lanes the closure reads (bit l = lane l of the (key lanes, val lanes) row)
unsigned proj_used_mask(const dbsp_proj& p, int nk_in) {
  unsigned mask = 0;
  auto use = [&](const dbsp_src& s) {
    if (s.kind == DBSP_SRC_KEY) mask |= 1u << s.idx;
    else if (s.kind == DBSP_SRC_LVAL || s.kind == DBSP_SRC_RVAL) mask |= 1u << (nk_in + s.idx);
  };
  int nl = p.out_schema.n_key_lanes + p.out_schema.n_val_lanes;
  for (int l = 0; l < nl; l++) { use(p.out[l].a); if (p.out[l].op >= DBSP_OP_ADD) use(p.out[l].b); }
  for (int i = 0; i < p.n_pred; i++) { use(p.pred[i].a); use(p.pred[i].b); }
  return mask;
}
static int used_lanes(const dbsp_proj& p, int n_in_lanes, int nk_in = 0) {
  int c = __builtin_popcount(proj_used_mask(p, nk_in) & ((1u << n_in_lanes) - 1));
  return c;
}

// project rows of (in cols) through proj, then consolidate.
int32_t project_and_consolidate(Ctx* ctx, const Cols& in, int nk_in, int n_in_lanes, const i64* w, u64 n,
                                const dbsp_proj& proj, Batch** out) {
  const dbsp_schema& os = proj.out_schema;
  int Lo = os.n_key_lanes + os.n_val_lanes;
  if (n == 0) { *out = batch_new_empty(ctx, os); return DBSP_OK; }
  ROWS32(n, "map_index / flat_map_index");
  const unsigned g = (unsigned)((n + PROJ_ROWS - 1) / PROJ_ROWS);
  const bool filtered = proj.n_pred > 0;
  const u64 m = n;   // upper bound when a filter is present
  u64* status = nullptr;
  u32* ticket = nullptr;
  u32* d_mw = nullptr;
  BufP cb;
  if (filtered) {
    // status[g] u64 | ticket u32, surviving-row count u32
    TRY(dev_alloc(ctx, (size_t)(g + 1) * 8, &cb));
    CUDA_TRY(cudaMemsetAsync(cb->p, 0, (size_t)(g + 1) * 8, lane(ctx).stream));
    status = (u64*)cb->p;
    ticket = (u32*)(status + g);
    d_mw = ticket + 1;   // stays on the device; the census of consolidate_rows returns it
  }
  const u32* d_m = d_mw;
  TmpRows t;
  TRY(tmp_alloc(ctx, Lo, m, &t));
  {
    // the lanes the closure names read once, the output rows written once (bound: every row survives)
    ProfScope ps(ctx, KID_PROJECT, n * (u64)(used_lanes(proj, n_in_lanes, nk_in) + (w ? 1 : 0)) * 8 + m * (u64)(Lo + 1) * 8);
    k_project_rows<<<g, TB, 0, lane(ctx).stream>>>(in, nk_in, w, n, proj, filtered ? 0 : 1, g, ticket, status, t.c, t.w, d_mw);
  }
  LAUNCH_COUNT(ctx);
  return consolidate_rows(ctx, os, t.cc(), t.w, m, &t.buf, out, d_m);
}

// Probe `delta` against (up to MAX_REFS) batches of `trace` and expand the matches.
// proj == nullptr: gather the matching trace rows unchanged.
static int32_t probe_chunk(Ctx* ctx, const Batch* delta, int nk, Batch* const* tb, int nb, const dbsp_proj* proj,
                           int delta_is_left, const dbsp_schema& out_schema, Batch** out) {
  cudaStream_t st = lane(ctx).stream;
  const u64 nd = delta->n;
  Flips f = delta->flips();
  BatchRefs refs;
  refs.nb = nb;
  u64 trace_rows = 0;
  ROWS32(nd, "join/gather delta");
  for (int b = 0; b < nb; b++) ROWS32(tb[b]->n, "join/gather trace batch");
  for (int b = 0; b < nb; b++) {
    refs.b[b].c = tb[b]->cols();
    refs.b[b].w = tb[b]->w;
    refs.b[b].n = tb[b]->n;
    trace_rows += tb[b]->n;
  }
  // lo, cnt: u32[nd * nb] (only the rows that start a segment are written) | ki: u32[nd]
  BufP kb, rb;
  TRY(dev_alloc(ctx, (size_t)nd * nb * 4 * 2 + (size_t)nd * 4, &kb));
  u32* lo = (u32*)kb->p;
  u32* cnt = lo + (size_t)nd * nb;
  u32* ki = cnt + (size_t)nd * nb;
  // ex[nd+1] u32 (padded to u64) | status[ntiles] u64 | ticket u64
  const u32 ntiles = (u32)((nd + PR_TILE - 1) / PR_TILE);
  const size_t ex_u64 = (size_t)(nd + 2) / 2 + 1;
  TRY(dev_alloc(ctx, (ex_u64 + ntiles + 1) * 8, &rb));
  u32* ex = (u32*)rb->p;
  u64* status = (u64*)rb->p + ex_u64;
  u32* ticket = (u32*)(status + ntiles);
  CUDA_TRY(cudaMemsetAsync(status, 0, (size_t)(ntiles + 1) * 8, st));
  const Mail mail = mail_begin(ctx);
  {
    // delta key lanes read once; ki, lo, cnt and ex written once; every search step touches one trace key row
    // (bounded by the trace's key bytes)
    u64 lg = 1; while ((1ull << lg) < trace_rows / std::max(nb, 1) + 1) lg++;
    const u64 touched = std::min<u64>(nd * (u64)nb * 2 * lg, trace_rows) * (u64)std::max(nk, 1) * 8;
    ProfScope ps(ctx, KID_PROBE_RANGES, nd * ((u64)nk * 8 + (u64)nb * 8 + 8) + touched);
    k_probe_ranges<<<ntiles, TB, 0, st>>>(delta->cols(), nd, refs, nk, f, ntiles, ticket, status, ki, lo, cnt, ex, mail);
  }
  LAUNCH_COUNT(ctx);
  u64 total;
  TRY(mail_finish(ctx, mail, &total, 1));
  if (total >= 0xffffffffull) {
    set_error("join/gather: 2^32-1 or more matches in one step (" + std::to_string(total) + "); feed the delta in smaller batches");
    return DBSP_ERR_UNSUPPORTED;
  }
  if (total == 0) { *out = batch_new_empty(ctx, out_schema); return DBSP_OK; }
  int Lo = out_schema.n_key_lanes + out_schema.n_val_lanes;
  dbsp_proj pj;
  if (proj) pj = *proj; else memset(&pj, 0, sizeof(pj));
  TmpRows t;
  TRY(tmp_alloc(ctx, Lo, total, &t));
  {
    // matched trace rows read once, delta rows read once, output rows written once
    ProfScope ps(ctx, KID_PROBE_FILL, (u64)total * (u64)(tb[0]->nl() - nk + 1) * 8 + nd * (u64)(delta->nl() + 1) * 8 +
                                          (u64)total * (u64)(Lo + 1) * 8);
    // slots per thread: as few as keep about two CTAs per SM busy, at most PF_IPT
    const u64 per_pass = (u64)256 * 2 * ctx->sm_count;
    const int ipt = (int)std::min<u64>(PF_IPT, std::max<u64>(1, (total + per_pass - 1) / per_pass));
    const u64 tile = (u64)ipt * 256;
    k_probe_fill<<<(unsigned)((total + tile - 1) / tile), 256, 0, st>>>(delta->cols(), delta->w, nd, refs, nk, delta->nl() - nk,
                                                                        tb[0]->nl() - nk, lo, cnt, ki, ex, total, ipt,
                                                                        proj ? 1 : 0, delta_is_left, pj, t.c, t.w);
  }
  LAUNCH_COUNT(ctx);
  // the Batcher of join.rs:845-858: usually sort-free (ordered slots)
  return consolidate_rows(ctx, out_schema, t.cc(), t.w, total, &t.buf, out);
}

static int32_t merge_tree(Ctx* ctx, std::vector<Batch*>& parts, const dbsp_schema& s, Batch** out);

static int32_t probe_spine(Ctx* ctx, const Batch* delta, int nk, const Spine* trace, const dbsp_proj* proj,
                           int delta_is_left, const dbsp_schema& out_schema, Batch** out) {
  const size_t nb = trace->batches.size();
  if (delta->n == 0 || nb == 0) { *out = batch_new_empty(ctx, out_schema); return DBSP_OK; }
  std::vector<Batch*> parts;
  for (size_t b0 = 0; b0 < nb; b0 += MAX_REFS) {
    int cnt = (int)std::min<size_t>(MAX_REFS, nb - b0);
    Batch* part = nullptr;
    int32_t rc = probe_chunk(ctx, delta, nk, trace->batches.data() + b0, cnt, proj, delta_is_left, out_schema, &part);
    if (rc) { for (Batch* p : parts) batch_unref(p); return rc; }
    parts.push_back(part);
  }
  return merge_tree(ctx, parts, out_schema, out);
}

// JoinTrace::eval (operator/join.rs:732-863)
int32_t op_join_delta_trace(Ctx* ctx, const Batch* delta, const Spine* trace, const dbsp_proj* proj, int delta_is_left,
                            Batch** out) {
  if (delta->s.n_key_lanes != trace->s.n_key_lanes) { set_error("join: key lanes differ"); return DBSP_ERR_INVALID; }
  return probe_spine(ctx, delta, delta->s.n_key_lanes, trace, proj, delta_is_left, proj->out_schema, out);
}

// Join::eval (operator/join.rs:436-473)
int32_t op_join_batches(Ctx* ctx, const Batch* l, const Batch* r, const dbsp_proj* proj, Batch** out) {
  Spine sp;
  sp.s = r->s;
  sp.ctx = ctx;
  if (r->n) sp.batches.push_back((Batch*)r);
  return op_join_delta_trace(ctx, l, &sp, proj, 1, out);
}

// distinct keys (first nk lanes) of a batch as an OrdZSet<K> batch with weight 1
static int32_t distinct_keys(Ctx* ctx, const Batch* b, int nk, Batch** out) {
  dbsp_schema ks;
  memset(&ks, 0, sizeof(ks));
  ks.n_key_lanes = nk;
  for (int l = 0; l < nk; l++) ks.lane_types[l] = b->s.lane_types[l];
  if (b->n == 0) { *out = batch_new_empty(ctx, ks); return DBSP_OK; }
  BufP fb;
  TRY(dev_alloc(ctx, (size_t)(b->n + 1) * 4, &fb));
  u32* flags = (u32*)fb->p;
  k_key_heads<<<blocks(b->n + 1), TB, 0, lane(ctx).stream>>>(b->cols(), b->n, nk, flags);
  LAUNCH_COUNT(ctx);
  return compact_ordered(ctx, ks, b->cols(), b->w, flags, b->n, out);
}

// AggregateIncremental::eval + Upsert::eval
// (operator/aggregate/mod.rs:479-547,600-684; operator/upsert.rs:161-208).
int32_t op_aggregate_delta(Ctx* ctx, const Batch* delta, const Spine* in_tr, const Spine* out_tr, int kind, Batch** out) {
  cudaStream_t st = lane(ctx).stream;
  const dbsp_schema& os = out_tr->s;
  int nk = os.n_key_lanes, nov = os.n_val_lanes;
  if (delta->n == 0) { *out = batch_new_empty(ctx, os); return DBSP_OK; }
  // 1. affected keys
  Batch* keys = nullptr;
  TRY(distinct_keys(ctx, delta, nk, &keys));
  int32_t rc;
  Batch* N = nullptr;
  // 2a. Max / Min: candidates straight from the batches' range ends
  if ((kind == DBSP_AGG_MAX || kind == DBSP_AGG_MIN) && in_tr->batches.size() <= (size_t)MAX_REFS && keys->n) {
    BatchRefs refs;
    refs.nb = (int)in_tr->batches.size();
    for (int b = 0; b < refs.nb; b++) {
      refs.b[b].c = in_tr->batches[b]->cols();
      refs.b[b].w = in_tr->batches[b]->w;
      refs.b[b].n = in_tr->batches[b]->n;
    }
    Flips tf;
    for (int l = 0; l < MAXL; l++)
      tf.f[l] = (l < nk + nov && in_tr->s.lane_types[l] == DBSP_I64) ? 0x8000000000000000ull : 0ull;
    BufP kb;
    TRY(dev_alloc(ctx, (size_t)(keys->n + 1) * 4, &kb));
    TmpRows nvr;
    TRY(tmp_alloc(ctx, nov, keys->n, &nvr));
    u64* slow = lane(ctx).d_scratch + 16;
    CUDA_TRY(cudaMemsetAsync(slow, 0, 8, st));
    {
      u64 lg = 1; while ((1ull << lg) < in_tr->batches[0]->n + 1) lg++;
      ProfScope ps(ctx, KID_AGG_PICK, keys->n * ((u64)nk * 8 + (u64)refs.nb * (lg * 8 + (u64)(nov + 1) * 8) + (u64)nov * 8));
      k_agg_extremum<<<blocks(keys->n + 1), TB, 0, st>>>(keys->cols(), keys->n, nk, nov, refs, tf, kind == DBSP_AGG_MAX,
                                                        (u32*)kb->p, nvr.c, slow);
    }
    LAUNCH_COUNT(ctx);
    u64 nslow;
    TRY(read_back(ctx, slow, 1, &nslow));
    if (nslow == 0) {
      Cols src;
      for (int l = 0; l < MAXL; l++) src.c[l] = nullptr;
      for (int l = 0; l < nk; l++) src.c[l] = keys->col[l];
      for (int l = 0; l < nov; l++) src.c[nk + l] = nvr.c.c[l];
      BufP ones;
      TRY(dev_alloc(ctx, (size_t)keys->n * 8, &ones));
      k_fill_i64<<<blocks(keys->n), TB, 0, st>>>((i64*)ones->p, keys->n, 1);
      LAUNCH_COUNT(ctx);
      rc = compact_ordered(ctx, os, src, (const i64*)ones->p, (u32*)kb->p, keys->n, &N);
      if (rc) { batch_unref(keys); return rc; }
    }
  }
  // 2b. general path: the keys' value groups, weights summed over batches
  Batch* G = nullptr;
  if (!N) {
    rc = probe_spine(ctx, keys, nk, in_tr, nullptr, 1, in_tr->s, &G);
    if (rc) { batch_unref(keys); return rc; }
  }
  // 3. aggregate per key -> rows (key, new value) with weight +1
  if (N) {
  } else if (G->n) {
    int gnk = nk, gnv = G->nl() - nk;
    if (kind == DBSP_AGG_WCOUNT2) gnv = 0;   // (K.., which) rows: `which` read as lane nk
    BufP kb, ps;
    TRY(dev_alloc(ctx, (size_t)(G->n + 1) * 4, &kb));
    u32* keep = (u32*)kb->p;
    const i64* psum = nullptr;
    if (kind == DBSP_AGG_FOLD_SUM) {
      TRY(dev_alloc(ctx, (size_t)G->n * 8, &ps));
      TRY(inclusive_scan_i64(ctx, (const i64*)G->col[nk], (i64*)ps->p, G->n));
      psum = (const i64*)ps->p;
    }
    TmpRows nv;
    TRY(tmp_alloc(ctx, nov, G->n, &nv));
    k_agg_pick<<<blocks(G->n + 1), TB, 0, st>>>(G->cols(), G->w, G->n, gnk, gnv, kind, psum, G->flips(), keep, nv.c, nov);
    LAUNCH_COUNT(ctx);
    // rows (key lanes of G, new value lanes), weight +1 (reuse delta-free ones array: build below)
    Cols src;
    for (int l = 0; l < MAXL; l++) src.c[l] = nullptr;
    for (int l = 0; l < nk; l++) src.c[l] = G->col[l];
    for (int l = 0; l < nov; l++) src.c[nk + l] = nv.c.c[l];
    // weights: all +1
    BufP ones;
    TRY(dev_alloc(ctx, (size_t)G->n * 8, &ones));
    k_fill_i64<<<blocks(G->n), TB, 0, st>>>((i64*)ones->p, G->n, 1);
    LAUNCH_COUNT(ctx);
    rc = compact_ordered(ctx, os, src, (const i64*)ones->p, keep, G->n, &N);
    if (rc) { batch_unref(keys); batch_unref(G); return rc; }
  } else {
    N = batch_new_empty(ctx, os);
  }
  if (G) batch_unref(G);
  // 4. current values of those keys in the output trace, negated
  Batch* O = nullptr;
  rc = probe_spine(ctx, keys, nk, out_tr, nullptr, 1, os, &O);
  batch_unref(keys);
  if (rc) { batch_unref(N); return rc; }
  // 5. consolidate(+new, -old) per key == merge of two consolidated batches
  Batch* On = nullptr;
  rc = op_neg(ctx, O, &On);
  batch_unref(O);
  if (rc) { batch_unref(N); return rc; }
  rc = merge_batches(ctx, N, On, out);
  batch_unref(N);
  batch_unref(On);
  return rc;
}

int32_t op_neg(Ctx* ctx, const Batch* a, Batch** out) {
  if (a->n == 0) { *out = batch_new_empty(ctx, a->s); return DBSP_OK; }
  BufP wb;
  TRY(dev_alloc(ctx, (size_t)a->n * 8, &wb));
  k_neg<<<blocks(a->n), TB, 0, lane(ctx).stream>>>(a->w, a->n, (i64*)wb->p);
  LAUNCH_COUNT(ctx);
  Batch* b = new Batch();
  b->s = a->s;
  b->n = a->n;
  b->ctx = ctx;
  for (int l = 0; l < MAXL; l++) b->col[l] = a->col[l];
  b->w = (const i64*)wb->p;
  b->bufs = a->bufs;   // share the lane storage
  b->bufs.push_back(wb);
  *out = b;
  return DBSP_OK;
}

// weigh (operator/aggregate/mod.rs:297-323)
int32_t op_weigh(Ctx* ctx, const Batch* b, const dbsp_expr* f, int mode, Batch** out) {
  int nk = b->s.n_key_lanes, nv = b->s.n_val_lanes;
  dbsp_schema os;
  memset(&os, 0, sizeof(os));
  os.n_key_lanes = nk + (mode == DBSP_WEIGH_AVG ? 1 : 0);
  for (int l = 0; l < nk; l++) os.lane_types[l] = b->s.lane_types[l];
  if (b->n == 0) { *out = batch_new_empty(ctx, os); return DBSP_OK; }
  u64 m = b->n * (mode == DBSP_WEIGH_AVG ? 2 : 1);
  ROWS32(m, "weigh");
  TmpRows t;
  TRY(tmp_alloc(ctx, os.n_key_lanes, m, &t));
  k_weigh<<<blocks(b->n), TB, 0, lane(ctx).stream>>>(b->cols(), b->w, b->n, nk, nv, *f, mode, t.c, t.w);
  LAUNCH_COUNT(ctx);
  return consolidate_rows(ctx, os, t.cc(), t.w, m, &t.buf, out);
}

// DistinctIncrementalTotal::eval (operator/distinct.rs:196-254)
int32_t op_distinct_delta(Ctx* ctx, const Batch* delta, const Spine* integral, Batch** out) {
  u64 n = delta->n;
  if (n == 0) { *out = batch_new_empty(ctx, delta->s); return DBSP_OK; }
  cudaStream_t st = lane(ctx).stream;
  BufP ab, kb;
  TRY(dev_alloc(ctx, (size_t)n * 8 * 2, &ab));
  TRY(dev_alloc(ctx, (size_t)(n + 1) * 4, &kb));
  i64* acc = (i64*)ab->p;
  i64* neww = acc + n;
  CUDA_TRY(cudaMemsetAsync(acc, 0, (size_t)n * 8, st));
  for (Batch* T : integral->batches) {
    k_lookup_add<<<blocks(n), TB, 0, st>>>(delta->cols(), n, T->cols(), T->w, T->n, delta->nl(), delta->flips(), acc);
    LAUNCH_COUNT(ctx);
  }
  k_distinct_decide<<<blocks(n + 1), TB, 0, st>>>(delta->w, acc, n, (u32*)kb->p, neww);
  LAUNCH_COUNT(ctx);
  return compact_ordered(ctx, delta->s, delta->cols(), neww, (u32*)kb->p, n, out);
}

// IndexedZSet::distinct (algebra/zset/mod.rs:14-38)
int32_t op_stream_distinct(Ctx* ctx, const Batch* b, Batch** out) {
  u64 n = b->n;
  if (n == 0) { *out = batch_new_empty(ctx, b->s); return DBSP_OK; }
  BufP ab, kb;
  TRY(dev_alloc(ctx, (size_t)n * 8, &ab));
  TRY(dev_alloc(ctx, (size_t)(n + 1) * 4, &kb));
  k_positive<<<blocks(n + 1), TB, 0, lane(ctx).stream>>>(b->w, n, (u32*)kb->p, (i64*)ab->p);
  LAUNCH_COUNT(ctx);
  return compact_ordered(ctx, b->s, b->cols(), (i64*)ab->p, (u32*)kb->p, n, out);
}

// SemiJoinStream::eval (operator/semijoin.rs:100-142)
int32_t op_semijoin(Ctx* ctx, const Batch* pairs, const Batch* keys, Batch** out) {
  u64 n = pairs->n;
  // Out: ZSet<Key = (Pairs::Key, Pairs::Val)> (semijoin.rs:47): same flat rows, every lane a key lane
  dbsp_schema os = pairs->s;
  os.n_key_lanes = (uint8_t)pairs->nl();
  os.n_val_lanes = 0;
  if (n == 0 || keys->n == 0) { *out = batch_new_empty(ctx, os); return DBSP_OK; }
  BufP ab, kb;
  TRY(dev_alloc(ctx, (size_t)n * 8, &ab));
  TRY(dev_alloc(ctx, (size_t)(n + 1) * 4, &kb));
  k_semijoin<<<blocks(n + 1), TB, 0, lane(ctx).stream>>>(pairs->cols(), pairs->w, n, keys->cols(), keys->w, keys->n,
                                                   pairs->s.n_key_lanes, pairs->flips(), (u32*)kb->p, (i64*)ab->p);
  LAUNCH_COUNT(ctx);
  return compact_ordered(ctx, os, pairs->cols(), (i64*)ab->p, (u32*)kb->p, n, out);
}

// Balanced merge of consolidated batches; consumes one reference of each part.
static int32_t merge_tree(Ctx* ctx, std::vector<Batch*>& parts, const dbsp_schema& s, Batch** out) {
  int32_t rc = DBSP_OK;
  while (parts.size() > 1) {
    std::vector<Batch*> nxt;
    size_t i = 0;
    for (; i + 1 < parts.size(); i += 2) {
      Batch* m = nullptr;
      if (rc == DBSP_OK) rc = merge_batches(ctx, parts[i], parts[i + 1], &m);
      batch_unref(parts[i]);
      batch_unref(parts[i + 1]);
      if (m) nxt.push_back(m);
    }
    if (i < parts.size()) nxt.push_back(parts[i]);
    parts.swap(nxt);
    if (rc != DBSP_OK) { for (Batch* b : parts) batch_unref(b); parts.clear(); return rc; }
  }
  *out = parts.empty() ? batch_new_empty(ctx, s) : parts[0];
  parts.clear();
  return DBSP_OK;
}

// Window::eval (operator/time_series/window.rs:144-222)
int32_t op_window_delta(Ctx* ctx, const Spine* trace, const Batch* delta, int has_prev, const u64* s0, const u64* e0,
                        const u64* s1, const u64* e1, Batch** out) {
  cudaStream_t st = lane(ctx).stream;
  const dbsp_schema& s = delta->s;
  int nk = s.n_key_lanes, L = delta->nl();
  auto lt = [&](const u64* a, const u64* b) {
    for (int l = 0; l < nk; l++) {
      u64 x = a[l], y = b[l];
      if (s.lane_types[l] == DBSP_I64) { x ^= 1ull << 63; y ^= 1ull << 63; }
      if (x != y) return x < y;
    }
    return false;
  };
  struct Range { const Batch* b; u64 lo, hi; int neg; };
  std::vector<Range> ranges;
  // queries: s0, s1, e0, e1 lower bounds in every batch (+ delta)
  u64 hq[4 * MAXL];
  memset(hq, 0, sizeof(hq));
  for (int l = 0; l < nk; l++) { hq[0 * MAXL + l] = s0[l]; hq[1 * MAXL + l] = s1[l]; hq[2 * MAXL + l] = e0[l]; hq[3 * MAXL + l] = e1[l]; }
  BufP qb;
  TRY(dev_alloc(ctx, sizeof(hq) + 4 * 8, &qb));
  u64* dq = (u64*)qb->p;
  u64* dres = dq + 4 * MAXL;
  CUDA_TRY(cudaMemcpyAsync(dq, hq, sizeof(hq), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaStreamSynchronize(st));   // hq is a stack buffer
  ctx->h2d_bytes += sizeof(hq);
  auto bounds = [&](const Batch* b, u64* r) -> int32_t {
    if (b->n == 0) { r[0] = r[1] = r[2] = r[3] = 0; return DBSP_OK; }
    k_lower_bounds<<<1, 32, 0, st>>>(b->cols(), b->n, nk, b->flips(), dq, 4, dres);
    LAUNCH_COUNT(ctx);
    return read_back(ctx, dres, 4, r);
  };
  u64 r[4];
  if (has_prev) {
    for (Batch* b : trace->batches) {
      TRY(bounds(b, r));
      u64 ps0 = r[0], ps1 = r[1], pe0 = r[2], pe1 = r[3];
      // region 1: [s0, min(s1, e0))
      u64 hi1 = std::min(ps1, pe0);
      if (hi1 > ps0) ranges.push_back({b, ps0, hi1, 1});
      // shrunk on the right: [e1, e0) when e1 < e0
      if (lt(e1, e0) && pe0 > pe1) ranges.push_back({b, pe1, pe0, 1});
      // region 3: [max(e0, s1), e1)
      u64 from = std::max(pe0, ps1);
      if (pe1 > from) ranges.push_back({b, from, pe1, 0});
    }
  }
  TRY(bounds(delta, r));
  if (r[3] > r[1]) ranges.push_back({delta, r[1], r[3], 0});
  // Every range is a slice of a consolidated batch: a zero-copy view (negated
  // for retractions), and Batch::from_tuples over their union is a merge tree.
  std::vector<Batch*> parts;
  int32_t rc = DBSP_OK;
  for (auto& g : ranges) {
    Batch* v = new Batch();
    v->s = s;
    v->ctx = ctx;
    v->n = g.hi - g.lo;
    for (int l = 0; l < L; l++) v->col[l] = g.b->col[l] + g.lo;
    v->w = g.b->w + g.lo;
    v->bufs = g.b->bufs;
    if (g.neg) {
      Batch* nv = nullptr;
      rc = op_neg(ctx, v, &nv);
      batch_unref(v);
      if (rc) break;
      v = nv;
    }
    parts.push_back(v);
  }
  if (rc != DBSP_OK) { for (Batch* b : parts) batch_unref(b); return rc; }
  return merge_tree(ctx, parts, s, out);
}

// Map/FlatMap/Index::eval + from_tuples (operator/filter_map.rs:563-577,700-724)
int32_t op_map_index(Ctx* ctx, const Batch* b, const dbsp_proj* proj, Batch** out) {
  return project_and_consolidate(ctx, b->cols(), b->s.n_key_lanes, b->nl(), b->w, b->n, *proj, out);
}

// shard_batch (operator/communication/shard.rs:165-199)
int32_t op_shard_partition(Ctx* ctx, const Batch* b, u32 P, Batch** outs) {
  for (u32 p = 0; p < P; p++) outs[p] = nullptr;
  if (b->n == 0) {
    for (u32 p = 0; p < P; p++) outs[p] = batch_new_empty(ctx, b->s);
    return DBSP_OK;
  }
  const u64 n = b->n;
  const int L = b->nl();
  CHECK_P(P <= 64, "shard_partition: at most 64 shards");
  ROWS32((n + 1) * (u64)P, "shard_partition");
  BufP fb;
  const u64 m = (u64)P * (n + 1);
  TRY(dev_alloc(ctx, (size_t)(m + 1) * 4 * 2, &fb));
  u32* flags = (u32*)fb->p;
  u32* pos = flags + (m + 1);
  k_shard_flags<<<blocks(n + 1), TB, 0, lane(ctx).stream>>>(b->cols(), n, b->s.n_key_lanes, P, flags);
  LAUNCH_COUNT(ctx);
  CUDA_TRY(cudaMemsetAsync(flags + m, 0, 4, lane(ctx).stream));
  TRY(exclusive_scan_u32(ctx, flags, pos, m));
  Batch* all;   // one buffer holding the P shards back to back; the shards are views
  MCols oc;
  i64* ow;
  TRY(batch_alloc(ctx, b->s, n, &all, &oc, &ow));
  u64* bounds = lane(ctx).d_scratch + 160;
  k_shard_scatter<<<blocks(std::max<u64>(n, P + 1)), TB, 0, lane(ctx).stream>>>(b->cols(), L, b->w, flags, pos, n, P, oc, ow, bounds);
  LAUNCH_COUNT(ctx);
  u64 hb[65];
  int32_t rc = read_back(ctx, bounds, P + 1, hb);
  if (rc) { batch_unref(all); return rc; }
  for (u32 p = 0; p < P; p++) {
    Batch* v = new Batch();
    v->s = b->s;
    v->ctx = ctx;
    v->n = hb[p + 1] - hb[p];
    for (int l = 0; l < L; l++) v->col[l] = all->col[l] + hb[p];
    v->w = all->w + hb[p];
    v->bufs = all->bufs;
    if (v->n == 0) v->nkeys = 0;
    outs[p] = v;
  }
  batch_unref(all);
  return DBSP_OK;
}

// CSR view: row index of every key's first tuple (OrderedLayer offs,
// trace/layers/ordered/mod.rs:32-44), built on demand.
int32_t batch_build_csr(Ctx* ctx, Batch* b) {
  if (b->nkeys != ~0ull) return DBSP_OK;
  if (b->n == 0) { b->nkeys = 0; return DBSP_OK; }
  ROWS32(b->n, "key_count / download_csr");
  int nk = b->s.n_key_lanes;
  BufP fb, pb;
  TRY(dev_alloc(ctx, (size_t)(b->n + 1) * 4 * 2, &fb));
  u32* flags = (u32*)fb->p;
  u32* pos = flags + (b->n + 1);
  k_key_heads<<<blocks(b->n + 1), TB, 0, lane(ctx).stream>>>(b->cols(), b->n, nk, flags);
  LAUNCH_COUNT(ctx);
  const Mail mail = mail_begin(ctx);
  TRY(exclusive_scan_u32(ctx, flags, pos, b->n, &mail));
  u64 nkeys64;
  TRY(mail_finish(ctx, mail, &nkeys64, 1));
  const u32 nkeys = (u32)nkeys64;
  TRY(dev_alloc(ctx, (size_t)(nkeys + 1) * 8, &pb));
  k_scatter_index<<<blocks(b->n), TB, 0, lane(ctx).stream>>>(flags, pos, b->n, (u64*)pb->p, nkeys);
  LAUNCH_COUNT(ctx);
  b->keystart = pb;
  b->nkeys = nkeys;
  return DBSP_OK;
}

// lower bound of one key tuple in a batch (host value)
int32_t batch_lower_bound(Ctx* ctx, const Batch* b, const u64* key, u64* pos) {
  if (b->n == 0) { *pos = 0; return DBSP_OK; }
  u64 hq[MAXL] = {0};
  for (int l = 0; l < b->s.n_key_lanes; l++) hq[l] = key[l];
  u64* dq = lane(ctx).d_scratch + 96;
  CUDA_TRY(cudaMemcpyAsync(dq, hq, sizeof(hq), cudaMemcpyHostToDevice, lane(ctx).stream));
  CUDA_TRY(cudaStreamSynchronize(lane(ctx).stream));
  k_lower_bounds<<<1, 32, 0, lane(ctx).stream>>>(b->cols(), b->n, b->s.n_key_lanes, b->flips(), dq, 1, lane(ctx).d_scratch + 120);
  LAUNCH_COUNT(ctx);
  return read_back(ctx, lane(ctx).d_scratch + 120, 1, pos);
}
