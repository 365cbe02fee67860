// consolidate.cu — K1/K2: Batch::from_tuples on the device.
//
// Replaces consolidation::consolidate (sort + sum equal keys + drop zeros,
// crates/dbsp/src/trace/consolidation/mod.rs:32-52,182-231), the MergeBatcher
// (trace/ord/merge_batcher/mod.rs:65-80,155-197) and the Builder
// (trace/layers/ordered/mod.rs:874-888) for rows of <= 8 integer lanes.
//
// B200-first design.
//  (1) One property pass over the rows reduces each lane's [min,max] and
//      counts order inversions, adjacent duplicates and zero weights.
//  (2) Rows that arrive already ordered (projections of sorted batches, join
//      and gather outputs, id-ordered event tables) skip the sort entirely;
//      if they are also duplicate- and zero-free the input buffer *becomes*
//      the batch (no copy).
//  (3) Otherwise the comparison sort the reference spends "90% of the work"
//      in (consolidation/mod.rs:101-104) is a radix sort over bit-packed
//      composite keys: the lanes' significant bits are concatenated (order
//      preserving, injective) into as few 64-bit words as possible and only
//      those bits are sorted, as (key word, row id) pairs, by the hand-written
//      passes of sort.cu (top digits in HBM, the rest in shared memory; no HBM
//      pass at all when the leading lane arrives ordered).  The Nexmark
//      schemas pack into one word of 30-60 bits.
//  (4) Epilogue: a two-pass reduce-by-key sums runs of equal rows and drops
//      zero sums; the duplicate-free case is one unpack/gather pass.
#include <cstdio>
#include <cstdlib>

#include "common.cuh"

namespace {

struct Plan {
  int L, W;
  int use_key;   // 1 / 2: the epilogue compares and unpacks the packed key word(s); 0: it goes through the row ids
  u64 mn[MAXL], flip[MAXL], mask[MAXL];
  unsigned char word[MAXL], shift[MAXL], bits[MAXL];
  unsigned char wbits[MAXL];
  signed char alias[MAXL];   // >= 0: the lane always equals that earlier lane (not packed; copied on unpack)
  unsigned char pos[MAXL];   // W <= 2: bit position of the lane inside the 128-bit concatenation (key1 : key0)
};

// mm[l] = min, mm[L+l] = max of flipped lane l; mm[2L] = # inversions
// (row i-1 > row i), mm[2L+1] = # adjacent duplicates, mm[2L+2] = # zero weights,
// mm[2L+3] = row count (when it lives on the device), mm[2L+4] = # inversions of lane 0 alone,
// mm[2L+5] = bit (l*(l-1)/2 + j) set when lane l differs from the earlier lane j in some row.
template <int L>   // compile-time lane count: the per-lane state stays in registers, every loop unrolls
__global__ void __launch_bounds__(256) k_props(Cols cols, Flips f, const i64* w, u64 n_host, const u32* dn, u64* mm, Mail mail) {
  // the producer may have left the exact row count on the device (dn): the
  // census then returns it with the lane ranges in the same read-back
  const u64 n = dn ? (u64)*dn : n_host;
  if (dn && blockIdx.x == 0 && threadIdx.x == 0) mm[2 * L + 3] = n;
  __shared__ u64 smin[MAXL], smax[MAXL];
  __shared__ unsigned s_cnt[4];
  if (threadIdx.x < MAXL) { smin[threadIdx.x] = ~0ull; smax[threadIdx.x] = 0; }
  if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  u64 lmin[L], lmax[L];
#pragma unroll
  for (int l = 0; l < L; l++) { lmin[l] = ~0ull; lmax[l] = 0; }
  unsigned inv = 0, dup = 0, zero = 0, inv0 = 0, neq = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    int c = 0;   // cmp(row i-1, row i)
    u64 raw[L];
#pragma unroll
    for (int l = 0; l < L; l++) {
      raw[l] = cols.c[l][i];
      u64 v = raw[l] ^ f.f[l];
      lmin[l] = min(lmin[l], v);
      lmax[l] = max(lmax[l], v);
      if (i > 0 && c == 0) {
        u64 pv = cols.c[l][i - 1] ^ f.f[l];
        if (pv != v) c = pv < v ? -1 : 1;
        if (l == 0) inv0 += pv > v;
      }
    }
    if (i > 0) { inv += c > 0; dup += c == 0; }
    if (w && w[i] == 0) zero++;
#pragma unroll
    for (int l = 1; l < L; l++)
#pragma unroll
      for (int j = 0; j < l; j++)
        if (raw[l] != raw[j]) neq |= 1u << (l * (l - 1) / 2 + j);
  }
#pragma unroll
  for (int l = 0; l < L; l++) {
    u64 a = lmin[l], b = lmax[l];
    for (int o = 16; o > 0; o >>= 1) {
      a = min(a, __shfl_xor_sync(0xffffffffu, a, o));
      b = max(b, __shfl_xor_sync(0xffffffffu, b, o));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin((unsigned long long*)&smin[l], (unsigned long long)a);
      atomicMax((unsigned long long*)&smax[l], (unsigned long long)b);
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    inv += __shfl_xor_sync(0xffffffffu, inv, o);
    dup += __shfl_xor_sync(0xffffffffu, dup, o);
    zero += __shfl_xor_sync(0xffffffffu, zero, o);
    inv0 += __shfl_xor_sync(0xffffffffu, inv0, o);
    neq |= __shfl_xor_sync(0xffffffffu, neq, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (neq) atomicOr((unsigned long long*)&mm[2 * L + 5], (unsigned long long)neq);
    if (inv) atomicAdd(&s_cnt[0], inv);
    if (dup) atomicAdd(&s_cnt[1], dup);
    if (zero) atomicAdd(&s_cnt[2], zero);
    if (inv0) atomicAdd(&s_cnt[3], inv0);
  }
  __syncthreads();
  if (threadIdx.x < L) {
    atomicMin((unsigned long long*)&mm[threadIdx.x], (unsigned long long)smin[threadIdx.x]);
    atomicMax((unsigned long long*)&mm[L + threadIdx.x], (unsigned long long)smax[threadIdx.x]);
  }
  if (threadIdx.x < 3 && s_cnt[threadIdx.x])
    atomicAdd((unsigned long long*)&mm[2 * L + threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
  if (threadIdx.x == 3 && s_cnt[3]) atomicAdd((unsigned long long*)&mm[2 * L + 4], (unsigned long long)s_cnt[3]);
  // the last block to finish publishes the census to the host mailbox (mm[2L+6] counts finished blocks)
  __shared__ unsigned s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd((unsigned long long*)&mm[2 * L + 6], 1ull) == (unsigned long long)(gridDim.x - 1);
  __syncthreads();
  if (s_last && threadIdx.x == 0) {
    __threadfence();
    u64 vals[2 * L + 6];
    for (int i = 0; i < 2 * L + 6; i++) vals[i] = ((volatile u64*)mm)[i];
    mail_publish(mail, vals, 2 * L + 6);
  }
}

__global__ void k_init_props(u64* mm, int L) {
  int t = threadIdx.x;
  if (t < L) mm[t] = ~0ull;
  else if (t < 2 * L + 7) mm[t] = 0;
}

// key[i] = word `wd` of row (idx ? idx[i] : i); writes idx_out[i] = i when idx == nullptr.
__global__ void k_pack(Cols cols, Plan p, int wd, const u32* idx, u64 n, u64* key, u32* idx_out) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 r = idx ? idx[i] : i;
  u64 k = 0;
  for (int l = 0; l < p.L; l++)
    if (p.word[l] == wd && p.bits[l]) k |= ((cols.c[l][r] ^ p.flip[l]) - p.mn[l]) << p.shift[l];
  key[i] = k;
  if (!idx) idx_out[i] = (u32)i;
}

// both words of a one- or two-word key in one read of the rows, plus the identity row ids.  The lanes' bits are
// packed back to back over the 128-bit concatenation (key1 : key0); a lane may straddle the word boundary.
__global__ void k_pack12(Cols cols, Plan p, u64 n, u64* key0, u64* key1, u32* idx_out) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 k0 = 0, k1 = 0;
  for (int l = 0; l < p.L; l++) {
    if (!p.bits[l]) continue;
    const u64 v = (cols.c[l][i] ^ p.flip[l]) - p.mn[l];
    const int ps = p.pos[l];
    if (ps >= 64) k1 |= v << (ps - 64);
    else {
      k0 |= v << ps;
      if (ps + p.bits[l] > 64) k1 |= v >> (64 - ps);
    }
  }
  key0[i] = k0;
  if (key1) key1[i] = k1;
  idx_out[i] = (u32)i;
}

__device__ __forceinline__ u64 unpack_lane(const Plan& p, int l, u64 key) {   // word-granular packing (W >= 3 path)
  u64 v = p.bits[l] ? ((key >> p.shift[l]) & p.mask[l]) : 0;
  return (v + p.mn[l]) ^ p.flip[l];
}
__device__ __forceinline__ u64 unpack_lane12(const Plan& p, int l, u64 k0, u64 k1) {
  u64 v = 0;
  if (p.bits[l]) {
    const int ps = p.pos[l];
    if (ps >= 64) v = k1 >> (ps - 64);
    else if (ps + p.bits[l] <= 64) v = k0 >> ps;
    else v = (k0 >> ps) | (k1 << (64 - ps));
    v &= p.mask[l];
  }
  return (v + p.mn[l]) ^ p.flip[l];
}

// ---------------------------------------------------------------------------
// k_reduce_emit — the dedup + retain of consolidate (consolidation/mod.rs:32-52) and the Builder
// (ordered/mod.rs:874-888) in ONE pass over the rows in sorted order (identity order, or through the row ids of
// the sort): every run of equal rows becomes one output row carrying the sum of the run's weights, zero sums are
// dropped.  Per tile of RE_TILE rows:
//   (1) head / tail flags and weights of the thread's rows; block scan with the (has-head, weight-since-last-head)
//       monoid gives every row the weight of the run open before it inside the tile;
//   (2) look-back #1 (same monoid, across tiles): the weight of the run that enters the tile.  A predecessor
//       that contains a head ends the walk, so the usual distance is one tile;
//   (3) run totals at the tails, kept flags (total != 0), block scan of the kept counts;
//   (4) look-back #2 (plain sum): the tile's first output slot;
//   (5) the kept rows are written (unpacked from the key word, or gathered through the row id), weights = totals.
// Tiles take their index from a ticket, so every predecessor a look-back waits on is already running.
constexpr int RE_THREADS = 256, RE_R = 4, RE_TILE = RE_THREADS * RE_R;
struct HS {
  u32 h;
  i64 s;
};
__device__ __forceinline__ HS hs_op(const HS& a, const HS& b) {   // a then b
  HS r;
  r.h = a.h | b.h;
  r.s = b.h ? b.s : (i64)((u64)a.s + (u64)b.s);
  return r;
}
// per-tile status: [0] aggregate {flag|h, s}, [1] inclusive prefix {flag|h, s}, [2] kept-count word (2-bit flag | value)
struct ReStatus {
  u64 agg_f, agg_s, pre_f, pre_s, cnt, pad_[3];
};
__device__ __forceinline__ u64 re_ld_acq(const u64* p) {
  u64 v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void re_st_rel(u64* p, u64 v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ u64 re_ld(const u64* p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void re_st(u64* p, u64 v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// result[0] = number of output rows; result[2] (the sort's fallback flag) != 0 on entry => nothing is done.
// Global traffic is coalesced on both sides: the tile's key words (or row ids) and gathered weights are loaded
// striped and staged in shared memory, the flag / scan work runs on the blocked arrangement out of shared memory,
// and the kept rows are staged by output rank and written striped.
__global__ void __launch_bounds__(RE_THREADS)
k_reduce_emit(Cols cols, Plan p, const u64* key, const u64* key1, const u32* idx, const i64* w, u64 n, ReStatus* status, u32* ticket,
              MCols out, i64* out_w, u64* result, Mail mail) {
  __shared__ u64 s_a[RE_TILE + 2];   // slot j+1 = row tile_s + j: key word 0 (use_key) or the row id; 0 / cnt+1 = halo rows
  __shared__ u64 s_b[RE_TILE + 2];   // key word 1 (use_key == 2)
  __shared__ i64 s_wt[RE_TILE];
  __shared__ HS s_warp_hs[RE_THREADS / 32];
  __shared__ u32 s_warp_u[RE_THREADS / 32];
  __shared__ u32 s_tile;
  __shared__ i64 s_cin;
  __shared__ u64 s_base;
  if (result[2]) {   // the sort raised its fallback flag: key / idx are not a permutation yet
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      const u64 vals[3] = {0, 0, result[2]};
      mail_publish(mail, vals, 3);
    }
    return;
  }
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const u32 tile = s_tile;
  const u64 tile_s = (u64)tile * RE_TILE;
  const u64 tile_e = tile_s + RE_TILE < n ? tile_s + RE_TILE : n;
  const int cnt = (int)(tile_e - tile_s);
  const int uk = p.use_key;

  // ---- striped, coalesced load into shared memory (+ one halo row on each side) ----
  auto stage = [&](int slot, u64 i) {
    if (uk) {
      s_a[slot] = key[i];
      if (uk == 2) s_b[slot] = key1[i];
    } else {
      s_a[slot] = idx ? (u64)idx[i] : i;
    }
  };
#pragma unroll
  for (int k = 0; k < RE_R; k++) {
    const int j = k * RE_THREADS + tid;
    if (j < cnt) {
      const u64 i = tile_s + j;
      stage(j + 1, i);
      s_wt[j] = w ? w[idx ? idx[i] : i] : 1;
    }
  }
  if (tid == 0 && tile_s > 0) stage(0, tile_s - 1);
  if (tid == 32 && tile_e < n) stage(cnt + 1, tile_e);
  __syncthreads();
  auto differs = [&](int sa, int sb) -> bool {   // staged rows in slots sa, sb
    if (uk == 1) return s_a[sa] != s_a[sb];
    if (uk == 2) return s_a[sa] != s_a[sb] || s_b[sa] != s_b[sb];
    const u64 a = s_a[sa], b = s_a[sb];
    for (int l = 0; l < p.L; l++)
      if (cols.c[l][a] != cols.c[l][b]) return true;
    return false;
  };

  // ---- blocked arrangement out of shared memory: thread t owns rows t*RE_R .. t*RE_R+RE_R-1 of the tile ----
  const int j0 = tid * RE_R;
  bool hd[RE_R], tl[RE_R], valid[RE_R];
  i64 wt[RE_R];
#pragma unroll
  for (int k = 0; k < RE_R; k++) {
    const int j = j0 + k;
    valid[k] = j < cnt;
    hd[k] = false; tl[k] = false; wt[k] = 0;
    if (valid[k]) {
      hd[k] = (tile_s + j == 0) || differs(j + 1, j);
      wt[k] = s_wt[j];
    }
  }
#pragma unroll
  for (int k = 0; k < RE_R; k++) {
    const int j = j0 + k;
    if (valid[k]) {
      if (k + 1 < RE_R && j + 1 < cnt) tl[k] = hd[k + 1];
      else tl[k] = (tile_s + j + 1 >= n) || differs(j + 2, j + 1);
    }
  }
  // (1) thread aggregate and block scan with the flag/sum monoid
  HS agg; agg.h = 0; agg.s = 0;
#pragma unroll
  for (int k = 0; k < RE_R; k++) {
    if (!valid[k]) continue;
    if (hd[k]) { agg.h = 1; agg.s = wt[k]; }
    else agg.s = (i64)((u64)agg.s + (u64)wt[k]);
  }
  HS incl = agg;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    HS v;
    v.h = __shfl_up_sync(0xffffffffu, incl.h, o);
    v.s = __shfl_up_sync(0xffffffffu, incl.s, o);
    if (lane >= o) incl = hs_op(v, incl);
  }
  if (lane == 31) s_warp_hs[wid] = incl;
  __syncthreads();
  HS wprefix; wprefix.h = 0; wprefix.s = 0;
  for (int k = 0; k < wid; k++) wprefix = hs_op(wprefix, s_warp_hs[k]);
  HS excl_in_warp;
  excl_in_warp.h = __shfl_up_sync(0xffffffffu, incl.h, 1);
  excl_in_warp.s = __shfl_up_sync(0xffffffffu, incl.s, 1);
  if (lane == 0) { excl_in_warp.h = 0; excl_in_warp.s = 0; }
  const HS excl = hs_op(wprefix, excl_in_warp);   // open run before this thread, within the tile

  // (2) look-back #1: weight of the run entering the tile
  if (tid == RE_THREADS - 1) {
    const HS tile_agg = hs_op(wprefix, incl);   // inclusive over the whole tile
    ReStatus* me = &status[tile];
    HS carry; carry.h = 0; carry.s = 0;   // fold of the tiles before this one, as far back as needed
    if (tile == 0) {
      re_st(&me->pre_s, (u64)tile_agg.s);
      re_st_rel(&me->pre_f, 2ull | ((u64)tile_agg.h << 2));
    } else {
      re_st(&me->agg_s, (u64)tile_agg.s);
      re_st_rel(&me->agg_f, 1ull | ((u64)tile_agg.h << 2));
      long long q = (long long)tile - 1;
      while (true) {
        const ReStatus* pr = &status[q];
        HS v;
        bool is_prefix;
        while (true) {
          const u64 pf = re_ld_acq(&pr->pre_f);
          if (pf & 3) { v.h = (u32)((pf >> 2) & 1); v.s = (i64)re_ld(&pr->pre_s); is_prefix = true; break; }
          const u64 af = re_ld_acq(&pr->agg_f);
          if (af & 3) { v.h = (u32)((af >> 2) & 1); v.s = (i64)re_ld(&pr->agg_s); is_prefix = false; break; }
        }
        carry = hs_op(v, carry);
        if (carry.h || is_prefix || q == 0) break;   // a head further back makes everything before it irrelevant
        q--;
      }
      const HS pre = hs_op(carry, tile_agg);
      re_st(&me->pre_s, (u64)pre.s);
      re_st_rel(&me->pre_f, 2ull | ((u64)pre.h << 2));
    }
    s_cin = carry.s;
  }
  __syncthreads();
  const i64 cin = s_cin;

  // (3) run totals at the tails, kept flags
  i64 run = excl.h ? excl.s : (i64)((u64)excl.s + (u64)cin);
  u32 kept = 0;
  i64 tot[RE_R];
  bool kp[RE_R];
#pragma unroll
  for (int k = 0; k < RE_R; k++) {
    kp[k] = false; tot[k] = 0;
    if (!valid[k]) continue;
    if (hd[k]) run = wt[k];
    else run = (i64)((u64)run + (u64)wt[k]);
    if (tl[k]) { tot[k] = run; kp[k] = run != 0; kept += kp[k]; }
  }
  u32 kincl = kept;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 v = __shfl_up_sync(0xffffffffu, kincl, o);
    if (lane >= o) kincl += v;
  }
  if (lane == 31) s_warp_u[wid] = kincl;
  // the kept rows' staged words are read before shared memory is reused for the output staging
  u64 ka[RE_R], kb[RE_R];
#pragma unroll
  for (int k = 0; k < RE_R; k++) {
    ka[k] = 0; kb[k] = 0;
    if (kp[k]) { ka[k] = s_a[j0 + k + 1]; if (uk == 2) kb[k] = s_b[j0 + k + 1]; }
  }
  __syncthreads();
  u32 woff = 0, tile_kept = 0;
#pragma unroll
  for (int k = 0; k < RE_THREADS / 32; k++) {
    const u32 v = s_warp_u[k];
    if (k < wid) woff += v;
    tile_kept += v;
  }
  // stage the kept rows by output rank
  {
    u32 lr = woff + kincl - kept;
#pragma unroll
    for (int k = 0; k < RE_R; k++) {
      if (!kp[k]) continue;
      s_a[lr] = ka[k];
      if (uk == 2) s_b[lr] = kb[k];
      s_wt[lr] = tot[k];
      lr++;
    }
  }
  // (4) look-back #2: first output slot of the tile.  Warp 0 inspects 32 predecessor status words per round trip
  // (tile q - lane per lane); aggregates of tiles that have not resolved their own prefix yet are summed on the way.
  if (wid == 0) {
    ReStatus* me = &status[tile];
    u64 base = 0;
    if (tile == 0) {
      if (lane == 0) re_st(&me->cnt, (2ull << 62) | (u64)tile_kept);
    } else {
      if (lane == 0) re_st(&me->cnt, (1ull << 62) | (u64)tile_kept);
      long long q0 = (long long)tile - 1;
      while (true) {
        const long long q = q0 - lane;
        u64 v = 2ull << 62;   // tiles before 0 contribute an empty prefix
        if (q >= 0) {
          do { v = re_ld(&status[q].cnt); } while ((v >> 62) == 0);
        }
        const unsigned isp = __ballot_sync(0xffffffffu, (v >> 62) == 2);
        const int first = isp ? (__ffs(isp) - 1) : 32;
        u64 c = (lane <= first) ? (v & ((1ull << 62) - 1)) : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        base += c;
        if (isp) break;
        q0 -= 32;
      }
      if (lane == 0) re_st(&me->cnt, (2ull << 62) | (base + tile_kept));
    }
    if (lane == 0) {
      s_base = base;
      if (tile_e == n) {   // the last tile knows the total: it goes straight to the host mailbox
        const u64 vals[3] = {base + tile_kept, 0, 0};
        result[0] = vals[0];
        mail_publish(mail, vals, 3);
      }
    }
  }
  __syncthreads();
  // (5) striped, coalesced output
  const u64 base = s_base;
  for (u32 o = tid; o < tile_kept; o += RE_THREADS) {
    const u64 pos = base + o;
    if (uk) {
      const u64 kk0 = s_a[o], kk1 = uk == 2 ? s_b[o] : 0;
      u64 v[MAXL];
      for (int l = 0; l < p.L; l++) {
        v[l] = p.alias[l] >= 0 ? v[p.alias[l]] : unpack_lane12(p, l, kk0, kk1);
        out.c[l][pos] = v[l];
      }
    } else {
      const u64 r = s_a[o];
      for (int l = 0; l < p.L; l++) out.c[l][pos] = cols.c[l][r];
    }
    out_w[pos] = s_wt[o];
  }
}

inline int bits_for(u64 range) { return range == 0 ? 0 : 64 - __builtin_clzll(range); }

}  // namespace

int32_t radix_sort_pairs(Ctx* ctx, int words, u64* k0a, u64* k0b, u64* k1a, u64* k1b, u32* ida, u32* idb, u64 n, int bits_lo, int bits_hi,
                         int presorted_top_bits, bool force_lsd, unsigned long long* fail, int* which, int* hbm_passes);

int32_t consolidate_rows(Ctx* ctx, const dbsp_schema& s, const Cols& cols, const i64* w, u64 n, const BufP* adopt,
                         Batch** out, const u32* d_n) {
  const int L = s.n_key_lanes + s.n_val_lanes;
  if (n == 0) { *out = batch_new_empty(ctx, s); return DBSP_OK; }   // with d_n: n is an upper bound
  if (n >= (1ull << 32)) { set_error("consolidate: more than 2^32-1 rows in one batch"); return DBSP_ERR_UNSUPPORTED; }
  cudaStream_t st = lane(ctx).stream;
  const int TB = 256;

  Flips f;
  for (int l = 0; l < MAXL; l++) f.f[l] = (l < L && s.lane_types[l] == DBSP_I64) ? 0x8000000000000000ull : 0;

  // ---- (1) lane ranges + order / duplicate / zero-weight census ---------------
  u64 mm[2 * MAXL + 6];
  {
    u64* dmm = lane(ctx).d_scratch + 64;
    k_init_props<<<1, 32, 0, st>>>(dmm, L);
    const Mail mail = mail_begin(ctx);
    int g = (int)std::min<u64>((n + TB - 1) / TB, (u64)ctx->sm_count * 8);
    {
      ProfScope ps(ctx, KID_MINMAX, n * (u64)(L + (w ? 1 : 0)) * 8);
      switch (L) {
        case 1: k_props<1><<<g, TB, 0, st>>>(cols, f, w, n, d_n, dmm, mail); break;
        case 2: k_props<2><<<g, TB, 0, st>>>(cols, f, w, n, d_n, dmm, mail); break;
        case 3: k_props<3><<<g, TB, 0, st>>>(cols, f, w, n, d_n, dmm, mail); break;
        case 4: k_props<4><<<g, TB, 0, st>>>(cols, f, w, n, d_n, dmm, mail); break;
        case 5: k_props<5><<<g, TB, 0, st>>>(cols, f, w, n, d_n, dmm, mail); break;
        case 6: k_props<6><<<g, TB, 0, st>>>(cols, f, w, n, d_n, dmm, mail); break;
        case 7: k_props<7><<<g, TB, 0, st>>>(cols, f, w, n, d_n, dmm, mail); break;
        default: k_props<8><<<g, TB, 0, st>>>(cols, f, w, n, d_n, dmm, mail); break;
      }
    }
    ctx->kernel_launches += 2;
    TRY(mail_finish(ctx, mail, mm, 2 * L + 6));
    if (d_n) {
      n = mm[2 * L + 3];
      if (n == 0) { *out = batch_new_empty(ctx, s); return DBSP_OK; }
    }
  }
  const unsigned nblk = (unsigned)((n + TB - 1) / TB);
  const u64 n_inv = mm[2 * L], n_dup = mm[2 * L + 1], n_zero = mm[2 * L + 2];

  Plan p;
  memset(&p, 0, sizeof(p));
  p.L = L;
  for (int l = 0; l < MAXL; l++) p.alias[l] = -1;
  u32* idx_cur = nullptr;
  const u64* key_sorted = nullptr;
  BufP kbuf, ibuf, tmp;

  if (n_inv == 0) {
    // ---- (2) already ordered: no sort ------------------------------------------
    if (n_dup == 0 && n_zero == 0 && adopt && w) {
      Batch* b = new Batch();   // the input buffer *is* the batch
      b->s = s;
      b->n = n;
      b->ctx = ctx;
      for (int l = 0; l < L; l++) b->col[l] = cols.c[l];
      b->w = w;
      b->bufs.push_back(*adopt);
      *out = b;
      return DBSP_OK;
    }
    p.W = 1;
    p.use_key = 0;   // compare / copy the lanes themselves, identity order
  } else {
    // ---- (3) bit-packing plan: lanes from last (least significant) to first ----
    // a lane that equals an earlier lane in every row never breaks a tie: it is left out of the key and copied
    // back when the rows are unpacked (q7's (price, auction, bidder, price, ..) rows)
    const u64 neq = mm[2 * L + 5];
    for (int l = 1; l < L; l++)
      for (int j = 0; j < l && p.alias[l] < 0; j++)
        if (!((neq >> (l * (l - 1) / 2 + j)) & 1)) p.alias[l] = (signed char)j;
    int total_bits = 0;
    for (int l = L - 1; l >= 0; l--) {
      const int b = p.alias[l] >= 0 ? 0 : bits_for(mm[L + l] - mm[l]);
      p.bits[l] = (unsigned char)b;
      p.mn[l] = mm[l];
      p.flip[l] = f.f[l];
      p.mask[l] = b >= 64 ? ~0ull : ((1ull << b) - 1);
      total_bits += b;
    }
    if (total_bits <= 128) {
      // one or two key words: the lanes' bits back to back, last lane least significant
      int at = 0;
      for (int l = L - 1; l >= 0; l--) { p.pos[l] = (unsigned char)at; at += p.bits[l]; }
      p.W = total_bits <= 64 ? 1 : 2;
      p.wbits[0] = (unsigned char)(total_bits <= 64 ? total_bits : 64);
      p.wbits[1] = (unsigned char)(total_bits <= 64 ? 0 : total_bits - 64);
    } else {
      // wider rows: whole lanes per word, sorted word by word
      int word = 0, used = 0;
      for (int l = L - 1; l >= 0; l--) {
        const int b = p.bits[l];
        if (used + b > 64) { word++; used = 0; }
        p.word[l] = (unsigned char)word;
        p.shift[l] = (unsigned char)used;
        used += b;
        p.wbits[word] = (unsigned char)used;
      }
      p.W = word + 1;
    }
    p.use_key = p.W <= 2 ? p.W : 0;
    static const bool debug_plan = getenv("DBSP_DEBUG_PLAN") != nullptr;
    if (debug_plan) {
      fprintf(stderr, "[dbsp plan] n=%llu L=%d W=%d neq=%llx inv0=%llu bits:", (unsigned long long)n, L, p.W, (unsigned long long)neq,
              (unsigned long long)mm[2 * L + 4]);
      for (int l = 0; l < L; l++) fprintf(stderr, " %d%s", (int)p.bits[l], p.alias[l] >= 0 ? "a" : "");
      fprintf(stderr, "\n");
    }
    TRY(dev_alloc(ctx, (size_t)n * 8 * 2 * (p.W == 2 ? 2 : 1), &kbuf));
    TRY(dev_alloc(ctx, (size_t)n * 4 * 2, &ibuf));
  }
  u64* const kbufs[2] = {kbuf ? (u64*)kbuf->p : nullptr, kbuf ? (u64*)kbuf->p + n : nullptr};
  u64* const k1bufs[2] = {(kbuf && p.W == 2) ? (u64*)kbuf->p + 2 * n : nullptr, (kbuf && p.W == 2) ? (u64*)kbuf->p + 3 * n : nullptr};
  u32* const ibufs[2] = {ibuf ? (u32*)ibuf->p : nullptr, ibuf ? (u32*)ibuf->p + n : nullptr};
  u64* const cnt = lane(ctx).d_scratch + 32;   // [0] output rows, [2] sort-fallback flag
  const u64* key1_sorted = nullptr;
  // lane 0 ordered on arrival (event tables come in time order): the top bits[0] bits of the key are non-decreasing
  // already, the sort needs no HBM pass (sort.cu)
  const int presorted = (p.W <= 2 && n_inv != 0 && mm[2 * L + 4] == 0) ? (int)p.bits[0] : 0;

  auto sort_rows = [&](bool force_lsd) -> int32_t {
    idx_cur = nullptr;
    if (p.W <= 2) {
      // one- or two-word keys: pack once, one sort over the whole key
      {
        ProfScope ps(ctx, KID_PACK, n * (u64)L * 8 + n * (u64)(8 * p.W + 4));
        k_pack12<<<nblk, TB, 0, st>>>(cols, p, n, kbufs[0], k1bufs[0], ibufs[0]);
      }
      LAUNCH_COUNT(ctx);
      int which = 0;
      TRY(radix_sort_pairs(ctx, p.W, kbufs[0], kbufs[1], k1bufs[0], k1bufs[1], ibufs[0], ibufs[1], n, (int)p.wbits[0],
                           p.W == 2 ? (int)p.wbits[1] : 0, presorted, force_lsd, (unsigned long long*)(cnt + 2), &which, nullptr));
      key_sorted = kbufs[which];
      key1_sorted = k1bufs[which];
      idx_cur = ibufs[which];
      return DBSP_OK;
    }
    // wider keys: word by word, least significant word first (every stage is stable)
    for (int wd = 0; wd < p.W; wd++) {
      // the keys of the previous word are dead: always pack into key buffer 0; the row ids stay where the
      // previous word's sort left them
      u64* kdst = kbufs[0];
      {
        ProfScope ps(ctx, KID_PACK, n * (u64)L * 8 + n * 12);
        if (wd == 0) {
          k_pack<<<nblk, TB, 0, st>>>(cols, p, wd, nullptr, n, kdst, ibufs[0]);
          idx_cur = ibufs[0];
        } else {
          k_pack<<<nblk, TB, 0, st>>>(cols, p, wd, idx_cur, n, kdst, nullptr);
        }
      }
      LAUNCH_COUNT(ctx);
      u32* iother = idx_cur == ibufs[0] ? ibufs[1] : ibufs[0];
      key_sorted = kdst;
      if (p.wbits[wd] > 0 && n > 1) {
        int which = 0;
        TRY(radix_sort_pairs(ctx, 1, kdst, kbufs[1], nullptr, nullptr, idx_cur, iother, n, (int)p.wbits[wd], 0, 0, force_lsd,
                             (unsigned long long*)(cnt + 2), &which, nullptr));
        key_sorted = which ? kbufs[1] : kdst;
        idx_cur = which ? iother : idx_cur;
      }
    }
    return DBSP_OK;
  };
  if (n_inv != 0) {
    CUDA_TRY(cudaMemsetAsync(cnt, 0, 24, st));
    TRY(sort_rows(false));
  }

  // ---- (4) epilogue: one pass — sum runs of equal rows, drop zero sums, build the batch -------
  const u32 ntiles = (u32)((n + RE_TILE - 1) / RE_TILE);
  BufP tbuf;
  TRY(dev_alloc(ctx, (size_t)ntiles * sizeof(ReStatus) + 16, &tbuf));
  ReStatus* status = (ReStatus*)tbuf->p;
  u32* ticket = (u32*)(status + ntiles);
  Batch* b = nullptr;
  MCols oc;
  i64* ow;
  TRY(batch_alloc(ctx, s, n, &b, &oc, &ow));   // capacity n: the exact count comes back with the kernel
  u64 res[3] = {0, 0, 0};
  Mail rmail_seq;
  for (int attempt = 0; attempt < 2; attempt++) {
    if (n_inv == 0) CUDA_TRY(cudaMemsetAsync(cnt, 0, 24, st));
    CUDA_TRY(cudaMemsetAsync(tbuf->p, 0, (size_t)ntiles * sizeof(ReStatus) + 16, st));
    {
      ProfScope pseg(ctx, KID_SEG_REDUCE, n * (u64)((p.use_key ? 8 * p.use_key + 4 : (L * 8 + (idx_cur ? 4 : 0))) + (w ? 8 : 0)) + n * (u64)(L + 1) * 8);
      const Mail rmail = mail_begin(ctx);
      k_reduce_emit<<<ntiles, RE_THREADS, 0, st>>>(cols, p, key_sorted, key1_sorted, idx_cur, w, n, status, ticket, oc, ow, cnt, rmail);
      LAUNCH_COUNT(ctx);
      rmail_seq = rmail;
    }
    int32_t rc = mail_finish(ctx, rmail_seq, res, 3);
    if (rc) { batch_unref(b); return rc; }
    if (res[2] == 0) break;
    // a bucket did not fit a shared-memory chunk (heavy key skew): redo the sort with the plain LSD sequence
    if (attempt == 1 || n_inv == 0) { batch_unref(b); set_error("consolidate: sort fallback failed"); return DBSP_ERR_CUDA; }
    CUDA_TRY(cudaMemsetAsync(cnt, 0, 24, st));
    rc = sort_rows(true);
    if (rc) { batch_unref(b); return rc; }
  }
  const u64 nout = res[0];
  if (nout == 0) { batch_unref(b); *out = batch_new_empty(ctx, s); return DBSP_OK; }
  b->n = nout;
  if (nout * 2 < n && n > 4096) {
    // heavy reduction: do not keep a capacity-n buffer alive behind a small batch
    Batch* small;
    MCols sc;
    i64* sw;
    int32_t rc = batch_alloc(ctx, s, nout, &small, &sc, &sw);
    if (rc) { batch_unref(b); return rc; }
    for (int l = 0; l < L; l++) cudaMemcpyAsync(sc.c[l], oc.c[l], nout * 8, cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(sw, ow, nout * 8, cudaMemcpyDeviceToDevice, st);
    batch_unref(b);
    b = small;
  }
  *out = b;
  return DBSP_OK;
}

// The epilogue alone: rows that are already in sorted order (equal rows adjacent) — sum the weights of equal rows,
// drop zero sums, build the batch.  One launch, one read-back.  Used by the receiver side of the exchange.
int32_t reduce_sorted_rows(Ctx* ctx, const dbsp_schema& s, const Cols& cols, const i64* w, u64 n, Batch** out) {
  const int L = s.n_key_lanes + s.n_val_lanes;
  if (n == 0) { *out = batch_new_empty(ctx, s); return DBSP_OK; }
  if (n >= (1ull << 32)) { set_error("reduce: more than 2^32-1 rows in one batch"); return DBSP_ERR_UNSUPPORTED; }
  cudaStream_t st = lane(ctx).stream;
  Plan p;
  memset(&p, 0, sizeof(p));
  p.L = L;
  p.W = 1;
  p.use_key = 0;
  for (int l = 0; l < MAXL; l++) p.alias[l] = -1;
  const u32 ntiles = (u32)((n + RE_TILE - 1) / RE_TILE);
  BufP tbuf;
  TRY(dev_alloc(ctx, (size_t)ntiles * sizeof(ReStatus) + 16, &tbuf));
  ReStatus* status = (ReStatus*)tbuf->p;
  u32* ticket = (u32*)(status + ntiles);
  u64* const cnt = lane(ctx).d_scratch + 32;
  Batch* b = nullptr;
  MCols oc;
  i64* ow;
  TRY(batch_alloc(ctx, s, n, &b, &oc, &ow));
  CUDA_TRY(cudaMemsetAsync(cnt, 0, 24, st));
  CUDA_TRY(cudaMemsetAsync(tbuf->p, 0, (size_t)ntiles * sizeof(ReStatus) + 16, st));
  const Mail rmail = mail_begin(ctx);
  {
    ProfScope pseg(ctx, KID_SEG_REDUCE, n * (u64)(L + 1) * 8 * 2);
    k_reduce_emit<<<ntiles, RE_THREADS, 0, st>>>(cols, p, nullptr, nullptr, nullptr, w, n, status, ticket, oc, ow, cnt, rmail);
  }
  LAUNCH_COUNT(ctx);
  u64 res[3];
  int32_t rc = mail_finish(ctx, rmail, res, 3);
  if (rc) { batch_unref(b); return rc; }
  if (res[0] == 0) { batch_unref(b); *out = batch_new_empty(ctx, s); return DBSP_OK; }
  b->n = res[0];
  *out = b;
  return DBSP_OK;
}

