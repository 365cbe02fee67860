// merge.cu — K3/K4: sorted 2-way merge of consolidated batches.
//
// Replaces ColumnLayerBuilder::push_merge
// (crates/dbsp/src/trace/layers/column_layer/builders.rs:98-169) and the
// two-level OrderedBuilder::merge_step / push_merge
// (trace/layers/ordered/mod.rs:344-396, 806-834): merging the flat
// (key lanes, val lanes) rows lexicographically is the same function as the
// reference's key-then-value-range merge; equal rows have their weights
// summed and zero sums are dropped.
//
// One pass over HBM.  A merge-path partition kernel cuts the merged sequence
// into tiles.  Each CTA first asks L2 to prefetch the inputs of a tile 148
// tiles ahead (cp.async.bulk.prefetch.L2), then stages the *lanes* of its A and
// B segments in shared memory with TMA bulk copies (cp.async.bulk + mbarrier:
// one thread issues 2*L copies, no registers, no per-thread address
// arithmetic).  Every thread merge-path-searches its own diagonal and serially
// merges IPT rows with both run heads in registers; kept rows are compacted as
// 16-bit slot ids, gathered and written back coalesced.  Weights: rows of one or
// two lanes stage them as one more lane (same TMA copies, partner sums folded in
// shared memory, coalesced stores); wider rows keep them out of shared memory
// (more rows in flight per SM) and fetch them in one batch of independent loads
// after the serial merge.  Because both inputs are consolidated, an equal pair
// is always (a, b) adjacent in merged order: the A row absorbs its partner's
// weight, the B row is skipped — also across thread and tile boundaries (one
// halo row on each side).  The tile's global output offset comes from a
// decoupled look-back over per-tile status words (tile index = an arrival
// ticket, so predecessors are always resident or done).
// Tile shapes, register caps, look-back width and prefetch distance were swept
// on the B200 (DESIGN.md §9, profiles/README.md).
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "common.cuh"

namespace {

#ifndef MERGE_THREADS_CFG
#define MERGE_THREADS_CFG 256
#endif
#ifndef MERGE_THREADS_NARROW
#define MERGE_THREADS_NARROW 128   // threads per CTA for two-lane rows (swept: 128 x 9 rows, weights staged: 63.0 -> 64.9 %)
#endif
#ifndef MERGE_NARROW_MAX
#define MERGE_NARROW_MAX 2   // rows up to this many lanes use the branch-free (select) search and serial merge
#endif
#ifndef MERGE_IPT_CFG
#define MERGE_IPT_CFG 9      // rows per thread, 1-2 lanes
#endif
#ifndef MERGE_IPT_MID
#define MERGE_IPT_MID 5      // rows per thread, 3-6 lanes
#endif
#ifndef MERGE_IPT_WIDE
#define MERGE_IPT_WIDE 3     // rows per thread, 7-8 lanes
#endif
#ifndef MERGE_L2_PREFETCH
#define MERGE_L2_PREFETCH 148   // tiles ahead whose inputs are prefetched into L2 (0 = off; swept: 148 > 444 > 740 > off)
#endif
#ifndef MERGE_LB_THREADS
#define MERGE_LB_THREADS 32   // look-back window: predecessor tiles inspected per round trip (measured: 32 > 64 > 128 > 256)
#endif
#ifndef MERGE_STAGE_W_MAXL
#define MERGE_STAGE_W_MAXL 2   // rows up to this many lanes stage their weights in shared memory as one more lane (0 = never;
                               // swept on the B200: 1 lane 48 -> 60 % of the HBM peak; 2 lanes 63 -> 61 % with 256
                               // threads, 64.9 % with 128 threads x 9 rows)
#endif
constexpr u64 ST_AGG = 1ull << 62, ST_PREFIX = 2ull << 62, ST_MASK = (1ull << 62) - 1;

// status words carry flag and value in one 64-bit word: relaxed device-scope
// accesses (L2, never a stale L1 line) are all the protocol needs
__device__ __forceinline__ u64 ld_relaxed(const u64* p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(u64* p, u64 v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
  unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gsrc, unsigned bytes, u64* mbar) {
  unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  unsigned m = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d),
               "l"(gsrc), "r"(bytes), "r"(m)
               : "memory");
}
// L2 prefetch of the 16-byte granules inside [p, p + bytes) (never past either end)
__device__ __forceinline__ void l2_prefetch(const void* p, u64 bytes) {
  const u64 a = ((u64)(size_t)p + 15ull) & ~15ull;
  const u64 e = ((u64)(size_t)p + bytes) & ~15ull;
  if (e > a) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"((unsigned)(e - a)) : "memory");
}
__device__ __forceinline__ void mbar_init(u64* mbar, unsigned count) {
  unsigned m = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(m), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64* mbar, unsigned bytes) {
  unsigned m = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(m), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64* mbar, unsigned parity) {
  unsigned m = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(m),
      "r"(parity)
      : "memory");
}

template <int L>
struct MergeCfg {
  // rows of one or two lanes (OrdZSet<u64>, OrdIndexedZSet<u64,u64>): the
  // configuration swept on the B200 (profiles/README.md) — 256 threads x 9 rows,
  // 5 CTAs/SM, selects instead of branches in search and serial merge
  static constexpr bool NARROW = L <= MERGE_NARROW_MAX;
  // odd rows/thread: the per-thread serial merge walks shared memory with a
  // stride of IPT 64-bit words between lanes of a warp -> bank-conflict free
  static constexpr int IPT = (L <= 2) ? MERGE_IPT_CFG : (L <= 6 ? MERGE_IPT_MID : MERGE_IPT_WIDE);
  static constexpr int THREADS = (L == 2) ? MERGE_THREADS_NARROW : MERGE_THREADS_CFG;
  static constexpr int TILE = THREADS * IPT;
  static constexpr int S = TILE + 8;   // staged slots per array (even; room for alignment slack + halos)
  // STAGE_W: the weights travel like one more lane — staged by the same TMA copies, summed with their partner in
  // shared memory, gathered with the kept rows and stored coalesced (no per-thread strided weight loads / stores).
  // Otherwise shared memory holds the staged lanes and 16-bit slot ids only, and the weights are read from and
  // written to HBM by the threads that need them (more rows in flight per SM).
  static constexpr bool STAGE_W = L <= MERGE_STAGE_W_MAXL;
  static constexpr int LS = L + (STAGE_W ? 1 : 0);   // staged arrays
  static constexpr size_t SMEM = (size_t)S * LS * 8 + (size_t)TILE * 2;
};

// a-count of the merge path at diagonal d: number of A rows among the first d
// merged rows (ties: A first).
template <int L>
__device__ __forceinline__ u64 diag_search_g(const Cols& A, u64 nA, const Cols& B, u64 nB, const Flips& f, u64 d) {
  u64 lo = d > nB ? d - nB : 0, hi = d < nA ? d : nA;
  while (lo < hi) {
    u64 mid = (lo + hi) >> 1;
    u64 j = d - 1 - mid;
    bool le = true;   // A[mid] <= B[j] ?
#pragma unroll
    for (int l = 0; l < L; l++) {
      u64 a = A.c[l][mid] ^ f.f[l], b = B.c[l][j] ^ f.f[l];
      if (a != b) { le = a < b; break; }
    }
    if (le) lo = mid + 1; else hi = mid;
  }
  return lo;
}

template <int L>
__global__ void k_merge_partition(Cols A, u64 nA, Cols B, u64 nB, Flips f, u32 tile, u32 ntiles, u64* part) {
  u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > ntiles) return;
  u64 total = nA + nB;
  u64 d = (u64)t * tile;
  if (d > total) d = total;
  part[t] = diag_search_g<L>(A, nA, B, nB, f, d);
}

// One merge-path split for the fuelled Merger: out[0] = a-count at diagonal d,
// out[1] = 1 when the cut would separate an equal pair (A[a-1] == B[d-a]): the
// caller then takes one more B row so that the pair's weights meet in one chunk.
template <int L>
__global__ void k_merge_split(Cols A, u64 nA, Cols B, u64 nB, Flips f, u64 d, u64* out) {
  u64 a = diag_search_g<L>(A, nA, B, nB, f, d);
  u64 j = d - a;
  u64 pair = 0;
  if (a > 0 && j < nB) {
    pair = 1;
#pragma unroll
    for (int l = 0; l < L; l++)
      if (A.c[l][a - 1] != B.c[l][j]) { pair = 0; break; }
  }
  out[0] = a;
  out[1] = pair;
}

// Scratch shared by the phases of one tile (static shared memory of the kernel).
struct TileScratch {
  u64* s_base;
  u32* s_warp;
  int* s_lb_first;
  u64* s_lb_all;
  u64* s_lb_upto;
};

// Everything after staging: per-thread merge path, serial merge, compaction,
// decoupled look-back, coalesced stores.  `sl` holds the staged lanes with the
// slot map of k_merge_tiles (A row a0+i at oa+i, B row b0+j at ob+j); `wAg` /
// `wBg` are the weight arrays offset to a0 / b0.  Input weights are never zero
// (batch invariant), so only a partner sum can cancel: the weight loads stay
// off the serial merge's critical path.
template <int L>
__device__ __forceinline__ void merge_process_tile(u64* sl, const i64* __restrict__ wAg, const i64* __restrict__ wBg,
                                                   unsigned short* perm, const int oa, const int ob, const int na,
                                                   const int nb, const bool has_prev, const bool has_next, const u32 t,
                                                   const u32 ntiles, u64* status, const MCols& O, i64* wO, u64* n_out,
                                                   const Flips& f, const TileScratch& sc, const Mail& mail) {
  constexpr int IPT = MergeCfg<L>::IPT;
  constexpr int S = MergeCfg<L>::S;
  const int tid = threadIdx.x;
  u64& s_base = *sc.s_base;
  u32* s_warp = sc.s_warp;
  int* s_lb_first = sc.s_lb_first;
  u64* s_lb_all = sc.s_lb_all;
  u64* s_lb_upto = sc.s_lb_upto;
  auto le = [&](int ia, int ib) {   // staged row ia <= staged row ib
    if constexpr (MergeCfg<L>::NARROW) {   // all lanes loaded at once, no branches
      u64 a[L], b[L];
#pragma unroll
      for (int l = 0; l < L; l++) { a[l] = sl[l * S + ia]; b[l] = sl[l * S + ib]; }
      bool r = true;
#pragma unroll
      for (int l = L - 1; l >= 0; l--) r = (a[l] < b[l]) | ((a[l] == b[l]) & r);
      return r;
    } else {
      bool r = true, open = true;   // first differing lane decides
#pragma unroll
      for (int l = 0; l < L; l++) {
        if (open) {
          u64 a = sl[l * S + ia], b = sl[l * S + ib];
          if (a != b) { r = a < b; open = false; }
        }
      }
      return r;
    }
  };

  // ---- per-thread merge path ------------------------------------------------
  const int n = na + nb;
  int dt = tid * IPT;
  if (dt > n) dt = n;
  int lo = dt > nb ? dt - nb : 0, hi = dt < na ? dt : na;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (le(oa + mid, ob + (dt - 1 - mid))) lo = mid + 1; else hi = mid;
  }
  int ai = lo, bi = dt - lo;

  // Serial merge with both run heads held in registers: one 3-way compare per
  // row, only the advanced side is re-read from shared memory.  `prev_eq`
  // says the previous merged row was an A row equal to the current B head.
  // The loop touches shared memory only; weights are fetched afterwards in one
  // batch of independent loads.
  u64 ka[L], kb[L];
  auto load_a = [&](int i) {
#pragma unroll
    for (int l = 0; l < L; l++) ka[l] = sl[l * S + oa + i];
  };
  auto load_b = [&](int j) {
#pragma unroll
    for (int l = 0; l < L; l++) kb[l] = sl[l * S + ob + j];
  };
  bool b_readable = (bi < nb) || (bi == nb && has_next);
  if (ai < na) load_a(ai);
  if (b_readable) load_b(bi);
  bool prev_eq = false;
  if ((ai > 0 || has_prev) && bi < nb) {   // A[ai-1] (slot oa+ai-1; halo at oa-1) vs B head
    prev_eq = true;
#pragma unroll
    for (int l = 0; l < L; l++) prev_eq = prev_eq && (sl[l * S + oa + ai - 1] == kb[l]);
  }

  u32 src[IPT];
  u32 keep = 0, pmask = 0;   // pmask bit k: row k is an A row whose equal B partner follows it
  if constexpr (MergeCfg<L>::NARROW) {
    // Narrow rows: branch-free formulation — every lane of the warp executes the
    // same instruction stream whichever side it consumes (selects instead of
    // divergent take-A / take-B paths).
#pragma unroll
    for (int k = 0; k < IPT; k++) {
    const bool valid = ai + bi < n;
    const bool a_ok = ai < na, b_in = bi < nb;
    bool lt = false, eq = true;   // A head < / == B head (meaningful when both are readable)
#pragma unroll
    for (int l = L - 1; l >= 0; l--) {
      lt = (ka[l] < kb[l]) | ((ka[l] == kb[l]) & lt);
      eq = eq & (ka[l] == kb[l]);
    }
    const bool both = a_ok & b_readable;
    const bool take_a = !b_in | (a_ok & (!both | lt | eq));
    const bool partner = take_a & b_readable & eq;
    src[k] = take_a ? (u32)(oa + ai) : (u32)(ob + bi);
    keep |= (u32)(valid & (take_a | !prev_eq)) << k;
    pmask |= (u32)(valid & partner) << k;
    prev_eq = valid ? partner : prev_eq;
    ai += (valid & take_a) ? 1 : 0;
    bi += (valid & !take_a) ? 1 : 0;
    b_readable = (bi < nb) | ((bi == nb) & has_next);
    const bool ld_ok = valid & (take_a ? (ai < na) : b_readable);
    const int slot = take_a ? (oa + ai) : (ob + bi);
    if (ld_ok) {
#pragma unroll
      for (int l = 0; l < L; l++) {
        const u64 nv = sl[l * S + slot];
        ka[l] = take_a ? nv : ka[l];
        kb[l] = take_a ? kb[l] : nv;
      }
    }
    }
  } else {
    // Wide rows: the selects would cost 2 * L moves per row; branch instead.
#pragma unroll
    for (int k = 0; k < IPT; k++) {
    src[k] = 0;
    if (ai + bi < n) {
      const bool a_ok = ai < na, b_in = bi < nb;
      int c = 0;   // cmp3(A head, B head) when both are readable
      if (a_ok && b_readable) {
#pragma unroll
        for (int l = 0; l < L; l++) {
          if (c == 0 && ka[l] != kb[l]) c = ka[l] < kb[l] ? -1 : 1;
        }
      }
      const bool take_a = !b_in || (a_ok && c <= 0);
      if (take_a) {
        const bool partner = b_readable && c == 0;
        src[k] = oa + ai;
        keep |= 1u << k;
        if (partner) pmask |= 1u << k;
        prev_eq = partner;
        ai++;
        if (ai < na) load_a(ai);
      } else {
        src[k] = ob + bi;
        if (!prev_eq) keep |= 1u << k;
        prev_eq = false;
        bi++;
        b_readable = (bi < nb) || (bi == nb && has_next);
        if (b_readable) load_b(bi);
      }
    }
    }
  }

  // ---- weights: one batch of independent global loads --------------------------
  // Row k's weight sits at wA[a0 + slot - oa] or wB[b0 + slot - ob].  The partner
  // of an A row is the next merged row: row k+1 of this thread, or — for the
  // thread's last row — the B head left over after the loop (possibly the first
  // row of the next thread / tile).  Input weights are never zero (batch
  // invariant), so only a partner sum can cancel.
  constexpr bool STAGE_W = MergeCfg<L>::STAGE_W;
  u64* const sw = sl + (size_t)L * S;   // staged weights (STAGE_W only)
  i64 wv[STAGE_W ? 1 : IPT];
  if constexpr (STAGE_W) {
    // An A row with a partner is owned by this thread and its partner (a B row: the next merged row) is never
    // written by anyone, so the sum can be folded into the A row's slot in place.
    if (pmask) {   // rare
#pragma unroll
      for (int k = 0; k < IPT; k++) {
        if (pmask & (1u << k)) {
          const u32 ps = (k + 1 < IPT && dt + k + 1 < n) ? src[k + 1 < IPT ? k + 1 : k] : (u32)(ob + bi);
          const u64 sum = sw[src[k]] + sw[ps];
          if (sum == 0) keep &= ~(1u << k);
          else sw[src[k]] = sum;
        }
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < IPT; k++) {
      wv[k] = 0;
      if (dt + k < n) {
        const int s = (int)src[k];
        wv[k] = (s >= ob) ? wBg[s - ob] : wAg[s - oa];
      }
    }
    if (pmask) {   // rare
      const i64 wlast = prev_eq ? wBg[bi] : 0;
#pragma unroll
      for (int k = 0; k < IPT; k++) {
        if (pmask & (1u << k)) {
          const i64 pw = (k + 1 < IPT && dt + k + 1 < n) ? wv[k + 1 < IPT ? k + 1 : k] : wlast;
          wv[k] = (i64)((u64)wv[k] + (u64)pw);
          if (wv[k] == 0) keep &= ~(1u << k);
        }
      }
    }
  }

  // ---- block exclusive scan of kept counts ------------------------------------
  const u32 cnt = __popc(keep);
  u32 incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    u32 v = __shfl_up_sync(0xffffffffu, incl, o);
    if ((tid & 31) >= o) incl += v;
  }
  if ((tid & 31) == 31) s_warp[tid >> 5] = incl;
  __syncthreads();
  u32 warp_off = 0, tile_total = 0;
#pragma unroll
  for (int wi = 0; wi < MergeCfg<L>::THREADS / 32; wi++) {
    u32 v = s_warp[wi];
    if (wi < (tid >> 5)) warp_off += v;
    tile_total += v;
  }
  u32 off = warp_off + incl - cnt;

  // ---- compact kept rows in shared memory -------------------------------------------
#pragma unroll
  for (int k = 0; k < IPT; k++) {
    if (keep & (1u << k)) {
      perm[off] = (unsigned short)src[k];
      off++;
    }
  }

  // ---- decoupled look-back for the tile's global output offset -------------------
  // The first LBT threads of the CTA inspect LBT predecessor status words per
  // round trip (tile p - tid per thread); aggregates of tiles that have not
  // resolved their own prefix yet are summed on the way.
  if (t == 0) {
    if (tid == 0) { st_relaxed(&status[0], ST_PREFIX | (u64)tile_total); s_base = 0; }
  } else {
    if (tid == 0) st_relaxed(&status[t], ST_AGG | (u64)tile_total);
    constexpr int LBT = MERGE_LB_THREADS < MergeCfg<L>::THREADS ? MERGE_LB_THREADS : MergeCfg<L>::THREADS;
    constexpr int NW = LBT / 32;
    u64 base_acc = 0;
    long long p = (long long)t - 1;   // window = tiles p, p-1, ..., p-(LBT-1)
    while (true) {
      if (tid < LBT) {
        const long long q = p - tid;
        u64 v = ST_PREFIX;               // tiles before 0 contribute an empty prefix
        if (q >= 0) {
          do { v = ld_relaxed(&status[q]); } while ((v >> 62) == 0);
        }
        const unsigned is_prefix = __ballot_sync(0xffffffffu, (v >> 62) == 2);
        const int wfirst = is_prefix ? (__ffs(is_prefix) - 1) : 32;
        u64 all = v & ST_MASK, upto = ((tid & 31) <= wfirst) ? (v & ST_MASK) : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          all += __shfl_xor_sync(0xffffffffu, all, o);
          upto += __shfl_xor_sync(0xffffffffu, upto, o);
        }
        if ((tid & 31) == 0) {
          s_lb_first[tid >> 5] = wfirst;
          s_lb_all[tid >> 5] = all;
          s_lb_upto[tid >> 5] = upto;
        }
      }
      __syncthreads();
      bool found = false;
      u64 add = 0;
#pragma unroll
      for (int wi = 0; wi < NW; wi++) {
        if (!found) {
          if (s_lb_first[wi] < 32) { add += s_lb_upto[wi]; found = true; }
          else add += s_lb_all[wi];
        }
      }
      base_acc += add;
      __syncthreads();   // s_lb_* are rewritten by the next window
      if (found) break;
      p -= LBT;
    }
    if (tid == 0) {
      st_relaxed(&status[t], ST_PREFIX | (base_acc + tile_total));
      s_base = base_acc;
    }
  }
  if (tid == 0 && t == ntiles - 1) {
    const u64 tot = s_base + tile_total;
    *n_out = tot;
    mail_publish(mail, &tot, 1);   // the output count goes straight to the host mailbox
  }
  __syncthreads();
  const u64 base = s_base;
  for (u32 o = tid; o < tile_total; o += MergeCfg<L>::THREADS) {
    u32 s = perm[o];
#pragma unroll
    for (int l = 0; l < L; l++) O.c[l][base + o] = sl[l * S + s] ^ f.f[l];
    if constexpr (STAGE_W) wO[base + o] = (i64)sw[s];
  }
  if constexpr (!STAGE_W) {   // weights: straight from registers to the thread's own (contiguous) output slots
    u64 wpos = base + (off - cnt);
#pragma unroll
    for (int k = 0; k < IPT; k++) {
      if (keep & (1u << k)) wO[wpos++] = wv[k];
    }
  }
}

// min CTAs/SM: narrow rows stage 41 KB per CTA -> 5 CTAs/SM, which caps the
// kernel at 48 registers (an uncapped schedule measured 2.5x slower)
#ifndef MERGE_MIN_CTAS
#define MERGE_MIN_CTAS 5
#endif
#ifndef MERGE_CTAS_MID
#define MERGE_CTAS_MID 6   // 3-4 lanes, swept: 3 -> 41 %, 6 -> 60 % of the HBM peak on 3-lane rows (register cap 40)
#endif
#ifndef MERGE_CTAS_WIDE
#define MERGE_CTAS_WIDE 4   // 5-8 lanes (5 lanes x 5 rows: 46 -> 61 %; 8 lanes x 3 rows: 57 %)
#endif
#ifndef MERGE_CTAS_L2
#define MERGE_CTAS_L2 7   // two-lane rows: 128 threads, 30 KB staged per CTA
#endif
#define MERGE_MIN_CTAS_FOR(L) ((L) == 1 ? MERGE_MIN_CTAS : ((L) == 2 ? MERGE_CTAS_L2 : ((L) <= 4 ? MERGE_CTAS_MID : MERGE_CTAS_WIDE)))
template <int L>
__global__ void __launch_bounds__(MergeCfg<L>::THREADS, MERGE_MIN_CTAS_FOR(L))
k_merge_tiles(Cols A, const i64* __restrict__ wA, u64 nA, Cols B, const i64* __restrict__ wB, u64 nB, Flips f,
              const u64* __restrict__ part, u32 ntiles, u64* status, MCols O, i64* wO, u64* n_out,
              int use_tma, Mail mail, u32* ticket) {
  constexpr int IPT = MergeCfg<L>::IPT;
  constexpr int TILE = MergeCfg<L>::TILE;
  constexpr int S = MergeCfg<L>::S;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  u64* sl = (u64*)smem_raw;                                   // L lanes of S staged slots
  unsigned short* perm = (unsigned short*)(sl + (size_t)MergeCfg<L>::LS * S);   // TILE staged-slot ids of kept rows
  __shared__ __align__(8) u64 s_mbar;
  __shared__ u64 s_base;
  __shared__ u32 s_warp[MergeCfg<L>::THREADS / 32];
  __shared__ int s_lb_first[MergeCfg<L>::THREADS / 32];
  __shared__ u64 s_lb_all[MergeCfg<L>::THREADS / 32], s_lb_upto[MergeCfg<L>::THREADS / 32];

  const int tid = threadIdx.x;
  // Tile index = arrival ticket: every predecessor a look-back waits on has taken its ticket earlier and is
  // therefore resident or finished — a forward-progress guarantee that does not rely on the order in which the
  // hardware dispatches blocks (MPS, preemption, compute-sanitizer).
  __shared__ u32 s_ticket;
  if (tid == 0) {
    s_ticket = atomicAdd(ticket, 1u);
    mbar_init(&s_mbar, 1);
  }
  __syncthreads();
  const u32 t = s_ticket;
  const u64 total = nA + nB;
  const u64 d0 = (u64)t * TILE;
  const u64 d1 = (d0 + TILE < total) ? d0 + TILE : total;
  const u64 a0 = part[t], a1 = part[t + 1];
  const u64 b0 = d0 - a0, b1 = d1 - a1;
  const int na = (int)(a1 - a0), nb = (int)(b1 - b0);
  const bool has_prev = a0 > 0, has_next = b1 < nB;
#if MERGE_L2_PREFETCH
  // Pull the inputs of the tile that will follow in this CTA slot (about one CTA
  // lifetime from now) into L2, so that its TMA staging does not wait on HBM.
  if (tid == 32 && t + MERGE_L2_PREFETCH < ntiles) {
    const u64 pa0 = part[t + MERGE_L2_PREFETCH], pa1 = part[t + MERGE_L2_PREFETCH + 1];
    const u64 pd0 = (u64)(t + MERGE_L2_PREFETCH) * TILE;
    const u64 pd1 = (pd0 + TILE < total) ? pd0 + TILE : total;
    const u64 pb0 = pd0 - pa0, pb1 = pd1 - pa1;
#pragma unroll
    for (int l = 0; l < L; l++) {
      l2_prefetch(A.c[l] + pa0, (pa1 - pa0) * 8);
      l2_prefetch(B.c[l] + pb0, (pb1 - pb0) * 8);
    }
    l2_prefetch(wA + pa0, (pa1 - pa0) * 8);
    l2_prefetch(wB + pb0, (pb1 - pb0) * 8);
  }
#endif
  bool any_flip = false;
#pragma unroll
  for (int l = 0; l < L; l++) any_flip = any_flip || (f.f[l] != 0);

  // ---- stage --------------------------------------------------------------------
  // Slot map: A row a0+i lives at slot oa+i (i = -1 is the A halo), B row b0+j at
  // slot ob+j (j = nb is the B halo).  The TMA path copies 16-byte aligned
  // super-ranges, which fixes oa/ob; the fallback uses oa = 1, ob = 1+na.
  int oa, ob;
  if (use_tma) {
    const long long fa = (long long)a0 - (has_prev ? 1 : 0);          // first A row needed
    const long long pa = (long long)(((unsigned long long)(size_t)A.c[0]) >> 3) & 1;
    const long long ga = fa - ((fa + pa) & 1);                        // aligned-down start (may be -1)
    const long long ea = (long long)a1;                               // end (exclusive)
    const int ca = (ea > fa) ? (int)(((ea - ga) + 1) & ~1ll) : 0;     // rows copied (even)
    oa = (int)((long long)a0 - ga);
    const int sb = (oa + na + 1) & ~1;                                // first slot of the B region (even)
    const long long eb = (long long)b1 + (has_next ? 1 : 0);
    const long long pb = (long long)(((unsigned long long)(size_t)B.c[0]) >> 3) & 1;
    const long long gb = (long long)b0 - (((long long)b0 + pb) & 1);
    const int cb = (eb > (long long)b0) ? (int)(((eb - gb) + 1) & ~1ll) : 0;
    ob = sb + (int)((long long)b0 - gb);
    if (tid == 0) {
      const unsigned bytes = (unsigned)(ca + cb) * 8u * MergeCfg<L>::LS;
      if (bytes) {
        mbar_expect_tx(&s_mbar, bytes);
        if (ca) {
#pragma unroll
          for (int l = 0; l < L; l++) tma_bulk_g2s(sl + l * S, A.c[l] + ga, (unsigned)ca * 8u, &s_mbar);
          if constexpr (MergeCfg<L>::STAGE_W) tma_bulk_g2s(sl + L * S, wA + ga, (unsigned)ca * 8u, &s_mbar);
        }
        if (cb) {
#pragma unroll
          for (int l = 0; l < L; l++) tma_bulk_g2s(sl + l * S + sb, B.c[l] + gb, (unsigned)cb * 8u, &s_mbar);
          if constexpr (MergeCfg<L>::STAGE_W) tma_bulk_g2s(sl + L * S + sb, wB + gb, (unsigned)cb * 8u, &s_mbar);
        }
      }
    }
    if ((ca + cb) > 0) mbar_wait(&s_mbar, 0);
  } else {
    oa = 1;
    ob = 1 + na;
    const int nslots = na + nb + 2;
#pragma unroll
    for (int k = 0; k < IPT + 1; k++) {
      const int x = tid + k * MergeCfg<L>::THREADS;
      if (x < nslots) {
        const bool from_a = x <= na;
        const bool skip = (x == 0 && !has_prev) || (x == nslots - 1 && !has_next);
        if (!skip) {
          const u64 g = from_a ? (a0 + x - 1) : (b0 + (x - 1 - na));
#pragma unroll
          for (int l = 0; l < L; l++) cp_async8(&sl[l * S + x], (from_a ? A.c[l] : B.c[l]) + g);
          if constexpr (MergeCfg<L>::STAGE_W) cp_async8(&sl[L * S + x], (from_a ? wA : wB) + g);
        }
      }
    }
    cp_async_wait_all();
  }
  if (any_flip) {   // i64 lanes: stage the order-preserving image
    __syncthreads();
    for (int x = tid; x < S; x += MergeCfg<L>::THREADS) {
#pragma unroll
      for (int l = 0; l < L; l++) sl[l * S + x] ^= f.f[l];
    }
  }
  __syncthreads();

  TileScratch sc{&s_base, s_warp, s_lb_first, s_lb_all, s_lb_upto};
  merge_process_tile<L>(sl, wA + a0, wB + b0, perm, oa, ob, na, nb, has_prev, has_next, t, ntiles, status, O, wO, n_out, f, sc, mail);
}


// all lanes of the batch share the 16-byte phase of element 0 (lanes of one
// allocation always do): precondition of the TMA path
bool uniform_phase(const Batch* b) {
  size_t ph = ((size_t)b->col[0] >> 3) & 1;
  for (int l = 1; l < b->nl(); l++)
    if ((((size_t)b->col[l] >> 3) & 1) != ph) return false;
  // the weights ride along with the lanes when they are staged
  return b->nl() > MERGE_STAGE_W_MAXL || (((size_t)b->w >> 3) & 1) == ph;
}

template <int L>
int32_t merge_launch(Ctx* ctx, const Batch* a, const Batch* b, Batch** out) {
  typedef MergeCfg<L> Cfg;
  cudaStream_t st = lane(ctx).stream;
  u64 total = a->n + b->n;
  u32 ntiles = (u32)((total + Cfg::TILE - 1) / Cfg::TILE);
  BufP aux;
  // part[ntiles+1] u64 | status[ntiles] u64 | n_out u64 | ticket u64
  size_t aux_u64 = (size_t)(ntiles + 1) + ntiles + 2;
  TRY(dev_alloc(ctx, aux_u64 * 8, &aux));
  u64* part = (u64*)aux->p;
  u64* status = part + (ntiles + 1);
  u64* n_out = status + ntiles;
  CUDA_TRY(cudaMemsetAsync(status, 0, (size_t)(ntiles + 2) * 8, st));
  Batch* o;
  MCols oc;
  i64* ow;
  TRY(batch_alloc(ctx, a->s, total, &o, &oc, &ow));
  Flips f = a->flips();
  // per *device* attribute and cheap: set on every launch (a process may drive several GPUs)
  CUDA_TRY(cudaFuncSetAttribute(k_merge_tiles<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
  static const bool tma_off = getenv("DBSP_MERGE_NO_TMA") != nullptr;
  const int use_tma = (!tma_off && uniform_phase(a) && uniform_phase(b)) ? 1 : 0;
  {
    ProfScope ps(ctx, KID_MERGE_PARTITION, (u64)(ntiles + 1) * 8);
    k_merge_partition<L><<<(ntiles + 1 + 127) / 128, 128, 0, st>>>(a->cols(), a->n, b->cols(), b->n, f, Cfg::TILE, ntiles, part);
  }
  ProfScope* ps = new ProfScope(ctx, KID_MERGE, 0);
  const Mail mail = mail_begin(ctx);
  k_merge_tiles<L><<<ntiles, MergeCfg<L>::THREADS, Cfg::SMEM, st>>>(a->cols(), a->w, a->n, b->cols(), b->w, b->n, f, part, ntiles,
                                                           status, oc, ow, n_out, use_tma, mail, (u32*)(n_out + 1));
  long ps_idx = ps->idx;
  delete ps;   // records the end event
  ctx->kernel_launches += 2;
  u64 nout;
  int32_t rc = mail_finish(ctx, mail, &nout, 1);
  if (rc != DBSP_OK) { batch_unref(o); return rc; }
  // algorithmic bytes: every input row read once, every output row written once
  if (ps_idx >= 0) lane(ctx).prof[ps_idx].bytes = (total + nout) * (u64)(L + 1) * 8;
  o->n = nout;
  if (nout == 0) { batch_unref(o); o = batch_new_empty(ctx, a->s); }
  *out = o;
  return DBSP_OK;
}

template <int L>
int32_t split_launch(Ctx* ctx, const Batch* a, const Batch* b, u64 d, u64* na, u64* nb) {
  u64* dout = lane(ctx).d_scratch + 124;
  k_merge_split<L><<<1, 1, 0, lane(ctx).stream>>>(a->cols(), a->n, b->cols(), b->n, a->flips(), d, dout);
  ctx->kernel_launches++;
  u64 h[2];
  TRY(read_back(ctx, dout, 2, h));
  *na = h[0];
  *nb = d - h[0] + h[1];
  return DBSP_OK;
}

}  // namespace

// Rows of a and b among the first d rows of merge(a, b) (never separating an
// equal pair): the chunk boundary of a fuelled merge.
int32_t merge_path_split(Ctx* ctx, const Batch* a, const Batch* b, u64 d, u64* na, u64* nb) {
  if (d >= a->n + b->n) { *na = a->n; *nb = b->n; return DBSP_OK; }
  if (a->n == 0) { *na = 0; *nb = d; return DBSP_OK; }
  if (b->n == 0) { *na = d; *nb = 0; return DBSP_OK; }
  switch (a->nl()) {
    case 1: return split_launch<1>(ctx, a, b, d, na, nb);
    case 2: return split_launch<2>(ctx, a, b, d, na, nb);
    case 3: return split_launch<3>(ctx, a, b, d, na, nb);
    case 4: return split_launch<4>(ctx, a, b, d, na, nb);
    case 5: return split_launch<5>(ctx, a, b, d, na, nb);
    case 6: return split_launch<6>(ctx, a, b, d, na, nb);
    case 7: return split_launch<7>(ctx, a, b, d, na, nb);
    case 8: return split_launch<8>(ctx, a, b, d, na, nb);
  }
  set_error("merge: unsupported lane count");
  return DBSP_ERR_UNSUPPORTED;
}

int32_t merge_batches(Ctx* ctx, const Batch* a, const Batch* b, Batch** out) {
  if (a->nl() != b->nl() || memcmp(&a->s, &b->s, sizeof(dbsp_schema)) != 0) {
    set_error("merge: schema mismatch");
    return DBSP_ERR_INVALID;
  }
  if (a->n == 0) { batch_ref((Batch*)b); *out = (Batch*)b; return DBSP_OK; }
  if (b->n == 0) { batch_ref((Batch*)a); *out = (Batch*)a; return DBSP_OK; }
  switch (a->nl()) {
    case 1: return merge_launch<1>(ctx, a, b, out);
    case 2: return merge_launch<2>(ctx, a, b, out);
    case 3: return merge_launch<3>(ctx, a, b, out);
    case 4: return merge_launch<4>(ctx, a, b, out);
    case 5: return merge_launch<5>(ctx, a, b, out);
    case 6: return merge_launch<6>(ctx, a, b, out);
    case 7: return merge_launch<7>(ctx, a, b, out);
    case 8: return merge_launch<8>(ctx, a, b, out);
  }
  set_error("merge: unsupported lane count");
  return DBSP_ERR_UNSUPPORTED;
}
