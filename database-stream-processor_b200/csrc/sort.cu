// sort.cu — the sort inside Batch::from_tuples (K1): hand-written radix / sample sort of (packed key, row id) pairs.
//
// Replaces the comparison sort of consolidation (crates/dbsp/src/trace/consolidation/mod.rs:92-111: "90% of the
// work done while joining or merging"; consolidation/quicksort.rs:12-33).  A key is W = 1 or 2 packed 64-bit words
// (consolidate.cu builds them: only the bits the lanes actually use); word 1 is the more significant one and word 0
// holds `bits_lo` valid bits.  Everything below is stable.
//
// Building blocks
//  (1) k_rs_pass — one 8-bit digit pass over HBM ("onesweep"): a tile of 3072 pairs is ranked in shared memory
//      (warp-private digit counters + warp match, no atomics), its 256 digit counts are published to a per-tile status
//      array and the tile's global offsets come from a decoupled look-back over the preceding tiles (one chain per
//      digit), so a pass reads every pair once and writes it once; pairs are staged in tile-sorted order in shared
//      memory so that the global stores are contiguous runs.  The digit comes either from the key bits or from a
//      16-bit bucket id carried along with the pair.  Histograms of all passes are taken up front by one kernel.
//  (2) k_chunk_sort — a whole range of rows ("chunk", <= 6144 pairs) is sorted inside one CTA with shared-memory
//      digit passes over both key words, skipping every digit that is constant inside the chunk.
//  (3) splitters — a strided sample of the keys is sorted (LSD, (1)), every 8th sample becomes a splitter, and every
//      row gets the bucket id 2*(#splitters < key) + (key == that splitter): ids are monotone in the key, odd ids hold
//      copies of one key only (heavy hitters need no sorting), even ids are the ranges between splitters and are small
//      whatever the key distribution.
//
// Plans (radix_sort_pairs)
//      n <= 3072 ............................ one chunk.
//      leading lane ordered on arrival ....... buckets exist already (runs of equal top bits): chunk sort only, ONE trip.
//      n < 256 K ............................ top digit in HBM (1 pass), chunks finish: 2 trips.
//      otherwise ............................ bucket ids from splitters, 2 passes over the ids, chunks finish: ~3.5 trips
//                                             for any key width and any skew, instead of ceil(bits / 8) trips.
//      a bucket that does not fit a chunk .... *fail is raised; the caller re-runs with force_lsd (plain LSD sequence).
#include "common.cuh"

namespace {

constexpr int RS_THREADS = 256, RS_IPT = 12, RS_TILE = RS_THREADS * RS_IPT, RS_WARPS = RS_THREADS / 32;
// chunk sort: 6144 pairs per CTA.  One-word keys: 512 threads x 12 pairs (64 registers, 2 CTAs/SM); two-word keys:
// 1024 threads x 6 pairs (64 registers, one CTA of 32 warps per SM — measured 1.6x faster than 512 x 12 at 128 registers).
constexpr int CS_CAP = 6144, CS_HALF = CS_CAP / 2;
template <int W> struct CsCfg {
  static constexpr int THREADS = W == 1 ? 512 : 1024;
  static constexpr int IPT = CS_CAP / THREADS;
  static constexpr int WARPS = THREADS / 32;
};
constexpr int MAX_PASSES = 16;
constexpr u64 RS_AGG = 1ull << 62, RS_PREFIX = 2ull << 62, RS_MASK = (1ull << 62) - 1;
constexpr u64 SPLITTER_MODE_MIN_ROWS = 262144;
constexpr int OVERSAMPLE = 8, MAX_BUCKETS = 32768;

struct PassList {
  int np;
  int lo[MAX_PASSES];
  unsigned mask[MAX_PASSES];
};

__device__ __forceinline__ u64 ldr(const u64* p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void str(u64* p, u64 v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// 8 (or fewer) bits at position `lo` of the concatenation (k1 : k0), k0 holding bits_lo valid bits (upper bits zero)
template <int W>
__device__ __forceinline__ unsigned key_digit(u64 k0, u64 k1, int lo, unsigned mask, int bits_lo) {
  if (W == 1) return (unsigned)(k0 >> lo) & mask;
  if (lo >= bits_lo) return (unsigned)(k1 >> (lo - bits_lo)) & mask;
  if (lo + 8 <= bits_lo) return (unsigned)(k0 >> lo) & mask;
  return (unsigned)((k0 >> lo) | (k1 << (bits_lo - lo))) & mask;
}
// do two keys agree on every bit at or above position `sh` of the concatenation?
template <int W>
__device__ __forceinline__ bool same_prefix(u64 a0, u64 a1, u64 b0, u64 b1, int sh, int bits_lo) {
  if (W == 1) return sh >= 64 ? true : (a0 >> sh) == (b0 >> sh);
  if (sh >= bits_lo) { const int s1 = sh - bits_lo; return s1 >= 64 ? true : (a1 >> s1) == (b1 >> s1); }
  return a1 == b1 && (a0 >> sh) == (b0 >> sh);
}

// digit histograms of every pass in one read of the keys (or of the bucket ids)
template <int W>
__global__ void __launch_bounds__(256)
k_rs_hist_all(const u64* __restrict__ k0, const u64* __restrict__ k1, const unsigned short* __restrict__ bid, u64 n, PassList pl,
              int bits_lo, u32* ghist) {
  __shared__ u32 s_h[MAX_PASSES][256];
  for (int k = threadIdx.x; k < pl.np * 256; k += 256) (&s_h[0][0])[k] = 0;
  __syncthreads();
  for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += (u64)gridDim.x * 256) {
    if (bid) {
      const unsigned b = bid[i];
      for (int p = 0; p < pl.np; p++) atomicAdd(&s_h[p][(b >> pl.lo[p]) & 0xffu], 1u);
    } else {
      const u64 a0 = k0[i], a1 = W > 1 ? k1[i] : 0;
      for (int p = 0; p < pl.np; p++) atomicAdd(&s_h[p][key_digit<W>(a0, a1, pl.lo[p], pl.mask[p], bits_lo)], 1u);
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < pl.np * 256; k += 256) {
    const u32 v = (&s_h[0][0])[k];
    if (v) atomicAdd(&ghist[k], v);
  }
}

// exclusive scan of the 256 bins of each pass (one CTA per pass)
__global__ void __launch_bounds__(256) k_rs_gscan(u32* ghist) {
  __shared__ u32 s_w[8];
  u32* h = ghist + (size_t)blockIdx.x * 256;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const u32 v = h[tid];
  u32 incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 x = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += x;
  }
  if (lane == 31) s_w[wid] = incl;
  __syncthreads();
  u32 off = 0;
  for (int k = 0; k < wid; k++) off += s_w[k];
  h[tid] = off + incl - v;
}

// Stable ranks of a warp's items among the items of the same digit that precede them in the warp's blocked range.
// s_wh[257] is this warp's private counter array (digit 256 = padding items).
template <int IPT>
__device__ __forceinline__ void warp_digit_ranks(const unsigned (&dig)[IPT], u32* s_wh, unsigned short (&rank)[IPT]) {
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1;
#pragma unroll
  for (int r = 0; r < IPT; r++) {
    const unsigned d = dig[r];
    const unsigned m = __match_any_sync(0xffffffffu, d);
    const int leader = __ffs(m) - 1;
    u32 old = 0;
    if (lane == leader) {
      old = s_wh[d];
      s_wh[d] = old + __popc(m);
    }
    old = __shfl_sync(0xffffffffu, old, leader);
    rank[r] = (unsigned short)(old + __popc(m & lt));
    __syncwarp();
  }
}

struct PairPtrs {
  const u64* k0;
  const u64* k1;
  const u32* id;
  const unsigned short* bid;
};
struct MPairPtrs {
  u64* k0;
  u64* k1;
  u32* id;
  unsigned short* bid;
};

// One digit pass over HBM.  BID: the digit is (bid >> lo) & 0xff and the bucket ids travel with the pairs.
// status: u64[ntiles * 256], zeroed; ticket: u32, zeroed; gbase: exclusive scan of the global histogram of this pass.
template <int W, bool BID>
__global__ void __launch_bounds__(RS_THREADS, W == 1 ? 4 : 2)
k_rs_pass(PairPtrs in, MPairPtrs out, u64 n, int lo, unsigned mask, int bits_lo, const u32* __restrict__ gbase, u64* status, u32* ticket) {
  extern __shared__ __align__(16) unsigned char rs_smem[];
  u64* s_key0 = (u64*)rs_smem;
  u64* s_key1 = s_key0 + RS_TILE;                                  // W == 2 only
  u32* s_id = (u32*)(s_key0 + (size_t)W * RS_TILE);
  unsigned short* s_bid = (unsigned short*)(s_id + RS_TILE);       // BID only
  u32* s_wh = (u32*)(s_bid + (BID ? RS_TILE : 0));                 // [RS_WARPS][257]
  __shared__ u32 s_dstart[256];
  __shared__ long long s_gb[256];
  __shared__ u32 s_wsum[RS_WARPS];
  __shared__ u32 s_tile;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);   // tiles ordered by arrival: every predecessor of a look-back is running
  for (int k = tid; k < RS_WARPS * 257; k += RS_THREADS) s_wh[k] = 0;
  __syncthreads();
  const u32 tile = s_tile;
  const u64 base = (u64)tile * RS_TILE;
  const int cnt = (int)((n - base) < (u64)RS_TILE ? (n - base) : (u64)RS_TILE);

  u64 key0[RS_IPT], key1[W > 1 ? RS_IPT : 1];
  u32 id[RS_IPT];
  unsigned short bidr[BID ? RS_IPT : 1];
  unsigned dig[RS_IPT];
  unsigned short rank[RS_IPT];
#pragma unroll
  for (int r = 0; r < RS_IPT; r++) {
    const int j = wid * (RS_IPT * 32) + r * 32 + lane;   // warp-blocked: item order = (warp, round, lane)
    const bool valid = j < cnt;
    key0[r] = valid ? in.k0[base + j] : 0;
    if (W > 1) key1[r] = valid ? in.k1[base + j] : 0;
    id[r] = valid ? in.id[base + j] : 0;
    if (BID) {
      bidr[r] = valid ? in.bid[base + j] : (unsigned short)0;
      dig[r] = valid ? (((unsigned)bidr[r] >> lo) & 0xffu) : 256u;
    } else {
      dig[r] = valid ? key_digit<W>(key0[r], W > 1 ? key1[r] : 0, lo, mask, bits_lo) : 256u;
    }
  }
  warp_digit_ranks<RS_IPT>(dig, s_wh + wid * 257, rank);
  __syncthreads();

  // per digit: exclusive prefix over the warps, tile count, look-back over the preceding tiles
  {
    const int d = tid;   // RS_THREADS == 256 digits
    u32 run = 0;
#pragma unroll
    for (int w = 0; w < RS_WARPS; w++) {
      const u32 v = s_wh[w * 257 + d];
      s_wh[w * 257 + d] = run;
      run += v;
    }
    const u32 tile_cnt = run;
    u32 incl = tile_cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const u32 x = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += x;
    }
    if (lane == 31) s_wsum[wid] = incl;
    u64 prev = 0;
    if (tile == 0) {
      str(&status[d], RS_PREFIX | (u64)tile_cnt);
    } else {
      str(&status[(u64)tile * 256 + d], RS_AGG | (u64)tile_cnt);
      long long p = (long long)tile - 1;
      while (true) {
        u64 v;
        do { v = ldr(&status[(u64)p * 256 + d]); } while ((v >> 62) == 0);
        prev += v & RS_MASK;
        if ((v >> 62) == 2) break;
        p--;
      }
      str(&status[(u64)tile * 256 + d], RS_PREFIX | (prev + tile_cnt));
    }
    __syncthreads();
    u32 off = 0;
    for (int k = 0; k < wid; k++) off += s_wsum[k];
    const u32 dstart = off + incl - tile_cnt;
    s_dstart[d] = dstart;
    s_gb[d] = (long long)gbase[d] + (long long)prev - (long long)dstart;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < RS_IPT; r++) {
    if (dig[r] < 256u) {
      const u32 li = s_dstart[dig[r]] + s_wh[wid * 257 + dig[r]] + rank[r];
      s_key0[li] = key0[r];
      if (W > 1) s_key1[li] = key1[r];
      s_id[li] = id[r];
      if (BID) s_bid[li] = bidr[r];
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < RS_IPT; k++) {
    const int j = k * RS_THREADS + tid;
    if (j < cnt) {
      const u64 a0 = s_key0[j], a1 = W > 1 ? s_key1[j] : 0;
      unsigned d;
      if (BID) d = ((unsigned)s_bid[j] >> lo) & 0xffu;
      else d = key_digit<W>(a0, a1, lo, mask, bits_lo);
      const long long o = s_gb[d] + j;
      out.k0[o] = a0;
      if (W > 1) out.k1[o] = a1;
      out.id[o] = s_id[j];
      if (BID) out.bid[o] = s_bid[j];
    }
  }
}
template <int W, bool BID>
constexpr size_t rs_smem_bytes() {
  return (size_t)RS_TILE * (8 * W + 4 + (BID ? 2 : 0)) + (size_t)RS_WARPS * 257 * 4;
}

// Finish a partitioned array in shared memory.  Buckets are contiguous and mutually ordered; row i starts a bucket when
//   BID : bid[i] != bid[i-1], or bid[i] is odd (copies of one key) and i is a multiple of CS_HALF (such a bucket may be
//         cut anywhere);
//   else: the bits at or above `bshift` of the key differ from row i-1's (bshift >= 128: one bucket).
// Window w = rows [w * CS_HALF, +CS_HALF); its CTA sorts the chunk from the first bucket start inside the window to the
// first bucket start inside the next window — whole buckets, at most CS_CAP rows when no bucket exceeds CS_HALF rows
// (else *fail is raised).
template <int W, bool BID>
__global__ void __launch_bounds__(CsCfg<W>::THREADS, W == 1 ? 2 : 1)
k_chunk_sort(PairPtrs in, MPairPtrs out, u64 n, int bits_total, int bits_lo, int bshift, unsigned long long* fail) {
  constexpr int CS_THREADS = CsCfg<W>::THREADS, CS_IPT = CsCfg<W>::IPT, CS_WARPS = CsCfg<W>::WARPS;
  extern __shared__ __align__(16) unsigned char cs_smem[];
  u64* s_key0 = (u64*)cs_smem;
  u64* s_key1 = s_key0 + CS_CAP;                                   // W == 2 only
  u32* s_id = (u32*)(s_key0 + (size_t)W * CS_CAP);
  u32* s_wh = s_id + CS_CAP;   // [CS_WARPS][257]
  __shared__ u32 s_dstart[256];
  __shared__ u32 s_wsum[8];
  __shared__ unsigned long long s_first[2];
  __shared__ unsigned long long s_vary[2];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const u64 x0 = (u64)blockIdx.x * CS_HALF;
  if (x0 >= n) return;
  if (tid == 0) { s_first[0] = ~0ull; s_first[1] = ~0ull; s_vary[0] = 0; s_vary[1] = 0; }
  __syncthreads();
#pragma unroll
  for (int side = 0; side < 2; side++) {
    const u64 from = x0 + (u64)side * CS_HALF;
    u64 best = ~0ull;
    for (int k = 0; k < CS_HALF / CS_THREADS; k++) {
      const u64 i = from + (u64)k * CS_THREADS + tid;
      if (i < n) {
        bool head = i == 0;
        if (!head) {
          if (BID) {
            const unsigned b = in.bid[i];
            head = (b != in.bid[i - 1]) || ((b & 1u) && (i % CS_HALF) == 0);
          } else if (bshift < 128) {
            head = !same_prefix<W>(in.k0[i], W > 1 ? in.k1[i] : 0, in.k0[i - 1], W > 1 ? in.k1[i - 1] : 0, bshift, bits_lo);
          }
        }
        if (head && i < best) best = i;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const u64 y = __shfl_xor_sync(0xffffffffu, best, o);
      best = y < best ? y : best;
    }
    if (lane == 0 && best != ~0ull) atomicMin(&s_first[side], (unsigned long long)best);
  }
  __syncthreads();
  u64 s = s_first[0], e = s_first[1];
  if (s == ~0ull) {
    // no bucket starts in this window: fine at the tail of the array (the previous chunk runs to n), else a bucket
    // longer than CS_HALF rows
    if (x0 + CS_HALF < n && tid == 0) atomicOr(fail, 1ull);
    return;
  }
  if (e == ~0ull) {
    if (x0 + 2 * (u64)CS_HALF < n) { if (tid == 0) atomicOr(fail, 1ull); return; }
    e = n;
  }
  const int m = (int)(e - s);
  if (m > CS_CAP) { if (tid == 0) atomicOr(fail, 1ull); return; }

  u64 key0[CS_IPT], key1[W > 1 ? CS_IPT : 1];
  u32 id[CS_IPT];
  unsigned dig[CS_IPT];
  unsigned short rank[CS_IPT];
  const u64 f0 = in.k0[s], f1 = W > 1 ? in.k1[s] : 0;
  u64 vary0 = 0, vary1 = 0;
#pragma unroll
  for (int r = 0; r < CS_IPT; r++) {
    const int j = wid * (CS_IPT * 32) + r * 32 + lane;
    const bool valid = j < m;
    key0[r] = valid ? in.k0[s + j] : f0;
    if (W > 1) key1[r] = valid ? in.k1[s + j] : f1;
    id[r] = valid ? in.id[s + j] : 0;
    vary0 |= key0[r] ^ f0;
    if (W > 1) vary1 |= key1[r] ^ f1;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    vary0 |= __shfl_xor_sync(0xffffffffu, vary0, o);
    if (W > 1) vary1 |= __shfl_xor_sync(0xffffffffu, vary1, o);
  }
  if (lane == 0) {
    if (vary0) atomicOr(&s_vary[0], (unsigned long long)vary0);
    if (W > 1 && vary1) atomicOr(&s_vary[1], (unsigned long long)vary1);
  }
  __syncthreads();
  vary0 = s_vary[0];
  vary1 = W > 1 ? s_vary[1] : 0;

  for (int lo = 0; lo < bits_total; lo += 8) {
    const unsigned mask = (bits_total - lo >= 8) ? 0xffu : ((1u << (bits_total - lo)) - 1);
    if (key_digit<W>(vary0, vary1, lo, mask, bits_lo) == 0) continue;   // digit constant inside the chunk (block-uniform)
    for (int k = tid; k < CS_WARPS * 257; k += CS_THREADS) s_wh[k] = 0;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < CS_IPT; r++) {
      const int j = wid * (CS_IPT * 32) + r * 32 + lane;
      dig[r] = j < m ? key_digit<W>(key0[r], W > 1 ? key1[r] : 0, lo, mask, bits_lo) : 256u;
    }
    warp_digit_ranks<CS_IPT>(dig, s_wh + wid * 257, rank);
    __syncthreads();
    if (tid < 256) {
      const int d = tid;
      u32 run = 0;
#pragma unroll
      for (int w = 0; w < CS_WARPS; w++) {
        const u32 v = s_wh[w * 257 + d];
        s_wh[w * 257 + d] = run;
        run += v;
      }
      u32 incl = run;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const u32 x = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += x;
      }
      if (lane == 31) s_wsum[wid] = incl;
      s_dstart[d] = incl - run;   // exclusive inside the warp of digits; the warp offsets are added below
    }
    __syncthreads();
    if (tid < 256) {
      u32 off = 0;
      for (int k = 0; k < wid; k++) off += s_wsum[k];
      s_dstart[tid] += off;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < CS_IPT; r++) {
      if (dig[r] < 256u) {
        const u32 li = s_dstart[dig[r]] + s_wh[wid * 257 + dig[r]] + rank[r];
        s_key0[li] = key0[r];
        if (W > 1) s_key1[li] = key1[r];
        s_id[li] = id[r];
      }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < CS_IPT; r++) {
      const int j = wid * (CS_IPT * 32) + r * 32 + lane;
      if (j < m) {
        key0[r] = s_key0[j];
        if (W > 1) key1[r] = s_key1[j];
        id[r] = s_id[j];
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < CS_IPT; r++) {
    const int j = wid * (CS_IPT * 32) + r * 32 + lane;
    if (j < m) {
      out.k0[s + j] = key0[r];
      if (W > 1) out.k1[s + j] = key1[r];
      out.id[s + j] = id[r];
    }
  }
}
template <int W>
constexpr size_t cs_smem_bytes() {
  return (size_t)CS_CAP * (8 * W + 4) + (size_t)CsCfg<W>::WARPS * 257 * 4;
}

// strided sample with a per-sample jitter (robust to periodic inputs)
template <int W>
__global__ void k_sample(const u64* __restrict__ k0, const u64* __restrict__ k1, u64 n, u32 m, u64* s0, u64* s1, u32* sid) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const u64 lo = (u64)j * n / m, hi = (u64)(j + 1) * n / m;
  u64 x = (u64)j * 0x9e3779b97f4a7c15ull;
  x ^= x >> 29;
  const u64 i = lo + (hi > lo ? x % (hi - lo) : 0);
  s0[j] = k0[i];
  if (W > 1) s1[j] = k1[i];
  sid[j] = j;
}
// splitter j = sorted sample[(j + 1) * OVERSAMPLE], j < ns
template <int W>
__global__ void k_pick_splitters(const u64* __restrict__ s0, const u64* __restrict__ s1, u32 ns, u64* sp0, u64* sp1) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= ns) return;
  sp0[j] = s0[(size_t)(j + 1) * OVERSAMPLE];
  if (W > 1) sp1[j] = s1[(size_t)(j + 1) * OVERSAMPLE];
}
// bucket id = 2 * (#splitters < key) + (key == splitter[that index]).  Two-level search: the last splitter of every
// group of 32 is staged in shared memory (<= 1024 entries), the group found there is finished with 5 steps inside
// two cache lines.
template <int W>
__global__ void __launch_bounds__(256)
k_bucket_ids(const u64* __restrict__ k0, const u64* __restrict__ k1, u64 n, const u64* __restrict__ sp0, const u64* __restrict__ sp1,
             u32 ns, unsigned short* bid) {
  __shared__ u64 s_c0[1024];
  __shared__ u64 s_c1[W > 1 ? 1024 : 1];
  const u32 nc = (ns + 31) / 32;
  for (u32 g = threadIdx.x; g < nc; g += 256) {
    const u32 j = g * 32 + 31 < ns ? g * 32 + 31 : ns - 1;
    s_c0[g] = sp0[j];
    if (W > 1) s_c1[g] = sp1[j];
  }
  __syncthreads();
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const u64 a0 = k0[i], a1 = W > 1 ? k1[i] : 0;
  u32 lo = 0, hi = nc;
  while (lo < hi) {   // first group whose last splitter >= key
    const u32 mid = (lo + hi) >> 1;
    bool less;
    if (W > 1) { const u64 b1 = s_c1[mid]; less = b1 < a1 || (b1 == a1 && s_c0[mid] < a0); }
    else less = s_c0[mid] < a0;
    if (less) lo = mid + 1; else hi = mid;
  }
  u32 res = ns;   // every splitter < key
  if (lo < nc) {
    u32 l2 = lo * 32, h2 = l2 + 32 < ns ? l2 + 32 : ns;
    while (l2 < h2) {   // first splitter >= key inside the group
      const u32 mid = (l2 + h2) >> 1;
      bool less;
      if (W > 1) { const u64 b1 = sp1[mid]; less = b1 < a1 || (b1 == a1 && sp0[mid] < a0); }
      else less = sp0[mid] < a0;
      if (less) l2 = mid + 1; else h2 = mid;
    }
    res = l2;
  }
  bool eq = false;
  if (res < ns) eq = sp0[res] == a0 && (W == 1 || sp1[res] == a1);
  bid[i] = (unsigned short)(2u * res + (eq ? 1u : 0u));
}

struct Bufs {   // the two ping-pong sets of a sort
  u64* k0[2];
  u64* k1[2];
  u32* id[2];
  unsigned short* bid[2];
};

template <int W, bool BID>
int32_t run_passes(Ctx* ctx, Bufs& B, int& cur, u64 n, const PassList& pl, int bits_lo, int* hbm_passes) {
  cudaStream_t st = lane(ctx).stream;
  if (pl.np == 0) return DBSP_OK;
  const u32 ntiles = (u32)((n + RS_TILE - 1) / RS_TILE);
  BufP aux;
  // ghist[np][256] u32 | tickets[np] u32 | status[np][ntiles*256] u64
  const size_t head_bytes = ((size_t)pl.np * 256 * 4 + (size_t)pl.np * 4 + 15) & ~15ull;
  const size_t status_bytes = (size_t)pl.np * ntiles * 256 * 8;
  TRY(dev_alloc(ctx, head_bytes + status_bytes, &aux));
  CUDA_TRY(cudaMemsetAsync(aux->p, 0, head_bytes + status_bytes, st));
  u32* ghist = (u32*)aux->p;
  u32* tickets = ghist + (size_t)pl.np * 256;
  u64* status = (u64*)((char*)aux->p + head_bytes);
  {
    ProfScope ps(ctx, KID_RADIX_SORT, n * (u64)(BID ? 2 : 8 * W));
    const unsigned g = (unsigned)std::min<u64>((n + 255) / 256, (u64)ctx->sm_count * 8);
    k_rs_hist_all<W><<<g, 256, 0, st>>>(B.k0[cur], B.k1[cur], BID ? B.bid[cur] : nullptr, n, pl, bits_lo, ghist);
    k_rs_gscan<<<pl.np, 256, 0, st>>>(ghist);
  }
  ctx->kernel_launches += 2;
  constexpr size_t SMEM = rs_smem_bytes<W, BID>();
  CUDA_TRY(cudaFuncSetAttribute(k_rs_pass<W, BID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
  for (int p = 0; p < pl.np; p++) {
    PairPtrs in{B.k0[cur], B.k1[cur], B.id[cur], B.bid[cur]};
    MPairPtrs out{B.k0[cur ^ 1], B.k1[cur ^ 1], B.id[cur ^ 1], B.bid[cur ^ 1]};
    {
      ProfScope ps(ctx, KID_RADIX_SORT, n * (u64)(2 * (8 * W + 4 + (BID ? 2 : 0))));   // every pair read once, written once
      k_rs_pass<W, BID><<<ntiles, RS_THREADS, SMEM, st>>>(in, out, n, pl.lo[p], pl.mask[p], bits_lo, ghist + (size_t)p * 256,
                                                          status + (size_t)p * ntiles * 256, tickets + p);
    }
    LAUNCH_COUNT(ctx);
    cur ^= 1;
  }
  if (hbm_passes) *hbm_passes += pl.np;
  return DBSP_OK;
}

template <int W, bool BID>
int32_t run_chunks(Ctx* ctx, Bufs& B, int& cur, u64 n, int bits_total, int bits_lo, int bshift, unsigned long long* fail, int* hbm_passes) {
  constexpr size_t SMEM = cs_smem_bytes<W>();
  CUDA_TRY(cudaFuncSetAttribute(k_chunk_sort<W, BID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
  const unsigned nwin = (unsigned)((n + CS_HALF - 1) / CS_HALF);
  PairPtrs in{B.k0[cur], B.k1[cur], B.id[cur], B.bid[cur]};
  MPairPtrs out{B.k0[cur ^ 1], B.k1[cur ^ 1], B.id[cur ^ 1], B.bid[cur ^ 1]};
  {
    ProfScope ps(ctx, KID_CHUNK_SORT, n * (u64)(2 * (8 * W + 4) + (BID ? 2 : 0)));
    k_chunk_sort<W, BID><<<nwin, CsCfg<W>::THREADS, SMEM, lane(ctx).stream>>>(in, out, n, bits_total, bits_lo, bshift, fail);
  }
  LAUNCH_COUNT(ctx);
  cur ^= 1;
  if (hbm_passes) *hbm_passes += 1;
  return DBSP_OK;
}

void lsd_passes(PassList& pl, int bits_total) {
  pl.np = 0;
  for (int lo = 0; lo < bits_total && pl.np < MAX_PASSES; lo += 8) {
    pl.lo[pl.np] = lo;
    pl.mask[pl.np] = (bits_total - lo >= 8) ? 0xffu : ((1u << (bits_total - lo)) - 1);
    pl.np++;
  }
}

template <int W>
int32_t sort_impl(Ctx* ctx, Bufs& B, u64 n, int bits_lo, int bits_hi, int presorted_top_bits, bool force_lsd, unsigned long long* fail,
                  int* cur_out, int* hbm_passes) {
  cudaStream_t st = lane(ctx).stream;
  const int bits_total = W == 1 ? bits_lo : bits_lo + bits_hi;
  int cur = 0;
  PassList pl;
  pl.np = 0;
  if (force_lsd) {
    lsd_passes(pl, bits_total);
    TRY((run_passes<W, false>(ctx, B, cur, n, pl, bits_lo, hbm_passes)));
  } else if (n <= (u64)CS_HALF) {
    TRY((run_chunks<W, false>(ctx, B, cur, n, bits_total, bits_lo, 128, fail, hbm_passes)));   // one chunk, one bucket
  } else if (presorted_top_bits > 0) {
    const int pb = presorted_top_bits < bits_total ? presorted_top_bits : bits_total;
    TRY((run_chunks<W, false>(ctx, B, cur, n, bits_total, bits_lo, bits_total - pb, fail, hbm_passes)));
  } else if (n > (u64)MAX_BUCKETS * 768) {
    // more rows than 32768 buckets of chunk size can hold: plain LSD
    lsd_passes(pl, bits_total);
    TRY((run_passes<W, false>(ctx, B, cur, n, pl, bits_lo, hbm_passes)));
  } else if (n < SPLITTER_MODE_MIN_ROWS) {
    if (bits_total > 16) {   // top digit in HBM, the chunks finish
      pl.np = 1;
      pl.lo[0] = bits_total - 8;
      pl.mask[0] = 0xffu;
      TRY((run_passes<W, false>(ctx, B, cur, n, pl, bits_lo, hbm_passes)));
      TRY((run_chunks<W, false>(ctx, B, cur, n, bits_total, bits_lo, bits_total - 8, fail, hbm_passes)));
    } else {
      lsd_passes(pl, bits_total);
      TRY((run_passes<W, false>(ctx, B, cur, n, pl, bits_lo, hbm_passes)));
    }
  } else {
    // ---- splitters from a sorted sample -------------------------------------------------------
    u32 nb = 256;
    while ((u64)nb * 768 < n && nb < (u32)MAX_BUCKETS) nb <<= 1;
    const u32 m = nb * OVERSAMPLE, ns = nb - 1;
    BufP sbuf;
    // sample keys (2 ping-pong sets of W words) + ids (2 sets) + splitters (W words)
    TRY(dev_alloc(ctx, (size_t)m * (8 * W + 4) * 2 + (size_t)nb * 8 * W + 64, &sbuf));
    Bufs S;
    u64* p64 = (u64*)sbuf->p;
    S.k0[0] = p64; p64 += m;
    S.k0[1] = p64; p64 += m;
    S.k1[0] = S.k1[1] = nullptr;
    if (W > 1) { S.k1[0] = p64; p64 += m; S.k1[1] = p64; p64 += m; }
    u64* sp0 = p64; p64 += nb;
    u64* sp1 = nullptr;
    if (W > 1) { sp1 = p64; p64 += nb; }
    S.id[0] = (u32*)p64;
    S.id[1] = S.id[0] + m;
    S.bid[0] = S.bid[1] = nullptr;
    k_sample<W><<<(m + 255) / 256, 256, 0, st>>>(B.k0[cur], B.k1[cur], n, m, S.k0[0], S.k1[0], S.id[0]);
    LAUNCH_COUNT(ctx);
    int scur = 0;
    PassList spl;
    lsd_passes(spl, bits_total);
    TRY((run_passes<W, false>(ctx, S, scur, m, spl, bits_lo, nullptr)));
    k_pick_splitters<W><<<(ns + 255) / 256, 256, 0, st>>>(S.k0[scur], S.k1[scur], ns, sp0, sp1);
    {
      ProfScope ps(ctx, KID_RADIX_SORT, n * (u64)(8 * W + 2));
      k_bucket_ids<W><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(B.k0[cur], B.k1[cur], n, sp0, sp1, ns, B.bid[cur]);
    }
    ctx->kernel_launches += 2;
    pl.np = 2;
    pl.lo[0] = 0; pl.mask[0] = 0xffu;
    pl.lo[1] = 8; pl.mask[1] = 0xffu;
    TRY((run_passes<W, true>(ctx, B, cur, n, pl, bits_lo, hbm_passes)));
    TRY((run_chunks<W, true>(ctx, B, cur, n, bits_total, bits_lo, 128, fail, hbm_passes)));
  }
  *cur_out = cur;
  return DBSP_OK;
}

}  // namespace

// Sorts n (key, id) pairs by key, stably.  The key is `words` (1 or 2) 64-bit words: k0 holds the low `bits_lo` bits
// (upper bits zero), k1 (words == 2) the next `bits_hi` bits.  The pairs are in (k0a, k1a, ida); (k0b, k1b, idb) are
// scratch of the same size.  presorted_top_bits > 0: that many leading bits of the key are already non-decreasing
// along the array.  force_lsd: plain LSD sequence (the fallback after *fail was raised).  *fail (device word, may be
// raised by this call) must be checked by the caller after the stream reaches the result.  *which = 0 / 1: the result
// is in the a / b set.
int32_t radix_sort_pairs(Ctx* ctx, int words, u64* k0a, u64* k0b, u64* k1a, u64* k1b, u32* ida, u32* idb, u64 n, int bits_lo, int bits_hi,
                         int presorted_top_bits, bool force_lsd, unsigned long long* fail, int* which, int* hbm_passes) {
  *which = 0;
  if (hbm_passes) *hbm_passes = 0;
  const int bits_total = words == 1 ? bits_lo : bits_lo + bits_hi;
  if (n <= 1 || bits_total <= 0) return DBSP_OK;
  if (n >= 0xffffffffull) { set_error("sort: 2^32-1 or more rows"); return DBSP_ERR_UNSUPPORTED; }
  if (words < 1 || words > 2 || bits_lo > 64 || bits_hi > 64) { set_error("sort: unsupported key width"); return DBSP_ERR_UNSUPPORTED; }
  Bufs B;
  B.k0[0] = k0a; B.k0[1] = k0b;
  B.k1[0] = k1a; B.k1[1] = k1b;
  B.id[0] = ida; B.id[1] = idb;
  B.bid[0] = B.bid[1] = nullptr;
  BufP bidbuf;
  if (!force_lsd && n >= SPLITTER_MODE_MIN_ROWS && n <= (u64)MAX_BUCKETS * 768 && presorted_top_bits <= 0) {
    TRY(dev_alloc(ctx, (size_t)((n + 7) & ~7ull) * 2 * 2, &bidbuf));
    B.bid[0] = (unsigned short*)bidbuf->p;
    B.bid[1] = B.bid[0] + ((n + 7) & ~7ull);
  }
  if (words == 1) return sort_impl<1>(ctx, B, n, bits_lo, 0, presorted_top_bits, force_lsd, fail, which, hbm_passes);
  return sort_impl<2>(ctx, B, n, bits_lo, bits_hi, presorted_top_bits, force_lsd, fail, which, hbm_passes);
}
