// goliath_b200/csrc/splat_bin_tiles.cu — tile binning for the fused render path, B200 formulation (sm_100a).
//
// Produces exactly what the key sort of csrc/splat_bin.cu produces for the fused render — per-tile
// [first,last) bins, the Gaussian ids of every tile in front-to-back order (ties: ascending id), and the
// packed blend records — i.e. the work gsplat 0.1.11 does in bin_and_sort_gaussians (called from
// rasterize_gaussians, call sites ca_code/utils/render_gsplat.py:65-78,90-104), but without a global sort of
// the I (tile, depth) intersection keys.  Two orderings, same outputs (gb_set_bin_sort_mode, GOLIATH_B200_BINSORT):
//
// TILE (default): bucket the pairs, sort each tile's short list on chip.
//   1. depth_keys_kernel<., false>   G threads: per-tile intersection COUNT of every visible Gaussian, and the min /
//                            max of the visible depth keys (sync[4..5]).  Counts are privatised per CTA in shared
//                            memory and flushed with one RED per (CTA, non-empty tile): the hot tiles of a head scene
//                            take ~2000 hits each, which serialise on the L2 atomic unit when issued one by one
//                            (measured: 118 us with one global RED per pair, 8 us privatised).
//   2. tile_scan_kernel + gb_tile_order / gb_tile_schedule, as below.
//   3. tile_scatter_kernel<true>     G threads: every (Gaussian, tile) pair writes the Gaussian's 32-bit depth key into
//                            its slot of tile_ranks and its id into the same slot of gids_sorted (slots claimed per
//                            CTA, order inside a bucket arbitrary); the 48-byte record goes to a table indexed BY ID.
//   4. tile_pair_sort_kernel one CTA per tile, longest first: composite (key - min key) << 32 | id — unique, and
//                            ordered as the key sort orders the tile (depth bits, ties by ascending id) — LSD radix
//                            sorted in shared memory over the KEY digits that vary inside the tile, then each run of
//                            equal keys put in id order (all digits when a run is long); sorted ids written back.  A list longer than kPairCap sorts in the
//                            tile's own slots of the records output (48 B per slot, 16 B used), written only by 5.
//   5. gather_records_kernel grid-wide: records[i] = table[gids_sorted[i]] (rec_colors_kernel first with late colours).
//   Workspace per intersection slot stays 4 bytes; no depth ranks, no cooperative launch, no per-tile G-bit bitmap.
//
// RANK: depth-rank the G Gaussians once, then order each tile's ranks with a bitmap.
//   1. depth_keys_kernel<., true>    as above, plus the key array and the digit-0 histogram of the rank sort.
//   2. rank_scatter_kernel   x4: stable LSD radix sort of the G depth keys (8-bit digits).  One kernel per
//                            pass: a CTA derives its own scatter bases from the per-CTA histogram table
//                            (column prefix read from L2) and accumulates the NEXT pass's table with global
//                            atomics while it scatters; a pass whose digit is the same for every key (the
//                            exponent byte of the depths) degenerates to a copy.  Result: rank_of[g] (unique,
//                            ties by ascending id) and rank_to_gid[rank].  This sorts G = 300k 4-byte keys
//                            instead of I = 1.08 M 12-byte (key, id) pairs through 6 passes.
//   3. tile_scan_kernel      one CTA: exclusive scan of the T counts -> tile_bins (clamped to the capacity),
//                            scatter cursors, total count, overflow flag.
//   4. tile_scatter_kernel   G threads: every (Gaussian, tile) pair drops the Gaussian's RANK into the
//                            tile's bucket (order inside the bucket arbitrary).  Slots are claimed per CTA:
//                            count in shared memory, one atomicAdd per (CTA, tile) on the global cursor, then
//                            shared-memory atomics hand out the slots.  The same threads write the 48-byte
//                            blend record of their Gaussian into a table indexed BY RANK (cull box computed
//                            once per Gaussian, not once per intersection).
//   5. tile_sort_pack_kernel one CTA per tile, longest first: the ranks of a bucket are unique integers
//                            < G, so sorting them is setting bits in a G-bit bitmap in shared memory
//                            (37.5 KB at 300k, 128 KB at 1 M) and reading the bits back in order:
//                            popcount prefix -> sorted ranks -> (Gaussian id, record copied from the by-rank
//                            table with monotonically increasing addresses), written linearly.
//
//   (2b is the default form of 2, one cooperative kernel; 5b the default form of 5, bitmap sort + grid-wide gather.)
//   gb_bin_tiles_ranked always takes this path: its blend reads records by depth rank.
//
// Integer/byte work with a BIT-EXACT contract: gids_sorted, tile_bins and records are identical to the
// key-sort path's under either ordering (tests/test_splat_gpu.py::test_bin_tiles_matches_key_sort,
// tests/test_bin_tiles_tilesort_gpu.py).
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "splat_record.cuh"

extern "C" int gb_tile_order(int num_tiles, const int32_t* tile_bins, int32_t* order, void* stream);
extern "C" int gb_tile_schedule(int num_tiles, const int32_t* tile_bins, int32_t* sched, void* stream);
GB_API int gb_bin_tiles_pack_ev(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                                const float* colors3, const float* opacity, const float* compensation, int img_h,
                                int img_w, int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order,
                                int tile_sched, int32_t* gids_sorted, float* records, int32_t* n_out, int32_t* overflow,
                                void* workspace, void* colors_ready, void* stream);

namespace {

constexpr int kRankBlock = 256;                       // 8 warps
constexpr int kRadix = 256;
constexpr int kRankPasses = 4;                        // 32 key bits
constexpr int kScatItems = 2;                         // Gaussians per thread in tile_scatter_kernel
constexpr int kSortThreads = 512;
constexpr int kCopyBatch = 2;                         // records copied per thread per round trip (register budget)
constexpr int kMaxBitmapBytes = 192 * 1024;           // bitmap of one tile must fit the SM's shared memory
constexpr int kMaxSmemTiles = 20 * 1024;              // per-CTA tile counters (x2 in the scatter) in shared memory

// keys per thread of the rank sort: 8 (2048 keys per CTA: 147 CTAs at 300k, one per SM) up to ~400k Gaussians,
// 16 beyond (the per-CTA column prefix over the histogram table grows with the square of the CTA count)
inline int rank_items(int G) { return G <= 2048 * 192 ? 8 : 16; }

// exclusive prefix of v over the CTA (any multiple of 32 threads up to 1024); total = CTA sum
__device__ __forceinline__ int block_exclusive_scan(int v, int* s_warp, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = (lane < (int)(blockDim.x >> 5)) ? s_warp[lane] : 0;
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    s_warp[lane] = winc - w;
    if (lane == 31) s_warp[32] = winc;
  }
  __syncthreads();
  total = s_warp[32];
  const int r = s_warp[warp] + inc - v;
  __syncthreads();
  return r;
}

// tile rectangle of a Gaussian: same arithmetic as map_to_intersects_kernel (csrc/splat_bin.cu)
__device__ __forceinline__ void tile_bbox(float cx, float cy, float radius, int tbx, int tby, int bw, int& x0,
                                          int& y0, int& x1, int& y1) {
  const float fb = (float)bw;
  const float tcx = __fdiv_rn(cx, fb), tcy = __fdiv_rn(cy, fb), tr = __fdiv_rn(radius, fb);
  x0 = min(max(0, __float2int_rz(__fsub_rn(tcx, tr))), tbx);
  x1 = min(max(0, __float2int_rz(__fadd_rn(__fadd_rn(tcx, tr), 1.f))), tbx);
  y0 = min(max(0, __float2int_rz(__fsub_rn(tcy, tr))), tby);
  y1 = min(max(0, __float2int_rz(__fadd_rn(__fadd_rn(tcy, tr), 1.f))), tby);
}

// ------------------------------------------------------------------ 1. keys, digit-0 histogram, tile counts
// smem_tiles = T: per-CTA counters in dynamic shared memory; 0: global atomics (more tiles than fit).
// A CTA covers one tile of the rank sort (kTileKeys keys) with kGaussBlock threads: few fat CTAs keep the number
// of counter flushes low, many threads per CTA keep enough loads in flight (the kernel is latency-bound).
// kRank = false (per-tile sort path): no key array and no digit-0 histogram, only the tile counts and sync[4..5].
constexpr int kGaussBlock = 1024;
template <int kTileKeys, bool kRank>
__global__ void __launch_bounds__(kGaussBlock) depth_keys_kernel(int G, const float2* __restrict__ xys,
                                                                 const float* __restrict__ depths,
                                                                 const int* __restrict__ radii, int tbx, int tby,
                                                                 int block_width, int smem_tiles,
                                                                 unsigned* __restrict__ keys,
                                                                 unsigned* __restrict__ hist0 /* [ctas][256] */,
                                                                 int* __restrict__ tile_counts,
                                                                 unsigned* __restrict__ key_bits /* [2], zeroed */) {
  constexpr int kItems = kTileKeys / kGaussBlock;
  extern __shared__ int s_cnt[];
  __shared__ unsigned s_hist[kRadix];
  __shared__ unsigned s_or, s_orc, s_max, s_maxc;
  if (threadIdx.x == 0) s_or = s_orc = s_max = s_maxc = 0u;
  if (threadIdx.x < kRadix) s_hist[threadIdx.x] = 0;
  for (int t = threadIdx.x; t < smem_tiles; t += kGaussBlock) s_cnt[t] = 0;
  const int base = blockIdx.x * kTileKeys;
  unsigned k[kItems];
  int r[kItems];
  float2 c[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {  // all loads first: independent, in flight together
    const int i = base + j * kGaussBlock + threadIdx.x;
    const bool in = i < G;
    k[j] = in ? __float_as_uint(depths[i]) : 0u;
    r[j] = in ? radii[i] : 0;
    c[j] = in ? xys[i] : make_float2(0.f, 0.f);
  }
  {  // OR of the VISIBLE keys and of their complements: a bit set in both differs between two visible keys, and the
     // rank sort only has to order those bits (culled Gaussians never reach a tile, where their rank lands is irrelevant)
    unsigned o = 0u, oc = 0u, mx = 0u, mxc = 0u;  // mxc = max of the complements = ~min
#pragma unroll
    for (int j = 0; j < kItems; ++j)
      if (r[j] > 0) { o |= k[j]; oc |= ~k[j]; mx = max(mx, k[j]); mxc = max(mxc, ~k[j]); }
    o = __reduce_or_sync(0xffffffffu, o);
    oc = __reduce_or_sync(0xffffffffu, oc);
    mx = __reduce_max_sync(0xffffffffu, mx);
    mxc = __reduce_max_sync(0xffffffffu, mxc);
    __syncthreads();  // the shared accumulators are initialised
    if ((threadIdx.x & 31) == 0 && (o | oc)) {
      atomicOr(&s_or, o); atomicOr(&s_orc, oc); atomicMax(&s_max, mx); atomicMax(&s_maxc, mxc);
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int i = base + j * kGaussBlock + threadIdx.x;
    if (i >= G) continue;
    if (kRank) {
      keys[i] = k[j];
      atomicAdd(&s_hist[k[j] & 0xffu], 1u);
    }
    if (r[j] > 0) {
      int x0, y0, x1, y1;
      tile_bbox(c[j].x, c[j].y, (float)r[j], tbx, tby, block_width, x0, y0, x1, y1);
      for (int ty = y0; ty < y1; ++ty)
        for (int tx = x0; tx < x1; ++tx) {
          if (smem_tiles) atomicAdd(&s_cnt[ty * tbx + tx], 1);
          else atomicAdd(&tile_counts[ty * tbx + tx], 1);
        }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && (s_or | s_orc)) {
    atomicOr(key_bits, s_or); atomicOr(key_bits + 1, s_orc);
    atomicMax(key_bits + 4, s_max); atomicMax(key_bits + 5, s_maxc);  // [4] = max visible key, [5] = ~min visible key
  }
  if (kRank && threadIdx.x < kRadix) hist0[(size_t)blockIdx.x * kRadix + threadIdx.x] = s_hist[threadIdx.x];
  for (int t = threadIdx.x; t < smem_tiles; t += kGaussBlock) {
    const int cnt = s_cnt[t];
    if (cnt) atomicAdd(&tile_counts[t], cnt);
  }
}

// ------------------------------------------------------------------ 2. one radix pass over the G depth keys
// warp w of a CTA owns the contiguous chunk [cta_base + w*32*kItems, +32*kItems), lane-strided inside the
// chunk, so that "earlier in memory" == (smaller item index j, then smaller lane): the ranking is stable.
template <int kItems>
__global__ void __launch_bounds__(kRankBlock) rank_scatter_kernel(
    int n, const unsigned* __restrict__ keys_in, const int* __restrict__ vals_in /* null: identity */,
    unsigned* __restrict__ keys_out /* null on the last pass */, int* __restrict__ vals_out, int shift, int ctas,
    const unsigned* __restrict__ hist_cur /* [ctas][256] of this pass's digit */,
    unsigned* __restrict__ hist_next /* [ctas][256], zeroed; null on the last pass */,
    int* __restrict__ rank_of /* last pass only: rank_of[val] = position */) {
  constexpr int kWarps = kRankBlock / 32;
  constexpr int kTile = kRankBlock * kItems;
  __shared__ unsigned s_whist[kWarps][kRadix];
  __shared__ int s_scan[33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  const int warp_base = blockIdx.x * kTile + warp * (32 * kItems);
  unsigned k[kItems];  // issued before the table reads below: both sets of loads are in flight together
  int v[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int i = warp_base + j * 32 + lane;
    k[j] = (i < n) ? keys_in[i] : 0xffffffffu;
    v[j] = (i < n) ? (vals_in ? vals_in[i] : i) : 0;
  }

  // scatter base of (digit d, this CTA): keys with smaller digits anywhere + keys with digit d in earlier CTAs.
  // Column sums of the CTA-major table, cooperatively: thread (g = t / 64, c = t % 64) adds rows g, g+4, ... of
  // the 16-byte column group c, so each thread keeps many independent 16-byte loads in flight (a one-thread-
  // per-digit loop over the rows is a chain of ~ctas/8 L2 round trips and dominated the pass).
  __shared__ uint4 s_part[2][4][kRadix / 4];
  {
    const int g = threadIdx.x >> 6, c4 = threadIdx.x & 63;
    const uint4* tab = reinterpret_cast<const uint4*>(hist_cur);
    uint4 tot = make_uint4(0u, 0u, 0u, 0u), bef = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll 8
    for (int b = g; b < ctas; b += 4) {
      const uint4 h = tab[(size_t)b * (kRadix / 4) + c4];
      tot.x += h.x; tot.y += h.y; tot.z += h.z; tot.w += h.w;
      if (b < (int)blockIdx.x) { bef.x += h.x; bef.y += h.y; bef.z += h.z; bef.w += h.w; }
    }
    s_part[0][g][c4] = tot;
    s_part[1][g][c4] = bef;
  }
  __syncthreads();
  unsigned before = 0, total = 0;
  {
    const unsigned* pt = reinterpret_cast<const unsigned*>(&s_part[0][0][0]);
    const unsigned* pb = reinterpret_cast<const unsigned*>(&s_part[1][0][0]);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      total += pt[g * kRadix + threadIdx.x];
      before += pb[g * kRadix + threadIdx.x];
    }
  }
  // a digit holding every key makes the pass the identity permutation (typical for the exponent byte)
  const bool copy_only = __syncthreads_or(total == (unsigned)n) != 0;

  if (copy_only) {
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      const int i = warp_base + j * 32 + lane;
      if (i < n) {
        if (keys_out) keys_out[i] = k[j];
        vals_out[i] = v[j];
        if (hist_next) atomicAdd(&hist_next[(size_t)blockIdx.x * kRadix + ((k[j] >> (shift + 8)) & 0xffu)], 1u);
        if (rank_of) rank_of[v[j]] = i;
      }
    }
    return;
  }
  int unused;
  const unsigned digit_base = (unsigned)block_exclusive_scan((int)total, s_scan, unused);
  const unsigned my_base = digit_base + before;

  for (int d = lane; d < kRadix; d += 32) s_whist[warp][d] = 0;
  __syncwarp();
  unsigned rank[kItems];  // rank among equal digits inside this warp's chunk
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int i = warp_base + j * 32 + lane;
    const bool valid = i < n;
    const unsigned dgt = (k[j] >> shift) & 0xffu;
    const unsigned peers = __match_any_sync(0xffffffffu, valid ? dgt : 0x100u);
    const unsigned lower = peers & ((1u << lane) - 1u);
    unsigned prev = 0;
    if (valid) prev = s_whist[warp][dgt];
    __syncwarp();
    rank[j] = prev + __popc(lower);
    if (valid && lower == 0u) s_whist[warp][dgt] = prev + __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  {  // per-warp counts -> per-warp scatter bases (exclusive over the warps, on top of the global base)
    const int d = threadIdx.x;
    unsigned run = my_base;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      const unsigned c = s_whist[w][d];
      s_whist[w][d] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int i = warp_base + j * 32 + lane;
    if (i < n) {
      const unsigned dgt = (k[j] >> shift) & 0xffu;
      const unsigned dst = s_whist[warp][dgt] + rank[j];
      if (keys_out) keys_out[dst] = k[j];
      vals_out[dst] = v[j];
      if (hist_next) atomicAdd(&hist_next[(size_t)(dst / kTile) * kRadix + ((k[j] >> (shift + 8)) & 0xffu)], 1u);
      if (rank_of) rank_of[v[j]] = (int)dst;
    }
  }
}


// ------------------------------------------------------------------ 2b. the whole rank sort as ONE cooperative kernel
// Round-1 launch list (profiles/r01_launches_pipe.txt): 4 x 17-19 us for the four radix passes over 300k keys, each
// a chain of L2 round trips at ~9 % issue utilisation with a kernel boundary in between.  Here the passes run inside
// one cooperative launch (grid <= SM count, every CTA co-resident), separated by a grid barrier (an L2 counter), and
// only the low bits in which the keys actually differ are sorted: depths of a head at ~1 m share their sign,
// exponent and leading mantissa bits, so 3 passes (or 2) replace 4 and no launch gap remains.  Data written by other
// CTAs inside the kernel (keys / ids ping-pong, histogram tables) is read with ld.global.cg (L2), never through the
// non-coherent path.  Same stable LSD ranking as rank_scatter_kernel, same outputs: rank_to_gid and rank_of.
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    target += gridDim.x;
    __threadfence();  // release this CTA's writes
    atomicAdd(counter, 1u);
    unsigned seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
    } while (seen < target);
    __threadfence();
  }
  __syncthreads();
}

template <int kItems>
__global__ void __launch_bounds__(kRankBlock) rank_sort_coop_kernel(
    int n, int tiles, unsigned* keys_a, unsigned* keys_b, int* vals_a, int* vals_b, unsigned* hist /* [4][tiles][256] */,
    const unsigned* key_bits, unsigned* barrier /* zeroed */, int* __restrict__ rank_to_gid, int* __restrict__ rank_of) {
  constexpr int kWarps = kRankBlock / 32;
  constexpr int kTile = kRankBlock * kItems;
  __shared__ unsigned s_whist[kWarps][kRadix];
  __shared__ int s_scan[33];
  __shared__ uint4 s_part[2][4][kRadix / 4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (key_bits[7] && !key_bits[6]) return;  // launched as the fallback of the bucket ranking, which did the job
  const unsigned diff = key_bits[0] & key_bits[1];  // written by depth_keys_kernel (previous launch): plain loads
  const int bits = diff ? 32 - __clz(diff) : 0;
  const int passes = (bits + 7) >> 3;  // 0 .. 4
  unsigned bar_target = 0;
  const size_t hs = (size_t)tiles * kRadix;

  if (passes == 0) {  // every visible key equal: the order is the id order
    for (int i = blockIdx.x * kRankBlock + threadIdx.x; i < n; i += gridDim.x * kRankBlock) {
      rank_to_gid[i] = i;
      rank_of[i] = i;
    }
    return;
  }
  // per-warp digit counts of one tile's keys (registers k[]), left in s_whist; rank[] = rank among equal digits
  // inside the warp's chunk.  "Earlier in memory" == (smaller item index j, then smaller lane): stable.
  auto warp_ranks = [&](const unsigned (&k)[kItems], int warp_base, int shift, unsigned (&rank)[kItems]) {
    for (int d = lane; d < kRadix; d += 32) s_whist[warp][d] = 0;
    __syncwarp();
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      const int i = warp_base + j * 32 + lane;
      const bool valid = i < n;
      const unsigned dgt = (k[j] >> shift) & 0xffu;
      const unsigned peers = __match_any_sync(0xffffffffu, valid ? dgt : 0x100u);
      const unsigned lower = peers & ((1u << lane) - 1u);
      unsigned prev = 0;
      if (valid) prev = s_whist[warp][dgt];
      __syncwarp();
      rank[j] = prev + __popc(lower);
      if (valid && lower == 0u) s_whist[warp][dgt] = prev + __popc(peers);
      __syncwarp();
    }
  };
  for (int p = 0; p < passes; ++p) {
    const bool last = (p == passes - 1);
    const int shift = 8 * p;
    const unsigned* kin = (p & 1) ? keys_b : keys_a;
    unsigned* kout = (p & 1) ? keys_a : keys_b;
    const int* vin = (p == 0) ? nullptr : ((p & 1) ? vals_b : vals_a);
    int* vout = last ? rank_to_gid : ((p & 1) ? vals_a : vals_b);
    unsigned* hist_cur = hist + (size_t)p * hs;
    // ---- phase A (passes > 0; pass 0's table was written by depth_keys_kernel): this pass's digit histogram of every
    // tile, from the keys as the previous pass left them.  No global atomics: round 2's first version accumulated the
    // next table with one RED per key while scattering, and the concentrated top digit of a head's depths put hundreds of
    // REDs on the same address per tile (ncu: 6 % issue-active, 18 us per pass).
    if (p > 0) {
      for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int warp_base = tile * kTile + warp * (32 * kItems);
        unsigned k[kItems], rank[kItems];
#pragma unroll
        for (int j = 0; j < kItems; ++j) {
          const int i = warp_base + j * 32 + lane;
          k[j] = (i < n) ? __ldcg(kin + i) : 0xffffffffu;
        }
        warp_ranks(k, warp_base, shift, rank);
        __syncthreads();
        {
          unsigned c = 0;
#pragma unroll
          for (int w = 0; w < kWarps; ++w) c += s_whist[w][threadIdx.x];
          hist_cur[(size_t)tile * kRadix + threadIdx.x] = c;
        }
        __syncthreads();
      }
      grid_barrier(barrier, bar_target);
    }
    // ---- phase B: column prefix over the tiles, then the stable scatter
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
      const int warp_base = tile * kTile + warp * (32 * kItems);
      unsigned k[kItems];
      int v[kItems];
#pragma unroll
      for (int j = 0; j < kItems; ++j) {
        const int i = warp_base + j * 32 + lane;
        k[j] = (i < n) ? __ldcg(kin + i) : 0xffffffffu;
        v[j] = (i < n) ? (vin ? __ldcg(vin + i) : i) : 0;
      }
      {  // column sums of the tile-major table (see rank_scatter_kernel)
        const int g = threadIdx.x >> 6, c4 = threadIdx.x & 63;
        const uint4* tab = reinterpret_cast<const uint4*>(hist_cur);
        uint4 tot = make_uint4(0u, 0u, 0u, 0u), bef = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll 8
        for (int b = g; b < tiles; b += 4) {
          const uint4 h = __ldcg(tab + (size_t)b * (kRadix / 4) + c4);
          tot.x += h.x; tot.y += h.y; tot.z += h.z; tot.w += h.w;
          if (b < tile) { bef.x += h.x; bef.y += h.y; bef.z += h.z; bef.w += h.w; }
        }
        s_part[0][g][c4] = tot;
        s_part[1][g][c4] = bef;
      }
      __syncthreads();
      unsigned before = 0, total = 0;
      {
        const unsigned* pt = reinterpret_cast<const unsigned*>(&s_part[0][0][0]);
        const unsigned* pb = reinterpret_cast<const unsigned*>(&s_part[1][0][0]);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          total += pt[g * kRadix + threadIdx.x];
          before += pb[g * kRadix + threadIdx.x];
        }
      }
      int unused;
      const unsigned digit_base = (unsigned)block_exclusive_scan((int)total, s_scan, unused);
      const unsigned my_base = digit_base + before;
      unsigned rank[kItems];
      warp_ranks(k, warp_base, shift, rank);
      __syncthreads();
      {
        const int d = threadIdx.x;
        unsigned run = my_base;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
          const unsigned c = s_whist[w][d];
          s_whist[w][d] = run;
          run += c;
        }
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < kItems; ++j) {
        const int i = warp_base + j * 32 + lane;
        if (i < n) {
          const unsigned dgt = (k[j] >> shift) & 0xffu;
          const unsigned dst = s_whist[warp][dgt] + rank[j];
          if (!last) kout[dst] = k[j];
          else rank_of[v[j]] = (int)dst;
          vout[dst] = v[j];
        }
      }
      __syncthreads();  // shared tables are reused by the next tile of this CTA
    }
    if (!last) grid_barrier(barrier, bar_target);
  }
}

// ------------------------------------------------------------------ 2c. depth ranks by buckets (option, measured slower)
// MEASURED (profiles/r02_launches_head_buckets.txt): steps (1)-(3) below take 8 + 5 + 12 us, but step (4), the n^2 in-bucket
// ranking, executes 25.6 M warp instructions and takes 65 us at 300 k keys -- the cooperative sort stays the default; the
// code is kept for GOLIATH_B200_RANKSORT=buckets and as the tested fallback protocol (device flag -> cooperative sort).
// The idea: the cooperative LSD sort above is latency-bound: 147 CTAs of 8 warps walk 3 passes of dependent L2 round trips and
// grid barriers (ncu: 6 % issue-active, 44 us for 300 k keys).  The ranks only have to order the VISIBLE Gaussians
// by (depth bits, id), so: (1) the visible keys are dealt into 2048 buckets that split [min key, max key] evenly
// (monotone in the key: bucket order == depth order), counts privatised per CTA; (2) one CTA scans the counts;
// (3) the (key, id) pairs are scattered into their bucket (slots claimed per CTA, order inside a bucket arbitrary);
// (4) one CTA per bucket ranks its ~150 pairs against each other in shared memory (n^2 compares on (key, id): exact,
// ties by id).  Independent kernels with a handful of round trips each instead of a 3-pass dependency chain.  A bucket
// larger than kBucketCap (degenerate depth distributions, e.g. every depth equal) raises a device flag: the bucket
// kernels then do nothing and the cooperative LSD sort, launched behind them, takes over (otherwise it exits at once).
constexpr int kBuckets = 2048;
constexpr int kBucketCap = 2048;   // pairs of one bucket held in shared memory (16 KB)
constexpr int kBucketThreads = 128;

__device__ __forceinline__ int bucket_of(unsigned key, unsigned kmin, unsigned long long range) {
  return (int)(((unsigned long long)(key - kmin) * (unsigned long long)kBuckets) / range);
}

template <int kTileKeys>
__global__ void __launch_bounds__(kGaussBlock) rank_bucket_count_kernel(int G, const unsigned* __restrict__ keys,
                                                                        const int* __restrict__ radii,
                                                                        const unsigned* __restrict__ key_bits,
                                                                        int* __restrict__ bcount) {
  constexpr int kItems = kTileKeys / kGaussBlock;
  __shared__ int s_cnt[kBuckets];
  for (int t = threadIdx.x; t < kBuckets; t += kGaussBlock) s_cnt[t] = 0;
  const unsigned kmax = key_bits[4], kmin = ~key_bits[5];
  const unsigned long long range = (unsigned long long)(kmax - kmin) + 1ull;
  __syncthreads();
  const int base = blockIdx.x * kTileKeys;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int i = base + j * kGaussBlock + threadIdx.x;
    if (i < G && radii[i] > 0) atomicAdd(&s_cnt[bucket_of(keys[i], kmin, range)], 1);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < kBuckets; t += kGaussBlock) {
    const int c = s_cnt[t];
    if (c) atomicAdd(&bcount[t], c);
  }
}

__global__ void __launch_bounds__(1024) rank_bucket_scan_kernel(const int* __restrict__ bcount, int* __restrict__ boffset,
                                                                int* __restrict__ bcursor, unsigned* __restrict__ flags) {
  __shared__ int s_warp[33];
  __shared__ int s_max;
  if (threadIdx.x == 0) s_max = 0;
  __syncthreads();
  int carry = 0;
  for (int base = 0; base < kBuckets; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = bcount[i];
    int total;
    const int ex = block_exclusive_scan(v, s_warp, total);
    boffset[i] = carry + ex;
    bcursor[i] = 0;
    atomicMax(&s_max, v);
    carry += total;
  }
  __syncthreads();
  if (threadIdx.x == 0) flags[6] = (s_max > kBucketCap) ? 1u : 0u;  // 1: the cooperative LSD sort must do the ranking
}

template <int kTileKeys>
__global__ void __launch_bounds__(kGaussBlock) rank_bucket_scatter_kernel(int G, const unsigned* __restrict__ keys,
                                                                          const int* __restrict__ radii,
                                                                          const unsigned* __restrict__ key_bits,
                                                                          const int* __restrict__ boffset,
                                                                          int* __restrict__ bcursor,
                                                                          unsigned* __restrict__ pair_keys,
                                                                          int* __restrict__ pair_ids) {
  constexpr int kItems = kTileKeys / kGaussBlock;
  __shared__ int s_cnt[kBuckets];
  __shared__ int s_base[kBuckets];
  if (key_bits[6]) return;  // fallback path active
  for (int t = threadIdx.x; t < kBuckets; t += kGaussBlock) s_cnt[t] = 0;
  const unsigned kmax = key_bits[4], kmin = ~key_bits[5];
  const unsigned long long range = (unsigned long long)(kmax - kmin) + 1ull;
  __syncthreads();
  const int base = blockIdx.x * kTileKeys;
  unsigned k[kItems];
  int b[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int i = base + j * kGaussBlock + threadIdx.x;
    b[j] = -1;
    if (i < G && radii[i] > 0) {
      k[j] = keys[i];
      b[j] = bucket_of(k[j], kmin, range);
      atomicAdd(&s_cnt[b[j]], 1);
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < kBuckets; t += kGaussBlock) {
    const int c = s_cnt[t];
    s_base[t] = c ? boffset[t] + atomicAdd(&bcursor[t], c) : 0;
    s_cnt[t] = 0;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    if (b[j] < 0) continue;
    const int pos = s_base[b[j]] + atomicAdd(&s_cnt[b[j]], 1);
    pair_keys[pos] = k[j];
    pair_ids[pos] = base + j * kGaussBlock + threadIdx.x;
  }
}

__global__ void __launch_bounds__(kBucketThreads) rank_bucket_sort_kernel(const int* __restrict__ bcount,
                                                                          const int* __restrict__ boffset,
                                                                          const unsigned* __restrict__ key_bits,
                                                                          const unsigned* __restrict__ pair_keys,
                                                                          const int* __restrict__ pair_ids,
                                                                          int* __restrict__ rank_to_gid, int* __restrict__ rank_of) {
  __shared__ unsigned s_k[kBucketCap];
  __shared__ int s_id[kBucketCap];
  if (key_bits[6]) return;
  const int n = bcount[blockIdx.x], off = boffset[blockIdx.x];
  if (n <= 0) return;
  for (int i = threadIdx.x; i < n; i += kBucketThreads) {
    s_k[i] = pair_keys[off + i];
    s_id[i] = pair_ids[off + i];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += kBucketThreads) {
    const unsigned ki = s_k[i];
    const int idi = s_id[i];
    int r = 0;
    for (int j = 0; j < n; ++j) {  // every lane reads the same s_k[j] / s_id[j]: shared-memory broadcasts
      const unsigned kj = s_k[j];
      r += (kj < ki || (kj == ki && s_id[j] < idi)) ? 1 : 0;
    }
    rank_to_gid[off + r] = idi;
    rank_of[idi] = off + r;
  }
}

// ------------------------------------------------------------------ 3. bins from the tile counts (one CTA)
__global__ void __launch_bounds__(1024) tile_scan_kernel(int T, long long cap, const int* __restrict__ counts,
                                                         int2* __restrict__ tile_bins, int* __restrict__ cursor,
                                                         int* __restrict__ n_out, int* __restrict__ overflow) {
  __shared__ int s_warp[33];
  int carry = 0;
  for (int base = 0; base < T; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const int v = (i < T) ? counts[i] : 0;
    int total;
    const int ex = block_exclusive_scan(v, s_warp, total);
    if (i < T) {
      const int s = carry + ex;
      cursor[i] = s;
      const int cs = (int)min((long long)s, cap), ce = (int)min((long long)s + v, cap);
      tile_bins[i] = (ce > cs) ? make_int2(cs, ce) : make_int2(0, 0);  // empty tiles read (0,0), as after torch.zeros
    }
    carry += total;
  }
  if (threadIdx.x == 0) {
    if (n_out) *n_out = carry;
    if (overflow && (long long)carry > cap) *overflow = 1;  // capacity exceeded: caller must re-run
  }
}

// ------------------------------------------------------------------ 4. pairs into the tile buckets + per-Gaussian records
// smem_tiles = T: slots claimed per CTA through shared memory (s_cnt | s_base, 2*T ints); 0: one global atomic
// per (Gaussian, tile).  kGaussBlock threads x kScatItems Gaussians per CTA (see depth_keys_kernel).
// kById = false (rank path): a slot receives the Gaussian's depth RANK, the record table is indexed by rank.
// kById = true (per-tile sort path): a slot receives the Gaussian's 32-bit depth key in tile_ranks and its id in the
// same slot of slot_ids (the gids_sorted output); the record table is indexed by id.
template <bool kById>
__global__ void __launch_bounds__(kGaussBlock) tile_scatter_kernel(
    int G, const float2* __restrict__ xys, const int* __restrict__ radii, const int* __restrict__ rank_of,
    const float* __restrict__ conics, const float* __restrict__ colors3, const float* __restrict__ depths,
    const float* __restrict__ opacity, const float* __restrict__ comp, int tbx, int tby, int block_width,
    long long cap, int smem_tiles, int* __restrict__ cursor, int* __restrict__ tile_ranks, int* __restrict__ slot_ids,
    float4* __restrict__ rec_by_rank) {
  extern __shared__ int s_cnt[];
  int* s_base = s_cnt + smem_tiles;
  for (int t = threadIdx.x; t < smem_tiles; t += kGaussBlock) s_cnt[t] = 0;
  const int base = blockIdx.x * (kGaussBlock * kScatItems);
  int rk[kScatItems], r[kScatItems];  // rk: what goes into tile_ranks (rank, or depth key bits when kById)
  float2 c[kScatItems];
#pragma unroll
  for (int j = 0; j < kScatItems; ++j) {  // all loads first: independent, in flight together
    const int i = base + j * kGaussBlock + threadIdx.x;
    const bool in = i < G;
    r[j] = in ? radii[i] : 0;
    c[j] = in ? xys[i] : make_float2(0.f, 0.f);
    if (kById) rk[j] = in ? __float_as_int(depths[i]) : 0;
    else rk[j] = in ? rank_of[i] : 0;
  }
  __syncthreads();
  unsigned bx[kScatItems], by[kScatItems];  // x0 | x1 << 16, y0 | y1 << 16 (tile coordinates < 65536)
#pragma unroll
  for (int j = 0; j < kScatItems; ++j) {
    const int i = base + j * kGaussBlock + threadIdx.x;
    bx[j] = by[j] = 0u;
    if (r[j] <= 0) continue;
    int x0, y0, x1, y1;
    tile_bbox(c[j].x, c[j].y, (float)r[j], tbx, tby, block_width, x0, y0, x1, y1);
    bx[j] = (unsigned)x0 | ((unsigned)x1 << 16);
    by[j] = (unsigned)y0 | ((unsigned)y1 << 16);
    gb::pack_record_fused(i, xys, conics, colors3, depths, opacity, comp, rec_by_rank + 3 * (size_t)(kById ? i : rk[j]));
    for (int ty = y0; ty < y1; ++ty)
      for (int tx = x0; tx < x1; ++tx) {
        if (smem_tiles) {
          atomicAdd(&s_cnt[ty * tbx + tx], 1);
        } else {
          const int pos = atomicAdd(&cursor[ty * tbx + tx], 1);
          if ((long long)pos < cap) {
            tile_ranks[pos] = rk[j];
            if (kById) slot_ids[pos] = i;
          }
        }
      }
  }
  if (!smem_tiles) return;
  __syncthreads();
  for (int t = threadIdx.x; t < smem_tiles; t += kGaussBlock) {
    const int cnt = s_cnt[t];
    s_base[t] = cnt ? atomicAdd(&cursor[t], cnt) : 0;
    s_cnt[t] = 0;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kScatItems; ++j) {
    const int x0 = bx[j] & 0xffffu, x1 = bx[j] >> 16, y0 = by[j] & 0xffffu, y1 = by[j] >> 16;
    for (int ty = y0; ty < y1; ++ty)
      for (int tx = x0; tx < x1; ++tx) {
        const int t = ty * tbx + tx;
        const int pos = s_base[t] + atomicAdd(&s_cnt[t], 1);
        if ((long long)pos < cap) {
          tile_ranks[pos] = rk[j];
          if (kById) slot_ids[pos] = base + j * kGaussBlock + threadIdx.x;
        }
      }
  }
}

// ------------------------------------------------------------------ 5. per-tile bitmap sort + record copy
__global__ void __launch_bounds__(kSortThreads, 3) tile_sort_pack_kernel(
    int words /* ceil(G/32) */, int chunk /* bitmap words per thread, odd */, const int* __restrict__ order,
    const int2* __restrict__ tile_bins, const int* __restrict__ tile_ranks, const int* __restrict__ rank_to_gid,
    const float4* __restrict__ rec_by_rank, int* __restrict__ gids_sorted, float4* __restrict__ rec) {
  extern __shared__ unsigned s_bits[];
  __shared__ int s_warp[33];
  const int tile = order ? order[blockIdx.x] : (int)blockIdx.x;
  const int2 range = tile_bins[tile];
  const int n = range.y - range.x;
  if (n <= 0) return;  // uniform over the CTA
  for (int w = threadIdx.x; w < words; w += kSortThreads) s_bits[w] = 0u;
  __syncthreads();
  for (int i0 = threadIdx.x; i0 < n; i0 += 4 * kSortThreads) {  // 4 independent loads in flight per thread
    int r[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * kSortThreads;
      r[u] = (i < n) ? tile_ranks[range.x + i] : -1;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (r[u] >= 0) atomicOr(&s_bits[r[u] >> 5], 1u << (r[u] & 31));
  }
  __syncthreads();
  // thread t owns bitmap words [t*chunk, (t+1)*chunk): odd chunk -> conflict-free shared-memory reads
  const int w0 = threadIdx.x * chunk, w1 = min(words, w0 + chunk);
  int cnt = 0;
  for (int w = w0; w < w1; ++w) cnt += __popc(s_bits[w]);
  int total;
  int pos = range.x + block_exclusive_scan(cnt, s_warp, total);
  for (int w = w0; w < w1; ++w) {  // sorted RANKS, parked in gids_sorted until the copy loop below
    unsigned m = s_bits[w];
    while (m) {
      const int b = __ffs(m) - 1;
      m &= m - 1;
      gids_sorted[pos++] = w * 32 + b;
    }
  }
  __syncthreads();  // the ranks written above are read back below by other threads of this CTA
  for (int i0 = threadIdx.x; i0 < n; i0 += kCopyBatch * kSortThreads) {  // kCopyBatch records per thread per round trip
    int r[kCopyBatch], g[kCopyBatch];
    float4 q[kCopyBatch][3];
#pragma unroll
    for (int u = 0; u < kCopyBatch; ++u) {
      const int i = i0 + u * kSortThreads;
      r[u] = (i < n) ? __ldcg(gids_sorted + (size_t)range.x + i) : -1;
    }
#pragma unroll
    for (int u = 0; u < kCopyBatch; ++u) {
      if (r[u] < 0) continue;
      g[u] = rank_to_gid[r[u]];
      const float4* src = rec_by_rank + 3 * (size_t)r[u];
      q[u][0] = gb::ld_nc_f4(src);
      q[u][1] = gb::ld_nc_f4(src + 1);
      q[u][2] = gb::ld_nc_f4(src + 2);
    }
#pragma unroll
    for (int u = 0; u < kCopyBatch; ++u) {
      if (r[u] < 0) continue;
      const size_t idx = (size_t)range.x + i0 + u * kSortThreads;
      gids_sorted[idx] = g[u];
      rec[3 * idx + 0] = q[u][0];
      rec[3 * idx + 1] = q[u][1];
      rec[3 * idx + 2] = q[u][2];
    }
  }
}

// ------------------------------------------------------------------ 5b. the same in two kernels (default)
// tile_sort_pack_kernel is bound by its heaviest tiles: one CTA walks bitmap clear -> bucket loads -> popcount scan ->
// rank write-out -> rank read-back -> gid load -> 48-byte record gather -> store, eight dependent global round trips
// per tile (profiles/r02_launches_head.txt: 51 us against ~12 us of traffic).  Split: the per-tile kernel stops after
// writing the SORTED RANKS in place over the tile's bucket; a grid-wide kernel then turns every intersection's rank
// into its Gaussian id and its record, three threads per record (48 B = 3 x 16 B), fully parallel over the 1.08 M
// intersections whatever the tile lengths are.
__global__ void __launch_bounds__(kSortThreads, 3) tile_sort_kernel(int words, int chunk, const int* __restrict__ order,
                                                                    const int2* __restrict__ tile_bins,
                                                                    int* __restrict__ tile_ranks) {
  extern __shared__ unsigned s_bits[];
  __shared__ int s_warp[33];
  const int tile = order ? order[blockIdx.x] : (int)blockIdx.x;
  const int2 range = tile_bins[tile];
  const int n = range.y - range.x;
  if (n <= 0) return;  // uniform over the CTA
  for (int w = threadIdx.x; w < words; w += kSortThreads) s_bits[w] = 0u;
  __syncthreads();
  for (int i0 = threadIdx.x; i0 < n; i0 += 4 * kSortThreads) {
    int r[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * kSortThreads;
      r[u] = (i < n) ? tile_ranks[range.x + i] : -1;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (r[u] >= 0) atomicOr(&s_bits[r[u] >> 5], 1u << (r[u] & 31));
  }
  __syncthreads();  // every rank of the bucket is in the bitmap: the bucket may now be overwritten
  const int w0 = threadIdx.x * chunk, w1 = min(words, w0 + chunk);
  int cnt = 0;
  for (int w = w0; w < w1; ++w) cnt += __popc(s_bits[w]);
  int total;
  int pos = range.x + block_exclusive_scan(cnt, s_warp, total);
  for (int w = w0; w < w1; ++w) {
    unsigned m = s_bits[w];
    while (m) {
      const int b = __ffs(m) - 1;
      m &= m - 1;
      tile_ranks[pos++] = w * 32 + b;
    }
  }
}

// ------------------------------------------------------------------ 5c. per-tile (depth key, id) sort (default)
// The tile's slots hold (32-bit depth key, Gaussian id) pairs in arbitrary order.  One CTA per tile, longest first, forms
// the 64-bit composite (key - min visible key) << 32 | id — unique, and ordered exactly as the key sort orders the
// tile (depth bits, ties by ascending id) — and radix-sorts it in 8-bit digits (pair_sort_tile: key digits first).  Up to
// kPairCap pairs live in shared memory; a longer tile sorts in the 48-byte record slots of its own range of the records
// output (16 B per pair used), which only the record gather writes, later.
constexpr int kPairThreads = 512;
constexpr int kPairWarps = kPairThreads / 32;
constexpr int kPairCap = 6144;  // 2 x 48 KB ping-pong + 16 KB warp histograms = 112 KB: two CTAs per SM
constexpr size_t kPairSmem = (size_t)2 * kPairCap * 8 + (size_t)kPairWarps * kRadix * 4;

// Stable LSD radix sort of a[0, n) over the 8-bit digits in which `varying` has a bit, ping-ponging between a and b;
// returns the buffer that holds the result.  Warp w owns the contiguous chunk [w*per, (w+1)*per) and walks it 32 pairs
// at a time, so "earlier in the buffer" == "earlier warp, or earlier in the same warp's walk": the scatter is stable.
__device__ __forceinline__ unsigned long long* pair_radix_sort(unsigned long long* a, unsigned long long* b, int n,
                                                               unsigned long long varying, unsigned* s_hist, int* s_warp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int per = (n + kPairWarps - 1) / kPairWarps;
  const int c0 = min(n, warp * per), c1 = min(n, c0 + per);
  const unsigned lt = (1u << lane) - 1u;
  unsigned* h = s_hist + warp * kRadix;
  for (int shift = 0; shift < 64; shift += 8) {
    if (((varying >> shift) & 0xffull) == 0ull) continue;  // the same digit for every pair: identity pass
    for (int d = lane; d < kRadix; d += 32) h[d] = 0u;
    __syncwarp();
    for (int i = c0 + lane; i < c1; i += 32) atomicAdd(&h[(unsigned)(a[i] >> shift) & 0xffu], 1u);
    __syncthreads();
    {  // scatter bases, digit-major then warp: smaller digits anywhere + the same digit in earlier warps
      const int d = threadIdx.x;
      unsigned tot = 0u;
      if (d < kRadix)
        for (int w = 0; w < kPairWarps; ++w) tot += s_hist[w * kRadix + d];
      int unused;
      unsigned run = (unsigned)block_exclusive_scan((int)tot, s_warp, unused);
      if (d < kRadix)
        for (int w = 0; w < kPairWarps; ++w) {
          const unsigned c = s_hist[w * kRadix + d];
          s_hist[w * kRadix + d] = run;
          run += c;
        }
    }
    __syncthreads();
    for (int i0 = c0; i0 < c1; i0 += 32) {  // uniform over the warp
      const int i = i0 + lane;
      const bool valid = i < c1;
      const unsigned long long v = valid ? a[i] : 0ull;
      const unsigned dg = valid ? ((unsigned)(v >> shift) & 0xffu) : 0x100u;
      const unsigned peers = __match_any_sync(0xffffffffu, dg);
      const unsigned lower = peers & lt;
      const unsigned at = valid ? h[dg] : 0u;
      __syncwarp();
      if (valid) {
        b[at + __popc(lower)] = v;
        if (lower == 0u) h[dg] = at + __popc(peers);
      }
      __syncwarp();
    }
    __syncthreads();
    unsigned long long* t = a;
    a = b;
    b = t;
  }
  return a;
}

// load -> sort -> sorted ids back in place.  Inlined twice: with shared-memory buffers and with global scratch.
// The composite is (key - kmin) << 32 | id.  Depth ties are rare, so the tile is first sorted on the KEY digits only
// (about half the passes: ties come out in bucket order), then every run of equal keys is put in id order by the thread
// that owns its first element (insertion sort, runs of up to kMaxRun).  A longer run (all-equal or quantised depths)
// makes the CTA sort the whole composite instead, id digits included.
constexpr int kMaxRun = 32;
__device__ __forceinline__ void pair_sort_tile(unsigned long long* a, unsigned long long* b, int2 range,
                                               unsigned kmin, const unsigned* __restrict__ tile_keys,
                                               int* __restrict__ gids_sorted, unsigned* s_hist, int* s_warp,
                                               unsigned long long* s_or_and) {
  const int n = range.y - range.x;
  unsigned long long o = 0ull, an = ~0ull;
  for (int i0 = threadIdx.x; i0 < n; i0 += 4 * kPairThreads) {  // 4 independent load pairs in flight per thread
    unsigned k[4];
    int g[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * kPairThreads;
      k[u] = (i < n) ? tile_keys[range.x + i] : kmin;
      g[u] = (i < n) ? gids_sorted[range.x + i] : 0;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * kPairThreads;
      if (i < n) {
        const unsigned long long c = ((unsigned long long)(k[u] - kmin) << 32) | (unsigned)g[u];
        a[i] = c;
        o |= c;
        an &= c;
      }
    }
  }
  const unsigned olo = __reduce_or_sync(0xffffffffu, (unsigned)o), ohi = __reduce_or_sync(0xffffffffu, (unsigned)(o >> 32));
  const unsigned alo = __reduce_and_sync(0xffffffffu, (unsigned)an),
                 ahi = __reduce_and_sync(0xffffffffu, (unsigned)(an >> 32));
  if ((threadIdx.x & 31) == 0) {
    atomicOr(&s_or_and[0], ((unsigned long long)ohi << 32) | olo);
    atomicAnd(&s_or_and[1], ((unsigned long long)ahi << 32) | alo);
  }
  __syncthreads();  // composites stored, OR / AND complete
  const unsigned long long varying = s_or_and[0] & ~s_or_and[1];
  unsigned long long* res = pair_radix_sort(a, b, n, varying & 0xffffffff00000000ull, s_hist, s_warp);
  bool long_run = false;
  for (int i = threadIdx.x; i < n; i += kPairThreads) {
    const unsigned key = (unsigned)(res[i] >> 32);
    if (i > 0 && (unsigned)(res[i - 1] >> 32) == key) continue;  // not the first element of its run
    int e = i + 1;
    while (e < n && e - i <= kMaxRun && (unsigned)(res[e] >> 32) == key) ++e;
    if (e - i > kMaxRun) {
      long_run = true;
    } else {
      for (int j = i + 1; j < e; ++j) {  // same key: order by id
        const unsigned long long v = res[j];
        int p = j - 1;
        while (p >= i && res[p] > v) {
          res[p + 1] = res[p];
          --p;
        }
        res[p + 1] = v;
      }
    }
  }
  if (__syncthreads_or(long_run)) res = pair_radix_sort(res, res == a ? b : a, n, varying, s_hist, s_warp);
  for (int i = threadIdx.x; i < n; i += kPairThreads) gids_sorted[range.x + i] = (int)(unsigned)res[i];
}

__global__ void __launch_bounds__(kPairThreads, 2) tile_pair_sort_kernel(
    const int* __restrict__ order, const int2* __restrict__ tile_bins,
    const unsigned* __restrict__ key_bits /* [5] = ~min visible key */, const unsigned* __restrict__ tile_keys,
    int* __restrict__ gids_sorted, float* __restrict__ records /* scratch of oversized tiles */) {
  extern __shared__ unsigned long long s_pairs[];  // [2][kPairCap] | [kPairWarps][kRadix] unsigned
  __shared__ int s_warp[33];
  __shared__ unsigned long long s_or_and[2];
  const int tile = order ? order[blockIdx.x] : (int)blockIdx.x;
  const int2 range = tile_bins[tile];
  const int n = range.y - range.x;
  if (n <= 1) return;  // uniform over the CTA; one pair is sorted
  if (threadIdx.x == 0) {
    s_or_and[0] = 0ull;
    s_or_and[1] = ~0ull;
  }
  __syncthreads();
  const unsigned kmin = ~key_bits[5];
  unsigned* s_hist = reinterpret_cast<unsigned*>(s_pairs + 2 * kPairCap);
  if (n <= kPairCap) {
    pair_sort_tile(s_pairs, s_pairs + kPairCap, range, kmin, tile_keys, gids_sorted, s_hist, s_warp, s_or_and);
  } else {
    unsigned long long* a = reinterpret_cast<unsigned long long*>(records + 12 * (size_t)range.x);  // 48 B per slot
    pair_sort_tile(a, a + n, range, kmin, tile_keys, gids_sorted, s_hist, s_warp, s_or_and);
  }
}

// Late colours (gb_bin_tiles_pack_ev with an event): tile_scatter leaves the colour quarter of the per-Gaussian records
// empty and this kernel fills it once the colours exist — colours are the only input of the binning that comes from
// the shade, so everything before it can run beside the shade forward.  rank_of = NULL: the table is indexed by id.
__global__ void __launch_bounds__(256) rec_colors_kernel(int G, const int* __restrict__ radii,
                                                         const int* __restrict__ rank_of,
                                                         const float* __restrict__ colors3,
                                                         const float* __restrict__ depths, float4* __restrict__ rec_by_rank) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G || radii[g] <= 0) return;
  const size_t at = rank_of ? (size_t)rank_of[g] : (size_t)g;
  rec_by_rank[3 * at + 2] = make_float4(colors3[3 * (size_t)g], colors3[3 * (size_t)g + 1], colors3[3 * (size_t)g + 2],
                                        depths[g]);
}

// rank_to_gid = NULL (per-tile sort path): `ranks_sorted` already holds the sorted Gaussian ids (it is gids_sorted),
// the table is indexed by id and only the records are written.
__global__ void __launch_bounds__(256) gather_records_kernel(long long cap, const int* __restrict__ n_dev,
                                                             const int* ranks_sorted, const int* __restrict__ rank_to_gid,
                                                             const float4* __restrict__ rec_by_rank, int* gids_sorted,
                                                             float4* __restrict__ rec) {
  const long long n = min((long long)*n_dev, cap);
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // float4 index: record j / 3, part j % 3
  if (j >= 3 * n) return;
  const long long i = j / 3;
  const int part = (int)(j - 3 * i);
  const int r = ranks_sorted[i];
  rec[j] = gb::ld_nc_f4(rec_by_rank + 3 * (size_t)r + part);
  if (rank_to_gid && part == 0) gids_sorted[i] = rank_to_gid[r];
}

struct Layout {
  size_t counts, hist, buckets, sync, zero_bytes, cursor, keys_a, keys_b, vals_a, vals_b, rank_to_gid, rank_of, rec_by_rank,
      tile_ranks, total;
};
inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
inline Layout make_layout(int G, int T, int64_t cap) {
  const int g1 = G > 0 ? G : 1;
  const size_t ctas = (size_t)gb::cdiv(g1, kRankBlock * rank_items(g1));
  const size_t g4 = align256((size_t)g1 * 4);
  Layout l;
  size_t o = 0;
  l.counts = o; o += align256((size_t)T * 4);
  l.hist = o;   o += align256(ctas * kRadix * 4 * kRankPasses);
  l.buckets = o; o += align256((size_t)3 * 2048 * 4);  // bucket ranking: counts | offsets | cursors
  l.sync = o;   o += 256;                 // [0..1]: OR of the visible keys / of their complements, [2]: grid-barrier counter
  l.zero_bytes = o;                       // [counts | hist | sync] are zeroed with one memset per call
  l.cursor = o; o += align256((size_t)T * 4);
  l.keys_a = o; o += g4;
  l.keys_b = o; o += g4;
  l.vals_a = o; o += g4;
  l.vals_b = o; o += g4;
  l.rank_to_gid = o; o += g4;
  l.rank_of = o; o += g4;
  l.rec_by_rank = o; o += align256((size_t)g1 * 48);
  l.tile_ranks = o; o += align256((size_t)(cap > 0 ? cap : 1) * 4);
  l.total = o;
  return l;
}

// 1: the four radix passes as separate launches (round 1), 0: one cooperative kernel (default), 2: 2048 key buckets +
// in-bucket n^2 ranking (measured slower: 65 us for the in-bucket pass at 300k, profiles/r02_launches_head_buckets.txt).
// GOLIATH_B200_RANKSORT=passes|coop|buckets
int g_tile_sort_mode = -1;  // 0: per-tile bitmap sort + grid-wide record gather (default), 1: one kernel per tile (round 1)
int tile_sort_mode() {
  if (g_tile_sort_mode < 0) {
    const char* e = getenv("GOLIATH_B200_TILESORT");
    g_tile_sort_mode = (e && strcmp(e, "fused") == 0) ? 1 : 0;
  }
  return g_tile_sort_mode;
}
int g_bin_sort_mode = -1;  // 0: per-tile (depth key, id) sort (default), 1: depth ranks + per-tile rank ordering
int bin_sort_mode() {
  if (g_bin_sort_mode < 0) {
    const char* e = getenv("GOLIATH_B200_BINSORT");
    g_bin_sort_mode = (e && strcmp(e, "rank") == 0) ? 1 : 0;
  }
  return g_bin_sort_mode;
}
int g_rank_sort_mode = -1;  // 0: cooperative LSD sort, 1: four separate radix passes (round 1), 2: bucket ranking (+ fallback)
int rank_sort_mode() {
  if (g_rank_sort_mode < 0) {
    const char* e = getenv("GOLIATH_B200_RANKSORT");
    g_rank_sort_mode = !e ? 0 : strcmp(e, "passes") == 0 ? 1 : strcmp(e, "buckets") == 0 ? 2 : 0;
  }
  return g_rank_sort_mode;
}
int sm_count() {
  static int n[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return gb::kNumSMs;
  if (!n[dev]) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v < 1) v = gb::kNumSMs;
    n[dev] = v;
  }
  return n[dev];
}

template <int kItems>
int launch_rank_sort(int G, int ctas, const float* xys, const float* depths, const int32_t* radii, int tbx, int tby,
                     int block_width, int smem_tiles, unsigned* keys_a, unsigned* keys_b, int* vals_a, int* vals_b,
                     unsigned* hist, int* counts, int* buckets, unsigned* sync, int* rank_to_gid, int* rank_of, cudaStream_t s) {
  const size_t hs = (size_t)ctas * kRadix;
  depth_keys_kernel<kRankBlock * kItems, true><<<ctas, kGaussBlock, (size_t)smem_tiles * 4, s>>>(
      G, (const float2*)xys, depths, radii, tbx, tby, block_width, smem_tiles, keys_a, hist, counts, sync);
  const int mode = rank_sort_mode();
  if (mode == 2) {  // bucket ranking
    int* bcount = buckets;
    int* boffset = bcount + kBuckets;
    int* bcursor = boffset + kBuckets;
    rank_bucket_count_kernel<kRankBlock * kItems><<<ctas, kGaussBlock, 0, s>>>(G, keys_a, radii, sync, bcount);
    rank_bucket_scan_kernel<<<1, 1024, 0, s>>>(bcount, boffset, bcursor, sync);
    rank_bucket_scatter_kernel<kRankBlock * kItems><<<ctas, kGaussBlock, 0, s>>>(G, keys_a, radii, sync, boffset, bcursor, keys_b,
                                                                               vals_b);
    rank_bucket_sort_kernel<<<kBuckets, kBucketThreads, 0, s>>>(bcount, boffset, sync, keys_b, vals_b, rank_to_gid, rank_of);
    gb::count_launches(4);
  }
  if (mode == 0 || mode == 2) {
    int n = G, tiles = ctas;
    const unsigned* key_bits = sync;
    unsigned* barrier = sync + 2;
    void* args[] = {&n, &tiles, &keys_a, &keys_b, &vals_a, &vals_b, &hist, &key_bits, &barrier, &rank_to_gid, &rank_of};
    const int grid = ctas < sm_count() ? ctas : sm_count();  // one CTA per SM at most: co-resident by construction
    // mode 2: sync[7] = 1 tells the cooperative kernel it is only the fallback (it exits unless sync[6] was raised)
    if (mode == 2) GB_CUDA(cudaMemsetAsync(sync + 7, 0xff, 4, s));
    GB_CUDA(cudaLaunchCooperativeKernel((const void*)rank_sort_coop_kernel<kItems>, dim3(grid), dim3(kRankBlock), args, 0, s));
    gb::count_launches(2);
    return 0;
  }
  // pass 0: a -> b (ids = identity), 1: b -> a, 2: a -> b, 3: b -> a (ids only) => rank_to_gid = vals_a
  rank_scatter_kernel<kItems><<<ctas, kRankBlock, 0, s>>>(G, keys_a, nullptr, keys_b, vals_b, 0, ctas, hist, hist + hs,
                                                          nullptr);
  rank_scatter_kernel<kItems><<<ctas, kRankBlock, 0, s>>>(G, keys_b, vals_b, keys_a, vals_a, 8, ctas, hist + hs,
                                                          hist + 2 * hs, nullptr);
  rank_scatter_kernel<kItems><<<ctas, kRankBlock, 0, s>>>(G, keys_a, vals_a, keys_b, vals_b, 16, ctas, hist + 2 * hs,
                                                          hist + 3 * hs, nullptr);
  rank_scatter_kernel<kItems><<<ctas, kRankBlock, 0, s>>>(G, keys_b, vals_b, nullptr, rank_to_gid, 24, ctas, hist + 3 * hs,
                                                          nullptr, rank_of);
  gb::count_launches(5);
  return 0;
}

// opt in to the large dynamic shared-memory window, once per device and kernel
template <typename K>
int opt_in_smem(K kernel, bool* done) {
  int dev = 0;
  GB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !done[dev]) {
    GB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxBitmapBytes));
    if (dev >= 0 && dev < 64) done[dev] = true;
  }
  return 0;
}

}  // namespace

// Ordering of gb_bin_tiles_pack[_ev]: 0 = per-tile sort of (depth key, id) pairs (default), 1 = depth ranks + per-tile
// rank ordering, whose variants the rank / tile sort modes below select (gb_bin_tiles_ranked always uses ranks).
// Identical outputs; the switches exist for A/B timing and the tests.
GB_API int gb_get_bin_sort_mode(void) { return bin_sort_mode(); }
GB_API void gb_set_bin_sort_mode(int mode) { g_bin_sort_mode = mode ? 1 : 0; }
// Depth-rank sort of the rank path: 0 = one cooperative kernel over the varying key bits (default), 1 = four
// radix passes as separate launches (round 1), 2 = bucket ranking.  Per-tile rank ordering: 0 = bitmap sort + grid-wide
// record gather (default), 1 = one kernel per tile (round 1).
GB_API int gb_get_tile_sort_mode(void) { return tile_sort_mode(); }
GB_API void gb_set_tile_sort_mode(int mode) { g_tile_sort_mode = mode ? 1 : 0; }
GB_API int gb_get_rank_sort_mode(void) { return rank_sort_mode(); }
GB_API void gb_set_rank_sort_mode(int mode) { g_rank_sort_mode = mode < 0 ? 0 : (mode > 2 ? 2 : mode); }

// 1 when gb_bin_tiles_pack supports G Gaussians (one tile's rank bitmap must fit in shared memory)
GB_API int gb_bin_tiles_supported(int G) { return G >= 1 && ((size_t)gb::cdiv(G, 32) * 4 <= (size_t)kMaxBitmapBytes); }

GB_API size_t gb_bin_tiles_workspace_bytes(int G, int num_tiles, int64_t cap) {
  return make_layout(G, num_tiles, cap).total;
}

// Binning + record packing of the fused render (see the header of this file).  Outputs: tile_bins [T,2],
// tile_order [T] (longest list first; with tile_sched = 1 an SM-affine schedule of gb_tile_schedule_ints(T)
// int32, see gb_tile_schedule), gids_sorted [cap], records [cap,12]; n_out (device int32, may be
// null) receives the true intersection count, *overflow is set to 1 when it exceeds `cap` (the excess is
// dropped).  Never allocates, never synchronises; capturable in a CUDA graph.
GB_API int gb_bin_tiles_pack(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                             const float* colors3, const float* opacity, const float* compensation, int img_h,
                             int img_w, int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order,
                             int tile_sched, int32_t* gids_sorted, float* records, int32_t* n_out, int32_t* overflow,
                             void* workspace, void* stream) {
  return gb_bin_tiles_pack_ev(G, xys, depths, radii, conics, colors3, opacity, compensation, img_h, img_w, block_width, cap,
                              tile_bins, tile_order, tile_sched, gids_sorted, records, n_out, overflow, workspace, nullptr,
                              stream);
}

// Same, with the colours allowed to arrive late: `colors_ready` (a cudaEvent_t recorded on the stream that produces
// colors3, or NULL) is waited for on `stream` just before the first kernel that reads colors3 — with the split tile
// sort (default) a small kernel that fills the colour quarter of the by-rank records after the per-tile sort — so depth
// ranks, tile buckets and the per-tile sort overlap the caller's shade.
static int bin_tiles_impl(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                          const float* colors3, const float* opacity, const float* compensation, int img_h, int img_w,
                          int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order, int tile_sched,
                          int32_t* gids_sorted, float* records, int32_t* n_out, int32_t* overflow, void* workspace,
                          void* colors_ready, void* stream, int32_t* ext_ranks, float* ext_rec, int32_t* ext_r2g);

GB_API int gb_bin_tiles_pack_ev(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                                const float* colors3, const float* opacity, const float* compensation, int img_h,
                                int img_w, int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order,
                                int tile_sched, int32_t* gids_sorted, float* records, int32_t* n_out, int32_t* overflow,
                                void* workspace, void* colors_ready, void* stream) {
  return bin_tiles_impl(G, xys, depths, radii, conics, colors3, opacity, compensation, img_h, img_w, block_width, cap,
                        tile_bins, tile_order, tile_sched, gids_sorted, records, n_out, overflow, workspace, colors_ready,
                        stream, nullptr, nullptr, nullptr);
}

// Binning WITHOUT the sorted-record gather, for the blend kernels that stage records by rank (gb_rasterize_ranked_*):
// ranks_sorted [cap] (per tile, the depth ranks in blend order), rec_by_rank [G,12] (one 48-byte record per Gaussian, at
// its depth rank) and rank_to_gid [G] are written to the CALLER's arrays (they must outlive the backward; the shared
// workspace does not).  Everything else as gb_bin_tiles_pack_ev.  Saves the 52 MB write + read of the sorted records
// and holds 14.4 + 4 I bytes per view for the backward instead of 52 I.
GB_API int gb_bin_tiles_ranked(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                               const float* colors3, const float* opacity, const float* compensation, int img_h,
                               int img_w, int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order,
                               int tile_sched, int32_t* ranks_sorted, float* rec_by_rank, int32_t* rank_to_gid,
                               int32_t* n_out, int32_t* overflow, void* workspace, void* colors_ready, void* stream) {
  if (!ranks_sorted || !rec_by_rank || !rank_to_gid) return (int)cudaErrorInvalidValue;
  return bin_tiles_impl(G, xys, depths, radii, conics, colors3, opacity, compensation, img_h, img_w, block_width, cap,
                        tile_bins, tile_order, tile_sched, nullptr, nullptr, n_out, overflow, workspace, colors_ready, stream,
                        ranks_sorted, rec_by_rank, rank_to_gid);
}

static int bin_tiles_impl(int G, const float* xys, const float* depths, const int32_t* radii, const float* conics,
                          const float* colors3, const float* opacity, const float* compensation, int img_h, int img_w,
                          int block_width, int64_t cap, int32_t* tile_bins, int32_t* tile_order, int tile_sched,
                          int32_t* gids_sorted, float* records, int32_t* n_out, int32_t* overflow, void* workspace,
                          void* colors_ready, void* stream, int32_t* ext_ranks, float* ext_rec, int32_t* ext_r2g) {
  if (!gb_bin_tiles_supported(G) || block_width < 1 || cap < 0) return (int)cudaErrorInvalidValue;
  cudaStream_t s = (cudaStream_t)stream;
  const int tbx = gb::cdiv(img_w, block_width), tby = gb::cdiv(img_h, block_width);
  const int T = tbx * tby;
  if (T < 1 || tbx > 65535 || tby > 65535) return (int)cudaErrorInvalidValue;
  const Layout l = make_layout(G, T, cap);
  char* ws = (char*)workspace;
  int* counts = (int*)(ws + l.counts);
  unsigned* hist = (unsigned*)(ws + l.hist);
  int* cursor = (int*)(ws + l.cursor);
  unsigned* keys_a = (unsigned*)(ws + l.keys_a);
  unsigned* keys_b = (unsigned*)(ws + l.keys_b);
  int* vals_a = (int*)(ws + l.vals_a);
  int* vals_b = (int*)(ws + l.vals_b);
  const bool ranked = ext_ranks != nullptr;  // outputs for the rank-staging blend: no sorted-record gather
  int* rank_to_gid = ranked ? ext_r2g : (int*)(ws + l.rank_to_gid);
  unsigned* sync = (unsigned*)(ws + l.sync);
  int* rank_of = (int*)(ws + l.rank_of);
  float4* rec_by_rank = ranked ? (float4*)ext_rec : (float4*)(ws + l.rec_by_rank);
  int* tile_ranks = ranked ? ext_ranks : (int*)(ws + l.tile_ranks);
  const int items = rank_items(G);
  const int ctas = gb::cdiv(G, kRankBlock * items);
  const int smem_tiles = (T <= kMaxSmemTiles) ? T : 0;
  // per-tile sort of (depth key, id) pairs: no depth ranks; the by-rank table becomes a by-id table
  const bool by_id = !ranked && bin_sort_mode() == 0;
  static bool s_opt_k8[64] = {}, s_opt_k16[64] = {}, s_opt_scat[64] = {}, s_opt_sort[64] = {}, s_opt_sort2[64] = {};
  static bool s_opt_k8i[64] = {}, s_opt_k16i[64] = {}, s_opt_scati[64] = {}, s_opt_pair[64] = {};
  if ((size_t)smem_tiles * 8 > 40 * 1024) {
    int e = by_id ? ((items == 8) ? opt_in_smem(depth_keys_kernel<kRankBlock * 8, false>, s_opt_k8i)
                                  : opt_in_smem(depth_keys_kernel<kRankBlock * 16, false>, s_opt_k16i))
                  : ((items == 8) ? opt_in_smem(depth_keys_kernel<kRankBlock * 8, true>, s_opt_k8)
                                  : opt_in_smem(depth_keys_kernel<kRankBlock * 16, true>, s_opt_k16));
    if (e) return e;
    e = by_id ? opt_in_smem(tile_scatter_kernel<true>, s_opt_scati) : opt_in_smem(tile_scatter_kernel<false>, s_opt_scat);
    if (e) return e;
  }

  GB_CUDA(cudaMemsetAsync(ws, 0, l.zero_bytes, s));
  if (by_id) {
    if (items == 8)
      depth_keys_kernel<kRankBlock * 8, false><<<ctas, kGaussBlock, (size_t)smem_tiles * 4, s>>>(
          G, (const float2*)xys, depths, radii, tbx, tby, block_width, smem_tiles, nullptr, nullptr, counts, sync);
    else
      depth_keys_kernel<kRankBlock * 16, false><<<ctas, kGaussBlock, (size_t)smem_tiles * 4, s>>>(
          G, (const float2*)xys, depths, radii, tbx, tby, block_width, smem_tiles, nullptr, nullptr, counts, sync);
    gb::count_launches(1);
  } else {
    const int es = (items == 8)
                       ? launch_rank_sort<8>(G, ctas, xys, depths, radii, tbx, tby, block_width, smem_tiles, keys_a, keys_b,
                                             vals_a, vals_b, hist, counts, (int*)(ws + l.buckets), sync, rank_to_gid, rank_of, s)
                       : launch_rank_sort<16>(G, ctas, xys, depths, radii, tbx, tby, block_width, smem_tiles, keys_a, keys_b,
                                              vals_a, vals_b, hist, counts, (int*)(ws + l.buckets), sync, rank_to_gid, rank_of, s);
    if (es) return es;
  }
  int* n_total = n_out ? n_out : (int*)(sync + 3);  // the record gather below needs the count on the device
  tile_scan_kernel<<<1, 1024, 0, s>>>(T, (long long)cap, counts, (int2*)tile_bins, cursor, n_total, overflow);
  gb::count_launches(1);
  GB_CHECK_LAUNCH();
  const int e = tile_sched ? gb_tile_schedule(T, tile_bins, tile_order, stream)
                           : gb_tile_order(T, tile_bins, tile_order, stream);
  if (e) return e;
  const bool split = by_id || ranked || tile_sort_mode() == 0;
  const bool late = split && colors_ready;  // the colour quarter of the per-Gaussian records is filled after the tile sort
  if (!late && colors_ready) GB_CUDA(cudaStreamWaitEvent(s, (cudaEvent_t)colors_ready, 0));
  const int scat_ctas = gb::cdiv(G, kGaussBlock * kScatItems);
  if (by_id) {
    // tile_ranks receives the depth keys, gids_sorted the ids; the table at rec_by_rank is indexed by id
    tile_scatter_kernel<true><<<scat_ctas, kGaussBlock, (size_t)smem_tiles * 8, s>>>(
        G, (const float2*)xys, radii, nullptr, conics, late ? nullptr : colors3, depths, opacity, compensation, tbx, tby,
        block_width, (long long)cap, smem_tiles, cursor, tile_ranks, gids_sorted, rec_by_rank);
    if (cap > 0) {
      const int e2 = opt_in_smem(tile_pair_sort_kernel, s_opt_pair);
      if (e2) return e2;
      tile_pair_sort_kernel<<<T, kPairThreads, kPairSmem, s>>>(tile_order, (const int2*)tile_bins, sync,
                                                               (const unsigned*)tile_ranks, gids_sorted, records);
    }
    if (late) {
      GB_CUDA(cudaStreamWaitEvent(s, (cudaEvent_t)colors_ready, 0));
      rec_colors_kernel<<<gb::cdiv(G, 256), 256, 0, s>>>(G, radii, nullptr, colors3, depths, rec_by_rank);
      gb::count_launches(1);
    }
    if (cap > 0)
      gather_records_kernel<<<(unsigned)gb::cdiv64(3 * cap, 256), 256, 0, s>>>((long long)cap, n_total, gids_sorted, nullptr,
                                                                               rec_by_rank, gids_sorted, (float4*)records);
    gb::count_launches(3);
    GB_CHECK_LAUNCH();
    return 0;
  }
  tile_scatter_kernel<false><<<scat_ctas, kGaussBlock, (size_t)smem_tiles * 8, s>>>(
      G, (const float2*)xys, radii, rank_of, conics, late ? nullptr : colors3, depths, opacity, compensation, tbx, tby,
      block_width, (long long)cap, smem_tiles, cursor, tile_ranks, nullptr, rec_by_rank);
  const int words = gb::cdiv(G, 32);
  const int chunk = gb::cdiv(words, kSortThreads) | 1;
  const size_t smem = (size_t)words * 4;
  if (split) {
    if (smem > 40 * 1024) {
      const int e2 = opt_in_smem(tile_sort_kernel, s_opt_sort2);
      if (e2) return e2;
    }
    tile_sort_kernel<<<T, kSortThreads, smem, s>>>(words, chunk, tile_order, (const int2*)tile_bins, tile_ranks);
    if (late) {
      GB_CUDA(cudaStreamWaitEvent(s, (cudaEvent_t)colors_ready, 0));
      rec_colors_kernel<<<gb::cdiv(G, 256), 256, 0, s>>>(G, radii, rank_of, colors3, depths, rec_by_rank);
      gb::count_launches(1);
    }
    if (cap > 0 && !ranked)
      gather_records_kernel<<<(unsigned)gb::cdiv64(3 * cap, 256), 256, 0, s>>>((long long)cap, n_total, tile_ranks, rank_to_gid,
                                                                             rec_by_rank, gids_sorted, (float4*)records);
    gb::count_launches(3);
    GB_CHECK_LAUNCH();
    return 0;
  }
  if (smem > 40 * 1024) {
    const int e2 = opt_in_smem(tile_sort_pack_kernel, s_opt_sort);
    if (e2) return e2;
  }
  tile_sort_pack_kernel<<<T, kSortThreads, smem, s>>>(words, chunk, tile_order, (const int2*)tile_bins, tile_ranks,
                                                      rank_to_gid, rec_by_rank, gids_sorted, (float4*)records);
  gb::count_launches(2);
  GB_CHECK_LAUNCH();
  return 0;
}
