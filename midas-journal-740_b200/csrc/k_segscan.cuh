// k_segscan.cuh — K2b: single-pass exclusive scan of the per-entry (vertex, face, active-corner) counts, kept
// at SEGMENT granularity.
//
// Replaces, for id assignment, the per-slice vertex lookup of the reference (VertexLookupMap h:273-313, used at
// txx:186-191): ids follow from an exclusive prefix sum, in voxel-raster order, of "corners first touched by
// this voxel" (vertex ids, nextVertexId txx:116,189-190) and "faces of this voxel" (cell ids, nextCellId
// txx:117,197-202).  The third quantity, active corners per corner word in corner-raster order, indexes the
// corner -> id map.
//
// K2a (k_sweep.cuh) leaves one packed count per entry of the [Zl+1][EY][EW] lattice (owned corners |
// faces << 10 | active corners << 20).  Round 1 expanded them into three dense offset arrays (4 B in, 12 B out
// per entry, 0.6 GB for 1024^3).  Every consumer (k_vertices, k_faces, k_points_raster) is organised as
// "one warp = 32 consecutive entries of a lattice row", so all it needs is the prefix at the START of its
// segment: the rest is a warp shuffle scan of counts it has in registers anyway.  This kernel therefore writes
// one uint4 {vertices, faces, active corners, -} per 32-entry segment of a row (NS = ceil(EW/32) segments per
// row): 4 B in, 0.5 B out per entry.  ONE dense array remains, the active-corner prefix cofs (the slot bases): it
// is gathered per VERTEX by k_vertices, which has no warp-per-row structure to scan in, and rebuilding it in
// k_faces with two more warp scans cost more issue slots than the four loads (measured in r2).  k_assign writes
// it (coalesced, its warp scan carries the counts along); this kernel can too (`cofs`), with strided stores.
//
// Structure: one large tile (whole lattice rows) per resident CTA, chained with decoupled look-back (flag +
// value in one 64-bit descriptor per tile and quantity, tiles handed out by an atomic ticket so that a tile
// only ever waits for tiles that started before it).  Inside a tile every warp owns a contiguous run of rows:
//   pass 1  the warp sums its rows (coalesced 16-byte loads)  -> CTA aggregate -> look-back -> tile prefix
//   pass 2  the warp walks its rows again (L1/L2), one lane per row, 32 rows at a time, and writes the segment bases.
#pragma once
#include <climits>

#include "cbr_common.cuh"

namespace cbr {

constexpr int kScanThreads = 256;
constexpr int kScanWarps = kScanThreads / 32;

constexpr uint64_t kFlagShift = 62;
constexpr uint64_t kFlagAggregate = 1ull << kFlagShift;
constexpr uint64_t kFlagPrefix = 2ull << kFlagShift;
constexpr uint64_t kValueMask = (1ull << kFlagShift) - 1ull;

// slots of the per-run info block in device memory (unsigned long long[kInfoWords]); everything the emission
// kernels need to know about the counts lives here, so that a step can be queued without a host round trip
enum {
  kInfoTotV = 0, kInfoTotF = 1, kInfoTotC = 2,      // totals of the scanned range
  kInfoMarkV = 3, kInfoMarkF = 4, kInfoMarkC = 5,   // prefixes at the first own entry / at the second own corner plane
  kInfoPoints = 6, kInfoQuads = 7,                  // what the handle's own range produces
  kInfoPointBase = 8, kInfoCellBase = 9,            // global id bases (cub_set_id_base / the count exchange)
  kInfoIdDelta = 10,                                // scan-relative vertex id -> final id (mod 2^64)
  kInfoGhostV = 11,                                 // scan-relative ids below this one belong to the slab underneath
  kInfoFlags = 12,                                  // bit 0: a result buffer was too small; bit 1: an interior slice of the range is empty
  kInfoWork = 13,                                   // work counter of the projection kernel
  kInfoSplitWork = 14,
  kInfoFits = 15,                                   // written by k_check_caps: the emission fits its buffers
  kInfoWords = 16
};
enum { kFlagBufferOverflow = 1, kFlagEmptyInteriorSlice = 2, kFlagIdOverflow = 4 };

// Capacities of the result buffers.  k_check_caps compares them with the device-side counts ONCE per emission, and
// every emission kernel reads its verdict: the whole emission is skipped (and flagged: cub_finish redoes it with
// larger buffers) if anything would not fit - no per-item checks.  An emission queued before the host knows the
// counts (cub_emit_async) can fail the check; one whose buffers were sized from the counts always passes it.
struct Caps {
  unsigned long long points, perm, quads;
  int raster;
};
// one thread, queued in front of every emission: the verdict every emission kernel reads
__global__ void k_check_caps(unsigned long long* info, Caps c) {
  pdl_enter();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const unsigned long long tv = info[kInfoTotV], tc = info[kInfoTotC], q = info[kInfoTotF] - info[kInfoMarkF];
  const bool fits = (c.raster ? tc : tv) <= c.points && (c.raster || tc <= c.perm) && q <= c.quads;
  info[kInfoFits] = fits ? 1ull : 0ull;
  if (!fits) info[kInfoFlags] |= (unsigned long long)kFlagBufferOverflow;
}
__device__ __forceinline__ bool emission_fits(const unsigned long long* __restrict__ info) {
  return __ldg(info + kInfoFits) != 0ull;
}

struct SegScanArgs {
  const uint32_t* cnt;
  uint4* seg;                    // [rows of the lattice][NS] exclusive prefixes at the start of every segment
  uint32_t* cofs;                // entry lattice: dense exclusive prefix of the active-corner counts, or null
  unsigned row_begin, n_rows;    // scanned lattice rows [row_begin, row_begin + n_rows): whole planes
  unsigned EW, NS;               // entries / segments per row
  unsigned ghost_row_end;        // active corners of rows below this one belong to the slab underneath: not counted
  unsigned mark_row_vf;          // row whose first segment base is the (vertex, face) mark, or UINT_MAX
  unsigned mark_row_c;           // ... the active-corner mark, or UINT_MAX
  unsigned rows_per_tile;        // a multiple of kScanWarps
  unsigned n_tiles;
  unsigned long long* status;    // [3][n_tiles] descriptors
  unsigned int* ticket;
  unsigned long long* info;      // kInfo* slots
};

__device__ __forceinline__ unsigned long long ld_relaxed(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// one warp: sum of the aggregates of all tiles before `tile`
__device__ __forceinline__ unsigned long long lookback(const unsigned long long* status, int tile, int lane) {
  unsigned long long exclusive = 0;
  int pos = tile - 1;
  while (true) {
    const int idx = pos - lane;
    unsigned long long d = kFlagPrefix;  // virtual tiles before tile 0: inclusive prefix 0
    if (idx >= 0) {
      d = ld_relaxed(status + idx);
      while ((d >> kFlagShift) == 0) d = ld_relaxed(status + idx);
    }
    const unsigned has_prefix = __ballot_sync(0xffffffffu, (d >> kFlagShift) == 2);
    const int first = has_prefix ? (__ffs(has_prefix) - 1) : 32;
    unsigned long long v = (lane <= first) ? (d & kValueMask) : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    exclusive += v;
    if (has_prefix) break;
    pos -= 32;
  }
  return exclusive;
}

__global__ void __launch_bounds__(kScanThreads) k_seg_scan(const SegScanArgs a) {
  pdl_enter();
  __shared__ unsigned int s_tile;
  __shared__ unsigned long long s_part[3][kScanWarps];
  __shared__ unsigned long long s_excl[3];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
  __syncthreads();
  const unsigned tile = s_tile;
  if (tile >= a.n_tiles) return;
  // rows of this warp: a contiguous run inside the tile
  const unsigned rpw = a.rows_per_tile / kScanWarps;
  const unsigned r0 = min(tile * a.rows_per_tile + warp * rpw, a.n_rows);
  const unsigned r1 = min(r0 + rpw, a.n_rows);

  // ---- pass 1: the warp's aggregate (coalesced 16-byte loads over its run of rows) ---------------------------
  unsigned long long sv = 0, sf = 0, sc = 0;
  {
    const size_t e0 = (size_t)(a.row_begin + r0) * a.EW, e1 = (size_t)(a.row_begin + r1) * a.EW;  // multiples of 4
    const size_t ghost_end = (size_t)a.ghost_row_end * a.EW;
    for (size_t e = e0 + 4 * (size_t)lane; e < e1; e += 128) {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(a.cnt + e));
      // three 10-bit fields; four entries fit a 32-bit accumulator per field (a group of 4 never straddles rows)
      const uint32_t v4 = (q.x & 0x3ffu) + (q.y & 0x3ffu) + (q.z & 0x3ffu) + (q.w & 0x3ffu);
      const uint32_t f4 = ((q.x >> 10) & 0x3ffu) + ((q.y >> 10) & 0x3ffu) + ((q.z >> 10) & 0x3ffu) + ((q.w >> 10) & 0x3ffu);
      const uint32_t c4 = (q.x >> 20) + (q.y >> 20) + (q.z >> 20) + (q.w >> 20);
      sv += v4; sf += f4;
      if (e >= ghost_end) sc += c4;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sv += __shfl_xor_sync(0xffffffffu, sv, o);
      sf += __shfl_xor_sync(0xffffffffu, sf, o);
      sc += __shfl_xor_sync(0xffffffffu, sc, o);
    }
  }
  if (lane == 0) { s_part[0][warp] = sv; s_part[1][warp] = sf; s_part[2][warp] = sc; }
  __syncthreads();
  if (warp < 3) {
    // warps 0..2 chain one quantity each, concurrently
    const int k = warp;
    unsigned long long aggk = 0;
#pragma unroll
    for (int i = 0; i < kScanWarps; ++i) aggk += s_part[k][i];
    unsigned long long* st = a.status + (size_t)k * a.n_tiles;
    if (lane == 0) st_relaxed(st + tile, (tile == 0 ? kFlagPrefix : kFlagAggregate) | aggk);
    unsigned long long ex = 0;
    if (tile > 0) {
      ex = lookback(st, (int)tile, lane);
      if (lane == 0) st_relaxed(st + tile, kFlagPrefix | (ex + aggk));
    }
    if (lane == 0) {
      s_excl[k] = ex;
      if (tile == a.n_tiles - 1) a.info[kInfoTotV + k] = ex + aggk;  // last tile: grand totals
    }
  }
  __syncthreads();
  // exclusive prefix of this warp's run
  unsigned long long run_v = s_excl[0], run_f = s_excl[1], run_c = s_excl[2];
  for (int i = 0; i < warp; ++i) { run_v += s_part[0][i]; run_f += s_part[1][i]; run_c += s_part[2][i]; }

  // ---- pass 2: segment bases.  One lane per row, 32 rows of the warp's run at a time: the lane sums its row
  // (all loads independent), a warp scan over the 32 rows gives every row's prefix, and the lane walks its row
  // once more (L1) to write the prefix at the start of every 32-entry segment. ------------------------------
  uint32_t v = (uint32_t)run_v, f = (uint32_t)run_f, c = (uint32_t)run_c;  // (a handle's totals fit 32 bits: cub_count checks)
  const unsigned ew4 = a.EW / 4;
  for (unsigned rb = r0; rb < r1; rb += 32) {
    const unsigned r = rb + lane;
    const bool live = r < r1;
    const unsigned row = a.row_begin + (live ? r : r1 - 1);
    const uint4* __restrict__ p = reinterpret_cast<const uint4*>(a.cnt + (size_t)row * a.EW);
    const bool counted = row >= a.ghost_row_end;
    uint32_t tv = 0, tf = 0, tc = 0;
    if (live) {
      for (unsigned k = 0; k < ew4; ++k) {
        const uint4 q = __ldg(p + k);
        tv += (q.x & 0x3ffu) + (q.y & 0x3ffu) + (q.z & 0x3ffu) + (q.w & 0x3ffu);
        tf += ((q.x >> 10) & 0x3ffu) + ((q.y >> 10) & 0x3ffu) + ((q.z >> 10) & 0x3ffu) + ((q.w >> 10) & 0x3ffu);
        tc += (q.x >> 20) + (q.y >> 20) + (q.z >> 20) + (q.w >> 20);
      }
      if (!counted) tc = 0;
    }
    uint32_t iv = tv, jf = tf, ic = tc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t x = __shfl_up_sync(0xffffffffu, iv, o), y = __shfl_up_sync(0xffffffffu, jf, o), z = __shfl_up_sync(0xffffffffu, ic, o);
      if (lane >= o) { iv += x; jf += y; ic += z; }
    }
    if (live) {
      uint32_t bv = v + iv - tv, bf = f + jf - tf, bc = c + ic - tc;  // prefix at the start of the lane's row
      if (row == a.mark_row_vf) { a.info[kInfoMarkV] = bv; a.info[kInfoMarkF] = bf; }
      if (row == a.mark_row_c) a.info[kInfoMarkC] = bc;
      uint4* __restrict__ out = a.seg + (size_t)row * a.NS;
      uint4* __restrict__ co = a.cofs ? reinterpret_cast<uint4*>(a.cofs + (size_t)row * a.EW) : nullptr;
      for (unsigned k = 0; k < ew4; ++k) {
        if ((k & 7u) == 0) out[k >> 3] = make_uint4(bv, bf, bc, 0u);   // segment k / 8 starts at entry 4 k
        const uint4 q = __ldg(p + k);
        bv += (q.x & 0x3ffu) + (q.y & 0x3ffu) + (q.z & 0x3ffu) + (q.w & 0x3ffu);
        bf += ((q.x >> 10) & 0x3ffu) + ((q.y >> 10) & 0x3ffu) + ((q.z >> 10) & 0x3ffu) + ((q.w >> 10) & 0x3ffu);
        if (co) {
          // the dense slot bases (exclusive prefix of the active-corner counts): k_vertices gathers them per vertex,
          // k_faces loads them per word
          uint4 o;
          const uint32_t m = counted ? 0xffffffffu : 0u;
          o.x = bc; o.y = o.x + ((q.x >> 20) & m); o.z = o.y + ((q.y >> 20) & m); o.w = o.z + ((q.z >> 20) & m);
          bc = o.w + ((q.w >> 20) & m);
          co[k] = o;
        } else if (counted) {
          bc += (q.x >> 20) + (q.y >> 20) + (q.z >> 20) + (q.w >> 20);
        }
      }
    }
    v += __shfl_sync(0xffffffffu, iv, 31); f += __shfl_sync(0xffffffffu, jf, 31); c += __shfl_sync(0xffffffffu, ic, 31);
  }
}

// The common case - at most two segments per lattice row (EW <= 64, i.e. X <= 1983) and at most 128 rows per warp -
// in ONE pass over the counts: a lane owns a row, a warp 32 rows at a time, up to four such batches; the row totals
// (and, for the second segment, the sum of the row's first 32 entries) stay in registers while the CTA aggregate
// goes through the look-back, then warp scans over the rows give every row's prefix and the lane writes its one or
// two segment bases.  Every count is read exactly once (the general kernel above reads them three times: 0.088 ms
// against 0.05 ms for the 151 MB of a 1024^3 lattice).
constexpr int kScanBatches = 4;

template <int NS>
__global__ void __launch_bounds__(kScanThreads) k_seg_scan_rows(const SegScanArgs a) {
  pdl_enter();
  __shared__ unsigned int s_tile;
  __shared__ unsigned long long s_part[3][kScanWarps];
  __shared__ unsigned long long s_excl[3];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
  __syncthreads();
  const unsigned tile = s_tile;
  if (tile >= a.n_tiles) return;
  const unsigned rpw = a.rows_per_tile / kScanWarps;   // <= 32 * kScanBatches
  const unsigned r0 = min(tile * a.rows_per_tile + warp * rpw, a.n_rows);
  const unsigned r1 = min(r0 + rpw, a.n_rows);
  const unsigned ew4 = a.EW / 4;

  uint32_t tv[kScanBatches], tf[kScanBatches], tc[kScanBatches], pv[kScanBatches], pf[kScanBatches], pc[kScanBatches];
#pragma unroll
  for (int b = 0; b < kScanBatches; ++b) {
    tv[b] = tf[b] = tc[b] = pv[b] = pf[b] = pc[b] = 0;
    const unsigned r = r0 + 32 * b + lane;
    if (r < r1) {
      const unsigned row = a.row_begin + r;
      const uint4* __restrict__ p = reinterpret_cast<const uint4*>(a.cnt + (size_t)row * a.EW);
      uint32_t v = 0, f = 0, c = 0;
      for (unsigned k = 0; k < ew4; ++k) {
        if (NS == 2 && k == 8) { pv[b] = v; pf[b] = f; pc[b] = c; }   // the second segment starts at entry 32
        const uint4 q = __ldg(p + k);
        v += (q.x & 0x3ffu) + (q.y & 0x3ffu) + (q.z & 0x3ffu) + (q.w & 0x3ffu);
        f += ((q.x >> 10) & 0x3ffu) + ((q.y >> 10) & 0x3ffu) + ((q.z >> 10) & 0x3ffu) + ((q.w >> 10) & 0x3ffu);
        c += (q.x >> 20) + (q.y >> 20) + (q.z >> 20) + (q.w >> 20);
      }
      const bool counted = row >= a.ghost_row_end;
      tv[b] = v; tf[b] = f; tc[b] = counted ? c : 0u;
      if (!counted) pc[b] = 0;
    }
  }
  // warp aggregate -> CTA aggregate -> look-back
  unsigned long long sv = 0, sf = 0, sc = 0;
#pragma unroll
  for (int b = 0; b < kScanBatches; ++b) { sv += tv[b]; sf += tf[b]; sc += tc[b]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sv += __shfl_xor_sync(0xffffffffu, sv, o);
    sf += __shfl_xor_sync(0xffffffffu, sf, o);
    sc += __shfl_xor_sync(0xffffffffu, sc, o);
  }
  if (lane == 0) { s_part[0][warp] = sv; s_part[1][warp] = sf; s_part[2][warp] = sc; }
  __syncthreads();
  if (warp < 3) {
    const int k = warp;
    unsigned long long aggk = 0;
#pragma unroll
    for (int i = 0; i < kScanWarps; ++i) aggk += s_part[k][i];
    unsigned long long* st = a.status + (size_t)k * a.n_tiles;
    if (lane == 0) st_relaxed(st + tile, (tile == 0 ? kFlagPrefix : kFlagAggregate) | aggk);
    unsigned long long ex = 0;
    if (tile > 0) {
      ex = lookback(st, (int)tile, lane);
      if (lane == 0) st_relaxed(st + tile, kFlagPrefix | (ex + aggk));
    }
    if (lane == 0) {
      s_excl[k] = ex;
      if (tile == a.n_tiles - 1) a.info[kInfoTotV + k] = ex + aggk;
    }
  }
  __syncthreads();
  unsigned long long run_v = s_excl[0], run_f = s_excl[1], run_c = s_excl[2];
  for (int i = 0; i < warp; ++i) { run_v += s_part[0][i]; run_f += s_part[1][i]; run_c += s_part[2][i]; }
  uint32_t v = (uint32_t)run_v, f = (uint32_t)run_f, c = (uint32_t)run_c;
#pragma unroll
  for (int b = 0; b < kScanBatches; ++b) {
    uint32_t iv = tv[b], jf = tf[b], ic = tc[b];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t x = __shfl_up_sync(0xffffffffu, iv, o), y = __shfl_up_sync(0xffffffffu, jf, o), z = __shfl_up_sync(0xffffffffu, ic, o);
      if (lane >= o) { iv += x; jf += y; ic += z; }
    }
    const unsigned r = r0 + 32 * b + lane;
    if (r < r1) {
      const unsigned row = a.row_begin + r;
      const uint32_t bv = v + iv - tv[b], bf = f + jf - tf[b], bc = c + ic - tc[b];  // prefix at the start of the lane's row
      if (row == a.mark_row_vf) { a.info[kInfoMarkV] = bv; a.info[kInfoMarkF] = bf; }
      if (row == a.mark_row_c) a.info[kInfoMarkC] = bc;
      uint4* __restrict__ out = a.seg + (size_t)row * NS;
      out[0] = make_uint4(bv, bf, bc, 0u);
      if (NS == 2) out[1] = make_uint4(bv + pv[b], bf + pf[b], bc + pc[b], 0u);
    }
    v += __shfl_sync(0xffffffffu, iv, 31); f += __shfl_sync(0xffffffffu, jf, 31); c += __shfl_sync(0xffffffffu, ic, 31);
  }
}

// Derived counts of the run: what the own range produces, the default id bases, and the empty-interior-slice check.
//   raster != 0: vertex ids are corner slots (CUB_ORDER_RASTER)
//   slice_any[z] != 0: voxel slice z of the scanned range has an inside voxel (set by k_sweep)
// An empty voxel slice between two occupied ones: the reference's lookup-plane rotation (txx:155-161) only
// advances on inside voxels, so it merges vertices of different corner planes there (SURVEY section 8a row 3);
// this library implements the intended rule and reports the case through cub_last_warning.
__global__ void __launch_bounds__(256) k_finalize_info(unsigned long long* info, int raster, const uint32_t* slice_any,
                                                       int z_begin, int z_end) {
  pdl_enter();
  __shared__ int s_first, s_last, s_hole;
  if (threadIdx.x == 0) { s_first = INT_MAX; s_last = -1; s_hole = 0; }
  __syncthreads();
  if (slice_any) {
    int first = INT_MAX, last = -1;
    for (int z = z_begin + (int)threadIdx.x; z < z_end; z += (int)blockDim.x)
      if (slice_any[z]) { first = min(first, z); last = max(last, z); }
    if (last >= 0) { atomicMin(&s_first, first); atomicMax(&s_last, last); }
    __syncthreads();
    for (int z = z_begin + (int)threadIdx.x; z < z_end; z += (int)blockDim.x)
      if (z > s_first && z < s_last && !slice_any[z]) s_hole = 1;
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  const unsigned long long ghost_v = raster ? info[kInfoMarkC] : info[kInfoMarkV];
  info[kInfoGhostV] = ghost_v;
  info[kInfoPoints] = (raster ? info[kInfoTotC] : info[kInfoTotV]) - ghost_v;
  info[kInfoQuads] = info[kInfoTotF] - info[kInfoMarkF];
  info[kInfoPointBase] = 0;
  info[kInfoCellBase] = 0;
  info[kInfoIdDelta] = 0ull - ghost_v;
  info[kInfoFlags] = s_hole ? (unsigned long long)kFlagEmptyInteriorSlice : 0ull;
  info[kInfoWork] = 0;
  info[kInfoSplitWork] = 0;
}

__global__ void k_set_bases(unsigned long long* info, unsigned long long point_base, unsigned long long cell_base) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  info[kInfoPointBase] = point_base;
  info[kInfoCellBase] = cell_base;
  info[kInfoIdDelta] = point_base - info[kInfoGhostV];
}

// Count exchange of a multi-GPU run: `gathered` holds every rank's (points, quads) (an all-gather of
// info[kInfoPoints..kInfoQuads]); the id bases of `rank` are the exclusive prefix (NCCL has no exscan).
__global__ void k_bases_from_gathered(unsigned long long* info, const unsigned long long* gathered, int rank,
                                      int cells_per_quad) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  unsigned long long p = 0, c = 0;
  for (int r = 0; r < rank; ++r) { p += gathered[2 * r]; c += gathered[2 * r + 1]; }
  info[kInfoPointBase] = p;
  info[kInfoCellBase] = c * (unsigned long long)cells_per_quad;
  info[kInfoIdDelta] = p - info[kInfoGhostV];
}

}  // namespace cbr
