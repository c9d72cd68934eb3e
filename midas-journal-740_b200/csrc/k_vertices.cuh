// k_vertices.cuh — K3a / K3b: vertex creation in the reference's order.
//
// Reference: the vertex creation loop txx:179-194 (voxels in raster order, local corners 0..7, a corner gets
// nextVertexId the first time it is touched) and AddVertex without the projection (txx:257-276):
// TransformIndexToPhysicalPoint, minus half a spacing, mesh->GetPoints()->InsertElement(id, vertex).
//
//   K3a k_assign   one warp per 32-word segment of a voxel row.  K2a (k_sweep.cuh) decided, per voxel word, which
//                  voxel owns which of its 8 local corners (8 masks, stored where the word owns anything); the
//                  first id of a word is the segment base of k_seg_scan plus a warp scan of the words' counts.
//                  The same scan carries the active-corner counts along and the warp writes the dense slot bases
//                  cofs of its lattice row, coalesced (k_seg_scan, whose lanes own one row each, could only write
//                  them with strided 16-byte stores: 0.21 ms against 0.08 ms without them).
//                  Lanes whose word owns a corner walk the masks - voxels in bit order, local corners 0..7 - and
//                  record for vertex id (first id + rank) the corner it sits on: cx | cy << 16 | oz << 31.
//   K3b k_vertices one thread per vertex id, perfectly balanced and coalesced: reads the 4-byte record, writes the
//                  12-byte point and stores its id at the corner's rank in corner-raster order,
//                      perm[cofs[corner word] + popc(act[corner word] & bits below)] = id,
//                  which is where the face kernel looks it up.  The owner slice of an id follows from the
//                  per-slice first ids (ids are handed out slice by slice; k_slice_index).
//
// r2 also tried ONE kernel for both (a warp walks the masks into a shared queue and then emits one vertex per
// lane, slots from warp scans of popc(act) of the four corner rows: no record array, no dense cofs): 0.75 ms
// against 0.48 ms for this pair - every warp then pays the corner context of all its 32 words, while k_assign
// drops the 57 % of words that own nothing after one load and k_vertices has no per-word work at all.
//
// In raster vertex order (the opt-in canonical order) ids ARE slots and k_points_raster writes the points
// straight from the active masks.
//
// k_assign, k_vertices and k_points_raster skip their work when k_check_caps found that the emission does not fit
// its buffers (k_segscan.cuh).
#pragma once
#include "cbr_common.cuh"
#include "k_segscan.cuh"

namespace cbr {

struct AssignArgs {
  const uint32_t* cnt;    // entry lattice: owned corners | faces << 10 | active corners << 20
  const uint4* own;       // entry lattice x 2: ownership masks O[0..3], O[4..7]
  const uint4* seg;       // [lattice rows][NS] segment bases {vertices, faces, active corners, -}
  uint32_t* cofs;         // entry lattice, written here: exclusive prefix of the active-corner counts (slot bases)
  int Wx, EY, EW, NS;
  int z_begin;            // first local plane of the scan range (blockIdx.z = 0)
  unsigned ghost_row_end; // active corners of lattice rows below this one are not counted (the slab underneath owns them)
  uint32_t* vtx;          // [n vertices] cx | cy << 16 | oz << 31
  unsigned long long* info;
};

constexpr int kAssignThreads = 128;  // (one row segment per warp)

// grid: x = 32-word segments of a voxel row, y = groups of kAssignThreads / 32 lattice rows (one row per warp),
// z = planes of the scan range (one more than its voxel slices: the top corner plane)
__global__ void __launch_bounds__(kAssignThreads) k_assign(const AssignArgs a) {
  pdl_enter();
  const bool fits = emission_fits(a.info);  // (looked at after the scan: see k_faces)
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.x * 32 + lane, y = blockIdx.y * (kAssignThreads / 32) + (threadIdx.x >> 5), z = a.z_begin + blockIdx.z;
  if (y >= a.EY) return;  // (warp-uniform)
  const uint32_t row = (uint32_t)z * (uint32_t)a.EY + (uint32_t)y;
  const uint32_t e = row * (uint32_t)a.EW + (uint32_t)w;
  const bool counted = row >= a.ghost_row_end;
  // (entries that are not voxel words - the column past the last voxel word, the row y = Y, the top plane - have
  //  no owned corners: K2a wrote 0 there)
  const uint32_t c = w < a.EW ? __ldg(a.cnt + e) : 0u;
  const uint4 sb = __ldg(a.seg + row * (uint32_t)a.NS + blockIdx.x);
  const uint32_t nv = c & 0x3ffu, na = counted ? c >> 20 : 0u;
  // the ownership masks are requested before the scan (the kernel is bound by this chain of dependent loads)
  uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
  if (nv) { lo = __ldcs(a.own + 2 * (size_t)e); hi = __ldcs(a.own + 2 * (size_t)e + 1); }
  // one warp scan, two 16-bit fields: owned corners (first id of the word) | active corners (slot base of the word)
  uint32_t incl = nv | (na << 16);
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const uint32_t excl = incl - (nv | (na << 16));
  if (!fits) return;
  if (w < a.EW) a.cofs[e] = sb.z + (excl >> 16);
  // the corner column past the last voxel word of the row, when it starts a segment of its own (X a multiple of 1024):
  // it is the first word of that segment, its slot base is the segment base (the words after it are padding)
  if (blockIdx.x == gridDim.x - 1 && lane == 0 && (int)(gridDim.x * 32) < a.EW)
    a.cofs[row * (uint32_t)a.EW + gridDim.x * 32u] = __ldg(&a.seg[row * (uint32_t)a.NS + gridDim.x].z);
  if (nv == 0) return;
  uint32_t n = sb.x + (excl & 0xffffu);
  const uint32_t O[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
  uint32_t U = O[0] | O[1] | O[2] | O[3] | O[4] | O[5] | O[6] | O[7];
  uint32_t* __restrict__ const out = a.vtx;
  const uint32_t xy0 = (uint32_t)(w * 32) | ((uint32_t)y << 16);
  while (U) {
    const int b = __ffs(U) - 1;
    U &= U - 1;
    const uint32_t bit = 1u << b;
    const uint32_t xy = xy0 + (uint32_t)b;
    // local corner l -> (ox, oy, oz) as in txx:236-254; a 32-bit running index (a predicated 64-bit pointer bump
    // costs 6 instructions per store)
    if (O[0] & bit) { out[n] = xy; ++n; }
    if (O[1] & bit) { out[n] = xy + 1u; ++n; }
    if (O[2] & bit) { out[n] = xy + 0x10001u; ++n; }
    if (O[3] & bit) { out[n] = xy + 0x10000u; ++n; }
    if (O[4] & bit) { out[n] = xy + 0x80000000u; ++n; }
    if (O[5] & bit) { out[n] = xy + 0x80000001u; ++n; }
    if (O[6] & bit) { out[n] = xy + 0x80010001u; ++n; }
    if (O[7] & bit) { out[n] = xy + 0x80010000u; ++n; }
  }
}

struct VertexArgs {
  const uint32_t* vtx;      // [n] packed corner of vertex id (scan-relative id): cx | cy << 16 | oz << 31
  const uint32_t* slice_first;  // [nz + 1] first id created by slice z_first + k; [nz] = UINT_MAX   (k_slice_index)
  const uint32_t* block_slice;  // [blocks of this launch] k of the block's first id                  (k_slice_index)
  unsigned long long* info;  // kInfoTotV = ghost vertices + own vertices, kInfoGhostV
  Caps caps;                // caps.points bounds the record loads issued before the counts are known
  int z_first;              // first local slice of the scan range
  int write_ghost_points;   // also write the points of the vertices that belong to the slab underneath
  const uint32_t* act;      // entry lattice [Zl+1][EY][EW]
  const uint32_t* cofs;
  int EY, EW;
  int plane_lo, plane_hi;   // local corner planes that faces of this handle reference (inclusive)
  int coff[3];              // image index of lattice corner (0, 0, 0): slab offset, region index, minus the pad of image_border_faces
  Geom geom;
  float* points;            // indexed by scan-relative vertex id
  uint32_t* perm;           // [active corners of planes plane_lo..plane_hi] -> scan-relative vertex id
};

// ids are handed out slice by slice, so the owner slice of an id follows from the per-slice first ids: this
// one-off kernel reads them out of the segment bases (the base of the first segment of a plane's first row) and
// bisects once per k_vertices block, so that the vertex threads only step forward from their block's slice
// (almost always zero steps).
struct SliceIndexArgs {
  const uint4* seg;
  size_t plane_segs;        // EY * NS: segments per plane
  int z_first, nz;          // local slices [z_first, z_first + nz) of the scan range
  uint32_t* slice_first;    // [nz + 1]
  uint32_t* block_slice;    // [n_blocks]
  uint32_t n_blocks, ids_per_block;
};

__global__ void __launch_bounds__(256) k_slice_index(const SliceIndexArgs a) {
  pdl_enter();
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t <= (uint32_t)a.nz) a.slice_first[t] = t < (uint32_t)a.nz ? __ldg(&a.seg[(size_t)(a.z_first + t) * a.plane_segs].x) : 0xffffffffu;
  if (t >= a.n_blocks) return;
  const uint32_t id = t * a.ids_per_block;
  int lo = 0, hi = a.nz - 1;  // largest k with first[k] <= id
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&a.seg[(size_t)(a.z_first + mid) * a.plane_segs].x) <= id) lo = mid; else hi = mid - 1;
  }
  a.block_slice[t] = (uint32_t)lo;
}

constexpr int kVertexPerThread = 4;                       // ids per thread: the loads of the 4 are in flight together
constexpr int kVertexBlockIds = 256 * kVertexPerThread;   // (the kernel is a chain of 3 dependent loads otherwise)

// The number of vertices comes from the device-side run info: the grid may be sized for the buffers' capacity
// (cub_emit_async), and the blocks past the count return.
template <bool ORIENTED>
__global__ void __launch_bounds__(256, ORIENTED ? 4 : 8) k_vertices(const VertexArgs a) {
  pdl_enter();
  const size_t id0 = (size_t)blockIdx.x * kVertexBlockIds + threadIdx.x;
  uint32_t v[kVertexPerThread];
  // the records are requested before the counts are looked at (any id below the capacity of the buffer is safe
  // to read), so that the two round trips overlap
#pragma unroll
  for (int j = 0; j < kVertexPerThread; ++j) {
    const size_t id = id0 + (size_t)j * 256;
    v[j] = id < a.caps.points ? __ldcs(a.vtx + id) : 0u;
  }
  if (!emission_fits(a.info)) return;
  const size_t n = (size_t)__ldg(a.info + kInfoTotV);
  if ((size_t)blockIdx.x * kVertexBlockIds >= n) return;
  const size_t first_point = a.write_ghost_points ? 0 : (size_t)__ldg(a.info + kInfoGhostV);
  int lo = (int)__ldg(a.block_slice + blockIdx.x);
  int cz[kVertexPerThread];
#pragma unroll
  for (int j = 0; j < kVertexPerThread; ++j) {
    const size_t id = id0 + (size_t)j * 256;
    if (id < n)
      while ((uint32_t)id >= __ldg(a.slice_first + lo + 1)) ++lo;
    cz[j] = a.z_first + lo + (int)(v[j] >> 31);
  }
  uint32_t co[kVertexPerThread], ac[kVertexPerThread];
#pragma unroll
  for (int j = 0; j < kVertexPerThread; ++j) {
    const size_t id = id0 + (size_t)j * 256;
    const int cx = (int)(v[j] & 0xffffu), cy = (int)((v[j] >> 16) & 0x7fffu);
    co[j] = ac[j] = 0;
    if (id < n && cz[j] >= a.plane_lo && cz[j] <= a.plane_hi) {
      const size_t e = ((size_t)cz[j] * a.EY + cy) * a.EW + (cx >> 5);
      co[j] = __ldg(a.cofs + e);
      ac[j] = __ldg(a.act + e);
    }
  }
#pragma unroll
  for (int j = 0; j < kVertexPerThread; ++j) {
    const size_t id = id0 + (size_t)j * 256;
    if (id >= n) break;
    const int cx = (int)(v[j] & 0xffffu), cy = (int)((v[j] >> 16) & 0x7fffu);
    if (id >= first_point) {
      // (r2 also tried per-axis coordinate tables - the position of a corner of a non-oriented image is separable -
      //  in place of the fp64 expressions: three more dependent loads per vertex, 205 -> 216 us)
      float* p = a.points + 3 * id;
      p[0] = corner_coord<ORIENTED>(a.geom, 0, cx + a.coff[0], cy + a.coff[1], cz[j] + a.coff[2]);
      p[1] = corner_coord<ORIENTED>(a.geom, 1, cx + a.coff[0], cy + a.coff[1], cz[j] + a.coff[2]);
      p[2] = corner_coord<ORIENTED>(a.geom, 2, cx + a.coff[0], cy + a.coff[1], cz[j] + a.coff[2]);
    }
    if (cz[j] >= a.plane_lo && cz[j] <= a.plane_hi) {
      const uint32_t below = (1u << (cx & 31)) - 1u;
      a.perm[co[j] + __popc(ac[j] & below)] = (uint32_t)id;
    }
  }
}

// Raster vertex order (CUB_ORDER_RASTER): vertex id = slot, so the points follow directly from the active
// masks: one thread per corner word, ids cseg[segment] + warp prefix + rank are consecutive inside a word.
struct RasterPointArgs {
  const uint32_t* act;
  uint32_t* cofs;           // entry lattice, written here: the slot base of every corner word (what k_assign writes in reference order)
  const uint4* seg;
  int EY, EW, NS, Wc;
  int plane_lo, plane_hi;   // local corner planes of the launch (inclusive)
  int point_plane_lo;       // first plane whose points are written (the bottom plane of a slab belongs to the slab underneath)
  int coff[3];              // as in VertexArgs
  Geom geom;
  float* points;            // indexed by slot
  unsigned long long* info;
};

template <bool ORIENTED>
__global__ void __launch_bounds__(256) k_points_raster(const RasterPointArgs a) {
  if (!emission_fits(a.info)) return;
  // grid: x = 32-word segments of a corner row, y = groups of 8 rows (one per warp), z = planes
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.x * 32 + lane, cy = blockIdx.y * 8 + (threadIdx.x >> 5), cz = a.plane_lo + blockIdx.z;
  if (cy >= a.EY) return;
  const size_t row = (size_t)cz * a.EY + cy;
  uint32_t m = w < a.Wc ? __ldg(a.act + row * a.EW + w) : 0u;   // (words Wc <= w < EW: never active)
  uint32_t incl = (uint32_t)__popc(m);
  const uint32_t mine = incl;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const uint32_t base = __ldg(&a.seg[row * a.NS + blockIdx.x].z) + (incl - mine);
  if (w < a.EW) a.cofs[row * a.EW + w] = base;
  if (!m || cz < a.point_plane_lo) return;
  size_t id = (size_t)base;
  while (m) {
    const int b = __ffs(m) - 1;
    m &= m - 1;
    float* p = a.points + 3 * id;
    const int cx = 32 * w + b;
    p[0] = corner_coord<ORIENTED>(a.geom, 0, cx + a.coff[0], cy + a.coff[1], cz + a.coff[2]);
    p[1] = corner_coord<ORIENTED>(a.geom, 1, cx + a.coff[0], cy + a.coff[1], cz + a.coff[2]);
    p[2] = corner_coord<ORIENTED>(a.geom, 2, cx + a.coff[0], cy + a.coff[1], cz + a.coff[2]);
    ++id;
  }
}

}  // namespace cbr
