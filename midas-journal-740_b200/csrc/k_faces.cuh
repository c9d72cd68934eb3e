// k_faces.cuh — K3c: quad / triangle emission straight into the mesh's cell buffer, one thread per
// 32-voxel word.
//
// Reference: faceHasQuad (txx:164-173), the face -> corner table (txx:197-202, 219-233) and AddQuadFace
// (txx:279-332).  Cell ids follow voxel raster x face index (nextCellId, txx:117): cell index =
// face base of the word + rank inside the word.  The four vertex ids of a face come from the corner -> id map:
//     slot(corner) = slot base of the corner word + popc(act[corner word] & bits below)      id = perm[slot]
// A warp owns one 32-word segment of a voxel row.  The face base of a word is the segment base of k_seg_scan plus
// a warp scan of the face counts (it rides in the scan of the surface-voxel counts the queue needs anyway: no
// dense face-offset array).  The slot bases of the four corner words around the word come from the dense cofs
// array: r2 also tried to rebuild them with two more warp scans of popc(act) - fewer bytes, but 100 more
// instructions per warp in a kernel that is bound by instruction issue (0.58 -> 0.71 ms).  All words are loaded
// once per word, up front (the kernel is bound by its chain of dependent loads, not by bytes).  The surface
// voxels of a warp's 32 words are then compacted into a shared-memory queue and emitted one voxel per lane.
#pragma once
#include "cbr_common.cuh"
#include "k_segscan.cuh"

namespace cbr {

enum { kEmitQuads = 0, kEmitTrisFixed = 1, kEmitScratchQuads = 2 };

struct FaceArgs {
  const uint32_t* bits;
  Grid g;
  int EY, EW, NS;
  int z_begin, z_end;          // local voxel slices whose faces are emitted (the handle's own range)
  const uint32_t* act;
  const uint32_t* cofs;        // entry lattice, exclusive scan of the active-corner counts (slot bases)
  const uint4* seg;            // [lattice rows][NS] segment bases {vertices, faces, active corners, -}
  const uint32_t* perm;        // slot -> scan-relative vertex id
  unsigned long long* info;    // kInfoMarkF: scan offset of the first own face; kInfoIdDelta: scan-relative vertex id -> final id
  void* cells;                 // final cells (IdT) or scratch quads (uint32 scan-relative ids)
  int mode;                    // kEmit*
  const void* vol;             // for cell data (may be null)
  int vX, vY, vpad, vzpad;     // cell data: buffer row / slice size; lattice (x, y, z) is voxel (x - vpad, y - vpad, z - vzpad)
  void* celldata;
  int pix_bytes;
};

// two triangles = 6 ids: 24 bytes (8-byte aligned) as three 8-byte stores, or 48 bytes as three 16-byte stores
template <typename IdT>
__device__ __forceinline__ void store_tri_pair(IdT* c, IdT a0, IdT a1, IdT a2, IdT b0, IdT b1, IdT b2) {
  if (sizeof(IdT) == 4) {
    uint2* d = reinterpret_cast<uint2*>(c);
    d[0] = make_uint2((uint32_t)a0, (uint32_t)a1);
    d[1] = make_uint2((uint32_t)a2, (uint32_t)b0);
    d[2] = make_uint2((uint32_t)b1, (uint32_t)b2);
  } else {
    ulonglong2* d = reinterpret_cast<ulonglong2*>(c);
    d[0] = make_ulonglong2((unsigned long long)a0, (unsigned long long)a1);
    d[1] = make_ulonglong2((unsigned long long)a2, (unsigned long long)b0);
    d[2] = make_ulonglong2((unsigned long long)b1, (unsigned long long)b2);
  }
}

// v0..v3: FINAL vertex ids (the id offset is added once per corner by the caller, not once per face)
template <typename IdT, int MODE>
__device__ __forceinline__ void write_cell(const FaceArgs& a, uint32_t fidx, IdT v0, IdT v1, IdT v2, IdT v3) {
  if (MODE == kEmitScratchQuads) {
    reinterpret_cast<uint4*>(a.cells)[fidx] = make_uint4((uint32_t)v0, (uint32_t)v1, (uint32_t)v2, (uint32_t)v3);
    return;
  }
  IdT* c = reinterpret_cast<IdT*>(a.cells);
  if (MODE == kEmitQuads) {
    c += (size_t)fidx * 4;
    if (sizeof(IdT) == 4) {
      *reinterpret_cast<uint4*>(c) = make_uint4((uint32_t)v0, (uint32_t)v1, (uint32_t)v2, (uint32_t)v3);
    } else {  // 32-byte cells: two 16-byte stores
      reinterpret_cast<ulonglong2*>(c)[0] = make_ulonglong2((unsigned long long)v0, (unsigned long long)v1);
      reinterpret_cast<ulonglong2*>(c)[1] = make_ulonglong2((unsigned long long)v2, (unsigned long long)v3);
    }
  } else {
    // unprojected quad: both diagonals are equal, `>=` takes the first split (txx:298-302)
    c += (size_t)fidx * 6;
    store_tri_pair<IdT>(c, v0, v1, v3, v1, v2, v3);
  }
}

// Cell data = the pixel of the generating voxel (both triangles of a quad get it).  The pixel is loaded once per
// voxel as raw bytes (1, 2, 4 or 8) and stored with one typed store per cell.
__device__ __forceinline__ unsigned long long load_pixel(const void* vol, size_t voxel, int pix_bytes) {
  switch (pix_bytes) {
    case 1: return __ldg(reinterpret_cast<const uint8_t*>(vol) + voxel);
    case 2: return __ldg(reinterpret_cast<const uint16_t*>(vol) + voxel);
    case 4: return __ldg(reinterpret_cast<const uint32_t*>(vol) + voxel);
    default: return __ldg(reinterpret_cast<const unsigned long long*>(vol) + voxel);
  }
}

template <int MODE>
__device__ __forceinline__ void write_celldata(const FaceArgs& a, uint32_t fidx, unsigned long long pix) {
  const bool two = (MODE != kEmitQuads);
  const size_t c = two ? 2 * (size_t)fidx : (size_t)fidx;
  switch (a.pix_bytes) {
    case 1: { uint8_t* d = reinterpret_cast<uint8_t*>(a.celldata) + c; d[0] = (uint8_t)pix; if (two) d[1] = (uint8_t)pix; break; }
    case 2: { uint16_t* d = reinterpret_cast<uint16_t*>(a.celldata) + c; d[0] = (uint16_t)pix; if (two) d[1] = (uint16_t)pix; break; }
    case 4: { uint32_t* d = reinterpret_cast<uint32_t*>(a.celldata) + c; d[0] = (uint32_t)pix; if (two) d[1] = (uint32_t)pix; break; }
    default: { unsigned long long* d = reinterpret_cast<unsigned long long*>(a.celldata) + c; d[0] = pix; if (two) d[1] = pix; break; }
  }
}

constexpr int kFaceThreads = 128;

// per-word context a warp shares through shared memory: 4 x uint4
//   [0] A[oz][oy]   active masks of the 4 corner words       [1] C[oz][oy]  their slot bases
//   [2] F0..F3      [3] F4, F5, face base, -
// (one array per uint4, the lane fastest: a lane stride of 16 bytes keeps the 128-bit stores of a warp free of bank
//  conflicts; [lane][4] - a 64-byte stride - made them 4-way conflicts and cost the kernel 15 %)
struct FaceSmem {
  uint4 ctx[4][kFaceThreads / 32][32];
  uint16_t queue[kFaceThreads / 32][1024];         // (lane << 5) | bit of every surface voxel of the warp's words
};

// One thread per 32-voxel word computes the face masks; the surface voxels of a warp's 32 words are then
// compacted into a queue and handled one per lane, so a word with ten surface voxels does not stall the 31
// lanes whose words have none.
template <typename IdT, int MODE, bool CD>
__global__ void __launch_bounds__(kFaceThreads, 12) k_faces(const FaceArgs a) {
  pdl_enter();
  __shared__ FaceSmem sm;
  // The verdict of k_check_caps (the device-side counts fit the buffers) is requested here and looked at after the
  // scan, when every other load of the thread has come back too (a branch on it up here would put one more L2 round
  // trip in front of each of these short-lived blocks).
  const bool fits = emission_fits(a.info);
  const Grid& g = a.g;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // grid: x = 32-word segments of a row, y = groups of 4 rows (one row per warp), z = own slices.  128-thread CTAs:
  // a CTA keeps its registers and shared memory until its last warp is done, and warps differ a lot here (r1: 256
  // threads 1.127 ms of emission, 128 threads 1.084, 64 threads 1.121)
  const int sgm = blockIdx.x, w = sgm * 32 + lane, y = blockIdx.y * (kFaceThreads / 32) + warp, zl = a.z_begin + blockIdx.z;

  // ---- face masks of the word (txx:164-173; clamped neighbours: no face on the image border) --------------
  uint32_t F[6] = {0, 0, 0, 0, 0, 0};
  // context of the word: active masks and slot bases of the 4 corner words around it (index oz*2+oy), the
  // segment base of its row {-, faces, -, -}
  const int plane = a.EY * a.EW;                           // entries per plane (< 2^31)
  const uint32_t e00 = ((uint32_t)zl * (uint32_t)a.EY + (uint32_t)y) * (uint32_t)a.EW + (uint32_t)w;  // corner word (w, y, z)
  uint32_t A[4] = {0, 0, 0, 0}, C[4] = {0, 0, 0, 0};
  uint32_t fseg = 0;
  // (requested with everything else: the id base of a multi-GPU run only exists on the device)
  const unsigned long long id_delta = __ldg(a.info + kInfoIdDelta);
  const uint32_t ghost_f = (uint32_t)__ldg(a.info + kInfoMarkF);
  {
    // all the words are requested together (no early-out on an empty word: that would make the neighbour
    // loads wait for the first one, and the kernel is bound by its chain of dependent loads)
    const bool valid = w < g.Wx && y < g.Y;
    if (y < g.Y) fseg = __ldg(&a.seg[((uint32_t)zl * (uint32_t)a.EY + (uint32_t)y) * (uint32_t)a.NS + (uint32_t)sgm].y);
    // word and entry indices fit 32 bits (cub_count checks the lattice size): one IMAD.WIDE per load
    const uint32_t* __restrict__ row = a.bits + (((uint32_t)zl * (uint32_t)g.Y + (uint32_t)y) * (uint32_t)g.Wp + (uint32_t)w);
    const int zgl = zl + g.zg0;
    const int sw = g.Y * g.Wp;  // words per slice (< 2^31: checked by cub_count)
    // neighbour rows / slices as signed word offsets from `row` (0 = clamped onto the row itself)
    const int dym = (y > 0) ? -g.Wp : 0, dyp = (y < g.Y - 1) ? g.Wp : 0;
    const int dzm = (zgl > 0 && zl > 0) ? -sw : 0, dzp = (zgl < g.Zg - 1 && zl < g.Zl - 1) ? sw : 0;
    uint32_t c0 = 0, nym = 0, nyp = 0, nzm = 0, nzp = 0, edge = 0;
    if (valid) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t e = e00 + (uint32_t)((k >> 1) * plane + (k & 1) * a.EW);
        A[k] = __ldg(a.act + e);
        C[k] = __ldg(a.cofs + e);
      }
      c0 = __ldg(row);
      nym = __ldg(row + dym); nyp = __ldg(row + dyp); nzm = __ldg(row + dzm); nzp = __ldg(row + dzp);
      // the x neighbours are the adjacent lanes' words, except across the ends of the warp's 32-word segment
      if (lane == 0 && w > 0) edge = __ldg(row - 1);
      if (lane == 31 && w < g.Wx - 1) edge = __ldg(row + 1);
    }
    const uint32_t up = __shfl_up_sync(0xffffffffu, c0, 1), dn = __shfl_down_sync(0xffffffffu, c0, 1);
    if (valid) {
      const uint32_t XB = g.X & 31;
      const uint32_t vc = (w == g.Wx - 1 && XB) ? ((1u << XB) - 1u) : ~0u;
      const uint32_t c = c0 & vc;
      const uint32_t prev = (w == 0) ? (c0 << 31) : (lane == 0 ? edge : up);
      const uint32_t next = (w == g.Wx - 1) ? (c0 >> 31) : (lane == 31 ? edge : dn);
      F[0] = c & ~__funnelshift_l(prev, c0, 1);
      F[1] = c & ~nym;
      F[2] = c & ~__funnelshift_r(c0, next, 1);
      F[3] = c & ~nyp;
      F[4] = c & ~nzm;
      F[5] = c & ~nzp;
    }
  }
  uint32_t U = F[0] | F[1] | F[2] | F[3] | F[4] | F[5];
  const uint32_t nvox = __popc(U);
  const uint32_t nf = __popc(F[0]) + __popc(F[1]) + __popc(F[2]) + __popc(F[3]) + __popc(F[4]) + __popc(F[5]);
  // one warp scan in two 16-bit fields: surface voxels (queue positions) | faces (cell ids)
  uint32_t s0 = nvox | (nf << 16);
  const uint32_t m0 = s0;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t0 = __shfl_up_sync(0xffffffffu, s0, o);
    if (lane >= o) s0 += t0;
  }
  const uint32_t total = __shfl_sync(0xffffffffu, s0, 31) & 0xffffu;
  if (!fits) return;
  if (total == 0) return;  // no surface voxel in the 1024 voxels of the segment

  if (U) {
    s0 -= m0;  // exclusive
    sm.ctx[0][warp][lane] = make_uint4(A[0], A[1], A[2], A[3]);
    sm.ctx[1][warp][lane] = make_uint4(C[0], C[1], C[2], C[3]);
    sm.ctx[2][warp][lane] = make_uint4(F[0], F[1], F[2], F[3]);
    sm.ctx[3][warp][lane] = make_uint4(F[4], F[5], fseg + (s0 >> 16) - ghost_f, 0u);
    uint32_t pos = s0 & 0xffffu;
    uint16_t* q = sm.queue[warp];
    const uint32_t tag = (uint32_t)lane << 5;
    while (U) {
      const int b = __ffs(U) - 1;
      U &= U - 1;
      q[pos++] = (uint16_t)(tag | (uint32_t)b);
    }
  }
  __syncwarp();

  for (uint32_t s = lane; s < total; s += 32) {
    const uint32_t it = sm.queue[warp][s];
    const uint32_t src = it >> 5, b = it & 31u;
    const uint4 A4 = sm.ctx[0][warp][src], C4 = sm.ctx[1][warp][src], Fa = sm.ctx[2][warp][src], Fb = sm.ctx[3][warp][src];
    const uint32_t A[4] = {A4.x, A4.y, A4.z, A4.w}, C[4] = {C4.x, C4.y, C4.z, C4.w};
    const uint32_t Fm[6] = {Fa.x, Fa.y, Fa.z, Fa.w, Fb.x, Fb.y};
    const uint32_t bit = 1u << b, below = bit - 1u;
    // index of the voxel's first face: faces of the voxels before it in the word
    uint32_t fi = Fb.z;  // faces of a handle < 2^32 (cub_count)
#pragma unroll
    for (int f = 0; f < 6; ++f) fi += __popc(Fm[f] & below);
    // slots of the 8 corners of voxel b; local l -> (ox, oy, oz) as in txx:236-254
    uint32_t vid[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int oz = k >> 1, oy = k & 1;
      const uint32_t s0 = C[k] + __popc(A[k] & below);                      // corner x
      const uint32_t s1 = s0 + ((A[k] >> b) & 1u);                          // corner x+1 (b = 31: bit 0 of the next corner word)
      vid[oz * 4 + (oy ? 3 : 0)] = s0;
      vid[oz * 4 + (oy ? 2 : 1)] = s1;
    }
    const bool f0 = Fm[0] & bit, f1 = Fm[1] & bit, f2 = Fm[2] & bit, f3 = Fm[3] & bit, f4 = Fm[4] & bit, f5 = Fm[5] & bit;
    if (a.perm) {
      // only the corners of present faces have a vertex (vertexHasQuad, txx:164-173)
      const bool need[8] = {f0 || f1 || f4, f1 || f2 || f4, f2 || f3 || f4, f0 || f3 || f4,
                            f0 || f1 || f5, f1 || f2 || f5, f2 || f3 || f5, f0 || f3 || f5};
#pragma unroll
      for (int l = 0; l < 8; ++l)
        if (need[l]) vid[l] = __ldg(a.perm + vid[l]);
    }
    // the voxel behind the face (cell data): word src of this warp's row
    const unsigned long long voxel =
        CD ? load_pixel(a.vol, ((size_t)(zl - a.vzpad) * a.vY + (size_t)(y - a.vpad)) * a.vX +
                                           (size_t)((sgm * 32 + src) * 32 + b - a.vpad), a.pix_bytes) : 0ull;
    // final ids: scan-relative id + id offset (scratch quads keep the scan-relative ids: K5 adds the offset)
    IdT fid[8];
#pragma unroll
    for (int l = 0; l < 8; ++l) fid[l] = MODE == kEmitScratchQuads ? (IdT)vid[l] : (IdT)(vid[l] + id_delta);
    if (f0) { write_cell<IdT, MODE>(a, fi, fid[0], fid[4], fid[7], fid[3]); if (CD) write_celldata<MODE>(a, fi, voxel); ++fi; }
    if (f1) { write_cell<IdT, MODE>(a, fi, fid[0], fid[1], fid[5], fid[4]); if (CD) write_celldata<MODE>(a, fi, voxel); ++fi; }
    if (f2) { write_cell<IdT, MODE>(a, fi, fid[1], fid[2], fid[6], fid[5]); if (CD) write_celldata<MODE>(a, fi, voxel); ++fi; }
    if (f3) { write_cell<IdT, MODE>(a, fi, fid[2], fid[3], fid[7], fid[6]); if (CD) write_celldata<MODE>(a, fi, voxel); ++fi; }
    if (f4) { write_cell<IdT, MODE>(a, fi, fid[0], fid[3], fid[2], fid[1]); if (CD) write_celldata<MODE>(a, fi, voxel); ++fi; }
    if (f5) { write_cell<IdT, MODE>(a, fi, fid[4], fid[5], fid[6], fid[7]); if (CD) write_celldata<MODE>(a, fi, voxel); ++fi; }
  }
}

// K5: triangle split of projected quads (AddQuadFace txx:286-321): reads the four PROJECTED points
// back, squared diagonal lengths in fp64 from the fp32 points in axis order (SURVEY Appendix A.5),
// `>=` tie -> first split.
template <typename IdT>
__global__ void __launch_bounds__(256) k_split_quads(const uint4* __restrict__ quads, const float* __restrict__ points,
                                                     IdT* __restrict__ tris, unsigned long long* __restrict__ info) {
  // the number of quads and the id offset come from the device-side run info (no host round trip needed)
  if (!emission_fits(info)) return;
  const size_t n_quads = (size_t)__ldg(info + kInfoQuads);
  const unsigned long long id_delta = __ldg(info + kInfoIdDelta);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_quads; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 q = quads[i];
    const uint32_t id[4] = {q.x, q.y, q.z, q.w};
    float p[4][3];
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int c = 0; c < 3; ++c) p[k][c] = __ldg(points + 3 * (size_t)id[k] + c);
    double d02 = 0.0, d13 = 0.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const double a = __dadd_rn((double)p[0][c], -(double)p[2][c]);
      d02 = __dadd_rn(d02, __dmul_rn(a, a));
      const double b = __dadd_rn((double)p[1][c], -(double)p[3][c]);
      d13 = __dadd_rn(d13, __dmul_rn(b, b));
    }
    IdT v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = (IdT)((unsigned long long)id[k] + id_delta);
    IdT* c = tris + i * 6;
    const bool first = d02 >= d13;  // (0,1,3),(1,2,3) else (0,1,2),(0,2,3)
    store_tri_pair<IdT>(c, v[0], v[1], first ? v[3] : v[2], first ? v[1] : v[0], v[2], v[3]);
  }
}

}  // namespace cbr
