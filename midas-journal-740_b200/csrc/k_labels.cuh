// k_labels.cuh — per-label voxel counts and bounding boxes of an integer label map (cub_label_bounds), and the box
// copy of cub_set_region_of_interest.
//
// k_label_bounds reads the volume once.  The cost of a label map is not its bytes but contention: most voxels are
// background and neighbours almost always share a label, so one atomic per voxel would serialise on the background
// entry.  Every lane therefore keeps two running aggregates {label, count, box} in registers, the current label and the
// one before, and folds each voxel into one of them: a row that crosses an object goes background -> label ->
// background without a flush.  Only a third label flushes the older aggregate, and the flushes of a warp are merged per
// label (__match_any_sync + warp reductions) before one lane issues the atomics.  A 16-byte load whose pixels all equal
// the lane's current label costs four 32-bit compares, or two 64-bit ones for 8-byte pixels.  Label keys and the
// pattern are as wide as the pixel: a 64-bit label is compared in 64 bits, so 2^32 + 5 is not label 5.
#pragma once
#include <type_traits>

#include "cbr_common.cuh"

namespace cbr {

constexpr int kLabelThreads = 256;
constexpr int kLabelCtasPerSm = 3;   // resident CTAs per SM at the register budget of __launch_bounds__

// the unsigned type of a label's window key and of its compare pattern: 32 bits up to 4-byte pixels, else 64
template <typename T>
using LabelKey = typename std::conditional<sizeof(T) == 8, unsigned long long, unsigned>::type;

template <typename K>
__device__ __forceinline__ constexpr K no_label() { return ~K(0); }

// Table entry of window label i: 8 words {count, ~xmin, ~ymin, ~zmin, xmax, ymax, zmax, 0}.  The minima are stored as
// 32-bit complements, so every field only grows and the whole table starts from one memset to 0 (the host undoes the
// complement).
template <typename K>
struct LabelAcc {
  K key;   // window index of the label, or no_label<K>()
  K pat;   // the label's pixel bits replicated over K (the compare of a whole 16-byte load)
  unsigned count;
  unsigned x0, x1, y0, y1, z0, z1;
};

__device__ __forceinline__ void label_max(unsigned long long* p, unsigned long long v) {
  // (a stale read only costs an atomic that changes nothing)
  if (*(volatile unsigned long long*)p < v) atomicMax(p, v);
}

// Warp-collective: every lane with `flush` adds its aggregate to the table, one atomic per label and field per warp.
template <typename K>
__device__ __forceinline__ void label_flush(unsigned long long* table, const LabelAcc<K>& a, bool flush) {
  const unsigned m = __match_any_sync(0xffffffffu, flush ? a.key : no_label<K>());
  if (!flush) return;
  const unsigned c = __reduce_add_sync(m, a.count);
  const unsigned nx0 = __reduce_max_sync(m, ~a.x0), ny0 = __reduce_max_sync(m, ~a.y0), nz0 = __reduce_max_sync(m, ~a.z0);
  const unsigned x1 = __reduce_max_sync(m, a.x1), y1 = __reduce_max_sync(m, a.y1), z1 = __reduce_max_sync(m, a.z1);
  if ((int)(threadIdx.x & 31) == __ffs(m) - 1) {
    unsigned long long* e = table + 8ull * a.key;
    atomicAdd(e, (unsigned long long)c);
    label_max(e + 1, nx0); label_max(e + 2, ny0); label_max(e + 3, nz0);
    label_max(e + 4, x1); label_max(e + 5, y1); label_max(e + 6, z1);
  }
}

template <typename T>
__device__ __forceinline__ LabelKey<T> label_pattern(T v) {
  if constexpr (sizeof(T) == 8) {
    return (unsigned long long)v;
  } else {
    const unsigned u = sizeof(T) == 1 ? (unsigned)(unsigned char)v : (sizeof(T) == 2 ? (unsigned)(unsigned short)v : (unsigned)v);
    return sizeof(T) == 1 ? u * 0x01010101u : (sizeof(T) == 2 ? u * 0x00010001u : u);
  }
}

template <typename T>
union LabelChunk {
  uint4 w;
  T v[16 / sizeof(T)];
};

// One chunk of a row: nv (<= V) pixels from x = x0.  Warp-collective: every lane of the warp calls it, nv = 0 for none.
template <typename T>
__device__ __forceinline__ void label_chunk(unsigned long long* table, LabelAcc<LabelKey<T>>& a, LabelAcc<LabelKey<T>>& b,
                                            const LabelChunk<T>& u, int nv, unsigned x0, unsigned y, unsigned z,
                                            LabelKey<T> first, unsigned n) {
  using K = LabelKey<T>;
  constexpr int V = 16 / sizeof(T);
  constexpr K kNoLabel = no_label<K>();
  // every pixel of a whole 16-byte load is the current label: four 32-bit compares, or two 64-bit ones
  bool same;
  if constexpr (sizeof(T) == 8)
    same = nv == 0 || (nv == V && a.key != kNoLabel && (((unsigned long long)u.w.y << 32) | u.w.x) == a.pat &&
                       (((unsigned long long)u.w.w << 32) | u.w.z) == a.pat);
  else
    same = nv == 0 || (nv == V && a.key != kNoLabel && u.w.x == a.pat && u.w.y == a.pat && u.w.z == a.pat &&
                       u.w.w == a.pat);
  if (__all_sync(0xffffffffu, same)) {
    if (nv) {
      a.count += V;
      a.x0 = min(a.x0, x0); a.x1 = max(a.x1, x0 + V - 1);
      a.y0 = min(a.y0, y); a.y1 = max(a.y1, y);
      a.z0 = min(a.z0, z); a.z1 = max(a.z1, z);
    }
    return;
  }
#pragma unroll
  for (int k = 0; k < V; ++k) {
    K key = (K)u.v[k] - first;   // (the window lies inside the type: no wrap-around reaches [0, n))
    if (k >= nv || key >= n) key = kNoLabel;
    const bool flush = key != kNoLabel && key != a.key && key != b.key && b.key != kNoLabel;
    if (__any_sync(0xffffffffu, flush)) label_flush(table, b, flush);
    if (key != kNoLabel) {
      const unsigned x = x0 + k;
      if (key != a.key) {
        const LabelAcc<K> older = b;
        b = a;
        if (key == older.key) {
          a = older;
        } else {
          a.key = key; a.pat = label_pattern(u.v[k]); a.count = 0;
          a.x0 = a.x1 = x; a.y0 = a.y1 = y; a.z0 = a.z1 = z;
        }
      }
      a.count++;
      a.x0 = min(a.x0, x); a.x1 = max(a.x1, x);
      a.y0 = min(a.y0, y); a.y1 = max(a.y1, y);
      a.z0 = min(a.z0, z); a.z1 = max(a.z1, z);
    }
  }
}

// Row r of the volume (y = r % Y, z = r / Y) is split into an unaligned head, 16-byte chunks and a tail; a warp reads
// 64 chunks of a row per step, two per lane, both loads in flight before either is used.  Counts in registers are
// 32-bit: the host sizes the grid so that a warp sees fewer than 2^32 voxels.
template <typename T>
__global__ void __launch_bounds__(kLabelThreads, kLabelCtasPerSm)
    k_label_bounds(const T* __restrict__ vol, unsigned X, unsigned Y, unsigned long long rows, LabelKey<T> first,
                   unsigned n, unsigned long long* __restrict__ table) {
  using K = LabelKey<T>;
  constexpr int V = 16 / sizeof(T);
  const int lane = threadIdx.x & 31;
  const unsigned long long warps = (unsigned long long)gridDim.x * (kLabelThreads / 32);
  LabelAcc<K> a{no_label<K>(), 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u}, b = a;   // the current label and the one before
  for (unsigned long long r = blockIdx.x * (unsigned long long)(kLabelThreads / 32) + (threadIdx.x >> 5); r < rows; r += warps) {
    const unsigned y = (unsigned)(r % Y), z = (unsigned)(r / Y);
    const T* row = vol + r * X;
    const unsigned head = min(X, (unsigned)(((16u - ((unsigned)reinterpret_cast<uintptr_t>(row) & 15u)) & 15u) / sizeof(T)));
    const unsigned n16 = (X - head) / V;
    const unsigned tail = X - head - n16 * V;
    const unsigned hh = head ? 1u : 0u;
    const unsigned chunks = hh + n16 + (tail ? 1u : 0u);
    for (unsigned base = 0; base < chunks; base += 64) {
      LabelChunk<T> u[2];
      int nv[2];
      unsigned x0[2];
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const unsigned c = base + 32 * s + lane;
        nv[s] = 0; x0[s] = 0;
        u[s].w = make_uint4(0, 0, 0, 0);
        if (c >= chunks) continue;
        if (c < hh) {
          nv[s] = (int)head;
        } else if (c - hh < n16) {
          x0[s] = head + (c - hh) * V;
          nv[s] = V;
          u[s].w = __ldg(reinterpret_cast<const uint4*>(row + x0[s]));
          continue;
        } else {
          x0[s] = head + n16 * V;
          nv[s] = (int)tail;
        }
#pragma unroll
        for (int k = 0; k < V; ++k)
          if (k < nv[s]) u[s].v[k] = row[x0[s] + k];
      }
      label_chunk<T>(table, a, b, u[0], nv[0], x0[0], y, z, first, n);
      label_chunk<T>(table, a, b, u[1], nv[1], x0[1], y, z, first, n);
    }
  }
  label_flush(table, a, a.key != no_label<K>());
  label_flush(table, b, b.key != no_label<K>());
}

// cub_set_region_of_interest: the box [lo, lo + size) of an x-fastest volume into a dense buffer, one CTA per row.
// Instantiated by pixel width: a copy does not care about the type.
template <typename W>
__global__ void k_gather_box(const W* __restrict__ src, W* __restrict__ dst, unsigned long long X, unsigned long long Y,
                             unsigned long long lx, unsigned long long ly, unsigned long long lz, unsigned long long sx,
                             unsigned long long sy, unsigned long long rows) {
  for (unsigned long long r = blockIdx.x; r < rows; r += gridDim.x) {
    const unsigned long long y = r % sy, z = r / sy;
    const W* s = src + ((z + lz) * Y + (y + ly)) * X + lx;
    W* d = dst + r * sx;
    for (unsigned long long x = threadIdx.x; x < sx; x += blockDim.x) d[x] = s[x];
  }
}

}  // namespace cbr
