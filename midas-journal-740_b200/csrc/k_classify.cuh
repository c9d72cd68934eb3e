// k_classify.cuh — K1: one pass over the volume -> 1 bit / voxel inside mask.
//
// Reference: the suitability test `center < m_IsoSurfaceValue -> skip` (txx:139-141) and the
// neighbour test `GetPixel(offset) < m_IsoSurfaceValue` (txx:167) compare pixels with the iso
// value in the pixel type; both are the same predicate, so it is evaluated ONCE per voxel here
// and every later kernel works on the bitmask (1/32 of the bytes for float input).
//
// HBM-bound streaming read: algorithmic bytes = X*Y*Zl*sizeof(T) read (+ X*Y*Zl/8 written).
// Each warp owns a task of kWordsPerTask consecutive words of one row; every lane issues
// kWordsPerTask independent coalesced loads (lane b of load k reads voxel 32*(w0+k)+b: one full
// 128-byte line per warp instruction for 4-byte pixels, immediate offsets from one base pointer)
// before the first ballot, so a resident SM keeps warps * kWordsPerTask * 128 B in flight.  A
// ballot of the predicate IS the output word - no shuffles; lane 0 stores the task's words with
// 16-byte stores.  Budget: ~4.5 issued instructions per 128 B of input (r1 profile: the first
// version spent 21 and was issue-bound at 74 % of the HBM roofline).
// Lanes past the end of a ragged row re-read the row's last voxel, which produces the "replicate
// bit X-1" padding the later kernels rely on (generic path only).
#pragma once
#include "cbr_common.cuh"

namespace cbr {

constexpr int kWordsPerTask = 16;

// The inside predicate, a template parameter of every classification kernel (K1 and the producers of k_fused.cuh).
// AtLeast is the reference's rule !(v < iso) (txx:139-141, 167).  Between is the inside-range mode of
// cub_set_inside_range, !(v < lo) && !(hi < v).  Both compare in the pixel type, so a NaN pixel is inside in either.
// A kernel takes In::Param and builds the predicate from it.  For AtLeast that is the plain iso value: a struct
// parameter would be loaded differently (as bytes for 8-bit pixels), and iso mode compiles to the same code as a
// kernel that takes `T iso`.
template <typename T>
struct AtLeast {
  static constexpr bool kRange = false;
  using Param = T;
  T iso;
  __host__ __device__ __forceinline__ Param param() const { return iso; }
  __device__ __forceinline__ bool operator()(const T v) const { return !(v < iso); }
  __device__ __forceinline__ T lower() const { return iso; }
};
template <typename T>
struct Between {
  static constexpr bool kRange = true;
  using Param = Between;
  T lo, hi;
  __host__ __device__ __forceinline__ Param param() const { return *this; }
  __device__ __forceinline__ bool operator()(const T v) const { return !(v < lo) && !(hi < v); }
  __device__ __forceinline__ T lower() const { return lo; }
};

template <typename T>
__device__ __forceinline__ T load_stream(const T* p) {
  return __ldcs(p);  // read-once data: evict-first
}

// FULL: X % 32 == 0 and Wx % kWordsPerTask == 0 (no clamping, no partial tasks)
template <typename T, bool FULL, typename In>
__global__ void __launch_bounds__(256) k_classify(const T* __restrict__ vol, uint32_t* __restrict__ bits, Grid g,
                                                  typename In::Param bounds, unsigned n_tasks, unsigned groups_per_row) {
  const In inside{bounds};
  const int lane = threadIdx.x & 31;
  const unsigned warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned n_warps = (gridDim.x * blockDim.x) >> 5;
  for (unsigned task = warp0; task < n_tasks; task += n_warps) {
    const unsigned row = task / groups_per_row;
    const int w0 = (int)(task - row * groups_per_row) * kWordsPerTask;
    const T* __restrict__ src = vol + (size_t)row * g.X + (size_t)w0 * 32 + lane;
    T v[kWordsPerTask];
    if (FULL) {
#pragma unroll
      for (int k = 0; k < kWordsPerTask; ++k) v[k] = load_stream(src + k * 32);
    } else {
      const int xmax = g.X - 1 - (w0 * 32 + lane);  // largest valid offset from src (may be negative)
#pragma unroll
      for (int k = 0; k < kWordsPerTask; ++k) {
        const int off = k * 32 < xmax ? k * 32 : xmax;
        v[k] = load_stream(src + off);
      }
    }
    uint32_t word[kWordsPerTask];
#pragma unroll
    for (int k = 0; k < kWordsPerTask; ++k) word[k] = __ballot_sync(0xffffffffu, inside(v[k]));
    if (lane == 0) {
      uint32_t* dst = bits + (size_t)row * g.Wp + w0;
      if (FULL) {
#pragma unroll
        for (int k = 0; k < kWordsPerTask; k += 4)
          *reinterpret_cast<uint4*>(dst + k) = make_uint4(word[k], word[k + 1], word[k + 2], word[k + 3]);
      } else {
#pragma unroll
        for (int k = 0; k < kWordsPerTask; ++k)
          if (w0 + k < g.Wx) dst[k] = word[k];
      }
    }
  }
}

// ---- 1- and 2-byte pixels: 4 bytes per lane per load -----------------------------------------------------
// With one pixel per lane a warp load of uint8 voxels moves 32 bytes and the kernel is bound by the number of
// load instructions (r1: 2.5 TB/s for uint8, 4.2 TB/s for int16).  Here a lane loads 4 bytes = VPL voxels, so a
// warp load is again one full 128-byte line = VPL words.  A task is 32 words of one row = G = 32 / VPL loads,
// all issued before the first compare.  The per-byte / per-halfword `>=` is done in-register (carry-free
// subtract, the result lands in each field's top bit), a multiply gathers the VPL flags, and the lane appends
// them to a 32-bit accumulator: after G loads lane m of a word group holds field k = its VPL bits of word
// (VPL * k + group).  A G x G transpose of the fields across the G lanes of the group (log2 G shuffle stages)
// turns that into: lane m holds the whole word VPL * m + group, and the task is written with one coalesced
// 128-byte store.  (A redux.sync per load over the G-lane groups was tried first: sub-warp masks serialise it.)
// Requires X % (32 * VPL) == 0 and a 4-byte aligned buffer (else: k_classify above).
template <typename T> struct PackedTraits;
// a pixel value in every 1- or 2-byte field of a word
template <typename T>
__device__ __forceinline__ uint32_t replicate(const T v) {
  return sizeof(T) == 1 ? 0x01010101u * (uint32_t)(uint8_t)v : 0x00010001u * (uint32_t)(uint16_t)v;
}
template <> struct PackedTraits<uint8_t>  { static constexpr bool is_signed = false; };
template <> struct PackedTraits<int8_t>   { static constexpr bool is_signed = true; };
template <> struct PackedTraits<uint16_t> { static constexpr bool is_signed = false; };
template <> struct PackedTraits<int16_t>  { static constexpr bool is_signed = true; };

template <typename T, typename In>
__global__ void __launch_bounds__(256) k_classify_packed(const T* __restrict__ vol, uint32_t* __restrict__ bits, Grid g,
                                                         typename In::Param bounds, unsigned n_tasks, unsigned tasks_per_row) {
  const In inside{bounds};
  constexpr int VPL = 4 / (int)sizeof(T);   // voxels per lane per load = words per warp load = bits per field
  constexpr int G = 32 / VPL;               // lanes per word = loads per task = fields per accumulator
  constexpr uint32_t H = sizeof(T) == 1 ? 0x80808080u : 0x80008000u;  // top bit of every pixel
  constexpr bool SGN = PackedTraits<T>::is_signed;
  const int lane = threadIdx.x & 31;
  const int grp = lane / G, m = lane % G;
  // iso in every pixel; signed compare == unsigned compare with the sign bits flipped (the lanes' sign flip is
  // folded into the final select below)
  uint32_t iso_rep = replicate<T>(inside.lower());
  if (SGN) iso_rep ^= H;
  const uint32_t iso_low = iso_rep & ~H;
  // range mode: the upper bound in every pixel, sign bits flipped like iso_rep, and with every top bit set
  uint32_t hi_rep = 0;
  if constexpr (In::kRange) hi_rep = replicate<T>(inside.hi) ^ (SGN ? H : 0u);
  const uint32_t hi_top = hi_rep | H;
  const unsigned warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned n_warps = (gridDim.x * blockDim.x) >> 5;
  for (unsigned task = warp0; task < n_tasks; task += n_warps) {
    const unsigned row = task / tasks_per_row;
    const int w0 = (int)(task - row * tasks_per_row) * 32;
    const int nload = min(G, (g.Wx - w0) / VPL);  // warp-uniform; Wx is a multiple of VPL
    const uint32_t* __restrict__ src =
        reinterpret_cast<const uint32_t*>(vol + (size_t)row * g.X + (size_t)w0 * 32) + lane;
    uint32_t v[G];
#pragma unroll
    for (int k = 0; k < G; ++k) v[k] = (k < nload) ? __ldcs(src + k * 32) : 0u;
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < G; ++k) {
      // per pixel a >= b:  t = (a | H) - (b & ~H) has, in each pixel's top bit, (low bits of a) >= (low bits of b),
      // with no borrow between pixels; the top bits decide unless they are equal
      const uint32_t a = v[k];
      const uint32_t t = (a | H) - iso_low;
      uint32_t ge;
      if (SGN) ge = (~a & ~iso_rep) | ((a ^ iso_rep) & t);   // a's sign bit flipped: a' = a ^ H
      else ge = (a & ~iso_rep) | (~(a ^ iso_rep) & t);
      if constexpr (In::kRange) {
        // per pixel hi >= a, the same compare with the operands swapped: u = (hi | H) - (a & ~H).  Every field of the
        // minuend is at least H and every field of the subtrahend below H, so no field borrows from the one above it;
        // u's top bit per pixel is (low bits of hi) >= (low bits of a), and the top bits decide unless they are equal
        const uint32_t u = hi_top - (a & ~H);
        if (SGN) ge &= (hi_rep & a) | ((hi_rep ^ a) & u);       // hi_rep is hi' = hi ^ H, a' = a ^ H
        else ge &= (hi_rep & ~a) | (~(hi_rep ^ a) & u);
      }
      // top bits of the VPL pixels -> the VPL top bits of the word -> field k
      uint32_t f;
      if (VPL == 4) f = ((ge & H) * 0x00204081u) >> 28;
      else f = ((ge & H) * 0x00008001u) >> 30;
      acc |= f << (VPL * k);
    }
    // transpose the G x G fields of each lane group: stage d swaps the blocks (lane bit d, field bit d)
#pragma unroll
    for (int d = 1; d < G; d <<= 1) {
      const uint32_t o = __shfl_xor_sync(0xffffffffu, acc, d);
      const int sh = VPL * d;
      // fields whose index has bit d clear, as a mask (d = 1: every other field, d = 2: pairs, ...)
      uint32_t lowmask = 0;
#pragma unroll
      for (int k = 0; k < G; ++k)
        if (!(k & d)) lowmask |= ((1u << VPL) - 1u) << (VPL * k);
      if (!(m & d)) acc = (acc & lowmask) | ((o << sh) & ~lowmask);   // keep my low-block fields, take theirs up
      else acc = (acc & ~lowmask) | ((o >> sh) & lowmask);            // keep my high-block fields, take theirs down
    }
    if (m < nload) bits[(size_t)row * g.Wp + w0 + VPL * m + grp] = acc;  // word VPL * m + grp of the task
  }
}

// ---- image_border_faces: the bitmask of the image padded with one outside layer ---------------------------
// Bit (x', y', z') of the padded grid is voxel (x'-1, y'-1, z'-zpad) of the buffer, or 0 (outside) beyond it.
// Every later kernel runs unchanged on the padded grid: its clamped neighbours at the padded border are outside
// on both sides, so no face is lost and none is invented.  One warp per 32-voxel word; the loads are one
// element off the 128-byte alignment, which costs this opt-in mode a few percent of bandwidth.
template <typename T, typename In>
__global__ void __launch_bounds__(256) k_classify_padded(const T* __restrict__ vol, uint32_t* __restrict__ bits, Grid gb,
                                                         int vX, int vY, int vZl, int zpad, typename In::Param bounds,
                                                         unsigned n_words_total) {
  const In inside{bounds};
  const int lane = threadIdx.x & 31;
  const unsigned warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned n_warps = (gridDim.x * blockDim.x) >> 5;
  for (unsigned task = warp0; task < n_words_total; task += n_warps) {
    const unsigned row = task / (unsigned)gb.Wx;       // padded row index: zb * gb.Y + yb
    const int w = (int)(task - row * (unsigned)gb.Wx);
    const int zb = (int)(row / (unsigned)gb.Y), yb = (int)(row - (unsigned)zb * (unsigned)gb.Y);
    const int x = 32 * w + lane - 1, y = yb - 1, z = zb - zpad;
    bool in = false;
    if (x >= 0 && x < vX && y >= 0 && y < vY && z >= 0 && z < vZl)
      in = inside(__ldcs(vol + ((size_t)z * vY + y) * vX + x));
    const uint32_t word = __ballot_sync(0xffffffffu, in);
    if (lane == 0) bits[(size_t)row * gb.Wp + w] = word;
  }
}

}  // namespace cbr
