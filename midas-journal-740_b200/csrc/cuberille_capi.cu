// cuberille_capi.cu — the C-ABI of include/cuberille_c.h: handle, buffers, kernel launches.
//
// Host-side orchestration of GenerateData() (txx:59-216) as a two-phase run:
//   cub_count : K1 classify -> K2a ownership sweep -> K2b segment scan (decoupled look-back)   (sizes are data dependent)
//   cub_emit  : K3a vertices (points + corner -> id map) -> K3c faces -> [K4 project] -> [K5 split projected quads]
// Everything is ordered on one CUDA stream.  The counts of a run live in a small device-side info block that the
// emission kernels read themselves, so a whole step can also be queued without a host round trip
// (cub_count_async / cub_emit_async / cub_finish).  There is no CPU implementation behind this file.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/cuberille_c.h"
#include "cbr_common.cuh"
#include "k_classify.cuh"
#include "k_segscan.cuh"
#include "k_generate.cuh"
#include "k_faces.cuh"
#include "k_project.cuh"
#include "k_sweep.cuh"
#include "k_fused.cuh"
#include "k_vertices.cuh"
#include "k_labels.cuh"

using namespace cbr;

namespace {

// tuning knobs, read from the environment ONCE per handle (cub_create) and clamped to sane values
struct Knobs {
  int k1_ctas = 32;          // CUB_K1_CTAS_PER_SM: grid cap of the classification kernel
  int fuse_tz = 0;           // CUB_FUSE_TZ: slices per sweep tile of the fused kernel (0: pick_tz)
  int fuse_ctas = 4;         // CUB_FUSE_CTAS_PER_SM
  int fuse_batch = 8;        // CUB_FUSE_BATCH: classification tasks (4 KB of a row each) per ticket and per publication
  int scan_ctas = 8;         // CUB_SCAN_CTAS_PER_SM
  int proj_ctas = 6;         // CUB_PROJ_CTAS_PER_SM
  int proj_refill = 18;      // CUB_PROJ_REFILL: lanes of a warp that keep iterating before the warp serves the idle ones
};

int env_int(const char* name, int dflt, int lo, int hi) {
  const char* v = getenv(name);
  if (!v || !*v) return dflt;
  const int x = atoi(v);
  return x < lo ? lo : (x > hi ? hi : x);
}

// slices per CTA sweep: long sweeps amortise the warm-up planes, but the grid must still fill the GPU
int pick_tz(int gx, int gy, int nz, int num_sms) {
  int tz = 32;
  while (tz > 4 && (long long)gx * gy * ((nz + tz - 1) / tz) < 6LL * num_sms) tz >>= 1;
  if (tz > nz) tz = nz;
  return tz < 1 ? 1 : tz;
}

// One instantiation of the sweep kernel (thread grid NTX x NTY, R corner rows per thread; k_sweep.cuh)
template <typename C>
cudaError_t launch_sweep(SweepArgs a, cudaStream_t stream, int num_sms) {
  using Smem = SweepSmem<C>;
  auto kern = k_sweep<C>;
  const int gx = (a.g.Wx + C::TXW - 1) / C::TXW, gy = (a.g.Y + C::TY - 1) / C::TY;
  const int nz = a.z_end - a.z_begin;
  a.tz = pick_tz(gx, gy, nz, num_sms);
  dim3 grid(gx, gy, (nz + a.tz - 1) / a.tz);
  kern<<<grid, C::NTP, sizeof(Smem), stream>>>(a);
  return cudaGetLastError();
}

// the sweep tile shapes: 16 voxel words per row for big volumes, 8 when a row has few words
using WideTile = SweepCfg<17, 7, 2>;
using NarrowTile = SweepCfg<9, 14, 2>;

constexpr size_t kCtrlHead = kInfoWords + 4;  // info block, two work counters, the scan's ticket (+ pad)

template <typename P>
struct DevBuf {
  P* p = nullptr;
  size_t cap = 0;  // elements
};

}  // namespace

struct cub_handle_s {
  int device = 0;
  int num_sms = 148;           // SMs of the handle's device: grid sizes are multiples of it
  Knobs knobs;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err = "";
  std::string warning = "";

  // volume
  const void* d_vol = nullptr;
  DevBuf<unsigned char> vol_owned;
  int dtype = -1, pix_bytes = 0;
  uint64_t dims[3] = {0, 0, 0};
  Geom geom{};
  bool has_volume = false;
  // inside-range mode (cub_set_inside_range): inside == !(v < range_lo) && !(range_hi < v) instead of !(v < iso)
  bool range_on = false;
  double range_lo = 0.0, range_hi = 0.0;
  // slab
  uint64_t image_nz = 0, local_z0 = 0, own_z0 = 0, own_z1 = 0;
  bool slab_set = false;
  // region of interest (cub_set_region_of_interest): while it is set, d_vol / dims / i0 describe the box and these
  // the whole volume; a box that is not whole rows and slices is a copy in roi_buf
  bool roi_on = false;
  const void* full_vol = nullptr;
  uint64_t full_dims[3] = {0, 0, 0};
  uint64_t roi_lo[3] = {0, 0, 0};
  DevBuf<unsigned char> roi_buf;
  // cub_label_bounds: the device table; cub_run_labels: the concatenation of the parts
  DevBuf<unsigned long long> label_table;
  DevBuf<float> cat_points;
  DevBuf<unsigned char> cat_cells, cat_celldata;

  // scratch
  DevBuf<uint32_t> bits, cnt, act, cofs, perm;
  // one control block, cleared with ONE memset per count: [info (kInfoWords + 2) | ticket | status (3 x tiles) | slice_any]
  DevBuf<unsigned long long> ctrl;
  uint32_t* d_slice_any = nullptr;
  unsigned* d_fuse_done = nullptr;
  unsigned* d_fuse_ctr = nullptr;
  bool fused_last = false;     // the last count ran K1 + K2a as the fused kernel
  bool pdl_on = false;         // the kernels of the current run are queued with programmatic dependent launch
  unsigned long long* d_status = nullptr;
  DevBuf<uint32_t> vtx;      // K3a -> K3b: the lattice corner of every vertex id
  DevBuf<uint32_t> vsl;      // k_slice_index: per-slice first ids, then the slice of each k_vertices block
  DevBuf<uint4> own;         // K2a -> K3a: the 8 ownership masks per voxel word (2 x uint4 per entry)
  DevBuf<uint4> seg;         // K2b -> K3: segment bases {vertices, faces, active corners, -}
  int EY = 0, EW = 0, NS = 0;
  uint64_t n_active = 0;     // active corners of the counted planes (size of the corner -> id map)
  bool raster = false;
  uint64_t bits_layout[3] = {0, 0, 0};
  unsigned int* d_ticket = nullptr;
  size_t ctrl_used = 0;
  unsigned long long* d_info = nullptr;  // kInfoWords (k_segscan.cuh) + 2 work counters
  unsigned long long* h_info = nullptr;  // pinned copy

  // results
  DevBuf<float> points;
  DevBuf<unsigned char> cells, celldata;
  DevBuf<uint4> quads;

  // state
  cub_params params{};
  Grid g{};    // the lattice every kernel after K1 works on: the buffer, or (image_border_faces) the buffer padded by one layer
  Grid gv{};   // the voxel buffer itself (K1, K4, cell data)
  long long i0[3] = {0, 0, 0};  // image index of buffer voxel (0, 0, 0): cub_set_region_index
  int pad = 0, zpad_lo = 0;  // image_border_faces: lattice (x, y, z) is voxel (x - pad, y - pad, z - zpad_lo)
  bool count_queued = false;    // the count kernels of the current run are on the stream
  bool counted = false;         // ... and the host knows their results
  bool emitted = false;
  bool emit_unverified = false; // the emission was queued with buffer sizes that the host has not checked yet (cub_emit_async)
  int zs0 = 0, zs1 = 0, owner_z_min = 0;
  bool vertices_done = false;   // the vertex stage of the current count has been queued (cub_emit_vertices)
  bool projected = false;       // the points of the current count have been projected in place
  bool caps_checked = false;    // k_check_caps of the current emission has been queued
  uint64_t n_points = 0, n_quads = 0, n_cells = 0, ghost_v = 0, ghost_f = 0;
  uint64_t point_base = 0, cell_base = 0;
  uint64_t flags = 0;
  cudaEvent_t wait_before_faces = nullptr;  // set by a queued count exchange (cuberille_comm.inl): the id bases are valid after it
  int id_bytes = 4, verts_per_cell = 4;
  double step_used = 0.0;

  bool timing = false;
  cudaEvent_t ev[10] = {};
  float ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  uint64_t launches = 0;
};

namespace {

int fail(cub_handle h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  return code;
}

#define CU_TRY(h, call)                                                                              \
  do {                                                                                               \
    cudaError_t e__ = (call);                                                                        \
    if (e__ != cudaSuccess)                                                                          \
      return fail(h, e__ == cudaErrorMemoryAllocation ? CUB_ERR_NOMEM : CUB_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                  cudaGetErrorString(e__), __FILE__, __LINE__);                                      \
  } while (0)

#define CUB_TRY(call)              \
  do {                             \
    int rc__ = (call);             \
    if (rc__ != CUB_OK) return rc__; \
  } while (0)

template <typename P>
int ensure(cub_handle h, DevBuf<P>& b, size_t n, bool zero_on_alloc = false) {
  if (n <= b.cap && b.p) return CUB_OK;
  if (b.p) {
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    CU_TRY(h, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  if (n == 0) n = 1;
  void* p = nullptr;
  CU_TRY(h, cudaMalloc(&p, n * sizeof(P)));
  b.p = static_cast<P*>(p);
  b.cap = n;
  if (zero_on_alloc) CU_TRY(h, cudaMemsetAsync(p, 0, n * sizeof(P), h->stream));
  return CUB_OK;
}

int pixel_bytes(int dtype) {
  switch (dtype) {
    case CUB_U8: case CUB_I8: return 1;
    case CUB_U16: case CUB_I16: return 2;
    case CUB_U32: case CUB_I32: case CUB_F32: return 4;
    case CUB_F64: case CUB_I64: case CUB_U64: return 8;
    default: return 0;
  }
}

#define DISPATCH_PIXEL(dtype, CALL)                          \
  switch (dtype) {                                           \
    case CUB_U8:  { typedef unsigned char  T; CALL; } break; \
    case CUB_I8:  { typedef signed char    T; CALL; } break; \
    case CUB_U16: { typedef unsigned short T; CALL; } break; \
    case CUB_I16: { typedef short          T; CALL; } break; \
    case CUB_U32: { typedef unsigned int   T; CALL; } break; \
    case CUB_I32: { typedef int            T; CALL; } break; \
    case CUB_F32: { typedef float          T; CALL; } break; \
    case CUB_F64: { typedef double         T; CALL; } break; \
    case CUB_I64: { typedef long long      T; CALL; } break; \
    case CUB_U64: { typedef unsigned long long T; CALL; } break; \
    default: break;                                          \
  }

// (double)(T)iso : m_IsoSurfaceValue is an InputPixelType (h:326).  An iso outside an integer T's range (or NaN) has
// no such value, and converting it to T would be undefined behaviour: it comes back as NaN, which equals no iso.
// The range is [min, max + 1) with max + 1 (a power of two) as the bound: for the 64-bit types (double)max rounds up
// to max + 1 itself, which does not convert.
template <typename T>
double iso_in_type(double iso) {
  if constexpr (std::is_integral<T>::value) {
    const double end = 2.0 * (double)(std::numeric_limits<T>::max() / 2 + 1);
    if (!(iso >= (double)std::numeric_limits<T>::min() && iso < end)) return std::numeric_limits<double>::quiet_NaN();
  }
  return (double)(T)iso;
}

double iso_as_pixel(int dtype, double iso) {
  double r = iso;
  DISPATCH_PIXEL(dtype, r = iso_in_type<T>(iso));
  return r;
}

struct Timer {
  cub_handle h;
  int slot;
  Timer(cub_handle h_, int slot_) : h(h_), slot(slot_) {
    if (h->timing) cudaEventRecord(h->ev[0], h->stream);
  }
  void stop() {
    if (h->timing) {
      cudaEventRecord(h->ev[1], h->stream);
      cudaEventSynchronize(h->ev[1]);
      float ms = 0;
      cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]);
      h->ms[slot] = ms;
    }
  }
};

// One kernel of a step on the handle's stream.  With programmatic dependent launch the kernel may be scheduled while
// its predecessor in the stream drains; every kernel launched through here starts with pdl_enter() (cbr_common.cuh).
template <typename... P, typename... A>
cudaError_t launch_step(cub_handle h, void (*kern)(P...), dim3 grid, dim3 block, bool pdl, A&&... args) {
  h->launches++;
  if (!h->pdl_on || !pdl) {
    kern<<<grid, block, 0, h->stream>>>(std::forward<A>(args)...);
    return cudaGetLastError();
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = h->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<A>(args)...);
}

// The kernels of one count, chosen from the input alone (choose_count_route)
enum class K1Route {
  fused,   // K1 + K2a as one kernel (k_fused.cuh)
  packed,  // k_classify_packed: 4 bytes per lane per load, for 8- and 16-bit pixels
  full,    // k_classify<T, true>: rows of whole tasks
  ragged,  // k_classify<T, false>
  padded,  // k_classify_padded: image_border_faces classifies into the padded lattice
};

struct CountRoute {
  K1Route k1 = K1Route::ragged;
  bool wide = true;         // sweep tiles of K2a and of the fused kernel's consumers: WideTile, else NarrowTile
  FuseArgs fuse{};          // k1 == fused: its tasks, batches and tiles (the launch adds the buffers and the sweep range)
  int fuse_tz = 0;
  unsigned fuse_blocks = 0;
  int scan_rows = 0;        // K2b: k_seg_scan_rows<scan_rows> for rows of one or two segments, 0: k_seg_scan
  bool pdl_on = false;
};

// k_classify_packed exists for the pixel types PackedTraits (k_classify.cuh) describes
template <typename T, typename = void> struct has_packed_kernel : std::false_type {};
template <typename T> struct has_packed_kernel<T, std::void_t<decltype(PackedTraits<T>::is_signed)>> : std::true_type {};

constexpr int kFuseStages = 3;

// Everything the count phase launches, from the lattice, the pixel type and the buffer's alignment.  Needs setup_grid
// and h->NS.
CountRoute choose_count_route(cub_handle h) {
  const Grid& g = h->g;
  const int pb = h->pix_bytes;
  const uintptr_t vol = reinterpret_cast<uintptr_t>(h->d_vol);
  CountRoute r;
  r.wide = g.Wx > 8;
  r.scan_rows = h->NS <= 2 ? h->NS : 0;
  // Programmatic dependent launch pays where the kernels are short.  Measured r2, gyroid f32, same box, off -> on:
  // 512^3 0.456 -> 0.444 ms per step, a 132-slice slab of 1024^2 rows 0.330 -> 0.319, Marschner-Lobb 512^3 0.405 -> 0.395;
  // 768^3 (453 M voxels) 1.112 -> 1.115, 1024^3 1.985 -> 2.02.  On below 300 M voxels per handle.
  r.pdl_on = (unsigned long long)g.X * g.Y * g.Zl < 300000000ull;

  bool packable = false;
  DISPATCH_PIXEL(h->dtype, packable = has_packed_kernel<T>::value);
  // k_classify_packed: rows must be whole warp loads and the buffer 4-byte aligned
  const bool packed = !h->pad && packable && g.X % (32 * (4 / pb)) == 0 && (vol & 3u) == 0;
  // the fused kernel: TMA bulk copies of 16-byte aligned rows; 8- and 16-bit pixels keep the packed kernel where it applies
  if (!h->pad && !packed && ((size_t)g.X * pb) % 16 == 0 && (vol & 15u) == 0) {
    FuseArgs& fa = r.fuse;
    const int wpt = kFuseStageBytes / (32 * pb);  // voxel words per task
    fa.groups_per_row = (unsigned)((g.Wx + wpt - 1) / wpt);
    fa.tasks_per_slice = fa.groups_per_row * (unsigned)g.Y;
    const unsigned long long tasks = (unsigned long long)fa.tasks_per_slice * (unsigned long long)g.Zl;
    // tasks per ticket / per publication: what the producer warps have in flight (2368 warps x batch x 4 KB) is how far
    // the consumers run behind, i.e. how long the bitmask words must survive in L2; a publication costs a release fence.
    // Measured on 1024^3 f32: 6 -> 0.842, 8 -> 0.831, 12 -> 0.839, 16 -> 0.856, 32 -> 0.895, 64 -> 0.924 ms.
    fa.batch = (unsigned)h->knobs.fuse_batch;
    const int txw = r.wide ? WideTile::TXW : NarrowTile::TXW, ty = r.wide ? WideTile::TY : NarrowTile::TY;
    const int gx = (g.Wx + txw - 1) / txw, gy = (g.Y + ty - 1) / ty;
    const int nz = h->zs1 - h->owner_z_min;
    // short sweeps: a tile can only start when the slice above its last one is classified, and what is still to sweep
    // when the producers finish is the kernel's tail; the two warm-up planes per tile cost issue slots the kernel has
    r.fuse_tz = std::min(h->knobs.fuse_tz > 0 ? h->knobs.fuse_tz : 8, pick_tz(gx, gy, nz, h->num_sms));
    const unsigned long long tiles = (unsigned long long)gx * gy * ((nz + r.fuse_tz - 1) / r.fuse_tz);
    if (tasks < (1ull << 32) - 256 && tiles < (1ull << 31)) {
      fa.n_tasks = (unsigned)tasks;
      fa.n_batches = (unsigned)((tasks + fa.batch - 1) / fa.batch);
      fa.n_tiles = (unsigned)tiles; fa.gx = (unsigned)gx; fa.gy = (unsigned)gy;
      // persistent: every CTA resident (4 per SM: 64 registers x 256 threads, ~47 KB of shared memory)
      const unsigned long long want = std::max<unsigned long long>((fa.n_batches + 3) / 4, fa.n_tiles);
      r.fuse_blocks = (unsigned)std::max<unsigned long long>(
          1, std::min<unsigned long long>(want, (unsigned long long)h->num_sms * h->knobs.fuse_ctas));
      r.k1 = K1Route::fused;
      return r;
    }
  }
  if (h->pad) r.k1 = K1Route::padded;
  else if (packed) r.k1 = K1Route::packed;
  else if (g.X % 32 == 0 && g.Wx % kWordsPerTask == 0) r.k1 = K1Route::full;
  else r.k1 = K1Route::ragged;
  return r;
}

// The inside predicate of the handle's mode, in the pixel type, handed to f: every classification route is instantiated
// for both (k_classify.cuh), and iso mode keeps its own instantiations rather than running as a range.
template <typename T, typename F>
auto with_inside(cub_handle h, F&& f) {
  return h->range_on ? f(Between<T>{(T)h->range_lo, (T)h->range_hi}) : f(AtLeast<T>{(T)h->params.iso_value});
}

template <typename T, typename C, typename In>
cudaError_t launch_fused(cub_handle h, In inside, const CountRoute& r, const SweepArgs& ca) {
  using Smem = FuseSmem<C, kFuseStages>;
  FuseArgs fa = r.fuse;
  fa.sw = ca;
  fa.sw.tz = r.fuse_tz;
  fa.vol = h->d_vol;
  fa.bits = h->bits.p;
  fa.ctr = h->d_fuse_ctr; fa.done = h->d_fuse_done;
  auto kern = k_classify_sweep<T, C, kFuseStages, In>;
  // (set on every launch: the attribute belongs to the current device, and one process may drive several)
  const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
  if (e != cudaSuccess) return e;
  kern<<<r.fuse_blocks, kFuseThreads, sizeof(Smem), h->stream>>>(fa, inside.param());
  h->launches++;
  return cudaGetLastError();
}

// K1 of the route on every local slice (rows are independent), with at most k1_ctas resident CTAs per SM; where the
// route fuses it, K1 + K2a
template <typename T, typename In>
cudaError_t launch_k1(cub_handle h, In inside, const CountRoute& r, const SweepArgs& ca) {
  if (r.k1 == K1Route::fused)
    return r.wide ? launch_fused<T, WideTile>(h, inside, r, ca) : launch_fused<T, NarrowTile>(h, inside, r, ca);
  const Grid& g = h->g;
  const T* vol = static_cast<const T*>(h->d_vol);
  const unsigned long long rows = (unsigned long long)g.Y * g.Zl;
  const unsigned long long max_blocks = (unsigned long long)h->num_sms * h->knobs.k1_ctas;
  auto blocks = [&](unsigned long long work) { return (unsigned)std::max(1ull, std::min((work + 7) / 8, max_blocks)); };
  h->launches++;
  if (r.k1 == K1Route::padded) {
    // g is the padded lattice, gv the voxel buffer
    const unsigned long long words = (unsigned long long)g.Wx * rows;  // < 2^32: checked by cub_count
    k_classify_padded<T, In><<<blocks(words), 256, 0, h->stream>>>(vol, h->bits.p, g, h->gv.X, h->gv.Y, h->gv.Zl,
                                                                   h->zpad_lo, inside.param(), (unsigned)words);
  } else if (r.k1 == K1Route::packed) {
    if constexpr (has_packed_kernel<T>::value) {  // (the only pixel types choose_count_route gives this route)
      const unsigned tasks_per_row = (unsigned)((g.Wx + 31) / 32);
      const unsigned long long tasks = rows * tasks_per_row;  // cub_count checks rows * groups < 2^32
      k_classify_packed<T, In><<<blocks(tasks), 256, 0, h->stream>>>(vol, h->bits.p, g, inside.param(), (unsigned)tasks,
                                                                     tasks_per_row);
    }
  } else {
    const unsigned groups = (unsigned)((g.Wx + kWordsPerTask - 1) / kWordsPerTask);
    const unsigned tasks = (unsigned)(rows * groups);  // dims < 2^31 and cub_count checks rows*groups < 2^32
    if (r.k1 == K1Route::full)
      k_classify<T, true, In><<<blocks(tasks), 256, 0, h->stream>>>(vol, h->bits.p, g, inside.param(), tasks, groups);
    else
      k_classify<T, false, In><<<blocks(tasks), 256, 0, h->stream>>>(vol, h->bits.p, g, inside.param(), tasks, groups);
  }
  return cudaGetLastError();
}

// capacities of the result buffers, for k_check_caps (and the early record loads of k_vertices)
Caps make_caps(cub_handle h, unsigned long long quads_cap) {
  Caps c;
  c.raster = h->raster ? 1 : 0;
  c.points = h->raster ? h->points.cap / 3 : std::min(h->points.cap / 3, h->vtx.cap);
  c.perm = h->perm.cap;
  c.quads = quads_cap;
  return c;
}

// K4 on `pts` (explicit count n), or - from_info - on the handle's point buffer with the range taken from the
// device-side run info (n = the capacity of the buffer)
int launch_project(cub_handle h, float* pts, size_t n, bool from_info, bool include_ghost) {
  if (n == 0) return CUB_OK;
  ProjArgs a;
  a.vol = h->d_vol;
  a.g = h->gv;
  a.geom = h->geom;
  for (int k = 0; k < 3; ++k) a.i0[k] = h->i0[k];
  a.iso = iso_as_pixel(h->dtype, h->params.iso_value);
  a.thr = h->params.surface_distance_threshold;
  a.step0 = h->step_used;
  a.relax = h->params.step_relaxation;
  a.max_steps = h->params.max_steps;
  a.points = pts;
  a.n_points = n;
  a.info = from_info ? h->d_info : nullptr;
  a.include_ghost = include_ghost ? 1 : 0;
  a.work = h->d_info + kInfoWords;
  a.refill = (unsigned)h->knobs.proj_refill;
  CU_TRY(h, cudaMemsetAsync(a.work, 0, sizeof(unsigned long long), h->stream));
  const size_t want = (n + 127) / 128;
  const unsigned blocks = (unsigned)std::min<size_t>(want, (size_t)h->num_sms * h->knobs.proj_ctas);
  const int method = h->params.projection_method;
  if (method != CUB_PROJECT_DEFAULT) {
    // the reference's compile-time alternates (USE_ADVANCED_PROJECTION / USE_LINESEARCH_PROJECTION)
    const unsigned ablocks = (unsigned)std::min<size_t>(want, (size_t)h->num_sms * 16);
    if (h->geom.oriented) { DISPATCH_PIXEL(h->dtype, (k_project_alt<T, true><<<ablocks, 128, 0, h->stream>>>(a, method))); }
    else { DISPATCH_PIXEL(h->dtype, (k_project_alt<T, false><<<ablocks, 128, 0, h->stream>>>(a, method))); }
  } else if (h->geom.oriented) { DISPATCH_PIXEL(h->dtype, (k_project<T, true><<<blocks, 128, 0, h->stream>>>(a))); }
  else { DISPATCH_PIXEL(h->dtype, (k_project<T, false><<<blocks, 128, 0, h->stream>>>(a))); }
  h->launches++;
  CU_TRY(h, cudaGetLastError());
  return CUB_OK;
}

// geometry of the run: Grid + own range in local coordinates
int setup_grid(cub_handle h) {
  if (!h->has_volume) return fail(h, CUB_ERR_INVALID, "no volume set");
  Grid& gv = h->gv;
  gv.X = (int)h->dims[0];
  gv.Y = (int)h->dims[1];
  gv.Zl = (int)h->dims[2];
  gv.Wx = (gv.X + 31) / 32;
  gv.Wp = (gv.Wx + 3) & ~3;
  gv.zg0 = (int)h->local_z0;
  gv.Zg = (int)h->image_nz;
  // image_border_faces: everything after K1 runs on the image padded with one outside layer (x and y always, z
  // where the local buffer touches the end of the image), in the padded image's coordinates
  const int pad = h->params.image_border_faces ? 1 : 0;
  const int zlo = (pad && h->local_z0 == 0) ? 1 : 0;
  const int zhi = (pad && h->local_z0 + h->dims[2] == h->image_nz) ? 1 : 0;
  h->pad = pad;
  h->zpad_lo = zlo;
  Grid& g = h->g;
  g.X = gv.X + 2 * pad;
  g.Y = gv.Y + 2 * pad;
  g.Zl = gv.Zl + zlo + zhi;
  g.Wx = (g.X + 31) / 32;
  g.Wp = (g.Wx + 3) & ~3;
  g.zg0 = gv.zg0 + pad - zlo;
  g.Zg = gv.Zg + 2 * pad;
  const long long own0 = (pad && h->own_z0 == 0) ? 0 : (long long)h->own_z0 + pad;
  const long long own1 = (pad && h->own_z1 == h->image_nz) ? (long long)h->image_nz + 2 : (long long)h->own_z1 + pad;
  h->zs0 = (int)(own0 - g.zg0);
  h->zs1 = (int)(own1 - g.zg0);
  h->owner_z_min = (h->own_z0 > 0) ? h->zs0 - 1 : h->zs0;
  return CUB_OK;
}

// txx:75-85: auto step length = max spacing * 0.25
double step_length_used(const cub_params& P, const Geom& G) {
  double ms = G.spacing[0];
  for (int a = 1; a < 3; ++a) ms = G.spacing[a] > ms ? G.spacing[a] : ms;
  return P.step_length < 0.0 ? ms * 0.25 : P.step_length;
}

void compute_step(cub_handle h) { h->step_used = step_length_used(h->params, h->geom); }

}  // namespace

extern "C" {

int cub_abi_version(void) { return CUB_ABI_VERSION; }

void cub_default_params(cub_params* p) {
  if (!p) return;
  memset(p, 0, sizeof *p);
  p->iso_value = 1.0;  // NumericTraits<InputPixelType>::One  (txx:34)
  p->generate_triangles = 1;
  p->project_vertices = 1;
  p->save_pixel_as_cell_data = 0;
  p->surface_distance_threshold = 0.5;
  p->step_length = -1.0;
  p->step_relaxation = 0.95;
  p->max_steps = 50;
}

int cub_create(int device, void* stream, cub_handle* out) {
  if (!out) return CUB_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return CUB_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return CUB_ERR_CUDA;
  cub_handle h = new (std::nothrow) cub_handle_s;
  if (!h) return CUB_ERR_NOMEM;
  h->device = device;
  if (stream) {
    h->stream = static_cast<cudaStream_t>(stream);
  } else {
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return CUB_ERR_CUDA; }
    h->own_stream = true;
  }
  {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) h->num_sms = sms;
    // the tuning knobs are read here, once, and clamped (a zero would make a launch with no blocks)
    h->knobs.k1_ctas = env_int("CUB_K1_CTAS_PER_SM", 32, 1, 32);
    h->knobs.fuse_tz = env_int("CUB_FUSE_TZ", 0, 0, 32);
    h->knobs.fuse_ctas = env_int("CUB_FUSE_CTAS_PER_SM", 4, 1, 4);
    h->knobs.fuse_batch = env_int("CUB_FUSE_BATCH", 8, 1, 256);
    h->knobs.scan_ctas = env_int("CUB_SCAN_CTAS_PER_SM", 8, 1, 32);
    h->knobs.proj_ctas = env_int("CUB_PROJ_CTAS_PER_SM", 6, 1, 16);
    h->knobs.proj_refill = env_int("CUB_PROJ_REFILL", 18, 1, 32);
  }
  bool ok = ensure(h, h->ctrl, kCtrlHead) == CUB_OK &&
            cudaMallocHost(&h->h_info, (kInfoWords + 2) * sizeof(unsigned long long)) == cudaSuccess;
  if (ok) { h->d_info = h->ctrl.p; h->d_ticket = reinterpret_cast<unsigned int*>(h->ctrl.p + kInfoWords + 2); }
  for (int i = 0; ok && i < 10; ++i) ok = cudaEventCreate(&h->ev[i]) == cudaSuccess;
  if (!ok) { cub_destroy(h); return CUB_ERR_CUDA; }
  cub_default_params(&h->params);
  *out = h;
  return CUB_OK;
}

int cub_destroy(cub_handle h) {
  if (!h) return CUB_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  cudaFree(h->vol_owned.p);
  cudaFree(h->bits.p); cudaFree(h->cnt.p); cudaFree(h->act.p); cudaFree(h->perm.p); cudaFree(h->own.p); cudaFree(h->seg.p);
  cudaFree(h->ctrl.p); cudaFree(h->cofs.p); cudaFree(h->vtx.p); cudaFree(h->vsl.p);
  if (h->h_info) cudaFreeHost(h->h_info);
  cudaFree(h->points.p); cudaFree(h->cells.p); cudaFree(h->celldata.p); cudaFree(h->quads.p);
  cudaFree(h->roi_buf.p); cudaFree(h->label_table.p);
  cudaFree(h->cat_points.p); cudaFree(h->cat_cells.p); cudaFree(h->cat_celldata.p);
  for (int i = 0; i < 10; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  if (h->own_stream) cudaStreamDestroy(h->stream);
  delete h;
  return CUB_OK;
}

const char* cub_last_error(cub_handle h) { return h ? h->err.c_str() : "null handle"; }

// spacing, direction cosines and the matrices built from them (null spacing / direction: 1 / identity), shared by
// cub_set_volume and cub_projection_halo_oriented so that the halo a slab is cut with and the halo cub_count checks come from
// the same geometry
static int make_geom(cub_handle h, const double spacing[3], const double direction[9], Geom& G) {
  for (int a = 0; a < 3; ++a) {
    const double s = spacing ? spacing[a] : 1.0;
    if (!(s > 0.0) || !std::isfinite(s)) return fail(h, CUB_ERR_INVALID, "spacing[%d] must be positive and finite", a);
    G.spacing[a] = s;
  }
  // direction cosines (itk::ImageBase::GetDirection): identity (or null) is the non-oriented image of the
  // reference's tests; anything else switches TransformIndexToPhysicalPoint, the continuous index and the
  // gradient to the oriented forms (cbr_common.cuh, k_project.cuh)
  static const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  bool ident = true;
  for (int i = 0; i < 9; ++i) {
    const double d = direction ? direction[i] : I[i];
    if (!std::isfinite(d)) return fail(h, CUB_ERR_INVALID, "direction[%d] is not finite", i);
    ident = ident && d == I[i];
  }
  G.oriented = ident ? 0 : 1;
  for (int k = 0; k < 9; ++k) {
    G.dir[k] = ident ? I[k] : direction[k];
    G.m[k] = G.dir[k] * G.spacing[k % 3];  // D * diag(spacing)
  }
  const double* m = G.m;  // cofactor inverse
  const double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
  const double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
  if (!(std::fabs(det) > 0.0) || !std::isfinite(det)) return fail(h, CUB_ERR_INVALID, "the direction matrix is singular");
  G.minv[0] = c00 / det; G.minv[1] = (m[2] * m[7] - m[1] * m[8]) / det; G.minv[2] = (m[1] * m[5] - m[2] * m[4]) / det;
  G.minv[3] = c01 / det; G.minv[4] = (m[0] * m[8] - m[2] * m[6]) / det; G.minv[5] = (m[2] * m[3] - m[0] * m[5]) / det;
  G.minv[6] = c02 / det; G.minv[7] = (m[1] * m[6] - m[0] * m[7]) / det; G.minv[8] = (m[0] * m[4] - m[1] * m[3]) / det;
  return CUB_OK;
}

static int set_geometry(cub_handle h, int dtype, const uint64_t dims[3], const double spacing[3],
                        const double origin[3], const double direction[9]) {
  if (!dims) return fail(h, CUB_ERR_INVALID, "dims is null");
  const int pb = pixel_bytes(dtype);
  if (!pb) return fail(h, CUB_ERR_INVALID, "unknown dtype %d", dtype);
  for (int a = 0; a < 3; ++a)
    if (dims[a] == 0 || dims[a] >= (1ull << 31)) return fail(h, CUB_ERR_INVALID, "dims[%d]=%llu out of range", a, (unsigned long long)dims[a]);
  CUB_TRY(make_geom(h, spacing, direction, h->geom));
  for (int a = 0; a < 3; ++a) {
    h->geom.origin[a] = origin ? origin[a] : 0.0;
    h->dims[a] = dims[a];
  }
  h->dtype = dtype;
  h->pix_bytes = pb;
  h->i0[0] = h->i0[1] = h->i0[2] = 0;
  h->range_on = false;
  h->roi_on = false;
  h->slab_set = false;
  h->image_nz = dims[2];
  h->local_z0 = 0;
  h->own_z0 = 0;
  h->own_z1 = dims[2];
  h->counted = h->emitted = h->count_queued = false;
  return CUB_OK;
}

int cub_set_volume(cub_handle h, const void* data, int dtype, const uint64_t dims[3], const double spacing[3],
                   const double origin[3], const double direction[9], int mem_kind) {
  if (!h) return CUB_ERR_INVALID;
  if (!data) return fail(h, CUB_ERR_INVALID, "data is null");
  CU_TRY(h, cudaSetDevice(h->device));
  h->has_volume = false;
  CUB_TRY(set_geometry(h, dtype, dims, spacing, origin, direction));
  const size_t bytes = (size_t)dims[0] * dims[1] * dims[2] * h->pix_bytes;
  if (mem_kind == CUB_MEM_DEVICE) {
    // every kernel loads whole pixels from the borrowed buffer
    if (reinterpret_cast<uintptr_t>(data) % (uintptr_t)h->pix_bytes != 0)
      return fail(h, CUB_ERR_INVALID, "device volume pointer %p is not aligned to the %d-byte pixel", data, h->pix_bytes);
    h->d_vol = data;
  } else if (mem_kind == CUB_MEM_HOST) {
    CUB_TRY(ensure(h, h->vol_owned, bytes));
    CU_TRY(h, cudaMemcpyAsync(h->vol_owned.p, data, bytes, cudaMemcpyHostToDevice, h->stream));
    h->d_vol = h->vol_owned.p;
  } else {
    return fail(h, CUB_ERR_INVALID, "bad mem_kind %d", mem_kind);
  }
  h->has_volume = true;
  return CUB_OK;
}

int cub_set_region_index(cub_handle h, const int64_t index[3]) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->has_volume) return fail(h, CUB_ERR_INVALID, "cub_set_region_index before cub_set_volume");
  for (int k = 0; k < 3; ++k) {
    const long long v = index ? (long long)index[k] : 0;
    if (v < -(1ll << 30) || v > (1ll << 30)) return fail(h, CUB_ERR_INVALID, "region index beyond +-2^30 is not supported");
    h->i0[k] = v + (h->roi_on ? (long long)h->roi_lo[k] : 0);
  }
  h->counted = h->emitted = h->count_queued = false;
  return CUB_OK;
}

int cub_set_inside_range(cub_handle h, int enable, double lower, double upper) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->has_volume) return fail(h, CUB_ERR_INVALID, "cub_set_inside_range before cub_set_volume");
  h->counted = h->emitted = h->count_queued = false;
  if (!enable) {
    h->range_on = false;
    return CUB_OK;
  }
  // the bounds are pixel values, checked by the rule cub_count applies to the iso value
  if (std::isnan(lower) || std::isnan(upper)) return fail(h, CUB_ERR_INVALID, "inside range bound is NaN");
  if (iso_as_pixel(h->dtype, lower) != lower || iso_as_pixel(h->dtype, upper) != upper)
    return fail(h, CUB_ERR_INVALID, "inside range [%.17g, %.17g] is not representable in the pixel type", lower, upper);
  if (!(lower <= upper)) return fail(h, CUB_ERR_INVALID, "inside range [%.17g, %.17g]: lower exceeds upper", lower, upper);
  h->range_on = true;
  h->range_lo = lower;
  h->range_hi = upper;
  return CUB_OK;
}

int cub_set_slab(cub_handle h, uint64_t image_nz, uint64_t local_z0, uint64_t own_z0, uint64_t own_z1) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->has_volume) return fail(h, CUB_ERR_INVALID, "cub_set_slab before cub_set_volume");
  if (h->roi_on) return fail(h, CUB_ERR_UNSUPPORTED, "a z-slab cannot be combined with a region of interest");
  const uint64_t zl = h->dims[2];
  if (image_nz == 0 || image_nz >= (1ull << 31) || local_z0 + zl > image_nz)
    return fail(h, CUB_ERR_INVALID, "local buffer [%llu,%llu) exceeds image_nz %llu", (unsigned long long)local_z0,
                (unsigned long long)(local_z0 + zl), (unsigned long long)image_nz);
  if (!(own_z0 < own_z1) || own_z1 > image_nz) return fail(h, CUB_ERR_INVALID, "bad own range");
  const uint64_t need_lo = own_z0 >= 2 ? own_z0 - 2 : 0;
  const uint64_t need_hi = own_z1 + 1 < image_nz ? own_z1 + 1 : image_nz;
  if (local_z0 > need_lo || local_z0 + zl < need_hi)
    return fail(h, CUB_ERR_INVALID, "local buffer must cover slices [%llu,%llu) (own range plus halo)",
                (unsigned long long)need_lo, (unsigned long long)need_hi);
  h->image_nz = image_nz;
  h->local_z0 = local_z0;
  h->own_z0 = own_z0;
  h->own_z1 = own_z1;
  h->slab_set = true;
  h->counted = h->emitted = h->count_queued = false;
  return CUB_OK;
}

}  // extern "C"

namespace {

// slices a projected vertex can reach below / above the plane it starts on: the travel is at most the geometric sum of
// the step lengths (max_steps + 2 moves, txx:464-469), trilinear interpolation reads one node further and the central
// differences one more (SURVEY section 7 "projection halo")
void projection_reach(const cub_params& P, double step_used, double z_index_per_unit, uint64_t* below, uint64_t* above) {
  const double spacing_z = 1.0 / z_index_per_unit;
  const double r = P.step_relaxation, n = (double)P.max_steps + 2.0;
  double travel = (r >= 1.0) ? step_used * n : step_used * (1.0 - std::pow(r, n)) / (1.0 - r);
  if (!(travel >= 0.0)) travel = 0.0;
  const double t = std::ceil(travel / spacing_z - 1e-9);
  const uint64_t ct = t > 1e9 ? (uint64_t)1e9 : (uint64_t)t;
  *below = ct + 3;  // (the ghost vertices of the plane under the own range are projected too, for the triangle split)
  *above = ct + 2;
}

// the halo of a z-slab of an image with this geometry: what cub_projection_halo_oriented reports and what count_launch requires
void slab_halo(const cub_params& P, const Geom& G, uint64_t* below, uint64_t* above) {
  if (!P.project_vertices) {
    *below = 2;
    *above = 1;
    return;
  }
  // index-space z travel per unit of physical travel: 1 / spacing_z, or the 1-norm of the z row of M^-1
  const double zpu = G.oriented ? std::fabs(G.minv[6]) + std::fabs(G.minv[7]) + std::fabs(G.minv[8]) : 1.0 / G.spacing[2];
  projection_reach(P, step_length_used(P, G), zpu, below, above);
}

// ---- the count phase, queued on the handle's stream (no host synchronisation) ----------------------------------
int count_launch(cub_handle h, const cub_params* p) {
  if (!p) return fail(h, CUB_ERR_INVALID, "params is null");
  CU_TRY(h, cudaSetDevice(h->device));
  h->counted = h->emitted = h->count_queued = h->emit_unverified = false;
  h->wait_before_faces = nullptr;
  h->params = *p;
  CUB_TRY(setup_grid(h));
  if (h->range_on) {
    // (the iso value plays no part in range mode)
    if (p->project_vertices)
      return fail(h, CUB_ERR_INVALID, "vertex projection needs an iso-surface and an inside range has none: turn "
                                      "project_vertices off, or leave range mode (cub_set_inside_range with enable = 0)");
  } else if (iso_as_pixel(h->dtype, p->iso_value) != p->iso_value) {
    return fail(h, CUB_ERR_INVALID, "iso value %.17g is not representable in the pixel type", p->iso_value);
  }
  if (p->projection_method < CUB_PROJECT_DEFAULT || p->projection_method > CUB_PROJECT_LINESEARCH || p->reserved != 0)
    return fail(h, CUB_ERR_INVALID, "unknown projection_method %d", (int)p->projection_method);
  compute_step(h);
  const Grid& g = h->g;
  // the halo contract (cub_set_slab checks it too; cub_generate_volume with a z offset does not go through it)
  {
    const uint64_t zl = h->dims[2];
    const uint64_t need_lo = h->own_z0 >= 2 ? h->own_z0 - 2 : 0;
    const uint64_t need_hi = h->own_z1 + 1 < h->image_nz ? h->own_z1 + 1 : h->image_nz;
    if (!(h->own_z0 < h->own_z1) || h->own_z1 > h->image_nz || h->local_z0 > need_lo || h->local_z0 + zl < need_hi ||
        h->owner_z_min < 0 || h->zs1 > g.Zl)
      return fail(h, CUB_ERR_INVALID, "the local buffer [%llu,%llu) does not cover the own range [%llu,%llu) plus its halo: call cub_set_slab",
                  (unsigned long long)h->local_z0, (unsigned long long)(h->local_z0 + zl), (unsigned long long)h->own_z0,
                  (unsigned long long)h->own_z1);
    if (p->project_vertices && (h->local_z0 > 0 || h->local_z0 + zl < h->image_nz)) {
      // a true slab: the projection must not run into the end of the local buffer (its reads would be clamped there
      // and the result would differ from the whole-image run without any error)
      uint64_t below = 0, above = 0;
      slab_halo(*p, h->geom, &below, &above);
      const uint64_t lo = h->own_z0 > below ? h->own_z0 - below : 0;
      const uint64_t hi = h->own_z1 + above < h->image_nz ? h->own_z1 + above : h->image_nz;
      if (h->local_z0 > lo || h->local_z0 + zl < hi)
        return fail(h, CUB_ERR_INVALID,
                    "projection needs a halo of %llu slices below and %llu above the own range (cub_projection_halo): the local "
                    "buffer must cover [%llu,%llu)", (unsigned long long)below, (unsigned long long)above,
                    (unsigned long long)lo, (unsigned long long)hi);
    }
  }
  if ((unsigned long long)g.Y * g.Zl * ((g.Wx + kWordsPerTask - 1) / kWordsPerTask) >= (1ull << 32))
    return fail(h, CUB_ERR_INVALID, "volume too large for one handle: split into z-slabs");
  if ((unsigned long long)g.Y * g.Wp >= (1ull << 31)) return fail(h, CUB_ERR_UNSUPPORTED, "x*y too large");
  if (g.X > 65534 || g.Y > 32766) return fail(h, CUB_ERR_UNSUPPORTED, "x size above 65534 or y size above 32766 voxels is not supported");
  if (h->zs1 + 1 - h->owner_z_min > 65535)
    return fail(h, CUB_ERR_UNSUPPORTED, "more than 65534 slices in one handle: split into z-slabs");
  const size_t words = (size_t)g.Zl * g.Y * g.Wp;
  const bool layout_changed = h->bits_layout[0] != (uint64_t)g.X || h->bits_layout[1] != (uint64_t)g.Y ||
                              h->bits_layout[2] != (uint64_t)g.Zl;
  const bool had = h->bits.p && h->bits.cap >= words;
  CUB_TRY(ensure(h, h->bits, words));
  if ((!had || layout_changed) && g.Wp != g.Wx) CU_TRY(h, cudaMemsetAsync(h->bits.p, 0, words * 4, h->stream));
  h->bits_layout[0] = g.X; h->bits_layout[1] = g.Y; h->bits_layout[2] = g.Zl;
  // entry lattice of the counts / active masks: one entry per corner word, (Zl+1) x (Y+1) x EW; NS segments of 32 per row
  const int Wc = (g.X + 32) / 32;
  h->EY = g.Y + 1;
  h->EW = (Wc + 1 + 3) & ~3;
  h->NS = (h->EW + 31) / 32;
  const size_t plane_entries = (size_t)h->EY * h->EW;
  const size_t entries = plane_entries * (size_t)(g.Zl + 1);
  const size_t lattice_rows = (size_t)h->EY * (size_t)(g.Zl + 1);
  if (entries + 4096 >= (1ull << 32)) return fail(h, CUB_ERR_INVALID, "volume too large for one handle: split into z-slabs");
  const bool had_e = h->cnt.p && h->cnt.cap >= entries && h->act.p && h->act.cap >= entries + 4;
  CUB_TRY(ensure(h, h->cnt, entries));
  CUB_TRY(ensure(h, h->act, entries + 4));
  CUB_TRY(ensure(h, h->seg, lattice_rows * h->NS));
  h->raster = p->vertex_order == CUB_ORDER_RASTER;
  CUB_TRY(ensure(h, h->cofs, entries + 4));
  if (!h->raster) CUB_TRY(ensure(h, h->own, 2 * entries));
  // entries that K2a never writes (padding columns) must read as zero counts / empty masks
  if (!had_e || layout_changed) {
    CU_TRY(h, cudaMemsetAsync(h->cnt.p, 0, entries * 4, h->stream));
    CU_TRY(h, cudaMemsetAsync(h->act.p, 0, (entries + 4) * 4, h->stream));
  }

  if (h->timing) cudaEventRecord(h->ev[2], h->stream);

  // K2 scan range = voxel slices [owner_z_min, zs1) and corner planes [zs0, zs1]
  const size_t row_begin = (size_t)h->owner_z_min * h->EY;
  const size_t n_rows = (size_t)(h->zs1 + 1 - h->owner_z_min) * h->EY;
  const CountRoute route = choose_count_route(h);
  // one large scan tile per resident CTA, so that every tile is in flight when the look-backs run; rows with at most
  // two segments take the one-pass kernel, whose warps hold at most 32 * kScanBatches rows (more tiles than resident
  // CTAs are fine: a tile only waits for tiles with earlier tickets)
  int scan_occ = 0;
  CU_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&scan_occ, k_seg_scan, kScanThreads, 0));
  const size_t max_tiles = (size_t)h->num_sms * std::max(1, std::min(scan_occ, h->knobs.scan_ctas));
  size_t rows_per_tile = ((n_rows + max_tiles - 1) / max_tiles + kScanWarps - 1) / kScanWarps * kScanWarps;
  if (rows_per_tile < (size_t)kScanWarps) rows_per_tile = kScanWarps;
  if (route.scan_rows) rows_per_tile = std::min<size_t>(rows_per_tile, (size_t)kScanWarps * 32 * kScanBatches);
  const size_t n_tiles = (n_rows + rows_per_tile - 1) / rows_per_tile;
  {
    const size_t slice_words = ((size_t)g.Zl + 2 + 1) / 2;  // one u32 per slice
    const size_t need = kCtrlHead + 3 * n_tiles + 2 * slice_words + 1;
    CUB_TRY(ensure(h, h->ctrl, need));
    h->d_info = h->ctrl.p;
    h->d_ticket = reinterpret_cast<unsigned int*>(h->ctrl.p + kInfoWords + 2);
    h->d_status = h->ctrl.p + kCtrlHead;
    h->d_slice_any = reinterpret_cast<uint32_t*>(h->d_status + 3 * n_tiles);
    h->d_fuse_done = reinterpret_cast<unsigned*>(h->d_status + 3 * n_tiles + slice_words);   // fused kernel: tasks done per slice
    h->d_fuse_ctr = reinterpret_cast<unsigned*>(h->d_status + 3 * n_tiles + 2 * slice_words);  // ... and its two tickets
    h->ctrl_used = need;
  }
  SweepArgs ca{};
  ca.bits = h->bits.p; ca.g = g; ca.Wc = Wc; ca.EY = h->EY; ca.EW = h->EW;
  ca.cnt = h->cnt.p; ca.act = h->act.p; ca.own = h->raster ? nullptr : h->own.p;
  ca.slice_any = h->d_slice_any;
  {
    h->pdl_on = route.pdl_on;
    // K1 + K2a: one warp-specialised kernel where the route fuses them (k_fused.cuh), else K1 then K2a on the handle's
    // stream.  The control block (tickets, per-slice progress, scan descriptors, slice occupancy) is cleared first.
    CU_TRY(h, cudaMemsetAsync(h->ctrl.p, 0, h->ctrl_used * sizeof(unsigned long long), h->stream));
    ca.z_begin = h->owner_z_min; ca.z_end = h->zs1;
    {
      Timer t(h, 0);
      cudaError_t k1_launch = cudaSuccess;
      DISPATCH_PIXEL(h->dtype, (k1_launch = with_inside<T>(h, [&](auto in) { return launch_k1<T>(h, in, route, ca); })));
      CU_TRY(h, k1_launch);
      t.stop();
    }
    h->fused_last = route.k1 == K1Route::fused;
    if (h->timing) cudaEventRecord(h->ev[0], h->stream);
    if (!h->fused_last) {
      CU_TRY(h, route.wide ? launch_sweep<WideTile>(ca, h->stream, h->num_sms)
                           : launch_sweep<NarrowTile>(ca, h->stream, h->num_sms));
      h->launches++;
    }
  }
  {
    if (h->timing) cudaEventRecord(h->ev[6], h->stream);
    SegScanArgs sa{};
    sa.cnt = h->cnt.p; sa.seg = h->seg.p; sa.cofs = nullptr;  // (k_assign / k_points_raster write the dense slot bases, coalesced)
    sa.row_begin = (unsigned)row_begin; sa.n_rows = (unsigned)n_rows;
    sa.EW = (unsigned)h->EW; sa.NS = (unsigned)h->NS;
    sa.ghost_row_end = (unsigned)((size_t)h->zs0 * h->EY);
    // the prefixes at the first own entry: what the ghost slice below contributed (slab runs)
    sa.mark_row_vf = (h->owner_z_min < h->zs0) ? (unsigned)((size_t)h->zs0 * h->EY) : 0xffffffffu;
    // raster order: the corners of the bottom plane of a slab's range belong to the slab underneath
    sa.mark_row_c = (h->own_z0 > 0) ? (unsigned)((size_t)(h->zs0 + 1) * h->EY) : 0xffffffffu;
    sa.rows_per_tile = (unsigned)rows_per_tile; sa.n_tiles = (unsigned)n_tiles;
    sa.status = h->d_status; sa.ticket = h->d_ticket; sa.info = h->d_info;
    if (route.scan_rows == 1) CU_TRY(h, launch_step(h, k_seg_scan_rows<1>, dim3((unsigned)n_tiles), dim3(kScanThreads), true, sa));
    else if (route.scan_rows == 2) CU_TRY(h, launch_step(h, k_seg_scan_rows<2>, dim3((unsigned)n_tiles), dim3(kScanThreads), true, sa));
    else CU_TRY(h, launch_step(h, k_seg_scan, dim3((unsigned)n_tiles), dim3(kScanThreads), true, sa));
    CU_TRY(h, launch_step(h, k_finalize_info, dim3(1), dim3(256), true, h->d_info, h->raster ? 1 : 0, (const uint32_t*)h->d_slice_any,
                          h->owner_z_min, h->zs1));
    if (h->timing) {
      cudaEventRecord(h->ev[1], h->stream);
      cudaEventSynchronize(h->ev[1]);
      cudaEventElapsedTime(&h->ms[1], h->ev[0], h->ev[1]);  // count sweep + scan
      cudaEventElapsedTime(&h->ms[7], h->ev[6], h->ev[1]);  // the scan alone
    }
  }
  h->point_base = h->cell_base = 0;
  h->count_queued = true;
  h->vertices_done = false;
  h->projected = false;
  h->caps_checked = false;
  return CUB_OK;
}

// ---- the host learns the counts: one device -> host copy and one synchronisation -----------------------------------
const char* const kEmptySliceRemark =
    "an empty voxel slice lies between occupied slices: the reference filter merges vertices of different corner "
    "planes there (its lookup-plane rotation only advances on inside voxels, txx:155-161); this mesh follows the "
    "intended rule and may differ from the reference's";

int count_finish(cub_handle h) {
  CU_TRY(h, cudaSetDevice(h->device));
  if (h->wait_before_faces) CU_TRY(h, cudaStreamWaitEvent(h->stream, h->wait_before_faces, 0));
  CU_TRY(h, cudaMemcpyAsync(h->h_info, h->d_info, kInfoWords * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  if (h->timing) {
    cudaEventRecord(h->ev[3], h->stream);
    cudaEventSynchronize(h->ev[3]);
    cudaEventElapsedTime(&h->ms[5], h->ev[2], h->ev[3]);
  }
  const uint64_t tot_v = h->h_info[kInfoTotV], tot_f = h->h_info[kInfoTotF];
  if (tot_v >= (1ull << 32) || tot_f >= (1ull << 32))
    return fail(h, CUB_ERR_OVERFLOW, "more than 2^32 vertices or faces in one handle (%llu, %llu): split into z-slabs",
                (unsigned long long)tot_v, (unsigned long long)tot_f);
  h->n_active = h->h_info[kInfoTotC];
  h->ghost_f = h->h_info[kInfoMarkF];
  // scan-relative vertex ids below ghost_v belong to the slab underneath (first-touch order: what the ghost
  // slice created; raster order: the corners of the shared bottom plane)
  h->ghost_v = h->h_info[kInfoGhostV];
  h->n_points = h->h_info[kInfoPoints];
  h->n_quads = h->h_info[kInfoQuads];
  h->point_base = h->h_info[kInfoPointBase];
  h->cell_base = h->h_info[kInfoCellBase];
  h->flags = h->h_info[kInfoFlags];
  h->warning.clear();
  if (h->flags & kFlagEmptyInteriorSlice) h->warning = kEmptySliceRemark;
  h->counted = true;
  return CUB_OK;
}

// The vertex stage of cub_emit: K3a (reference order) or k_points_raster.  It needs the counts but not the id
// base, so a multi-GPU caller can queue it before the ranks have exchanged their counts (cub_emit_vertices).
// exact: the host knows the counts, sizes the buffers and the grids from them; otherwise the buffers keep their
// sizes and the grids cover their capacity (k_check_caps flags an emission that does not fit).  Either way the
// kernels read the counts from the device-side run info.
const int kNeedSizes = -1000;

// quads, triangles with the fixed split, or quads into a scratch buffer that K5 splits by the diagonal test.
// Unprojected quads of a non-oriented image are axis-aligned rectangles: both diagonals are equal in fp64 whatever
// the spacing, `>=` takes the first split (txx:298-302), so the face kernel writes the triangles directly.  Projected
// points, and the rounded points of an oriented image, need the test.
int emit_mode(cub_handle h) {
  const cub_params& P = h->params;
  if (!P.generate_triangles) return kEmitQuads;
  return (P.project_vertices || h->geom.oriented) ? kEmitScratchQuads : kEmitTrisFixed;
}

int size_vertex_buffers(cub_handle h) {
  const size_t n_pts_all = (size_t)(h->ghost_v + h->n_points);
  CUB_TRY(ensure(h, h->points, 3 * (n_pts_all + n_pts_all / 16)));
  if (!h->raster) {
    CUB_TRY(ensure(h, h->perm, (size_t)h->n_active + (size_t)h->n_active / 16));
    CUB_TRY(ensure(h, h->vtx, h->points.cap / 3));
  }
  return CUB_OK;
}

int emit_vertex_stage(cub_handle h, bool exact) {
  const Grid& g = h->g;
  const int mode = emit_mode(h);
  const int nz = h->zs1 - h->owner_z_min;
  if (exact) {
    CUB_TRY(size_vertex_buffers(h));
    if (h->n_quads == 0) { h->vertices_done = true; return CUB_OK; }
  } else if (!h->points.p || (!h->raster && (!h->perm.p || !h->vtx.p))) {
    return kNeedSizes;
  }
  h->vertices_done = true;
  h->projected = false;
  if (!h->caps_checked) {
    // the vertex stage queued ahead of the emission (cub_emit_vertices): the vertex buffers are checked now, the
    // quads with the cell buffers of the emission, in emit_launch
    CU_TRY(h, launch_step(h, k_check_caps, dim3(1), dim3(32), true, h->d_info, make_caps(h, ~0ull)));
  }
  // the points of the vertices the slab underneath owns are only needed by the projected triangle split
  const bool ghost_points = (mode == kEmitScratchQuads) && h->owner_z_min < h->zs0;
  if (!h->raster) {
    // the vertex kernels run over what the buffers can hold when the host does not know the counts (cub_emit_async)
    const size_t cap = std::min(h->points.cap / 3, h->vtx.cap);
    const size_t n_ids = exact ? (size_t)(h->ghost_v + h->n_points) : cap;
    const unsigned n_blocks = (unsigned)((n_ids + kVertexBlockIds - 1) / kVertexBlockIds);
    CUB_TRY(ensure(h, h->vsl, (size_t)nz + 1 + (cap + kVertexBlockIds - 1) / kVertexBlockIds + 1));
    {
      // K3a: vertex id -> lattice corner, walking the ownership masks K2a stored (reference creation order)
      AssignArgs a{};
      a.cnt = h->cnt.p; a.own = h->own.p; a.seg = h->seg.p; a.cofs = h->cofs.p;
      a.Wx = g.Wx; a.EY = h->EY; a.EW = h->EW; a.NS = h->NS; a.z_begin = h->owner_z_min;
      a.ghost_row_end = (unsigned)((size_t)h->zs0 * h->EY);
      a.vtx = h->vtx.p; a.info = h->d_info;
      const int rows = kAssignThreads / 32;
      const dim3 grid((g.Wx + 31) / 32, (h->EY + rows - 1) / rows, nz + 1);
      CU_TRY(h, launch_step(h, k_assign, grid, dim3(kAssignThreads), true, a));
    }
    if (n_blocks > 0) {
      // K3b: points + corner -> id map
      SliceIndexArgs si{};
      si.seg = h->seg.p; si.plane_segs = (size_t)h->EY * h->NS; si.z_first = h->owner_z_min; si.nz = nz;
      si.slice_first = h->vsl.p; si.block_slice = h->vsl.p + nz + 1; si.n_blocks = n_blocks; si.ids_per_block = kVertexBlockIds;
      const unsigned si_threads = n_blocks > (unsigned)nz + 1 ? n_blocks : (unsigned)nz + 1;
      CU_TRY(h, launch_step(h, k_slice_index, dim3((si_threads + 255) / 256), dim3(256), true, si));
      VertexArgs a{};
      a.vtx = h->vtx.p; a.caps = make_caps(h, ~0ull); a.write_ghost_points = ghost_points ? 1 : 0;
      a.info = h->d_info;
      a.slice_first = si.slice_first; a.block_slice = si.block_slice; a.z_first = h->owner_z_min;
      a.act = h->act.p; a.cofs = h->cofs.p; a.EY = h->EY; a.EW = h->EW;
      a.plane_lo = h->zs0; a.plane_hi = h->zs1; a.geom = h->geom;
      a.coff[0] = (int)(h->i0[0] - h->pad); a.coff[1] = (int)(h->i0[1] - h->pad); a.coff[2] = (int)(h->i0[2] + g.zg0 - h->pad);
      a.points = h->points.p; a.perm = h->perm.p;
      CU_TRY(h, launch_step(h, h->geom.oriented ? k_vertices<true> : k_vertices<false>, dim3(n_blocks), dim3(256), true, a));
    }
  } else {
    // raster order: vertex id = corner slot, points straight from the active masks
    RasterPointArgs a{};
    a.act = h->act.p; a.cofs = h->cofs.p; a.seg = h->seg.p; a.EY = h->EY; a.EW = h->EW; a.NS = h->NS; a.Wc = (g.X + 32) / 32;
    a.plane_lo = h->zs0; a.plane_hi = h->zs1;
    a.point_plane_lo = (ghost_points || h->own_z0 == 0) ? h->zs0 : h->zs0 + 1;
    a.coff[0] = (int)(h->i0[0] - h->pad); a.coff[1] = (int)(h->i0[1] - h->pad); a.coff[2] = (int)(h->i0[2] + g.zg0 - h->pad);
    a.geom = h->geom; a.points = h->points.p; a.info = h->d_info;
    const dim3 grid((unsigned)h->NS, (h->EY + 7) / 8, a.plane_hi - a.plane_lo + 1);
    auto kern = h->geom.oriented ? k_points_raster<true> : k_points_raster<false>;
    kern<<<grid, 256, 0, h->stream>>>(a);
    h->launches++;
    CU_TRY(h, cudaGetLastError());
  }
  return CUB_OK;
}

int emit_launch(cub_handle h, int id_bytes, bool exact) {
  CU_TRY(h, cudaSetDevice(h->device));
  const cub_params& P = h->params;
  const Grid& g = h->g;
  const bool tri = P.generate_triangles != 0, proj = P.project_vertices != 0, cd = P.save_pixel_as_cell_data != 0;
  const int mode = emit_mode(h);
  h->verts_per_cell = tri ? 3 : 4;
  h->id_bytes = id_bytes;
  const size_t quad_bytes = (size_t)(tri ? 6 : 4) * id_bytes;   // cell bytes per quad
  const size_t cd_bytes = (size_t)(tri ? 2 : 1) * h->pix_bytes;
  if (exact) {
    h->n_cells = tri ? 2 * h->n_quads : h->n_quads;
    if (id_bytes == 4 && h->point_base + h->n_points > (1ull << 32))
      return fail(h, CUB_ERR_OVERFLOW, "point ids up to %llu do not fit 32 bits", (unsigned long long)(h->point_base + h->n_points));
    const size_t nq = (size_t)h->n_quads + (size_t)h->n_quads / 16;
    CUB_TRY(ensure(h, h->cells, nq * quad_bytes));
    if (mode == kEmitScratchQuads) CUB_TRY(ensure(h, h->quads, nq));
    if (cd) CUB_TRY(ensure(h, h->celldata, nq * cd_bytes));
  } else if (!h->cells.p || (mode == kEmitScratchQuads && !h->quads.p) || (cd && !h->celldata.p)) {
    return kNeedSizes;
  }
  size_t quads_cap = h->cells.cap / quad_bytes;
  if (mode == kEmitScratchQuads) quads_cap = std::min(quads_cap, h->quads.cap);
  if (cd) quads_cap = std::min(quads_cap, h->celldata.cap / cd_bytes);
  // a second emit of the same count (another id width, new id bases) starts from unprojected points again
  if (proj && h->projected) h->vertices_done = false;
  // (the check below covers the vertex buffers of a vertex stage that runs with this emission)
  if (exact && !h->vertices_done) CUB_TRY(size_vertex_buffers(h));

  if (h->timing) cudaEventRecord(h->ev[4], h->stream);
  // one comparison of the device-side counts with the capacity of the buffers, for every kernel of the emission
  // (buffers sized from the counts always pass it)
  CU_TRY(h, launch_step(h, k_check_caps, dim3(1), dim3(32), true, h->d_info, make_caps(h, quads_cap)));
  h->caps_checked = true;
  const bool ghost_points = (mode == kEmitScratchQuads) && h->owner_z_min < h->zs0;
  if (!exact || h->n_quads > 0) {
    Timer t(h, 2);
    if (!h->vertices_done) {
      const int rc = emit_vertex_stage(h, exact);
      if (rc != CUB_OK) return rc;
    }
    {
      // K3c: faces (the only consumer of the id base: a queued count exchange has to be through)
      if (h->wait_before_faces) CU_TRY(h, cudaStreamWaitEvent(h->stream, h->wait_before_faces, 0));
      FaceArgs a{};
      a.bits = h->bits.p; a.g = g; a.EY = h->EY; a.EW = h->EW; a.NS = h->NS;
      a.z_begin = h->zs0; a.z_end = h->zs1;
      a.act = h->act.p; a.cofs = h->cofs.p; a.seg = h->seg.p; a.perm = h->raster ? nullptr : h->perm.p;
      a.info = h->d_info;
      a.cells = (mode == kEmitScratchQuads) ? (void*)h->quads.p : (void*)h->cells.p;
      a.mode = mode;
      a.vol = cd ? h->d_vol : nullptr;
      a.vX = h->gv.X; a.vY = h->gv.Y; a.vpad = h->pad; a.vzpad = h->zpad_lo;
      a.celldata = cd ? h->celldata.p : nullptr;
      a.pix_bytes = h->pix_bytes;
      const dim3 blocks((g.Wx + 31) / 32, (g.Y + kFaceThreads / 32 - 1) / (kFaceThreads / 32), h->zs1 - h->zs0);
      // (behind an event of another stream the launch is an ordinary one: the id base comes from the count exchange)
      const bool pdl = h->wait_before_faces == nullptr;
      void (*kern)(FaceArgs);
      if (mode == kEmitScratchQuads) kern = cd ? k_faces<uint32_t, kEmitScratchQuads, true> : k_faces<uint32_t, kEmitScratchQuads, false>;
      else if (mode == kEmitQuads && id_bytes == 4) kern = cd ? k_faces<uint32_t, kEmitQuads, true> : k_faces<uint32_t, kEmitQuads, false>;
      else if (mode == kEmitQuads) kern = cd ? k_faces<unsigned long long, kEmitQuads, true> : k_faces<unsigned long long, kEmitQuads, false>;
      else if (id_bytes == 4) kern = cd ? k_faces<uint32_t, kEmitTrisFixed, true> : k_faces<uint32_t, kEmitTrisFixed, false>;
      else kern = cd ? k_faces<unsigned long long, kEmitTrisFixed, true> : k_faces<unsigned long long, kEmitTrisFixed, false>;
      CU_TRY(h, launch_step(h, kern, blocks, dim3(kFaceThreads), pdl, a));
    }
    t.stop();
  }
  if (proj && (!exact || h->n_points > 0)) {
    Timer t(h, 3);
    CUB_TRY(launch_project(h, h->points.p, h->points.cap / 3, true, ghost_points));
    h->projected = true;
    t.stop();
  }
  if (mode == kEmitScratchQuads && (!exact || h->n_quads > 0)) {
    Timer t(h, 4);
    const size_t want = exact ? (size_t)h->n_quads : quads_cap;
    const unsigned blocks = (unsigned)std::max<size_t>(1, std::min<size_t>((want + 255) / 256, (size_t)h->num_sms * 16));
    if (id_bytes == 4)
      k_split_quads<uint32_t><<<blocks, 256, 0, h->stream>>>(h->quads.p, h->points.p, (uint32_t*)h->cells.p, h->d_info);
    else
      k_split_quads<unsigned long long><<<blocks, 256, 0, h->stream>>>(h->quads.p, h->points.p, (unsigned long long*)h->cells.p, h->d_info);
    h->launches++;
    CU_TRY(h, cudaGetLastError());
    t.stop();
  }
  if (h->timing) {
    cudaEventRecord(h->ev[5], h->stream);
    cudaEventSynchronize(h->ev[5]);
    cudaEventElapsedTime(&h->ms[6], h->ev[4], h->ev[5]);
  }
  h->emitted = true;
  h->emit_unverified = !exact;
  return CUB_OK;
}

// after an emission that was queued without the host knowing the counts: learn them, and redo the emission with
// buffers of the right size in the (rare) case that one was too small
int verify_emit(cub_handle h) {
  if (!h->counted) CUB_TRY(count_finish(h));
  if (h->emit_unverified) {
    h->emit_unverified = false;
    const cub_params& P = h->params;
    h->n_cells = P.generate_triangles ? 2 * h->n_quads : h->n_quads;
    if (h->flags & kFlagBufferOverflow) {
      h->vertices_done = false;
      // (the id bases live on the device; finalize/the exchange wrote them, emit_launch does not touch them)
      CUB_TRY(emit_launch(h, h->id_bytes, true));
      CU_TRY(h, cudaStreamSynchronize(h->stream));
    } else if (h->id_bytes == 4 && h->point_base + h->n_points > (1ull << 32)) {
      return fail(h, CUB_ERR_OVERFLOW, "point ids up to %llu do not fit 32 bits", (unsigned long long)(h->point_base + h->n_points));
    }
  }
  return CUB_OK;
}

}  // namespace

extern "C" {

int cub_count(cub_handle h, const cub_params* p, uint64_t* n_points, uint64_t* n_quads) {
  if (!h) return CUB_ERR_INVALID;
  CUB_TRY(count_launch(h, p));
  CUB_TRY(count_finish(h));
  if (n_points) *n_points = h->n_points;
  if (n_quads) *n_quads = h->n_quads;
  return CUB_OK;
}

int cub_count_async(cub_handle h, const cub_params* p) {
  if (!h) return CUB_ERR_INVALID;
  return count_launch(h, p);
}

int cub_projection_halo_oriented(const cub_params* p, const double spacing[3], const double direction[9],
                                 uint64_t* below, uint64_t* above) {
  if (!p || !below || !above) return CUB_ERR_INVALID;
  Geom G{};
  CUB_TRY(make_geom(nullptr, spacing, direction, G));
  slab_halo(*p, G, below, above);
  return CUB_OK;
}

int cub_projection_halo(const cub_params* p, const double spacing[3], uint64_t* below, uint64_t* above) {
  return cub_projection_halo_oriented(p, spacing, nullptr, below, above);
}

int cub_set_id_base(cub_handle h, uint64_t point_id_base, uint64_t cell_id_base) {
  if (!h) return CUB_ERR_INVALID;
  h->point_base = point_id_base;
  h->cell_base = cell_id_base;
  if (h->count_queued) {
    CU_TRY(h, cudaSetDevice(h->device));
    k_set_bases<<<1, 32, 0, h->stream>>>(h->d_info, point_id_base, cell_id_base);
    h->launches++;
    CU_TRY(h, cudaGetLastError());
  }
  return CUB_OK;
}

int cub_emit_vertices(cub_handle h) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->count_queued) return fail(h, CUB_ERR_INVALID, "cub_emit_vertices before cub_count");
  CU_TRY(h, cudaSetDevice(h->device));
  if (h->vertices_done || h->timing) return CUB_OK;  // (per-kernel timing keeps the whole emission inside cub_emit)
  const int rc = emit_vertex_stage(h, h->counted);
  return rc == kNeedSizes ? CUB_OK : rc;  // (first run of an asynchronous pipeline: cub_emit_async sizes the buffers)
}

int cub_emit(cub_handle h, int id_bytes) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->count_queued) return fail(h, CUB_ERR_INVALID, "cub_emit before cub_count");
  if (id_bytes != 4 && id_bytes != 8) return fail(h, CUB_ERR_INVALID, "id_bytes must be 4 or 8");
  if (!h->counted) CUB_TRY(count_finish(h));
  return emit_launch(h, id_bytes, true);
}

int cub_emit_async(cub_handle h, int id_bytes) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->count_queued) return fail(h, CUB_ERR_INVALID, "cub_emit_async before cub_count_async");
  if (id_bytes != 4 && id_bytes != 8) return fail(h, CUB_ERR_INVALID, "id_bytes must be 4 or 8");
  if (!h->counted && !h->timing) {
    const int rc = emit_launch(h, id_bytes, false);
    if (rc != kNeedSizes) return rc;
  }
  // first run (or per-kernel timing): the buffers have to be sized from the counts
  if (!h->counted) CUB_TRY(count_finish(h));
  return emit_launch(h, id_bytes, true);
}

int cub_finish(cub_handle h, uint64_t* n_points, uint64_t* n_cells) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->count_queued) return fail(h, CUB_ERR_INVALID, "cub_finish: nothing has been queued");
  CUB_TRY(verify_emit(h));
  if (!h->emit_unverified) CU_TRY(h, cudaStreamSynchronize(h->stream));
  if (n_points) *n_points = h->n_points;
  if (n_cells) *n_cells = h->params.generate_triangles ? 2 * h->n_quads : h->n_quads;
  return CUB_OK;
}

int cub_device_counts(cub_handle h, const uint64_t** counts) {
  if (!h || !counts) return CUB_ERR_INVALID;
  *counts = reinterpret_cast<const uint64_t*>(h->d_info + kInfoPoints);
  return CUB_OK;
}

const char* cub_last_warning(cub_handle h) { return h ? h->warning.c_str() : ""; }

int cub_run(cub_handle h, const cub_params* p, int id_bytes, uint64_t* n_points, uint64_t* n_cells) {
  uint64_t np = 0, nq = 0;
  CUB_TRY(cub_count(h, p, &np, &nq));
  CUB_TRY(cub_emit(h, id_bytes));
  if (n_points) *n_points = h->n_points;
  if (n_cells) *n_cells = h->n_cells;
  return CUB_OK;
}

int cub_fetch_async(cub_handle h, float* points, void* cells, void* cell_data, int mem_kind) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->emitted) return fail(h, CUB_ERR_INVALID, "cub_fetch before cub_emit");
  CU_TRY(h, cudaSetDevice(h->device));
  CUB_TRY(verify_emit(h));
  const cudaMemcpyKind k = mem_kind == CUB_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  if (points && h->n_points)
    CU_TRY(h, cudaMemcpyAsync(points, h->points.p + 3 * (size_t)h->ghost_v, (size_t)h->n_points * 12, k, h->stream));
  if (cells && h->n_cells)
    CU_TRY(h, cudaMemcpyAsync(cells, h->cells.p, (size_t)h->n_cells * h->verts_per_cell * h->id_bytes, k, h->stream));
  if (cell_data && h->n_cells) {
    if (!h->params.save_pixel_as_cell_data) return fail(h, CUB_ERR_INVALID, "cell data was not requested");
    CU_TRY(h, cudaMemcpyAsync(cell_data, h->celldata.p, (size_t)h->n_cells * h->pix_bytes, k, h->stream));
  }
  return CUB_OK;
}

int cub_synchronize(cub_handle h) {
  if (!h) return CUB_ERR_INVALID;
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  return CUB_OK;
}

int cub_fetch(cub_handle h, float* points, void* cells, void* cell_data, int mem_kind) {
  CUB_TRY(cub_fetch_async(h, points, cells, cell_data, mem_kind));
  return cub_synchronize(h);
}

int cub_device_buffers(cub_handle h, const float** points, const void** cells, const void** cell_data,
                       uint64_t* n_points, uint64_t* n_cells, int* verts_per_cell, int* id_bytes) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->emitted) return fail(h, CUB_ERR_INVALID, "no mesh has been emitted");
  CUB_TRY(verify_emit(h));
  if (points) *points = h->points.p + 3 * (size_t)h->ghost_v;
  if (cells) *cells = h->cells.p;
  if (cell_data) *cell_data = h->params.save_pixel_as_cell_data ? h->celldata.p : nullptr;
  if (n_points) *n_points = h->n_points;
  if (n_cells) *n_cells = h->n_cells;
  if (verts_per_cell) *verts_per_cell = h->verts_per_cell;
  if (id_bytes) *id_bytes = h->id_bytes;
  return CUB_OK;
}

int cub_debug_bitmask(cub_handle h, uint32_t* out, uint64_t* words_per_row) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->count_queued) return fail(h, CUB_ERR_INVALID, "cub_debug_bitmask before cub_count");
  if (h->pad) return fail(h, CUB_ERR_UNSUPPORTED, "cub_debug_bitmask: the bitmask of image_border_faces runs is that of the padded image");
  if (words_per_row) *words_per_row = (uint64_t)h->g.Wp;
  if (out) {
    CU_TRY(h, cudaSetDevice(h->device));
    const size_t words = (size_t)h->g.Zl * h->g.Y * h->g.Wp;
    CU_TRY(h, cudaMemcpyAsync(out, h->bits.p, words * 4, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
  }
  return CUB_OK;
}

int cub_debug_project_points(cub_handle h, const cub_params* p, float* points_xyz, uint64_t n_points) {
  if (!h) return CUB_ERR_INVALID;
  if (!p || !points_xyz) return fail(h, CUB_ERR_INVALID, "null argument");
  if (h->range_on)
    return fail(h, CUB_ERR_INVALID, "vertex projection needs an iso-surface and an inside range has none: leave range mode "
                                    "(cub_set_inside_range with enable = 0)");
  CU_TRY(h, cudaSetDevice(h->device));
  h->params = *p;
  CUB_TRY(setup_grid(h));
  compute_step(h);
  h->counted = h->emitted = h->count_queued = false;
  CUB_TRY(ensure(h, h->points, 3 * (size_t)n_points));
  CU_TRY(h, cudaMemcpyAsync(h->points.p, points_xyz, (size_t)n_points * 12, cudaMemcpyHostToDevice, h->stream));
  CUB_TRY(launch_project(h, h->points.p, (size_t)n_points, false, true));
  CU_TRY(h, cudaMemcpyAsync(points_xyz, h->points.p, (size_t)n_points * 12, cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  return CUB_OK;
}

int cub_generate_volume(cub_handle h, int kind, const uint64_t dims[3], const uint64_t image_dims[3], uint64_t z_offset,
                        double param0, double param1, uint64_t seed) {
  if (!h) return CUB_ERR_INVALID;
  if (!dims || !image_dims) return fail(h, CUB_ERR_INVALID, "null dims");
  if (kind < 0 || kind > 2) return fail(h, CUB_ERR_INVALID, "unknown generator %d", kind);
  CU_TRY(h, cudaSetDevice(h->device));
  h->has_volume = false;
  CUB_TRY(set_geometry(h, CUB_F32, dims, nullptr, nullptr, nullptr));
  if (z_offset + dims[2] > image_dims[2] || dims[0] != image_dims[0] || dims[1] != image_dims[1])
    return fail(h, CUB_ERR_INVALID, "slab does not fit the image");
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  CUB_TRY(ensure(h, h->vol_owned, n * 4));
  GenArgs a;
  a.out = reinterpret_cast<float*>(h->vol_owned.p);
  a.X = (int)dims[0]; a.Y = (int)dims[1]; a.Zl = (int)dims[2];
  a.IX = (int)image_dims[0]; a.IY = (int)image_dims[1]; a.IZ = (int)image_dims[2];
  a.zg0 = (int)z_offset;
  a.kind = kind;
  a.p0 = (float)param0; a.p1 = (float)param1;
  a.seed = seed;
  size_t blocks = (n + 255) / 256;
  if (blocks > (size_t)h->num_sms * 32) blocks = (size_t)h->num_sms * 32;
  k_generate<<<(unsigned)blocks, 256, 0, h->stream>>>(a);
  h->launches++;
  CU_TRY(h, cudaGetLastError());
  h->d_vol = h->vol_owned.p;
  h->has_volume = true;
  h->image_nz = image_dims[2];
  h->local_z0 = z_offset;
  // own range defaults to the whole local buffer; callers with halos follow up with cub_set_slab
  h->own_z0 = z_offset;
  h->own_z1 = z_offset + dims[2];
  return CUB_OK;
}

int cub_download_volume(cub_handle h, void* out, uint64_t bytes) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->has_volume || !out) return fail(h, CUB_ERR_INVALID, "no volume / null buffer");
  const uint64_t have = h->dims[0] * h->dims[1] * h->dims[2] * (uint64_t)h->pix_bytes;
  if (bytes != have) return fail(h, CUB_ERR_INVALID, "size mismatch: volume has %llu bytes", (unsigned long long)have);
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaMemcpyAsync(out, h->d_vol, bytes, cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  return CUB_OK;
}

// Device memory for callers that do not link the CUDA runtime themselves (the destination buffers of
// cub_comm_gather_mesh, CUB_MEM_DEVICE volumes): plain cudaMalloc / cudaFree / cudaMemcpyAsync on the handle's device.
int cub_device_alloc(cub_handle h, uint64_t bytes, void** out) {
  if (!h || !out) return CUB_ERR_INVALID;
  *out = nullptr;
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaMalloc(out, bytes ? (size_t)bytes : 1));
  return CUB_OK;
}

int cub_device_free(cub_handle h, void* p) {
  if (!h) return CUB_ERR_INVALID;
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  CU_TRY(h, cudaFree(p));
  return CUB_OK;
}

int cub_device_copy(cub_handle h, void* dst, const void* src, uint64_t bytes, int dst_kind, int src_kind) {
  if (!h || (!dst && bytes) || (!src && bytes)) return CUB_ERR_INVALID;
  CU_TRY(h, cudaSetDevice(h->device));
  const cudaMemcpyKind k = dst_kind == CUB_MEM_DEVICE ? (src_kind == CUB_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice)
                                                      : (src_kind == CUB_MEM_DEVICE ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost);
  CU_TRY(h, cudaMemcpyAsync(dst, src, (size_t)bytes, k, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  return CUB_OK;
}

// Page-lock / unlock a caller buffer (cudaHostRegister): host <-> device copies of pageable memory run at a
// fraction of the PCIe rate.
int cub_host_register(cub_handle h, void* p, uint64_t bytes) {
  if (!h || !p) return CUB_ERR_INVALID;
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaHostRegister(p, (size_t)bytes, cudaHostRegisterDefault));
  return CUB_OK;
}

// Page-locked host memory (cudaHostAlloc / cudaFreeHost): staging buffers for cub_fetch at the full PCIe rate.
int cub_host_alloc(cub_handle h, uint64_t bytes, void** out) {
  if (!h || !out) return CUB_ERR_INVALID;
  *out = nullptr;
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaHostAlloc(out, bytes ? (size_t)bytes : 1, cudaHostAllocDefault));
  return CUB_OK;
}

int cub_host_free(cub_handle h, void* p) {
  if (!h) return CUB_ERR_INVALID;
  if (!p) return CUB_OK;
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  CU_TRY(h, cudaFreeHost(p));
  return CUB_OK;
}

int cub_host_unregister(cub_handle h, void* p) {
  if (!h || !p) return CUB_ERR_INVALID;
  CU_TRY(h, cudaSetDevice(h->device));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  CU_TRY(h, cudaHostUnregister(p));
  return CUB_OK;
}

int cub_enable_timing(cub_handle h, int on) {
  if (!h) return CUB_ERR_INVALID;
  h->timing = on != 0;
  return CUB_OK;
}

int cub_get_timings(cub_handle h, float ms[8]) {
  if (!h || !ms) return CUB_ERR_INVALID;
  for (int i = 0; i < 8; ++i) ms[i] = h->ms[i];
  return CUB_OK;
}

uint64_t cub_launch_count(cub_handle h) { return h ? h->launches : 0; }
int cub_count_was_fused(cub_handle h) { return (h && h->fused_last) ? 1 : 0; }

}  // extern "C"

// ---- label maps: per-label bounds, a region of interest, and every label meshed in its box ----------------------
namespace {

// the value range of an integer pixel type, as far as a long long holds it (uint64: [0, 2^63 - 1], the labels an
// int64 first_label reaches); false for the float types
template <typename T>
bool type_range(long long* lo, long long* hi) {
  if constexpr (std::is_integral<T>::value) {
    const unsigned long long max = (unsigned long long)std::numeric_limits<T>::max();
    *lo = (long long)std::numeric_limits<T>::min();
    *hi = max > (unsigned long long)std::numeric_limits<long long>::max() ? std::numeric_limits<long long>::max() : (long long)max;
    return true;
  }
  return false;
}

bool integer_range(int dtype, long long* lo, long long* hi) {
  bool integral = false;
  DISPATCH_PIXEL(dtype, integral = type_range<T>(lo, hi));
  return integral;
}

// a z-slab: cub_set_slab, or a generated slab of a taller image
bool has_slab(cub_handle h) { return h->slab_set || h->local_z0 != 0 || h->image_nz != h->dims[2]; }

// k_label_bounds over the current volume into out[n * 8] (host), then the host form of the table
int label_bounds(cub_handle h, long long first, uint32_t n, uint64_t* out) {
  CU_TRY(h, cudaSetDevice(h->device));
  CUB_TRY(ensure(h, h->label_table, (size_t)n * 8));
  CU_TRY(h, cudaMemsetAsync(h->label_table.p, 0, (size_t)n * 8 * sizeof(unsigned long long), h->stream));
  const unsigned long long X = h->dims[0], rows = h->dims[1] * h->dims[2];
  // a warp sums its lanes' counts in 32 bits: more warps until one sees fewer than 2^32 voxels
  unsigned long long blocks = std::min<unsigned long long>((rows + 7) / 8, (unsigned long long)h->num_sms * kLabelCtasPerSm);
  const unsigned long long warp_rows = (1ull << 32) / X - 1;
  blocks = std::max(blocks, (rows + warp_rows * 8 - 1) / (warp_rows * 8));
  if (blocks >= (1ull << 31)) return fail(h, CUB_ERR_UNSUPPORTED, "volume too large for cub_label_bounds");
  switch (h->dtype) {
#define CUB_LABEL_BOUNDS(CODE, T)                                                                                      \
    case CODE:                                                                                                         \
      k_label_bounds<T><<<(unsigned)blocks, kLabelThreads, 0, h->stream>>>(static_cast<const T*>(h->d_vol), (unsigned)X, \
                                                                         (unsigned)h->dims[1], rows,                  \
                                                                         (LabelKey<T>)(unsigned long long)first, n,   \
                                                                         h->label_table.p);                           \
      break;
    CUB_LABEL_BOUNDS(CUB_U8, unsigned char)
    CUB_LABEL_BOUNDS(CUB_I8, signed char)
    CUB_LABEL_BOUNDS(CUB_U16, unsigned short)
    CUB_LABEL_BOUNDS(CUB_I16, short)
    CUB_LABEL_BOUNDS(CUB_U32, unsigned int)
    CUB_LABEL_BOUNDS(CUB_I32, int)
    CUB_LABEL_BOUNDS(CUB_I64, long long)
    CUB_LABEL_BOUNDS(CUB_U64, unsigned long long)
#undef CUB_LABEL_BOUNDS
    default: return fail(h, CUB_ERR_UNSUPPORTED, "label bounds need an integer pixel type");
  }
  h->launches++;
  CU_TRY(h, cudaGetLastError());
  CU_TRY(h, cudaMemcpyAsync(out, h->label_table.p, (size_t)n * 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(h, cudaStreamSynchronize(h->stream));
  for (size_t i = 0; i < n; ++i) {
    uint64_t* e = out + 8 * i;
    if (e[0] == 0) {
      for (int k = 1; k < 8; ++k) e[k] = 0;
    } else {
      for (int k = 1; k < 4; ++k) e[k] = (uint64_t)(~(uint32_t)e[k]);
    }
  }
  return CUB_OK;
}

// back to the whole volume (the region index stays the caller's)
void clear_roi(cub_handle h) {
  if (!h->roi_on) return;
  h->d_vol = h->full_vol;
  for (int k = 0; k < 3; ++k) {
    h->dims[k] = h->full_dims[k];
    h->i0[k] -= (long long)h->roi_lo[k];
    h->roi_lo[k] = 0;
  }
  h->image_nz = h->own_z1 = h->dims[2];
  h->roi_on = false;
}

// the box [lo, lo + size) of the whole volume becomes the volume: in place when it is whole rows and slices, else a
// copy (k_gather_box); the region index moves by lo
int apply_roi(cub_handle h, const uint64_t lo[3], const uint64_t size[3]) {
  clear_roi(h);
  const uint64_t* d = h->dims;
  const size_t pb = (size_t)h->pix_bytes;
  if (lo[0] == 0 && lo[1] == 0 && size[0] == d[0] && size[1] == d[1]) {
    h->full_vol = h->d_vol;
    h->d_vol = static_cast<const unsigned char*>(h->d_vol) + (size_t)lo[2] * d[0] * d[1] * pb;
  } else {
    CUB_TRY(ensure(h, h->roi_buf, (size_t)size[0] * size[1] * size[2] * pb));
    const unsigned long long rows = size[1] * size[2];
    const unsigned blocks = (unsigned)std::min<unsigned long long>(rows, (unsigned long long)h->num_sms * 32);
    const unsigned threads = size[0] >= 256 ? 256 : (size[0] >= 64 ? 64 : 32);
    switch (pb) {
#define CUB_GATHER(W)                                                                                                       \
      k_gather_box<W><<<blocks, threads, 0, h->stream>>>(static_cast<const W*>(h->d_vol), reinterpret_cast<W*>(h->roi_buf.p), \
                                                         d[0], d[1], lo[0], lo[1], lo[2], size[0], size[1], rows)
      case 1: CUB_GATHER(uint8_t); break;
      case 2: CUB_GATHER(uint16_t); break;
      case 4: CUB_GATHER(uint32_t); break;
      default: CUB_GATHER(unsigned long long); break;
#undef CUB_GATHER
    }
    h->launches++;
    CU_TRY(h, cudaGetLastError());
    h->full_vol = h->d_vol;
    h->d_vol = h->roi_buf.p;
  }
  for (int k = 0; k < 3; ++k) {
    h->full_dims[k] = d[k];
    h->roi_lo[k] = lo[k];
    h->i0[k] += (long long)lo[k];
  }
  for (int k = 0; k < 3; ++k) h->dims[k] = size[k];
  h->image_nz = h->own_z1 = size[2];
  h->local_z0 = h->own_z0 = 0;
  h->roi_on = true;
  return CUB_OK;
}

// device-to-device append at `used` elements, growing the buffer (and keeping its contents) when needed
template <typename P>
int append(cub_handle h, DevBuf<P>& b, size_t used, const P* src, size_t n) {
  if (n == 0) return CUB_OK;
  if (!b.p || used + n > b.cap) {
    const size_t cap = std::max(used + n, b.cap + b.cap / 2);
    void* p = nullptr;
    CU_TRY(h, cudaMalloc(&p, cap * sizeof(P)));
    if (used) CU_TRY(h, cudaMemcpyAsync(p, b.p, used * sizeof(P), cudaMemcpyDeviceToDevice, h->stream));
    if (b.p) {
      CU_TRY(h, cudaStreamSynchronize(h->stream));
      CU_TRY(h, cudaFree(b.p));
    }
    b.p = static_cast<P*>(p);
    b.cap = cap;
  }
  CU_TRY(h, cudaMemcpyAsync(b.p + used, src, n * sizeof(P), cudaMemcpyDeviceToDevice, h->stream));
  return CUB_OK;
}

std::string label_text(double v) {
  char buf[32];
  snprintf(buf, sizeof buf, "%.17g", v);
  return buf;
}

// cub_run_labels after its checks: one bounds pass per window of 65536 label values, then count -> emit of every
// label on its grown box with the running totals as id bases, appended to the concatenation buffers
int run_labels(cub_handle h, const cub_params* p, const double* labels, uint64_t n, int id_bytes, uint64_t* point_offsets,
               uint64_t* cell_offsets) {
  std::vector<long long> sorted(n);
  for (uint64_t i = 0; i < n; ++i) sorted[i] = (long long)labels[i];
  std::sort(sorted.begin(), sorted.end());
  std::vector<uint64_t> bounds(8 * (size_t)n), window;
  for (size_t i = 0; i < sorted.size();) {
    size_t j = i;
    // (label distances in unsigned arithmetic: two int64 labels can be more than 2^63 apart)
    auto dist = [&](size_t k) { return (unsigned long long)sorted[k] - (unsigned long long)sorted[i]; };
    while (j < sorted.size() && dist(j) < 65536) ++j;
    const uint32_t span = (uint32_t)(dist(j - 1) + 1);
    window.resize(8 * (size_t)span);
    CUB_TRY(label_bounds(h, sorted[i], span, window.data()));
    for (size_t k = i; k < j; ++k) std::copy_n(&window[8 * (size_t)dist(k)], 8, &bounds[8 * k]);
    i = j;
  }
  const bool tri = p->generate_triangles != 0, cd = p->save_pixel_as_cell_data != 0;
  const size_t cell_bytes = (size_t)(tri ? 3 : 4) * id_bytes;
  const uint64_t whole[3] = {h->dims[0], h->dims[1], h->dims[2]};
  uint64_t n_points = 0, n_cells = 0;
  std::string warned;
  for (uint64_t i = 0; i < n; ++i) {
    point_offsets[i] = n_points;
    cell_offsets[i] = n_cells;
    const long long k = (long long)labels[i];
    const uint64_t* b = &bounds[8 * (size_t)(std::lower_bound(sorted.begin(), sorted.end(), k) - sorted.begin())];
    if (b[0] == 0) continue;
    // the label's bounding box grown by one voxel and clipped to the image: the same mesh as on the whole volume
    uint64_t lo[3], size[3];
    for (int a = 0; a < 3; ++a) {
      lo[a] = b[1 + a] > 0 ? b[1 + a] - 1 : 0;
      size[a] = std::min(b[4 + a] + 1, whole[a] - 1) + 1 - lo[a];
    }
    CUB_TRY(apply_roi(h, lo, size));
    h->range_on = true;
    h->range_lo = h->range_hi = labels[i];
    CUB_TRY(count_launch(h, p));
    CUB_TRY(count_finish(h));
    if (h->flags & kFlagEmptyInteriorSlice) warned += (warned.empty() ? "" : ", ") + label_text(labels[i]);
    CUB_TRY(cub_set_id_base(h, n_points, n_cells));
    CUB_TRY(emit_launch(h, id_bytes, true));
    CUB_TRY(append(h, h->cat_points, 3 * (size_t)n_points, h->points.p + 3 * (size_t)h->ghost_v, 3 * (size_t)h->n_points));
    CUB_TRY(append(h, h->cat_cells, (size_t)n_cells * cell_bytes, h->cells.p, (size_t)h->n_cells * cell_bytes));
    if (cd) CUB_TRY(append(h, h->cat_celldata, (size_t)n_cells * h->pix_bytes, h->celldata.p, (size_t)h->n_cells * h->pix_bytes));
    n_points += h->n_points;
    n_cells += h->n_cells;
  }
  point_offsets[n] = n_points;
  cell_offsets[n] = n_cells;
  // the concatenation becomes the handle's result (cub_fetch, cub_device_buffers); the per-label buffers are the
  // concatenation buffers of the next call
  std::swap(h->points, h->cat_points);
  std::swap(h->cells, h->cat_cells);
  if (cd) std::swap(h->celldata, h->cat_celldata);
  h->params = *p;
  h->n_points = n_points;
  h->n_cells = n_cells;
  h->n_quads = tri ? n_cells / 2 : n_cells;
  h->ghost_v = 0;
  h->verts_per_cell = tri ? 3 : 4;
  h->id_bytes = id_bytes;
  h->count_queued = false;
  h->counted = h->emitted = true;
  h->emit_unverified = false;
  h->warning = warned.empty() ? std::string() : std::string(kEmptySliceRemark) + " (label " + warned + ")";
  return CUB_OK;
}

}  // namespace

extern "C" {

int cub_label_bounds(cub_handle h, int64_t first_label, uint32_t n_labels, uint64_t* out) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->has_volume) return fail(h, CUB_ERR_INVALID, "cub_label_bounds before cub_set_volume");
  long long lo = 0, hi = 0;
  if (!integer_range(h->dtype, &lo, &hi)) return fail(h, CUB_ERR_UNSUPPORTED, "label bounds need an integer pixel type");
  if (!out) return fail(h, CUB_ERR_INVALID, "out is null");
  if (h->roi_on || has_slab(h)) return fail(h, CUB_ERR_INVALID, "cub_label_bounds runs on a whole volume: no region of interest or z-slab");
  if (n_labels < 1 || n_labels > 65536) return fail(h, CUB_ERR_INVALID, "n_labels = %u is not in [1, 65536]", n_labels);
  // (the distance to hi in unsigned arithmetic: first_label + n_labels - 1 may not fit a long long)
  if (first_label < lo || first_label > hi || (unsigned long long)hi - (unsigned long long)first_label < n_labels - 1ull)
    return fail(h, CUB_ERR_INVALID, "label window of %u labels from %lld is not inside the pixel type's range [%lld, %lld]",
                n_labels, (long long)first_label, lo, hi);
  return label_bounds(h, first_label, n_labels, out);
}

int cub_set_region_of_interest(cub_handle h, const uint64_t lo[3], const uint64_t size[3]) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->has_volume) return fail(h, CUB_ERR_INVALID, "cub_set_region_of_interest before cub_set_volume");
  CU_TRY(h, cudaSetDevice(h->device));
  h->counted = h->emitted = h->count_queued = false;
  if (!lo) {
    clear_roi(h);
    return CUB_OK;
  }
  if (!h->roi_on && has_slab(h)) return fail(h, CUB_ERR_UNSUPPORTED, "a region of interest cannot be combined with a z-slab");
  if (!size) return fail(h, CUB_ERR_INVALID, "size is null");
  const uint64_t* d = h->roi_on ? h->full_dims : h->dims;
  for (int a = 0; a < 3; ++a)
    if (size[a] == 0 || lo[a] >= d[a] || size[a] > d[a] - lo[a])
      return fail(h, CUB_ERR_INVALID, "region of interest [%llu, %llu + %llu) on axis %d is empty or leaves the volume (%llu)",
                  (unsigned long long)lo[a], (unsigned long long)lo[a], (unsigned long long)size[a], a, (unsigned long long)d[a]);
  return apply_roi(h, lo, size);
}

int cub_run_labels(cub_handle h, const cub_params* p, const double* labels, uint64_t n_labels, int id_bytes,
                   uint64_t* point_offsets, uint64_t* cell_offsets) {
  if (!h) return CUB_ERR_INVALID;
  if (!h->has_volume) return fail(h, CUB_ERR_INVALID, "cub_run_labels before cub_set_volume");
  long long lo = 0, hi = 0;
  if (!integer_range(h->dtype, &lo, &hi)) return fail(h, CUB_ERR_UNSUPPORTED, "label meshes need an integer pixel type");
  if (!p || (n_labels && !labels) || !point_offsets || !cell_offsets) return fail(h, CUB_ERR_INVALID, "null argument");
  if (p->project_vertices)
    return fail(h, CUB_ERR_INVALID, "vertex projection needs an iso-surface and a label has none: turn project_vertices off");
  if (h->roi_on) return fail(h, CUB_ERR_INVALID, "cub_run_labels runs on the whole volume: clear the region of interest");
  if (has_slab(h)) return fail(h, CUB_ERR_INVALID, "cub_run_labels does not run on a z-slab");
  if (id_bytes != 4 && id_bytes != 8) return fail(h, CUB_ERR_INVALID, "id_bytes must be 4 or 8");
  for (uint64_t i = 0; i < n_labels; ++i) {
    if (std::isnan(labels[i]) || iso_as_pixel(h->dtype, labels[i]) != labels[i])
      return fail(h, CUB_ERR_INVALID, "label %.17g is not representable in the pixel type", labels[i]);
    // (the windows of cub_label_bounds, and the keys run_labels sorts, are long longs: uint64 labels end at 2^63 - 1,
    // and (double)hi rounds up to 2^63, so the bound is 2^63 itself)
    if (hi == std::numeric_limits<long long>::max() && !(labels[i] < 0x1p63))
      return fail(h, CUB_ERR_INVALID, "label %.17g is above %lld, the largest label a window reaches", labels[i], hi);
  }
  {
    std::vector<double> s(labels, labels + n_labels);
    std::sort(s.begin(), s.end());
    for (size_t i = 1; i < s.size(); ++i)
      if (s[i] == s[i - 1]) return fail(h, CUB_ERR_INVALID, "label %.17g is given twice", s[i]);
  }
  CU_TRY(h, cudaSetDevice(h->device));
  const bool range_on = h->range_on;
  const double range_lo = h->range_lo, range_hi = h->range_hi;
  const int rc = run_labels(h, p, labels, n_labels, id_bytes, point_offsets, cell_offsets);
  clear_roi(h);
  h->range_on = range_on;
  h->range_lo = range_lo;
  h->range_hi = range_hi;
  if (rc != CUB_OK) h->counted = h->emitted = h->count_queued = false;
  return rc;
}

}  // extern "C"

#include "cuberille_comm.inl"
