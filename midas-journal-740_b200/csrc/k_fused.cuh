// k_fused.cuh — K1 + K2a in ONE persistent, warp-specialised kernel: the HBM-bound classification pass and the
// issue-bound ownership sweep run side by side on every SM.
//
// Reference: the suitability / neighbour predicate (txx:139-141, 167; k_classify.cuh) and the vertex lookup of the hot
// loop (txx:179-194; k_sweep.cuh).  Nothing changes in what is computed: the bitmask, the packed counts, the active
// masks and the ownership records are the ones the two separate kernels write (tests/test_gpu_fused.py compares them).
//
// Why: run one after the other, K1 keeps the memory system at the copy peak with a quarter of the issue slots, then K2a
// fills two thirds of the issue slots while HBM idles (0.66 + 0.39 ms for 1024^3 float32).  Here every CTA holds both
// roles (0.83 ms, bound by the DRAM traffic of the two together):
//   * warpgroup 0 = four PRODUCER warps.  Each owns a private ring of kFuseStages 4 KB shared-memory stages that one
//     elected lane fills with TMA bulk copies (cp.async.bulk global -> shared, completion on an mbarrier), so the
//     bytes in flight per SM are set by shared memory, not by registers or by the number of resident warps; the warp
//     reads a landed stage one voxel per lane, the ballot of the inside predicate is the output word (as in k_classify), and
//     lane 0 stores the words with an L2 evict-last hint (the consumers read them a few slices later).
//     Tasks (<= 4 KB of one row) are handed out in raster order, `batch` at a time through one atomic ticket (the next
//     ticket is requested while the current batch is issued); a finished batch is published with one release-add per
//     slice it touches into done[z].
//   * warpgroup 1 = four CONSUMER warps = one sweep tile at a time (sweep_tile of k_sweep.cuh on named barrier 1),
//     tiles taken in z-major order through a second ticket; before a tile starts, one of its warps waits (acquire
//     loads, growing back-off) until every slice the tile reads is complete (done[z] == tasks per slice).
//   * setmaxnreg moves registers from the producers (32) to the consumers (96): four CTAs = four sweep tiles per SM.
// Producers never wait for anything but their own copies and every CTA has producers, so the kernel cannot deadlock,
// whatever part of the grid is resident.
// What bounds it (r2, ncu): 4.50 GB read + 0.85 GB written in 0.87 ms = 94 % of the measured copy peak before the
// evict-last hint and the smaller batches; how far the consumers run behind the producers (what all producer warps
// have in flight: 2368 warps x batch x 4 KB) decides whether the bitmask words are still in L2 when they are read.
#pragma once
#include "k_classify.cuh"
#include "k_sweep.cuh"

namespace cbr {

constexpr int kFuseStageBytes = 4096;   // one task: 32 words of 4-byte pixels, 16 words of 8-byte pixels
constexpr int kFuseProducerWarps = 4;
constexpr int kFuseThreads = 256;
constexpr int kFuseProducerRegs = 32, kFuseConsumerRegs = 96;   // 128 * (32 + 96) = 256 * 64

struct FuseArgs {
  SweepArgs sw;
  const void* vol;
  uint32_t* bits;
  unsigned n_tasks, groups_per_row, tasks_per_slice, n_batches;
  unsigned batch;             // tasks per ticket and per publication (8: one release + atomic per 32 KB)
  unsigned n_tiles, gx, gy;   // sweep tiles; ticket -> (bx, by, bz), bz slowest
  unsigned* ctr;              // [0] producer ticket, [1] consumer ticket (zeroed before the launch)
  unsigned* done;             // [Zl] classification tasks completed per slice (zeroed before the launch)
};

template <int S>
struct FuseProducerSmem {
  alignas(128) unsigned char stage[kFuseProducerWarps][S][kFuseStageBytes];
  alignas(16) uint4 meta[kFuseProducerWarps][S];
  alignas(8) unsigned long long full[kFuseProducerWarps][S];
};

template <typename C, int S>
struct FuseSmem {
  FuseProducerSmem<S> p;
  SweepSmem<C> sw;
  uint32_t tile;
};

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* b, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* b, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(b)), "r"(bytes) : "memory");
}
// (an L2 evict-first hint on these copies - the volume is read once - was measured: 0.88 -> 1.05 ms; plain copies it is)
__device__ __forceinline__ void bulk_load(void* dst, const void* src, unsigned bytes, unsigned long long* b) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
               "l"(src), "r"(bytes), "r"(smem_addr(b))
               : "memory");
}
// the bitmask words are read again a few slices later by the consumers: ask L2 to keep them
__device__ __forceinline__ unsigned long long l2_evict_last_policy() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void st_keep(uint32_t* p, const uint4 v, unsigned long long policy) {
  asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w),
               "l"(policy)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* b, unsigned parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_addr(b)), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---- producer warp: classification tasks through the warp's private TMA ring ---------------------------------------
template <typename T, int S, typename In>
__device__ __forceinline__ void fused_producer(const FuseArgs& a, const typename In::Param bounds, FuseProducerSmem<S>& sm,
                                               const int warp, const int lane) {
  const In inside{bounds};
  constexpr int WPT = kFuseStageBytes / (32 * (int)sizeof(T));  // words per task
  static_assert(WPT >= 4 && WPT % 4 == 0, "16-byte stores of the words of a task");
  const T* __restrict__ vol = static_cast<const T*>(a.vol);
  const Grid& g = a.sw.g;
  unsigned long long* full = sm.full[warp];
  uint4* meta = sm.meta[warp];   // per stage: {row, first word, task, voxels}
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncwarp();

  // the batch being issued: tasks [icur, iend), icur = group igrp of row irow (kept incrementally: no division per task)
  unsigned icur = 0, iend = 0, irow = 0, igrp = 0;
  const unsigned long long keep = l2_evict_last_policy();
  // the ticket of the NEXT batch is requested while the current one is being issued (lane 0 holds it; an atomic's
  // round trip is worth several tasks)
  unsigned next_b = 0;
  if (lane == 0) next_b = atomicAdd(a.ctr, 1u);
  bool more = true;
  unsigned sig_first = 0, sig_n = 0;  // consumed, not yet published: tasks [sig_first, sig_first + sig_n)

  // queue the next task into stage s (warp-uniform result: false once the tickets are used up)
  auto issue = [&](const int s) -> bool {
    if (icur == iend) {
      if (!more) return false;
      const unsigned b = __shfl_sync(0xffffffffu, next_b, 0);
      if (b >= a.n_batches) {
        more = false;
        return false;
      }
      if (lane == 0) next_b = atomicAdd(a.ctr, 1u);
      icur = b * a.batch;
      iend = min(icur + a.batch, a.n_tasks);
      irow = icur / a.groups_per_row;
      igrp = icur - irow * a.groups_per_row;
    }
    if (lane == 0) {
      const int w0 = (int)igrp * WPT;
      const int nvox = min(WPT * 32, g.X - w0 * 32);
      meta[s] = make_uint4(irow, (unsigned)w0, icur, (unsigned)nvox);
      const unsigned bytes = (unsigned)nvox * (unsigned)sizeof(T);  // a multiple of 16 (checked by the host)
      mbar_expect_tx(&full[s], bytes);
      bulk_load(sm.stage[warp][s], vol + (size_t)irow * g.X + (size_t)w0 * 32, bytes, &full[s]);
    }
    ++icur;
    if (++igrp == a.groups_per_row) {
      igrp = 0;
      ++irow;
    }
    return true;
  };
  // publish the finished tasks: the bitmask words were stored by lane 0, so its release-add orders them
  auto publish = [&]() {
    if (lane == 0 && sig_n) {
      unsigned t0 = sig_first, left = sig_n;
      while (left) {
        const unsigned z = t0 / a.tasks_per_slice;
        const unsigned n = min(left, (z + 1) * a.tasks_per_slice - t0);
        red_release_add(a.done + z, n);
        t0 += n;
        left -= n;
      }
    }
    sig_n = 0;
  };

  int inflight = 0;
#pragma unroll
  for (int s = 0; s < S; ++s)
    if (issue(s)) ++inflight;
  uint32_t phases = 0;
  int head = 0;
  while (inflight > 0) {
    mbar_wait(&full[head], (phases >> head) & 1u);
    phases ^= 1u << head;
    const uint4 m = meta[head];
    const unsigned task = m.z;
    const int nvox = (int)m.w;
    const T* __restrict__ sp = reinterpret_cast<const T*>(sm.stage[warp][head]) + lane;
    uint32_t* __restrict__ dst = a.bits + (size_t)m.x * g.Wp + m.y;
    if (nvox == WPT * 32) {
#pragma unroll
      for (int k4 = 0; k4 < WPT; k4 += 4) {
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = __ballot_sync(0xffffffffu, inside(sp[(k4 + k) * 32]));
        if (lane == 0) st_keep(dst + k4, make_uint4(w[0], w[1], w[2], w[3]), keep);
      }
    } else {
      // ragged end of a row: lanes past it re-read the row's last voxel ("replicate bit X-1", k_classify.cuh)
      const int nw = (nvox + 31) >> 5, last = nvox - 1 - lane;
      for (int k = 0; k < nw; ++k) {
        const uint32_t w = __ballot_sync(0xffffffffu, inside(sp[min(k * 32, last)]));
        if (lane == 0) dst[k] = w;
      }
    }
    __syncwarp();  // every lane has read the stage before it is filled again
    if (sig_n && task != sig_first + sig_n) publish();
    if (!sig_n) sig_first = task;
    if (++sig_n == a.batch) publish();
    if (!issue(head)) --inflight;
    head = (head + 1 == S) ? 0 : head + 1;
  }
  publish();
}

// ---- consumer warpgroup: sweep tiles in z-major order, each after the slices it reads are complete -----------------
template <typename C>
__device__ __forceinline__ void fused_consumer(const FuseArgs& a, SweepSmem<C>& sm, uint32_t* tile_slot, const int t) {
  const int lane = t & 31;
  const Grid& g = a.sw.g;
  const int zlo = max(0, -g.zg0), zhi = min(g.Zl - 1, g.Zg - 1 - g.zg0);  // the clamp of the sweep's slice loads
  for (;;) {
    // (every thread read the slot of the previous tile before that tile's second barrier below: no barrier needed here)
    if (t == 0) *tile_slot = atomicAdd(a.ctr + 1, 1u);
    asm volatile("bar.sync 1, %0;" ::"n"(C::NTP) : "memory");
    const unsigned tile = *tile_slot;
    if (tile >= a.n_tiles) break;  // (uniform: every thread of the warpgroup reads the same slot)
    const unsigned bz = tile / (a.gx * a.gy), rem = tile - bz * (a.gx * a.gy);
    const unsigned by = rem / a.gx, bx = rem - by * a.gx;
    const int zs = a.sw.z_begin + (int)bz * a.sw.tz, ze = min(zs + a.sw.tz, a.sw.z_end);
    const int need_lo = min(max(zs - 1, zlo), zhi), need_hi = min(max(ze, zlo), zhi);
    // One warp polls, with a growing back-off (every consumer of the GPU watches the same few counters: a tight
    // loop in all of them would queue up in front of the one L2 slice that also serves the producers' publications):
    // first the top slice alone - batches finish roughly in raster order - then all of them.
    if (t < 32) {
      unsigned ns = 256;
      while (ld_acquire(a.done + need_hi) < a.tasks_per_slice) {
        __nanosleep(ns);
        if (ns < 4096) ns <<= 1;
      }
      for (int z = need_lo + lane; z < need_hi; z += 32)
        while (ld_acquire(a.done + z) < a.tasks_per_slice) __nanosleep(1024);
    }
    asm volatile("bar.sync 1, %0;" ::"n"(C::NTP) : "memory");  // (orders the other warps' loads after the acquires)
    sweep_tile<C, true>(a.sw, sm, t, (int)bx, (int)by, (int)bz);
  }
}

template <typename T, typename C, int S, typename In>
__global__ void __launch_bounds__(kFuseThreads, 4) k_classify_sweep(const FuseArgs a, const typename In::Param bounds) {
  pdl_enter();
  static_assert(C::NTP == 128, "the consumer role is one warpgroup");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  FuseSmem<C, S>& sm = *reinterpret_cast<FuseSmem<C, S>*>(smem_raw);
  if (threadIdx.x < 32 * kFuseProducerWarps) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kFuseProducerRegs));
    fused_producer<T, S, In>(a, bounds, sm.p, (int)(threadIdx.x >> 5), (int)(threadIdx.x & 31));
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kFuseConsumerRegs));
    fused_consumer<C>(a, sm.sw, &sm.tile, (int)threadIdx.x - 32 * kFuseProducerWarps);
  }
}

}  // namespace cbr
