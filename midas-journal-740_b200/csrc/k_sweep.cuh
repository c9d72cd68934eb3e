// k_sweep.cuh — K2a: corner-centric first-touch ownership, shared through shared memory, swept along z.
//
// Reference: the "Create vertices" part of the hot loop (txx:179-194) and the two-plane vertex lookup it
// relies on (VertexLookupMap h:273-313, txx:128-131,155-161,186-191).
//
// Ownership rule (SURVEY §8a row 8): a lattice corner gets its vertex from the first voxel, in raster
// order, among the 2x2x2 voxels around it that has an active face touching it.  For the eight inside
// bits i0..i7 of that block (block raster order, coordinates clamped to the image) this is the closed form
//     i0 == 0 : the first inside voxel
//     i0 == 1 : 0 if !(i1&i2&i4), else 1 if !(i3&i5), else 2 if !i6, else 3 if !i7, else none
// (equal to "first p with i_p & ~(i_{p^1} & i_{p^2} & i_{p^4})" for all 256 inputs, and for blocks clipped
// by the image border once an out-of-image alias hands its claim to its in-image twin;
// tests/test_ownership_rule.py enumerates both).  It is evaluated for 32 corners at a time, ONCE per
// corner word, by the thread that owns that corner word; the eight one-hot masks it yields are exactly the
// eight "my local corner l is new" masks of the <=4 voxel words around it, so neighbouring threads swap
// them through shared memory instead of re-deriving them (the first version did, at 3.5x the cost).
//
// A CTA is a grid of NTX x NTY threads; thread (i, j) owns corner word i of R consecutive corner rows and
// walks along z, like the reference walks slices with its two lookup planes.  Per z step a thread loads
// the R+1 voxel rows under its corner rows for the new slice (one step ahead of their use), evaluates the
// closed form for corner plane z+1, publishes what its -x / -y neighbours need (6 words per thread,
// whatever R), and assembles the 8 ownership masks of its R voxel words in slice z.
// Output per entry of the [Zl+1][EY][EW] lattice: one packed count (owned corners | faces << 10 | active corners << 20),
// the active-corner mask and, for words that own a corner, the 8 ownership masks themselves (k_vertices.cuh walks
// them).  Round 1 also had a second instantiation that swept the volume again to number the vertices; storing the
// masks made it redundant (0.52 ms against 0.07 ms here) and it is gone.
#pragma once
#include "cbr_common.cuh"

namespace cbr {

struct SweepArgs {
  const uint32_t* bits;
  Grid g;
  int Wc;              // corner words per row = ceil((X+1)/32)
  int EY, EW;          // entry lattice: EY = Y+1 rows, EW = roundup(Wc, 4) words per row, Zl+1 planes
  int z_begin, z_end;  // local z range of the voxel slices assembled by the launch (the scan range)
  int tz;              // slices per CTA
  // --- count
  uint32_t* cnt;       // [Zl+1][EY][EW] packed owned corners | faces << 10 | active corners << 20
  uint32_t* act;       // [Zl+1][EY][EW] active-corner mask of the corner word
  uint4* own;          // [Zl+1][EY][EW][2] the 8 ownership masks of the voxel word, written where it owns a corner
                       // (may be null: raster vertex order does not need them)
  uint32_t* slice_any;  // [Zl] set to 1 where voxel slice z has an inside voxel (the empty-interior-slice check), may be null
};

template <int NTX_, int NTY_, int R_>
struct SweepCfg {
  static constexpr int NTX = NTX_, NTY = NTY_, R = R_;
  static constexpr int NT = NTX * NTY;               // live threads
  static constexpr int NTP = (NT + 31) / 32 * 32;    // launched threads
  static constexpr int NW = NTP / 32;
  static constexpr int MINB = (NTP == 128 && R_ == 2) ? 5 : 1;  // (forcing 6 CTAs/SM = 80 registers on the (17, 7, 2) tile was measured in r2: 388 -> 404 us)
  static constexpr int LO = 0;
  static constexpr int CR = NTY * R;                 // corner rows per CTA
  static constexpr int TXW = NTX - 1 - 2 * LO;       // voxel words (x) whose results the CTA produces
  static constexpr int TY = CR - 1 - 2 * LO;         // voxel rows  (y)
  static_assert(R >= 1 && R <= 4, "nibble word holds 5 bits per row");
};

template <typename C>
struct SweepSmem {
  uint32_t ex[2][6][C::NT];  // exchange: P0,P1,P4,P5 of the thread's lowest corner row, its c word, bit-0 nibbles
};

// closed-form first-touch owner of 32 corners: in[p] = inside word of block voxel p = qz*4+qy*2+qx;
// vm = corners of this word that exist
__device__ __forceinline__ void corner_owners(const uint32_t in[8], uint32_t vm, uint32_t own[8]) {
  uint32_t r = in[0];
#pragma unroll
  for (int p = 1; p < 8; ++p) {
    own[p] = in[p] & ~r & vm;
    r |= in[p];
  }
  const uint32_t a = in[1] & in[2] & in[4];
  own[0] = in[0] & ~a & vm;
  const uint32_t t = in[0] & a & vm;
  const uint32_t b = in[3] & in[5];
  own[1] |= t & ~b;
  const uint32_t t2 = t & b;
  own[2] |= t2 & ~in[6];
  own[3] |= t2 & in[6] & ~in[7];
}

// One tile of the sweep: thread t of the C::NTP threads that share `sm`, tile (bx, by) of the x-y plane, z chunk bz.
// FUSED: the caller is one warpgroup of k_classify_sweep (k_fused.cuh) - the threads meet at named barrier 1 instead of
// the CTA barrier, and the bitmask, written by other SMs earlier in the SAME kernel, is read past the (incoherent) L1.
template <typename C, bool FUSED>
__device__ __forceinline__ void sweep_tile(const SweepArgs& a, SweepSmem<C>& sm, const int t, const int bx, const int by,
                                           const int bz) {
  constexpr int NTX = C::NTX, NTY = C::NTY, R = C::R, NT = C::NT, CR = C::CR;
  const Grid& g = a.g;
  const bool alive = t < NT;
  const int tt = alive ? t : 0;
  const int i = tt % NTX, j = tt / NTX;
  const int w0 = bx * C::TXW, y0 = by * C::TY;
  const int cw = w0 + i;
  const int rr0 = j * R;          // first corner row of the thread, CTA-relative
  const int cy0 = y0 + rr0;       // ... and in the image
  const int zs = a.z_begin + bz * a.tz;
  const int ze = min(zs + a.tz, a.z_end);

  // ---- per-thread constants ---------------------------------------------------------------------------
  const int XW = g.X >> 5, XB = g.X & 31;
  const bool col_ok = alive && cw < a.Wc;
  const uint32_t vmx = !col_ok ? 0u : (cw < XW ? ~0u : ((2u << XB) - 1u));       // corners cx <= X of this word
  const uint32_t vc = (cw == g.Wx - 1 && XB) ? ((1u << XB) - 1u) : ~0u;           // voxels x < X of this word
  const bool first = cw == 0, synth = cw >= g.Wx;  // no voxel word on the left / this corner word is the x = X replicate
  const int cwl = min(cw, g.Wx - 1);
  const bool xcomplete = alive && i <= NTX - 2;    // the +x neighbour thread exists
  const bool word_ok = xcomplete && cw < g.Wx;
  // the corner column one past the last voxel word belongs to the last tile in x
  const bool xcorner = col_ok && (i <= NTX - 2 || cw >= g.Wx);
  const size_t slice_words = (size_t)g.Y * g.Wp;
  const size_t plane_entries = (size_t)a.EY * a.EW;
  int rowoff[R + 1];
#pragma unroll
  for (int k = 0; k <= R; ++k) rowoff[k] = min(max(cy0 - 1 + k, 0), g.Y - 1) * g.Wp + cwl;
  const int dprev = (first || synth) ? 0 : 1;
  // local slice indices are clamped to the image (globally) and, for memory safety, to the local buffer
  const int zlo = max(0, -g.zg0), zhi = min(g.Zl - 1, g.Zg - 1 - g.zg0);
  const int e0 = cy0 * a.EW + cw;       // entry index of (cw, cy0) inside a plane of the entry lattice
  // per-row predicates, one bit per k: voxel row complete & inside the image / corner row counted by this CTA
  uint32_t rowok_bits = 0, corner_bits = 0;
#pragma unroll
  for (int k = 0; k < R; ++k) {
    const int rr = rr0 + k, cy = cy0 + k;
    if (word_ok && rr <= CR - 2 && cy < g.Y) rowok_bits |= 1u << k;
    // rows one past the last voxel row belong to the last tile in y
    if (xcorner && cy <= g.Y && (rr <= CR - 2 || cy >= g.Y)) corner_bits |= 1u << k;
  }
  const int exo = alive ? t : 0;

  // raw words (this corner word and the one to its left) of the R+1 window rows of one slice; fetched one
  // step ahead of their use so that the L2/HBM latency overlaps the previous step
  auto fetch_slice = [&](int zl, uint32_t (&cwv)[R + 1], uint32_t (&pwv)[R + 1]) {
    const uint32_t* __restrict__ sl = a.bits + (size_t)min(max(zl, zlo), zhi) * slice_words;
#pragma unroll
    for (int k = 0; k <= R; ++k) {
      cwv[k] = FUSED ? __ldcg(sl + rowoff[k]) : __ldg(sl + rowoff[k]);
      pwv[k] = FUSED ? __ldcg(sl + rowoff[k] - dprev) : __ldg(sl + rowoff[k] - dprev);
    }
  };
  // -> c (voxel x = corner x) and l (voxel x-1) words, edge-replicated in x
  auto decode_slice = [&](const uint32_t (&cwv)[R + 1], const uint32_t (&pwv)[R + 1], uint32_t (&c)[R + 1], uint32_t (&l)[R + 1]) {
#pragma unroll
    for (int k = 0; k <= R; ++k) {
      const uint32_t rep = 0u - (cwv[k] >> 31);
      const uint32_t pw = first ? (cwv[k] << 31) : pwv[k];
      c[k] = synth ? rep : cwv[k];
      l[k] = synth ? rep : __funnelshift_l(pw, cwv[k], 1);
    }
  };

  // rolling voxel words of the window rows: "lo" = slice cz-1, "hi" = slice cz
  uint32_t lo_c[R + 1], lo_l[R + 1], hi_c[R + 1], hi_l[R + 1];
  uint32_t below_c[R];  // voxel rows of slice cz-2 (the -z neighbours of the voxel words being assembled)
#pragma unroll
  for (int k = 0; k <= R; ++k) lo_c[k] = lo_l[k] = 0;
  uint32_t nx_c[R + 1], nx_p[R + 1];  // prefetched raw words of the next slice
  fetch_slice(zs - 1, nx_c, nx_p);
  decode_slice(nx_c, nx_p, hi_c, hi_l);
  fetch_slice(zs, nx_c, nx_p);
  // kept from the previous plane: own P4..P7 per row, the +y neighbour's P4,P5, the neighbours' nibbles, active masks
  uint32_t sv[R][4], su4 = 0, su5 = 0, nr_prev = 0, nur_prev = 0, act_prev[R];
#pragma unroll
  for (int k = 0; k < R; ++k) {
    sv[k][0] = sv[k][1] = sv[k][2] = sv[k][3] = 0;
    act_prev[k] = 0;
  }

  uint32_t occupied = 0;  // bit k: voxel slice zs + k has an inside voxel in this thread's words (a.tz <= 32)
  for (int cz = zs; cz <= ze; ++cz) {
    const int buf = cz & 1;
    // ---- 1. slide the window, decode slice cz (fetched during the previous step), closed form for plane cz ---
#pragma unroll
    for (int k = 0; k < R; ++k) below_c[k] = lo_c[k + 1];
#pragma unroll
    for (int k = 0; k <= R; ++k) { lo_c[k] = hi_c[k]; lo_l[k] = hi_l[k]; }
    decode_slice(nx_c, nx_p, hi_c, hi_l);
    if (cz < ze) fetch_slice(cz + 1, nx_c, nx_p);
    const int czg = cz + g.zg0;
    uint32_t own[R][8];
    uint32_t nib = 0;
#pragma unroll
    for (int k = 0; k < R; ++k) {
      const int cy = cy0 + k;
      const uint32_t in[8] = {lo_l[k], lo_c[k], lo_l[k + 1], lo_c[k + 1], hi_l[k], hi_c[k], hi_l[k + 1], hi_c[k + 1]};
      corner_owners(in, cy <= g.Y ? vmx : 0u, own[k]);
      if (cy == 0 || czg == 0 || cw == 0) {  // clipped blocks: out-of-image aliases hand over to their in-image twins
        if (cy == 0) {
          own[k][2] |= own[k][0]; own[k][3] |= own[k][1]; own[k][6] |= own[k][4]; own[k][7] |= own[k][5];
          own[k][0] = own[k][1] = own[k][4] = own[k][5] = 0;
        }
        if (czg == 0) {
          own[k][4] |= own[k][0]; own[k][5] |= own[k][1]; own[k][6] |= own[k][2]; own[k][7] |= own[k][3];
          own[k][0] = own[k][1] = own[k][2] = own[k][3] = 0;
        }
        if (cw == 0) {
#pragma unroll
          for (int p = 0; p < 8; p += 2) {
            own[k][p + 1] |= own[k][p] & 1u;
            own[k][p] &= ~1u;
          }
        }
      }
      nib |= ((own[k][0] & 1u) | ((own[k][2] & 1u) << 1) | ((own[k][4] & 1u) << 2) | ((own[k][6] & 1u) << 3) |
              ((lo_c[k + 1] & 1u) << 4)) << (5 * k);
    }
    uint32_t* __restrict__ exw = &sm.ex[buf][0][exo];
    if (alive) {
      exw[0 * NT] = own[0][0];
      exw[1 * NT] = own[0][1];
      exw[2 * NT] = own[0][4];
      exw[3 * NT] = own[0][5];
      exw[4 * NT] = lo_c[1];
      exw[5 * NT] = nib;
    }
    // does slice cz-1 have an inside voxel at all (the empty-interior-slice check)?  One bit per slice of the CTA's
    // sweep in a per-thread mask, reduced and stored once after the sweep.
    {
      uint32_t any_in = 0;
#pragma unroll
      for (int k = 0; k < R; ++k)
        if ((rowok_bits >> k) & 1u) any_in |= lo_c[k + 1] & vc;
      if (any_in != 0 && cz > zs) occupied |= 1u << (cz - 1 - zs);
    }
    if (FUSED) asm volatile("bar.sync 1, %0;" ::"n"(C::NTP) : "memory");
    else __syncthreads();

    uint32_t act[R];
#pragma unroll
    for (int k = 0; k < R; ++k)
      act[k] = own[k][0] | own[k][1] | own[k][2] | own[k][3] | own[k][4] | own[k][5] | own[k][6] | own[k][7];
    // what the neighbours published for this plane
    uint32_t p0u = 0, p1u = 0, p4u = 0, p5u = 0, upc = 0, nr = 0, nur = 0;
    if (xcomplete) {
      nr = exw[5 * NT + 1];                       // thread (i+1, j)
      if (j <= NTY - 2) {
        const uint32_t* __restrict__ exu = exw + NTX;  // thread (i, j+1)
        p0u = exu[0 * NT]; p1u = exu[1 * NT]; p4u = exu[2 * NT]; p5u = exu[3 * NT];
        upc = exu[4 * NT];
        nur = exu[5 * NT + 1];                    // thread (i+1, j+1)
      }
    }

    if (cz > zs) {
      const int z = cz - 1;  // the voxel slice being assembled
      // ownership masks of voxel row k (corner rows k and k+1 of planes z [kept] and z+1 [fresh])
      auto assemble = [&](int k, uint32_t (&O)[8]) {
        const bool top = (k == R - 1);
        const int ku = top ? 0 : k + 1;
        const uint32_t s4 = top ? su4 : sv[ku][0], s5 = top ? su5 : sv[ku][1];
        const uint32_t f0 = top ? p0u : own[ku][0], f1 = top ? p1u : own[ku][1];
        const uint32_t nup = top ? nur : (nr >> (5 * ku)), nup_prev = top ? nur_prev : (nr_prev >> (5 * ku));
        O[0] = sv[k][3];
        O[1] = __funnelshift_r(sv[k][2], nr_prev >> (5 * k + 3), 1);
        O[2] = __funnelshift_r(s4, nup_prev >> 2, 1);
        O[3] = s5;
        O[4] = own[k][3];
        O[5] = __funnelshift_r(own[k][2], nr >> (5 * k + 1), 1);
        O[6] = __funnelshift_r(f0, nup, 1);
        O[7] = f1;
      };

      uint32_t* __restrict__ cntz = a.cnt + (size_t)z * plane_entries;
      uint32_t* __restrict__ actz = a.act + (size_t)z * plane_entries;
#pragma unroll
      for (int k = 0; k < R; ++k) {
        const bool vox = (rowok_bits >> k) & 1u, cor = (corner_bits >> k) & 1u;
        if (!(vox || cor)) continue;
        uint32_t packed = 0;
        if (vox) {
          uint32_t O[8];
          assemble(k, O);
          const uint32_t c = lo_c[k + 1] & vc;
          const uint32_t nf = __popc(c & ~lo_l[k + 1]) + __popc(c & ~lo_c[k]) +
                              __popc(c & ~__funnelshift_r(lo_c[k + 1], nr >> (5 * k + 4), 1)) +
                              __popc(c & ~((k == R - 1) ? upc : lo_c[(k == R - 1) ? 0 : k + 2])) +
                              __popc(c & ~below_c[k]) + __popc(c & ~hi_c[k + 1]);
          uint32_t nv = 0;
#pragma unroll
          for (int l = 0; l < 8; ++l) nv += __popc(O[l]);
          packed = nv | (nf << 10);
          // (r2 also tried two 16-byte half records, each written only where it has a bit: fewer bytes stored, but a
          //  16-byte store leaves half a 32-byte L2 sector to be filled from DRAM - the fused kernel went 0.88 -> 0.98 ms)
          if (nv && a.own) {  // k_assign walks these instead of sweeping again
            uint4* __restrict__ o = a.own + 2 * ((size_t)z * plane_entries + (size_t)(e0 + k * a.EW));
            __stcs(o, make_uint4(O[0], O[1], O[2], O[3]));
            __stcs(o + 1, make_uint4(O[4], O[5], O[6], O[7]));
          }
        }
        if (cor) {
          packed |= (uint32_t)__popc(act_prev[k]) << 20;
          actz[e0 + k * a.EW] = act_prev[k];
        }
        cntz[e0 + k * a.EW] = packed;
      }
      if (cz == ze && ze == a.z_end) {  // the top corner plane of the range has no voxel slice of its own
#pragma unroll
        for (int k = 0; k < R; ++k) {
          if ((corner_bits >> k) & 1u) {
            (a.cnt + (size_t)cz * plane_entries)[e0 + k * a.EW] = (uint32_t)__popc(act[k]) << 20;
            (a.act + (size_t)cz * plane_entries)[e0 + k * a.EW] = act[k];
          }
        }
      }
    }

    // ---- what the next plane needs from this one ------------------------------------------------------------
#pragma unroll
    for (int k = 0; k < R; ++k) {
      sv[k][0] = own[k][4]; sv[k][1] = own[k][5]; sv[k][2] = own[k][6]; sv[k][3] = own[k][7];
      act_prev[k] = act[k];
    }
    su4 = p4u; su5 = p5u;
    nr_prev = nr; nur_prev = nur;
  }
  if (a.slice_any) {
    occupied = __reduce_or_sync(0xffffffffu, occupied);
    const int lane = t & 31;
    if (((occupied >> lane) & 1u) && zs + lane < ze) a.slice_any[zs + lane] = 1u;
  }
}

template <typename C>
__global__ void __launch_bounds__(C::NTP, C::MINB) k_sweep(const SweepArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  sweep_tile<C, false>(a, *reinterpret_cast<SweepSmem<C>*>(smem_raw), (int)threadIdx.x, (int)blockIdx.x, (int)blockIdx.y,
                       (int)blockIdx.z);
}

}  // namespace cbr
