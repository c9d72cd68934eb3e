// k_project.cuh — K4: ProjectVertexToIsoSurface, one thread per vertex.
//
// Reference: txx:440-474 (default branch) on top of ComputeGradientImage (txx:479-498).  The
// reference materialises a 12 B/voxel fp32 gradient image for the whole volume and interpolates
// it; here the central differences (GradientImageFilter semantics, SURVEY Appendix A.3) are
// evaluated on the fly at the <=8 lattice nodes a vertex touches, with exactly the arithmetic of
// the oracle: fp32 differences, fp64 trilinear weights in ITK 3.x neighbour order with the
// zero-overlap skip and the `totalOverlap == 1` early exit (Appendix A.4), fp32 normal,
// fp64 norm / step / sign, fp32 vertex.  The library is compiled with -fmad=false so that no
// multiply-add is contracted; double division and sqrt are IEEE in CUDA.  The result is
// bit-identical to oracle/cuberille_oracle.cpp::project_vertex (tests/test_gpu_parity.py).
//
// Divergence from the reference, shared with the oracle: out-of-image neighbour indices are
// clamped (the reference reads out of bounds) and a zero gradient stops the vertex where it is
// (the reference divides by zero).
#pragma once
#include <climits>

#include "cbr_common.cuh"
#include "k_segscan.cuh"

namespace cbr {

struct ProjArgs {
  const void* vol;
  Grid g;
  Geom geom;
  double iso;    // (double)(T)iso
  double thr;    // m_ProjectVertexSurfaceDistanceThreshold
  double step0;  // m_ProjectVertexStepLength (after the auto rule txx:82-85)
  double relax;  // m_ProjectVertexStepLengthRelaxationFactor
  unsigned max_steps;
  float* points;
  size_t n_points;           // number of points (info == null)
  unsigned long long* info;  // when set: the points are [ghost ? 0 : info[kInfoGhostV], info[kInfoGhostV] + info[kInfoPoints]),
                             // and nothing is projected unless k_check_caps found that the emission fits its buffers
  int include_ghost;
  long long i0[3];           // image index of buffer voxel (0, 0, 0) (cub_set_region_index): continuous indices are image indices
  unsigned long long* work;  // device counter (zeroed before the launch): next vertex to hand out
  unsigned refill;           // lanes of a warp that must still be iterating for the warp to skip the service phase (1..32)
};

template <typename T>
struct VolView {
  const T* __restrict__ d;
  int X, Y, Zl, zg0, Zg;
  __device__ __forceinline__ T at(int x, int y, int zg) const {  // image-clamped (zg is a GLOBAL z index)
    x = x < 0 ? 0 : (x > X - 1 ? X - 1 : x);
    y = y < 0 ? 0 : (y > Y - 1 ? Y - 1 : y);
    zg = zg < 0 ? 0 : (zg > Zg - 1 ? Zg - 1 : zg);
    int z = zg - zg0;
    z = z < 0 ? 0 : (z > Zl - 1 ? Zl - 1 : z);  // memory safety only (halo contract of cub_set_slab)
    return __ldg(d + ((size_t)z * Y + y) * X + x);
  }
};

template <typename T> struct is_fp { static constexpr bool value = false; };
template <> struct is_fp<float> { static constexpr bool value = true; };
template <> struct is_fp<double> { static constexpr bool value = true; };

// GradientImageFilter at one node: sum = 0; sum += (-c)*I[-1]; sum += 0*I[0]; sum += c*I[+1]  (fp32)
template <typename T>
__device__ __forceinline__ void gradient_at(const VolView<T>& v, const float c[3], int x, int y, int z, float g[3]) {
  // the 0*I[0] term only matters for non-finite float pixels; integer pixels skip the load
  const float mid = is_fp<T>::value ? (float)v.at(x, y, z) : 0.0f;
  {
    float s = 0.0f;
    s += (-c[0]) * (float)v.at(x - 1, y, z);
    s += 0.0f * mid;
    s += c[0] * (float)v.at(x + 1, y, z);
    g[0] = s;
  }
  {
    float s = 0.0f;
    s += (-c[1]) * (float)v.at(x, y - 1, z);
    s += 0.0f * mid;
    s += c[1] * (float)v.at(x, y + 1, z);
    g[1] = s;
  }
  {
    float s = 0.0f;
    s += (-c[2]) * (float)v.at(x, y, z - 1);
    s += 0.0f * mid;
    s += c[2] * (float)v.at(x, y, z + 1);
    g[2] = s;
  }
}

// GradientImageFilter::m_UseImageDirection on an oriented image: every gradient pixel is rotated into physical space,
// TransformLocalVectorToPhysicalVector: fp64 row sums (from 0) of D * fp32 gradient, rounded to fp32
__device__ __forceinline__ void rotate_gradient(const Geom& geom, float g[3]) {
  float r[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double sum = 0.0;
#pragma unroll
    for (int j = 0; j < 3; ++j) sum += geom.dir[3 * i + j] * (double)g[j];
    r[i] = (float)sum;
  }
  g[0] = r[0]; g[1] = r[1]; g[2] = r[2];
}

__device__ __forceinline__ int clampi(long long v, int hi) { return v < 0 ? 0 : (v > hi ? hi : (int)v); }

// Persistent lanes: the number of moves varies from 0 to max_steps+2 between vertices, so a lane that finishes
// its vertex immediately takes the next one from a global counter instead of idling until the slowest vertex of
// its warp is done.  The arithmetic per vertex is unchanged (and so are the results, bit for bit).
template <typename T, bool ORIENTED>
__global__ void __launch_bounds__(128, ORIENTED ? 5 : 6) k_project(const ProjArgs a) {
  VolView<T> v{static_cast<const T*>(a.vol), a.g.X, a.g.Y, a.g.Zl, a.g.zg0, a.g.Zg};
  float gc[3];
  double inv_sp[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    inv_sp[k] = 1.0 / a.geom.spacing[k];
    gc[k] = (float)(0.5 * inv_sp[k]);
  }
  size_t n_points = a.n_points;
  float* const points = a.points + (a.info && !a.include_ghost ? 3 * (size_t)__ldg(a.info + kInfoGhostV) : 0);
  if (a.info) {
    if (!emission_fits(a.info)) return;
    const size_t ghost = (size_t)__ldg(a.info + kInfoGhostV);
    const size_t all = ghost + (size_t)__ldg(a.info + kInfoPoints);
    n_points = a.include_ghost ? all : all - ghost;
  }
  size_t i = 0;
  bool have = false, exhausted = false;
  float vert[3] = {0.f, 0.f, 0.f};
  double step = a.step0;
  unsigned numberOfSteps = 0;

  // The 8 lattice nodes around the vertex: their pixel values and fp32 central-difference gradients are kept
  // in registers and only re-fetched when the vertex crosses into another cell (a step is a fraction of a
  // voxel, so most iterations stay in the cell: the first version re-read 64 voxels per iteration).
  long long cell[3] = {LLONG_MIN, LLONG_MIN, LLONG_MIN};
  double nval[8];
  // the 24 gradient components live in shared memory, already widened to fp64 (exact), one column per thread: the
  // interpolation then reads them with LDS.64 instead of converting them again on every pass (r2 profile: 24 of the
  // ~50 conversions of a pass, on a conversion pipe that was 56 % busy), and 24 registers are free
  __shared__ double s_ngrad[24][128];
  double (*const ng)[128] = reinterpret_cast<double (*)[128]>(&s_ngrad[0][threadIdx.x]);  // ng[3 * node + axis][0]
  // continuous index of `vert`: base index (buffer-relative) and distances (shared by both interpolators)
  // (32-bit saturated base indices were measured in r2: same register count, 5.15 -> 5.33 ms)
  long long base[3] = {0, 0, 0};
  double dist[3] = {0.0, 0.0, 0.0};
  auto locate = [&]() {
    double ci[3];
    if (!ORIENTED) {
#pragma unroll
      for (int k = 0; k < 3; ++k) ci[k] = ((double)vert[k] - a.geom.origin[k]) * inv_sp[k];
    } else {
      // TransformPhysicalPointToContinuousIndex of an oriented image: M^-1 * (point - origin), row sums from 0
      double c[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) c[k] = (double)vert[k] - a.geom.origin[k];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < 3; ++j) sum += a.geom.minv[3 * i + j] * c[j];
        ci[i] = sum;
      }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double f = floor(ci[k]);
      base[k] = (long long)f - a.i0[k];  // buffer-relative
      dist[k] = ci[k] - f;
    }
  };

  // Two phases per round (the per-vertex arithmetic is the reference's loop body, unchanged):
  //   SERVICE  lanes without a vertex take the next one from the global counter; lanes whose vertex is in a cell
  //            other than the cached one (a new vertex, or one that crossed a cell face) load the cell
  //   ITERATE  passes of the reference's `while ( !done )` body (txx:448-473) for the lanes whose cell is cached,
  //            repeated while at least a.refill lanes of the warp still have one to make
  // so that the long cell load runs for many lanes at a time instead of once per lane event (r1/r2: every pass of a
  // warp went through it with one or two lanes active, and it took as many issue slots as the iterations).
  while (true) {
    if (!have && !exhausted) {
      i = (size_t)atomicAdd(a.work, 1ull);
      if (i >= n_points) {
        exhausted = true;
      } else {
        vert[0] = points[3 * i]; vert[1] = points[3 * i + 1]; vert[2] = points[3 * i + 2];
        step = a.step0;
        numberOfSteps = 0;
        have = true;
        locate();
      }
    }
    if (__all_sync(0xffffffffu, !have)) break;
    if (have && (base[0] != cell[0] || base[1] != cell[1] || base[2] != cell[2])) {
      cell[0] = base[0]; cell[1] = base[1]; cell[2] = base[2];
      const long long zl0 = base[2] - v.zg0;  // local slice of node z = 0
      const bool nodes_inside = base[0] >= 0 && base[0] + 1 <= v.X - 1 && base[1] >= 0 && base[1] + 1 <= v.Y - 1 &&
                                base[2] >= 0 && base[2] + 1 <= v.Zg - 1 && zl0 >= 0 && zl0 + 1 <= v.Zl - 1;
      if (nodes_inside) {
        // The 8 nodes are in the image, so only their outward 6-neighbours can clamp, and clamp(node +- 1) is the
        // node itself there.  The nodes and their 6-neighbours are 32 distinct voxels (a 4x2x2 block along each
        // axis sharing the 2x2x2 nodes), fetched once from 12 row pointers.  Same values and the same arithmetic
        // as the general path below (which remains for vertices that have left the image).
        const T* __restrict__ p = v.d + ((size_t)zl0 * v.Y + (size_t)base[1]) * v.X + (size_t)base[0];
        const ptrdiff_t sx = (ptrdiff_t)v.X, sxy = (ptrdiff_t)v.X * v.Y;
        const ptrdiff_t xm = base[0] >= 1 ? -1 : 0, xp = base[0] + 2 <= v.X - 1 ? 2 : 1;
        const ptrdiff_t ym = base[1] >= 1 ? -sx : 0, yp = base[1] + 2 <= v.Y - 1 ? 2 * sx : sx;
        const ptrdiff_t zm = (base[2] >= 1 && zl0 >= 1) ? -sxy : 0;
        const ptrdiff_t zp = (base[2] + 2 <= v.Zg - 1 && zl0 + 2 <= v.Zl - 1) ? 2 * sxy : sxy;
        float ax[2][2][4], ay[2][2][2], az[2][2][2];  // [oz][oy][x = -1..2], [oz][y = -1 | 2][ox], [z = -1 | 2][oy][ox]
#pragma unroll
        for (int oz = 0; oz < 2; ++oz)
#pragma unroll
          for (int oy = 0; oy < 2; ++oy) {
            const T* __restrict__ r = p + oz * sxy + oy * sx;
            const T n0 = __ldg(r), n1 = __ldg(r + 1);
            ax[oz][oy][0] = (float)__ldg(r + xm); ax[oz][oy][1] = (float)n0;
            ax[oz][oy][2] = (float)n1;            ax[oz][oy][3] = (float)__ldg(r + xp);
            nval[oz * 4 + oy * 2] = (double)n0; nval[oz * 4 + oy * 2 + 1] = (double)n1;
          }
#pragma unroll
        for (int oz = 0; oz < 2; ++oz)
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const T* __restrict__ r = p + oz * sxy + (j ? yp : ym);
            ay[oz][j][0] = (float)__ldg(r); ay[oz][j][1] = (float)__ldg(r + 1);
          }
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int oy = 0; oy < 2; ++oy) {
            const T* __restrict__ r = p + oy * sx + (j ? zp : zm);
            az[j][oy][0] = (float)__ldg(r); az[j][oy][1] = (float)__ldg(r + 1);
          }
#pragma unroll
        for (int counter = 0; counter < 8; ++counter) {
          const int ox = counter & 1, oy = (counter >> 1) & 1, oz = counter >> 2;
          const float mid = is_fp<T>::value ? ax[oz][oy][ox + 1] : 0.0f;
          const float xm = ax[oz][oy][ox], xp = ax[oz][oy][ox + 2];
          const float ym = oy == 0 ? ay[oz][0][ox] : ax[oz][0][ox + 1], yp = oy == 0 ? ax[oz][1][ox + 1] : ay[oz][1][ox];
          const float zm = oz == 0 ? az[0][oy][ox] : ax[0][oy][ox + 1], zp = oz == 0 ? ax[1][oy][ox + 1] : az[1][oy][ox];
          // sum = 0; sum += (-c) * I[-1]; sum += 0 * I[0]; sum += c * I[+1].  The middle term only matters for a
          // non-finite centre pixel (0 * inf = NaN): for a finite one it adds +-0 to a sum that is never -0 (the
          // first addition to +0 cleared the sign), i.e. nothing.
          const bool odd = is_fp<T>::value && !(fabsf(mid) <= 3.402823466e38f);
          float gt[3];
          { float s = 0.0f; s += (-gc[0]) * xm; if (odd) s += 0.0f * mid; s += gc[0] * xp; gt[0] = s; }
          { float s = 0.0f; s += (-gc[1]) * ym; if (odd) s += 0.0f * mid; s += gc[1] * yp; gt[1] = s; }
          { float s = 0.0f; s += (-gc[2]) * zm; if (odd) s += 0.0f * mid; s += gc[2] * zp; gt[2] = s; }
          if (ORIENTED) rotate_gradient(a.geom, gt);
          ng[3 * counter + 0][0] = (double)gt[0]; ng[3 * counter + 1][0] = (double)gt[1]; ng[3 * counter + 2][0] = (double)gt[2];
        }
      } else {
#pragma unroll 1
        for (int counter = 0; counter < 8; ++counter) {
          const int cx = clampi(base[0] + ((counter & 1) ? 1 : 0), v.X - 1);
          const int cy = clampi(base[1] + ((counter & 2) ? 1 : 0), v.Y - 1);
          const int cz = clampi(base[2] + ((counter & 4) ? 1 : 0), v.Zg - 1);
          float gtmp[3];
          gradient_at(v, gc, cx, cy, cz, gtmp);
          if (ORIENTED) rotate_gradient(a.geom, gtmp);
          const double nv = (double)v.at(cx, cy, cz);
          ng[3 * counter + 0][0] = (double)gtmp[0]; ng[3 * counter + 1][0] = (double)gtmp[1]; ng[3 * counter + 2][0] = (double)gtmp[2];
          // (dynamic index into the register cache: written through a switch so that it stays in registers)
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (q == counter) nval[q] = nv;
        }
      }
    }
    unsigned n_active;
    do {
      if (have && base[0] == cell[0] && base[1] == cell[1] && base[2] == cell[2]) {
        bool done = false;  // one pass of the reference's `while ( !done )` body (txx:448-473)
        double gd[3] = {0.0, 0.0, 0.0};
        double value = 0.0, total = 0.0;
        bool open = true;
        // overlap = ((1 * wx) * wy) * wz in the reference's order; 1 * wx is wx, and the four wx * wy products are shared
        // by the two z layers (same values, same association: bit-identical, 12 multiplications instead of 24)
        const double wx[2] = {1.0 - dist[0], dist[0]}, wy[2] = {1.0 - dist[1], dist[1]}, wz[2] = {1.0 - dist[2], dist[2]};
        const double wxy[4] = {wx[0] * wy[0], wx[1] * wy[0], wx[0] * wy[1], wx[1] * wy[1]};
    #pragma unroll
        for (int counter = 0; counter < 8; ++counter) {
          if (open) {
            const double overlap = wxy[counter & 3] * wz[counter >> 2];
            if (overlap != 0.0) {
              gd[0] += overlap * ng[3 * counter + 0][0];
              gd[1] += overlap * ng[3 * counter + 1][0];
              gd[2] += overlap * ng[3 * counter + 2][0];
              value += overlap * nval[counter];
              total += overlap;
            }
            if (total == 1.0) open = false;
          }
        }
        // normal = (CovariantVector<float,3>) gradient; normal.Normalize()        txx:451-452
        float normal[3] = {(float)gd[0], (float)gd[1], (float)gd[2]};
        double sq = 0.0;
    #pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double c = (double)normal[k];
          sq += c * c;
        }
        if (sq == 0.0) {   // norm == 0 (the square root of a positive double is positive)
          done = true;  // zero gradient: the vertex stays where it is (DESIGN.md section 2)
        } else {
          done |= fabs(value - a.iso) < a.thr;  // txx:456  (the normalised normal is only used by the move below)
          if (!done) {
            // normal[k] = (float)((double)normal[k] / sqrt(sq)), txx:452: an IEEE square root and three IEEE divisions
            // (~120 instructions).  Fast path: q = normal[k] * rsqrt(sq) is within a few ulp (double) of the exact
            // quotient, so it rounds to the same float unless it lies within 64 ulp of a float rounding boundary (the low
            // 29 mantissa bits near 2^28) or the float result would be subnormal; only then (2.4e-7 of the cases) the
            // exact expressions run.  The result is bit-identical to the oracle's either way.
            const double r = rsqrt(sq);
            float fast[3];
            bool risky = !(sq >= 1e-280 && sq <= 1e280);
    #pragma unroll
            for (int k = 0; k < 3; ++k) {
              const double q = (double)normal[k] * r;
              fast[k] = (float)q;
              // low 29 mantissa bits within 64 of the rounding boundary 2^28; |q| below the smallest normal float
              // (biased exponent < 1023 - 126) unless it is an exact zero
              const unsigned lo = (unsigned)__double2loint(q), hi = (unsigned)__double2hiint(q) & 0x7fffffffu;
              risky |= ((lo & 0x1fffffffu) - (0x10000000u - 64u) < 128u) || (hi < 0x38100000u && (hi | lo) != 0u);
            }
            if (risky) {
              const double norm = sqrt(sq);
    #pragma unroll
              for (int k = 0; k < 3; ++k) normal[k] = (float)((double)normal[k] / norm);
            } else {
              normal[0] = fast[0]; normal[1] = fast[1]; normal[2] = fast[2];
            }
            const double sign = (value < a.iso) ? +1.0 : -1.0;  // txx:463
    #pragma unroll
            for (int k = 0; k < 3; ++k) vert[k] = (float)((double)vert[k] + ((double)normal[k] * sign) * step);  // txx:466
            step *= a.relax;                                  // txx:468
            done |= numberOfSteps++ > a.max_steps;            // txx:469
          }
        }
        if (done) {
          points[3 * i] = vert[0];
          points[3 * i + 1] = vert[1];
          points[3 * i + 2] = vert[2];
          have = false;
        } else {
          locate();
        }
      }
      n_active = __popc(__ballot_sync(0xffffffffu, have && base[0] == cell[0] && base[1] == cell[1] && base[2] == cell[2]));
    } while (n_active >= a.refill);
  }
}

// ---- the reference's compile-time alternates (h:22-23): USE_ADVANCED_PROJECTION txx:340-397 and
// USE_LINESEARCH_PROJECTION txx:398-438.  No test of the reference enables them; they are offered at run time
// (cub_params.projection_method), one thread per vertex, with the same interpolation arithmetic as the default
// branch (general clamped path, no cell cache: these variants are not the hot configuration), bit-identical to
// oracle/cuberille_oracle.cpp::project_vertex_advanced / project_vertex_linesearch.
enum { kProjectDefault = 0, kProjectAdvanced = 1, kProjectLineSearch = 2 };

template <typename T, bool ORIENTED>
struct Sampler {
  VolView<T> v;
  const ProjArgs& a;
  float gc[3];
  double inv_sp[3];
  __device__ __forceinline__ Sampler(const ProjArgs& a_) : v{static_cast<const T*>(a_.vol), a_.g.X, a_.g.Y, a_.g.Zl, a_.g.zg0, a_.g.Zg}, a(a_) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      inv_sp[k] = 1.0 / a.geom.spacing[k];
      gc[k] = (float)(0.5 * inv_sp[k]);
    }
  }
  // interpolated value and (optionally) gradient at a Point<float>: ITK 3.x N-d linear interpolation (Appendix A.4)
  template <bool GRAD>
  __device__ __forceinline__ double sample(const float pt[3], double gd[3]) const {
    double ci[3];
    if (!ORIENTED) {
#pragma unroll
      for (int k = 0; k < 3; ++k) ci[k] = ((double)pt[k] - a.geom.origin[k]) * inv_sp[k];
    } else {
      double c[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) c[k] = (double)pt[k] - a.geom.origin[k];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < 3; ++j) sum += a.geom.minv[3 * i + j] * c[j];
        ci[i] = sum;
      }
    }
    long long base[3];
    double dist[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double f = floor(ci[k]);
      base[k] = (long long)f - a.i0[k];
      dist[k] = ci[k] - f;
    }
    double value = 0.0, total = 0.0;
    if (GRAD) gd[0] = gd[1] = gd[2] = 0.0;
#pragma unroll 1
    for (int counter = 0; counter < 8; ++counter) {
      double overlap = 1.0;
      overlap *= (counter & 1) ? dist[0] : 1.0 - dist[0];
      overlap *= (counter & 2) ? dist[1] : 1.0 - dist[1];
      overlap *= (counter & 4) ? dist[2] : 1.0 - dist[2];
      if (overlap != 0.0) {
        const int cx = clampi(base[0] + ((counter & 1) ? 1 : 0), v.X - 1);
        const int cy = clampi(base[1] + ((counter & 2) ? 1 : 0), v.Y - 1);
        const int cz = clampi(base[2] + ((counter & 4) ? 1 : 0), v.Zg - 1);
        if (GRAD) {
          float g[3];
          gradient_at(v, gc, cx, cy, cz, g);
          if (ORIENTED) rotate_gradient(a.geom, g);
          gd[0] += overlap * (double)g[0];
          gd[1] += overlap * (double)g[1];
          gd[2] += overlap * (double)g[2];
        } else {
          value += overlap * (double)v.at(cx, cy, cz);
        }
        total += overlap;
      }
      if (total == 1.0) break;
    }
    return value;
  }
  // normal = gradient interpolated at the vertex, normalised (txx:351-352); false: zero gradient
  __device__ __forceinline__ bool unit_normal(const float vertex[3], float normal[3]) const {
    double gd[3];
    sample<true>(vertex, gd);
    double sq = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      normal[k] = (float)gd[k];
      const double c = (double)normal[k];
      sq += c * c;
    }
    const double norm = sqrt(sq);
    if (norm == 0.0) return false;
#pragma unroll
    for (int k = 0; k < 3; ++k) normal[k] = (float)((double)normal[k] / norm);
    return true;
  }
  __device__ __forceinline__ double value_at(const float pt[3]) const { return sample<false>(pt, nullptr); }
};

template <typename T, bool ORIENTED>
__global__ void __launch_bounds__(128) k_project_alt(const ProjArgs a, int method) {
  const Sampler<T, ORIENTED> S(a);
  size_t n_points = a.n_points;
  float* const points = a.points + (a.info && !a.include_ghost ? 3 * (size_t)__ldg(a.info + kInfoGhostV) : 0);
  if (a.info) {
    if (!emission_fits(a.info)) return;
    const size_t ghost = (size_t)__ldg(a.info + kInfoGhostV);
    const size_t all = ghost + (size_t)__ldg(a.info + kInfoPoints);
    n_points = a.include_ghost ? all : all - ghost;
  }
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_points; i += (size_t)gridDim.x * blockDim.x) {
    float vertex[3] = {points[3 * i], points[3 * i + 1], points[3 * i + 2]};
    if (method == kProjectAdvanced) {
      // txx:340-397
      bool done = false;
      double step = a.step0;
      unsigned numberOfSteps = 0, swaps = 0;
      int previousi = -1;
      while (!done) {
        float normal[3];
        if (!S.unit_normal(vertex, normal)) break;
        float t0[3], t1[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          t0[k] = (float)((double)vertex[k] + ((double)normal[k] * +1.0) * step);
          t1[k] = (float)((double)vertex[k] + ((double)normal[k] * -1.0) * step);
        }
        step *= a.relax;
        const double d0 = fabs(S.value_at(t0) - a.iso), d1 = fabs(S.value_at(t1) - a.iso);
        const int side = (d0 <= d1) ? 0 : 1;
        if (previousi < 0) previousi = side;
        swaps += (unsigned)(previousi != side);
#pragma unroll
        for (int k = 0; k < 3; ++k) vertex[k] = side ? t1[k] : t0[k];
        done |= (side ? d1 : d0) < a.thr;
        if (done) break;
        done |= numberOfSteps++ > a.max_steps;
        if (done) break;
        done |= swaps >= 5;
      }
    } else {
      // txx:398-438
      float normal[3];
      if (S.unit_normal(vertex, normal)) {
        float best[3] = {vertex[0], vertex[1], vertex[2]};
        double bestMetric = 10000;
        const unsigned half = a.max_steps / 2;
        for (int s = 0; s < 2; ++s) {
          const double sign = s == 0 ? -1.0 : 1.0;
          for (unsigned j = 1; j < half; ++j) {
            const double d = (double)j / ((double)a.max_steps / 2.0);
            float temp[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) temp[k] = (float)((double)vertex[k] + (((double)normal[k] * sign) * a.step0) * d);
            const double metric = fabs(S.value_at(temp) - a.iso);
            if (metric < bestMetric) {
              bestMetric = metric;
              best[0] = temp[0]; best[1] = temp[1]; best[2] = temp[2];
            }
          }
        }
        vertex[0] = best[0]; vertex[1] = best[1]; vertex[2] = best[2];
      }
    }
    points[3 * i] = vertex[0];
    points[3 * i + 1] = vertex[1];
    points[3 * i + 2] = vertex[2];
  }
}

}  // namespace cbr
