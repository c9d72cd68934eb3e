// oracle64.cpp — the CPU oracle (oracle/cuberille_oracle.cpp) for int64 and uint64 pixels.  TEST INFRASTRUCTURE.
//
// The oracle's algorithm is a template over the pixel type; its C entry points dispatch the eight types of the first
// pixel-code set.  This translation unit compiles the oracle unchanged and adds entry points for pixel codes 8 (int64)
// and 9 (uint64), with the signatures of orc_cuberille / orc_classify / orc_project_points / orc_sample.  Like the
// library, the 64-bit instantiations convert a pixel with (float)v for the gradient and (double)v for interpolation,
// each a single correctly rounded conversion (tests/oracle64.py builds it; tests/test_int64_oracle.py checks it).
#include "../oracle/cuberille_oracle.cpp"

#define ORC64_DISPATCH(dtype, CALL)                      \
  switch (dtype) {                                       \
    case 8: { typedef int64_t  T; CALL; } return 0;      \
    case 9: { typedef uint64_t T; CALL; } return 0;      \
    default: return 1;                                   \
  }

extern "C" {

orc_mesh* orc64_cuberille(const void* data, int dtype, const uint64_t dims[3], const double spacing[3],
                          const double origin[3], const orc_params* P) {
  const Geometry g = make_geometry(dims, spacing, origin, P->region_index, P->direction);
  orc_mesh* m = nullptr;
  auto run = [&]() -> int { ORC64_DISPATCH(dtype, m = run_typed<T>(data, g, *P)); };
  run();
  return m;
}

int orc64_classify(const void* data, int dtype, const uint64_t dims[3], double iso, uint32_t* out, uint64_t words_per_row) {
  const Geometry g = make_geometry(dims, nullptr, nullptr);
  if (words_per_row * 32 < dims[0]) return 1;
  ORC64_DISPATCH(dtype, classify_typed<T>(data, g, iso, out, words_per_row));
}

int orc64_project_points(const void* data, int dtype, const uint64_t dims[3], const double spacing[3],
                         const double origin[3], const orc_params* P, float* pts, uint64_t n) {
  const Geometry g = make_geometry(dims, spacing, origin, P->region_index, P->direction);
  ORC64_DISPATCH(dtype, project_typed<T>(data, g, *P, pts, n));
}

int orc64_sample(const void* data, int dtype, const uint64_t dims[3], const double spacing[3],
                 const double origin[3], const double* pts, uint64_t n, double* val, double* grad) {
  const Geometry g = make_geometry(dims, spacing, origin);
  ORC64_DISPATCH(dtype, sample_typed<T>(data, g, pts, n, val, grad));
}

}  // extern "C"
