/* cuberille_c.h — C-ABI of libcuberille_cuda.so (B200 / sm_100a).
 *
 * This is the drop-in boundary for the hot path of
 * itk::CuberilleImageToMeshFilter::GenerateData()
 *   (reference: Source/itkCuberilleImageToMeshFilter.txx:59-216 and the helpers
 *    it calls, txx:219-498).
 * The host side (include/itkCuberilleImageToMeshFilter.h, C++) keeps the
 * filter's ITK API and calls only the functions below; nothing here exposes a
 * CUDA, torch or C++ type.  Plain pointers and sizes, int status codes, no
 * exceptions cross this boundary, no global state: one handle per host
 * thread / stream.
 *
 * Every entry point names the reference interface it replaces (file:line under
 * the reference tree; "h" = Source/itkCuberilleImageToMeshFilter.h,
 * "txx" = Source/itkCuberilleImageToMeshFilter.txx).
 *
 * There is NO CPU fallback behind this interface: if no CUDA device is usable
 * cub_create() fails with CUB_ERR_CUDA and nothing else can be called.
 */
#ifndef CUBERILLE_C_H
#define CUBERILLE_C_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CUB_ABI_VERSION 3

/* ---- status codes ------------------------------------------------------- */
enum {
  CUB_OK = 0,
  CUB_ERR_INVALID = 1,    /* bad argument / call order                        */
  CUB_ERR_CUDA = 2,       /* a CUDA runtime call failed (see cub_last_error)  */
  CUB_ERR_NOMEM = 3,      /* device or pinned-host allocation failed          */
  CUB_ERR_OVERFLOW = 4,   /* ids do not fit the requested id width            */
  CUB_ERR_UNSUPPORTED = 5 /* e.g. an image too wide for one handle, no NCCL    */
};

/* ---- pixel types: TInputImage::PixelType (h:150) ------------------------ */
enum {
  CUB_U8 = 0, CUB_I8 = 1, CUB_U16 = 2, CUB_I16 = 3,
  CUB_U32 = 4, CUB_I32 = 5, CUB_F32 = 6, CUB_F64 = 7,
  CUB_I64 = 8, CUB_U64 = 9   /* label maps of ITK's IdentifierType and numpy's default int;
                                an older library of the same ABI version answers
                                CUB_ERR_INVALID "unknown dtype" */
};

/* ---- where a caller buffer lives ---------------------------------------- */
enum {
  CUB_MEM_HOST = 0,        /* pageable or pinned host memory                  */
  CUB_MEM_DEVICE = 1       /* device memory on the handle's device            */
};

/* ---- ProjectVertexToIsoSurface variants (h:22-23) ---------------------------- */
enum { CUB_PROJECT_DEFAULT = 0, CUB_PROJECT_ADVANCED = 1, CUB_PROJECT_LINESEARCH = 2 };

/* ---- vertex numbering ----------------------------------------------------- */
enum { CUB_ORDER_REFERENCE = 0, CUB_ORDER_RASTER = 1 };

typedef struct cub_handle_s *cub_handle;

/* Filter parameters: the member variables of the reference filter
 * (h:326-335) with the constructor defaults of txx:31-41.                    */
typedef struct cub_params {
  double   iso_value;           /* m_IsoSurfaceValue (h:180-181); must be exactly
                                   representable in the pixel type              */
  int32_t  generate_triangles;  /* m_GenerateTriangleFaces (h:193-195)          */
  int32_t  project_vertices;    /* m_ProjectVerticesToIsoSurface (h:199-201)    */
  int32_t  save_pixel_as_cell_data; /* SavePixelAsCellData (north-star knob; the
                                   reference only has commented stubs txx:314,321,330) */
  int32_t  vertex_order;        /* CUB_ORDER_REFERENCE (default): vertex ids in the reference's
                                   first-touch creation order (txx:179-194);
                                   CUB_ORDER_RASTER: ids in raster order of the lattice corners -
                                   same points and connectivity up to that renumbering, about a
                                   third less work (no ownership sweep, no corner->id map)      */
  double   surface_distance_threshold; /* h:209-210, default 0.5                */
  double   step_length;         /* h:215-216; < 0 means auto = max spacing*0.25
                                   (txx:82-85)                                  */
  double   step_relaxation;     /* h:222-223, default 0.95                      */
  uint32_t max_steps;           /* h:227-228, default 50                        */
  uint32_t image_border_faces;  /* 0 (default): the reference's behaviour, a neighbour outside
                                 * the image reads the clamped pixel, so the image border never
                                 * gets a face (open mesh there, h:55-57).  1: a neighbour outside
                                 * the image counts as outside the surface, i.e. the mesh of the
                                 * image padded with one outside layer: always closed (the
                                 * "handle voxels on the edge of the image" TODO, txx:133)       */
  int32_t  projection_method;   /* CUB_PROJECT_DEFAULT: the branch the reference compiles (txx:440-474).
                                 * CUB_PROJECT_ADVANCED / CUB_PROJECT_LINESEARCH: its compile-time alternates
                                 * USE_ADVANCED_PROJECTION (txx:340-397) and USE_LINESEARCH_PROJECTION
                                 * (txx:398-438), h:22-23 - off in the reference, offered here at run time     */
  int32_t  reserved;            /* must be 0                                                                  */
} cub_params;

/* Fills *p with the constructor defaults of txx:31-41
 * (iso 1, triangles on, projection on, thr 0.5, step -1, relax 0.95, 50).     */
void cub_default_params(cub_params *p);

/* Replaces CuberilleImageToMeshFilter::New() (h:121) as far as device state
 * goes.  `device` is a CUDA ordinal; `stream` is a cudaStream_t cast to void*
 * (NULL = the handle creates and owns a non-blocking stream).  All work of the
 * handle is ordered on that stream.                                           */
int cub_create(int device, void *stream, cub_handle *out);

/* Replaces ~CuberilleImageToMeshFilter() (txx:43-48).                          */
int cub_destroy(cub_handle h);

/* Last error text of this handle (never NULL).  Replaces the
 * itk::ExceptionObject description the driver prints (Testing/CuberilleTest01.cxx:207-212). */
const char *cub_last_error(cub_handle h);

/* Replaces SetInput(const InputImageType*) (h:184, txx:53-56) plus the image
 * geometry GenerateData reads (txx:71-79, 266-270).
 *   data      : x-fastest voxel buffer of dims[0]*dims[1]*dims[2] pixels
 *   mem_kind  : CUB_MEM_HOST -> copied to the device on the handle's stream;
 *               CUB_MEM_DEVICE -> borrowed (must stay valid until the next
 *               cub_set_volume / cub_destroy), no copy; the pointer must be
 *               aligned to the pixel size (else CUB_ERR_INVALID).  Any such
 *               offset is accepted: the kernels that need a 4- or 16-byte
 *               aligned buffer give way to others when it is not.
 *   direction : row-major 3x3 direction cosines (itk::ImageBase::GetDirection), or
 *               NULL = identity.  The identity is the non-oriented image every test
 *               of the reference has.  Any other (non-singular) matrix gives the
 *               oriented-image semantics of ITK: TransformIndexToPhysicalPoint with
 *               M = direction*diag(spacing) into the float point (txx:266), the
 *               continuous index through M^-1, gradients rotated into physical
 *               space (GradientImageFilter's UseImageDirection); the reference's
 *               half-spacing shift stays axis-aligned in physical space, exactly as
 *               written at txx:268-270.
 * The volume may be a z-slab of a larger image, see cub_set_slab.              */
int cub_set_volume(cub_handle h, const void *data, int dtype, const uint64_t dims[3],
                   const double spacing[3], const double origin[3],
                   const double direction[9], int mem_kind);

/* Image index of the buffer's first voxel (itk::ImageRegion::GetIndex of the
 * buffered region; every test of the reference has 0).  The points are
 * TransformIndexToPhysicalPoint(index + region index) (txx:266) and the
 * interpolators' continuous indices are image indices.  Call after
 * cub_set_volume (which resets it to 0).  For a z-slab it is the index of the
 * WHOLE image's first voxel.                                                   */
int cub_set_region_index(cub_handle h, const int64_t index[3]);

/* Inside-range mode (no counterpart in the reference): with enable != 0 a
 * voxel is inside when !(v < lower) && !(upper < v), compared in the pixel
 * type, instead of !(v < iso_value).  A label k of a label map is the range
 * [k, k]; a range of several labels meshes the surface of their union, and with
 * save_pixel_as_cell_data every cell carries the value of the voxel that made
 * it.  A NaN pixel is inside, as in iso mode.  [iso, type maximum] (or +inf)
 * gives the mask of iso mode with that iso.  Both bounds must be pixel values
 * of the current volume's type (the rule cub_count applies to iso_value), not
 * NaN, and lower <= upper; else CUB_ERR_INVALID.  While the mode is on,
 * cub_params.iso_value is ignored, and cub_count / cub_count_async with
 * project_vertices != 0 and cub_debug_project_points return CUB_ERR_INVALID:
 * the projection needs an iso-surface.  enable == 0 returns to iso mode.
 * Call after cub_set_volume, which turns the mode off.                         */
int cub_set_inside_range(cub_handle h, int enable, double lower, double upper);

/* z-slab decomposition (no counterpart in the reference: GenerateData is a
 * single raster loop txx:136-206; concatenating z-slabs preserves its order).
 *   image_nz      : z size of the WHOLE image
 *   local_z0      : global z index of the local buffer's slice 0
 *   own_z0/own_z1 : global half-open z range whose voxels this handle emits
 * The local buffer must contain slices [own_z0-2, own_z1+1) clipped to the
 * image (2 slices below: one for face/corner classification, one so that the
 * first-touch owner of a shared corner is computed identically on both sides;
 * 1 slice above for the +z faces; more is harmless);
 * with projection the halo must cover the travel of a vertex, up to
 * step_length / (1 - step_relaxation) = 5 x the largest spacing by default, i.e.
 * >= 8 slices for isotropic voxels and more when the z spacing is the small one.  Default
 * (never called): the buffer is the whole image.                               */
int cub_set_slab(cub_handle h, uint64_t image_nz, uint64_t local_z0,
                 uint64_t own_z0, uint64_t own_z1);

/* Label maps (no counterpart in the reference).
 *
 * cub_label_bounds: one pass over the current volume on the device that finds,
 * for every label k of the window [first_label, first_label + n_labels), its
 * voxel count and bounding box.  out is a host buffer of n_labels x 8 values:
 * {count, xmin, ymin, zmin, xmax, ymax, zmax, 0} of label first_label + i at
 * out[8 * i], in buffer indices, maxima inclusive; a label with count 0 has all
 * six bounds 0.  Pixels outside the window are ignored.  Integer pixel types
 * only (CUB_ERR_UNSUPPORTED for float32 / float64); 1 <= n_labels <= 65536 and
 * the window must lie inside the pixel type's range, else CUB_ERR_INVALID, as
 * while a region of interest or a z-slab is set.  Labels are compared in the
 * pixel type's width, so label 2^32 + 5 of an int64 map is not label 5.  For
 * uint64 the window must lie in [0, 2^63 - 1], what first_label can express;
 * pixels above it are ignored like any other pixel outside the window.
 * Synchronises.                                                                */
int cub_label_bounds(cub_handle h, int64_t first_label, uint32_t n_labels, uint64_t *out);

/* Region of interest: from now on cub_count / cub_count_async (and
 * cub_debug_bitmask, cub_download_volume, cub_debug_project_points) work on the
 * box [lo, lo + size) of the current volume.  The result is exactly that of
 * cub_set_volume on a copy of the box followed by cub_set_region_index(region
 * index + lo), in every mode: interpolation and gradients of the projection
 * clamp at the box, as for an image cut out with ITK's ExtractImageFilter.  A
 * box of whole rows and slices (full x and y extent) is used in place; any
 * other box is copied, on the handle's stream, into a buffer the handle owns.
 * lo == NULL returns to the whole volume.  An empty box, one that leaves the
 * volume, or a call before cub_set_volume returns CUB_ERR_INVALID; combining
 * the box with cub_set_slab, in either order, CUB_ERR_UNSUPPORTED.
 * cub_set_volume and cub_generate_volume clear the box; cub_set_region_index
 * stays the index of the whole buffer, and the box's lo adds to it.             */
int cub_set_region_of_interest(cub_handle h, const uint64_t lo[3], const uint64_t size[3]);

/* Every label of a label map in one call: labels[i] is meshed as the inside
 * range [k, k] and the meshes are concatenated in the given order, point ids of
 * label i offset by the points of labels 0..i-1.  point_offsets and
 * cell_offsets (n_labels + 1 entries each) receive the start of every label's
 * part and, last, the totals.  The result is read with cub_fetch /
 * cub_device_buffers like any other run; its cell data, when asked for, is the
 * label.  Each part is bit-identical to cub_set_inside_range(k, k) + cub_count
 * + cub_set_id_base(point_offsets[i], cell_offsets[i]) + cub_emit on the whole
 * volume, in every emit mode, because each label is meshed in its bounding box
 * grown by one voxel and clipped to the image (DESIGN.md §2): one
 * cub_label_bounds pass finds the boxes, and a label without voxels gives an
 * empty part and launches nothing.  The labels must be pixel values of the
 * volume's integer type (the rule of cub_set_inside_range), each given once,
 * else CUB_ERR_INVALID.  A label is a double, so of int64 / uint64 maps only
 * the labels a double holds exactly can be given: every one up to 2^53 in
 * magnitude, and beyond that the even ones, then multiples of 4, ...; and of
 * uint64 maps only labels up to 2^63 - 1, the windows of cub_label_bounds.
 * project_vertices != 0 (a label has no iso-surface), a set region of
 * interest and a z-slab return CUB_ERR_INVALID too.  A float volume returns
 * CUB_ERR_UNSUPPORTED.  The handle's own inside-range setting is left as it
 * was.  cub_last_warning names the labels whose mesh has an empty interior
 * slice.  Synchronises once per label.                                         */
int cub_run_labels(cub_handle h, const cub_params *p, const double *labels, uint64_t n_labels,
                   int id_bytes, uint64_t *point_offsets, uint64_t *cell_offsets);

/* Phase 1 of GenerateData (txx:136-173 without the emission): classify every
 * voxel against iso, find faces and first-touch corner owners, scan.
 * Returns the number of points / quads this handle's own z-range produces.
 * (n_cells of the final mesh is n_quads, or 2*n_quads with triangles.)         */
int cub_count(cub_handle h, const cub_params *p, uint64_t *n_points, uint64_t *n_quads);

/* Slices of halo a z-slab needs below / above its own range for these parameters
 * and the image's geometry (spacing and direction as given to cub_set_volume;
 * null: 1 and the identity): 2 / 1 without projection; with projection the reach
 * of a vertex (the geometric sum of its <= max_steps + 2 moves, txx:464-469, in
 * slices: over spacing[2], or for an oriented image times the 1-norm of the z row
 * of (D * diag(spacing))^-1) plus the interpolation and central-difference
 * footprints.  cub_count requires exactly this halo of a slab of an image with
 * the same geometry, and refuses a shorter buffer (a clamped read would silently
 * change the mesh).  CUB_ERR_INVALID for a spacing that is not positive and
 * finite, or a singular or non-finite direction.                               */
int cub_projection_halo_oriented(const cub_params *p, const double spacing[3], const double direction[9],
                                 uint64_t *below, uint64_t *above);

/* cub_projection_halo_oriented of a non-oriented image (identity direction).   */
int cub_projection_halo(const cub_params *p, const double spacing[3],
                        uint64_t *below, uint64_t *above);

/* Global id bases for z-slab runs: the exclusive scan over ranks of the
 * (n_points, n_cells) returned by cub_count.  Default 0, 0.  The bases live on
 * the device (the emission kernels read them there); this call queues the
 * update on the handle's stream.                                               */
int cub_set_id_base(cub_handle h, uint64_t point_id_base, uint64_t cell_id_base);

/* Optional early half of cub_emit: queues the vertex stage (vertex creation
 * order + AddVertex positions, txx:179-194, 257-276) of the current count on
 * the handle's stream.  It needs the counts but not the id base, so a rank of a
 * multi-GPU run calls it right after cub_count and exchanges its counts with
 * the other ranks while it runs; cub_emit then skips the stage.  No effect if
 * already done (or while cub_enable_timing is on).                            */
int cub_emit_vertices(cub_handle h);

/* Phase 2 of GenerateData: AddVertex (txx:257-276), ProjectVertexToIsoSurface
 * (txx:440-474) with ComputeGradientImage (txx:479-498) evaluated on the fly,
 * AddQuadFace (txx:279-332).  Results stay in device buffers owned by the
 * handle until the next cub_count.  id_bytes = 4 or 8 (PointIdentifier is
 * unsigned long in the reference; 4 is the fast path and fails with
 * CUB_ERR_OVERFLOW when an id would not fit).                                  */
int cub_emit(cub_handle h, int id_bytes);

/* cub_count + cub_emit with id bases 0: the whole of GenerateData().
 * n_cells counts final cells (triangles when generate_triangles).              */
int cub_run(cub_handle h, const cub_params *p, int id_bytes,
            uint64_t *n_points, uint64_t *n_cells);

/* The same two phases WITHOUT a host round trip in between.  The counts stay in
 * device memory, where the emission kernels (and the multi-GPU count exchange,
 * cub_comm_exchange_counts) read them; nothing blocks the calling thread until
 * cub_finish.  cub_emit_async writes into the result buffers the handle already
 * has (they only grow: the first run of a handle sizes them through one
 * synchronisation); should a later run produce more than they hold, the kernels
 * stop at the end of the buffers and cub_finish redoes the emission with larger
 * ones - the caller never sees a truncated mesh.
 *   cub_count_async  : queues phase 1
 *   cub_device_counts: device pointer to {n_points, n_quads} of the own range
 *   cub_emit_async   : queues phase 2
 *   cub_finish       : synchronises, returns the counts, validates the emission
 * cub_fetch / cub_device_buffers call cub_finish themselves when needed.       */
int cub_count_async(cub_handle h, const cub_params *p);
int cub_device_counts(cub_handle h, const uint64_t **counts);
int cub_emit_async(cub_handle h, int id_bytes);
int cub_finish(cub_handle h, uint64_t *n_points, uint64_t *n_cells);

/* Non-fatal remark about the last count (never NULL, "" if none).  Currently:
 * an empty voxel slice between occupied ones, where the reference's lookup-plane
 * rotation (txx:155-161, it only advances on inside voxels) merges vertices of
 * different corner planes and this library does not (SURVEY section 8a row 3).   */
const char *cub_last_warning(cub_handle h);

/* Copies the mesh out: what mesh->GetPoints()->InsertElement (txx:275) and
 * mesh->SetCell (txx:313,320,329) received, in the reference's id order.
 *   points    : n_points * 3 floats (itk::Mesh default Point<float,3>), or NULL
 *   cells     : n_cells * (3|4) ids of id_bytes each, or NULL
 *   cell_data : n_cells pixels of the input dtype (only when
 *               save_pixel_as_cell_data), or NULL
 *   mem_kind  : where those three buffers live                                 */
int cub_fetch(cub_handle h, float *points, void *cells, void *cell_data, int mem_kind);

/* cub_fetch without the final synchronisation: the copies are only ordered on the
 * handle's stream; call cub_synchronize before reading the destination buffers.
 * Lets a caller that streams z-slabs through several handles overlap the
 * device->host copy of one slab with the host->device copy of the next.        */
int cub_fetch_async(cub_handle h, float *points, void *cells, void *cell_data, int mem_kind);

/* Blocks until everything issued on the handle's stream has finished.          */
int cub_synchronize(cub_handle h);

/* Zero-copy access to the result buffers on the device (valid until the next
 * cub_count on this handle).  Any out pointer may be NULL.                     */
int cub_device_buffers(cub_handle h, const float **points, const void **cells,
                       const void **cell_data, uint64_t *n_points, uint64_t *n_cells,
                       int *verts_per_cell, int *id_bytes);

/* ---- multi-GPU: z-slabs over NCCL (SURVEY section 8e) -----------------------
 * No counterpart in the reference (GenerateData is one raster loop on one core,
 * txx:136-206).  One handle per GPU, each with its slab (cub_set_slab); a
 * communicator binds the handle to its rank.  NCCL is loaded at run time
 * (libnccl.so.2), single-GPU users do not need it.
 *   cub_comm_unique_id      : ncclGetUniqueId (rank 0; the host distributes the 128 bytes)
 *   cub_comm_create         : ncclCommInitRank on the handle's device (collective)
 *   cub_comm_exchange_counts: after cub_count / cub_count_async.  All-gather of the
 *                             (points, quads) of every rank's own range, device to
 *                             device on a side stream; the exclusive prefix becomes
 *                             the handle's id bases (what cub_set_id_base would set).
 *                             Nothing blocks the host: cub_emit(_async) orders its
 *                             face kernel after the exchange by itself.
 *   cub_comm_counts         : the gathered counts on the host, 2 * world values
 *                             (points, quads per rank); synchronises the exchange
 *   cub_comm_gather_mesh    : "allgatherv" over NVLink: every rank receives the whole
 *                             mesh into DEVICE buffers sized for the totals (points:
 *                             3 floats each; cells: verts_per_cell ids of id_bytes;
 *                             cell_data: pixels), each rank's part at its id base -
 *                             the concatenation IS the single-GPU mesh.  Queued on the
 *                             handle's stream (cub_synchronize to wait).  Any buffer
 *                             may be NULL on ALL ranks alike.                         */
typedef struct cub_comm_s *cub_comm;
int cub_comm_unique_id(unsigned char id[128]);
int cub_comm_create(cub_handle h, const unsigned char id[128], int world, int rank, cub_comm *out);
int cub_comm_destroy(cub_comm c);
int cub_comm_exchange_counts(cub_comm c);
int cub_comm_counts(cub_comm c, uint64_t *counts);
int cub_comm_gather_mesh(cub_comm c, float *points, void *cells, void *cell_data);

/* Device memory for hosts that do not link the CUDA runtime themselves (the
 * destination buffers of cub_comm_gather_mesh, CUB_MEM_DEVICE volumes):
 * cudaMalloc / cudaFree / a blocking copy (kinds: CUB_MEM_*) on the handle's
 * device and stream.                                                           */
int cub_device_alloc(cub_handle h, uint64_t bytes, void **out);
int cub_device_free(cub_handle h, void *p);
int cub_device_copy(cub_handle h, void *dst, const void *src, uint64_t bytes, int dst_kind, int src_kind);

/* Page-lock / unlock a caller's host buffer (cudaHostRegister / cudaHostUnregister):
 * an itk::Image buffer is pageable, and host <-> device copies of pageable memory
 * run at a fraction of the PCIe rate.                                          */
int cub_host_register(cub_handle h, void *p, uint64_t bytes);
int cub_host_unregister(cub_handle h, void *p);
/* Page-locked host memory (cudaHostAlloc / cudaFreeHost), e.g. staging buffers that
 * cub_fetch fills at the full PCIe rate (the C++ adapter keeps a grow-only pair).  */
int cub_host_alloc(cub_handle h, uint64_t bytes, void **out);
int cub_host_free(cub_handle h, void *p);

/* Diagnostics for parity tests of the individual kernels.
 * cub_debug_bitmask: the 1-bit/voxel inside mask of the local buffer after
 * cub_count; words_per_row receives the row stride in 32-bit words; `out` (host)
 * must hold dims[2]*dims[1]*words_per_row words (call with out=NULL to query). */
int cub_debug_bitmask(cub_handle h, uint32_t *out, uint64_t *words_per_row);

/* Projects caller-supplied points in place with the current volume and params
 * (the K4 kernel alone; ProjectVertexToIsoSurface txx:440-474).  Host buffer.  */
int cub_debug_project_points(cub_handle h, const cub_params *p, float *points_xyz,
                             uint64_t n_points);

/* Device-side synthetic volume generators (bench only; SURVEY §8d configs 3-5).
 * Writes a float32 volume of dims into device memory owned by the handle and
 * makes it the current volume (as cub_set_volume with CUB_MEM_DEVICE would).
 * The field is evaluated at GLOBAL voxel coordinates (x, y, local z + z_offset)
 * of an image of size image_dims, so slabs of one image agree bit for bit.     */
enum { CUB_GEN_GYROID = 0, CUB_GEN_MARSCHNER_LOBB = 1, CUB_GEN_BLOBS = 2 };
int cub_generate_volume(cub_handle h, int kind, const uint64_t dims[3],
                        const uint64_t image_dims[3], uint64_t z_offset,
                        double param0, double param1, uint64_t seed);

/* Copies the current volume to a host buffer (parity runs feed the same bytes
 * to the CPU oracle).  `bytes` must equal the volume size in bytes.            */
int cub_download_volume(cub_handle h, void *out, uint64_t bytes);

/* Per-kernel device times (ms, CUDA events on the handle's stream) of the last
 * cub_count/cub_emit: [0]=classify [1]=count sweep + scan [2]=emit (assign sweep,
 * vertices, faces) [3]=project [4]=triangle split [5]=total count phase
 * [6]=total emit phase [7]=the look-back scan alone.  Only filled
 * when timing was enabled with cub_enable_timing(h, 1) (adds event records and
 * one synchronize per phase; off by default).                                  */
int cub_enable_timing(cub_handle h, int on);
int cub_get_timings(cub_handle h, float ms[8]);

/* Number of kernel launches issued by this handle so far.                      */
uint64_t cub_launch_count(cub_handle h);

/* 1 if the last cub_count ran classification + ownership sweep as the one fused
 * kernel (k_classify_sweep; [0] of cub_get_timings is then that kernel and [1]
 * the scan alone), 0 if it ran them as two kernels.  Diagnostic only.           */
int cub_count_was_fused(cub_handle h);

int cub_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CUBERILLE_C_H */
