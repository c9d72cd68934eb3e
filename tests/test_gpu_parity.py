"""GPU: the CUDA path, called through the C-ABI, against the CPU oracle on the same inputs.
Bar: bit-exact connectivity, vertex count, vertex order and positions (projected ones included:
the kernel reproduces the oracle's arithmetic, which is tighter than the 1e-5 x spacing of the spec)."""
import numpy as np
import pytest

from util import KAT, KAT_ARGS, assert_mesh_equal, assert_mesh_equal_up_to_vertex_order, gyroid, oracle, pkg, random_volume, read_fixture, run_filter, smooth_volume

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("row", KAT, ids=[r[0] for r in KAT])
def test_reference_known_answers_on_gpu(row):
    """the reference's 19 CTest rows (Testing/CMakeLists.txt:10-331) through the filter interface"""
    name, fixture, iso, exp_points, exp_cells, tri, proj, max_steps = row
    img = read_fixture(fixture)
    mesh = run_filter(img, iso, triangles=tri, project=proj, max_steps=max_steps, **KAT_ARGS)
    assert mesh.GetNumberOfPoints() == exp_points
    assert mesh.GetNumberOfCells() == exp_cells
    ref = oracle().cuberille(img.data, iso, triangles=tri, project=proj, max_steps=max_steps, **KAT_ARGS)
    assert_mesh_equal(mesh, ref, name)


@pytest.mark.parametrize("dtype", [np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.float32, np.float64])
# the last five shapes have whole-warp-load rows: 1- and 2-byte pixels take the packed kernel there (one, several
# and partial 32-word tasks per row)
@pytest.mark.parametrize("shape", [(7, 9, 33), (5, 6, 1), (3, 1, 70), (1, 8, 8), (6, 5, 32), (4, 4, 31), (9, 13, 131),
                                   (3, 5, 128), (2, 3, 64), (2, 2, 1152), (1, 2, 192), (2, 1, 2176)])
def test_bitmask_matches_oracle(dtype, shape):
    """K1: inside == !(v < iso) for every pixel type and ragged row lengths"""
    P, O = pkg(), oracle()
    vol, iso = random_volume(shape, dtype, seed=sum(shape))
    h = P.capi.Handle(0)
    h.set_volume(vol)
    p = P.capi.default_params()
    p.iso_value = float(iso)
    h.count(p)
    got = h.bitmask()
    wpr = got.shape[2]
    ref = O.classify(vol, iso, wpr)
    nx = shape[2]
    valid = np.zeros(wpr * 32, bool)
    valid[:nx] = True
    mask = np.packbits(valid.reshape(-1, 32)[:, ::-1], axis=1).view(">u4").astype(np.uint32).reshape(-1)
    assert np.array_equal(got & mask, ref & mask)
    # padding bits of the last valid word replicate voxel X-1 (DESIGN.md §3)
    if nx % 32:
        w, b = (nx - 1) // 32, (nx - 1) % 32
        last = (got[:, :, w] >> b) & 1
        pad = got[:, :, w] >> (b + 1)
        assert np.array_equal(pad, np.where(last == 1, np.uint32(0xFFFFFFFF) >> (b + 1), 0))
    h.close()


@pytest.mark.parametrize("dtype", [np.uint8, np.int16, np.uint16, np.float32, np.float64, np.int32])
@pytest.mark.parametrize("shape,fill", [((6, 7, 8), 0.5), ((9, 33, 65), 0.5), ((17, 20, 97), 0.2), ((12, 40, 200), 0.8),
                                        ((2, 3, 4), 0.5), ((1, 1, 1), 0.5), ((3, 3, 1), 0.5), ((1, 5, 40), 0.5),
                                        # rows that end on a word boundary: the corner column x = X starts a corner word
                                        ((5, 6, 32), 0.5), ((24, 8, 96), 0.7), ((4, 9, 64), 0.3)])
def test_noise_volumes_ids_and_connectivity(dtype, shape, fill):
    """iid noise exercises every corner configuration of the first-touch rule, with inside voxels on
    the image border (no faces there); quads and fixed-split triangles, unprojected: exact positions"""
    O = oracle()
    vol, iso = random_volume(shape, dtype, seed=shape[2] * 7 + int(fill * 10), fill=fill)
    for tri in (False, True):
        ref = O.cuberille(vol, iso, triangles=tri, project=False, mode=O.CLOSED_FORM)
        mesh = run_filter(vol, iso, triangles=tri, project=False)
        assert_mesh_equal(mesh, ref, f"{dtype.__name__} {shape} tri={tri}")


@pytest.mark.parametrize("shape", [(3, 2, 40000), (2, 30000, 5), (3000, 6, 7), (2, 2, 65534)])
def test_extreme_aspect_ratios(shape):
    """long rows / many rows / many slices: the 16 + 15 bit corner records, the per-slice id index, 32-bit indices"""
    O = oracle()
    vol, iso = random_volume(shape, np.uint8, seed=shape[0] + shape[1], fill=0.5)
    for tri, order in ((False, 0), (True, 0)):
        ref = O.cuberille(vol, iso, triangles=tri, project=False, mode=O.CLOSED_FORM)
        assert_mesh_equal(run_filter(vol, iso, triangles=tri, project=False), ref, f"{shape} tri={tri}")


@pytest.mark.parametrize("dtype,shape,fill", [(np.uint8, (6, 7, 8), 0.5), (np.int16, (9, 33, 65), 0.5), (np.float32, (12, 40, 200), 0.8),
                                              (np.uint8, (1, 1, 1), 0.9), (np.uint8, (3, 4, 5), 1.0), (np.uint16, (5, 2, 130), 0.6)])
def test_image_border_faces(dtype, shape, fill):
    """opt-in closed mesh: the image padded with one outside layer (bit-exact against the oracle's flag)"""
    O = oracle()
    vol, iso = random_volume(shape, dtype, seed=shape[2] + 3, fill=fill)
    if fill >= 1.0:
        vol[...] = np.asarray(iso).astype(vol.dtype)  # everything inside: a closed box
    for tri, cd in ((False, False), (True, True)):
        ref = O.cuberille(vol, iso, triangles=tri, project=False, cell_data=cd, mode=O.CLOSED_FORM, border_faces=True)
        mesh = run_filter(vol, iso, triangles=tri, project=False, cell_data=cd, border_faces=True)
        assert_mesh_equal(mesh, ref, f"border faces {np.dtype(dtype).name} {shape} tri={tri}")
        assert ref.cells.shape[0] > 0


def test_image_border_faces_with_projection_slabs_and_raster_order():
    P, O = pkg(), oracle()
    vol = gyroid((41, 30, 50), 13.0, border=False)
    ref = O.cuberille(vol, 0.0, triangles=True, project=True, thr=0.01, mode=O.CLOSED_FORM, border_faces=True,
                      spacing=(0.5, 1.0, 2.0), origin=(3.0, -2.0, 7.0))
    mesh = run_filter(P.Image(vol, (0.5, 1.0, 2.0), (3.0, -2.0, 7.0)), 0.0, triangles=True, project=True, thr=0.01, border_faces=True)
    assert_mesh_equal(mesh, ref, "border faces + projection")
    img = P.Image(vol, (0.5, 1.0, 2.0), (3.0, -2.0, 7.0))
    ras = run_filter(img, 0.0, triangles=True, project=True, thr=0.01, border_faces=True, raster_order=True)
    ras0 = run_filter(img, 0.0, triangles=True, project=False, border_faces=True, raster_order=True)
    ref0 = O.cuberille(vol, 0.0, triangles=True, project=False, mode=O.CLOSED_FORM, border_faces=True,
                       spacing=(0.5, 1.0, 2.0), origin=(3.0, -2.0, 7.0))
    assert_mesh_equal_up_to_vertex_order(ras, ref, ras0, ref0, "border faces + raster order")
    # z-slabs
    nz = vol.shape[0]
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices, p.surface_distance_threshold, p.image_border_faces = 0.0, 1, 1, 0.01, 1
    pts, cells, pbase, cbase = [], [], 0, 0
    for z0, z1 in ((0, 13), (13, 14), (14, 30), (30, 41)):
        lo, hi = max(0, z0 - 9), min(nz, z1 + 9)
        h = P.capi.Handle(0)
        h.set_volume(vol[lo:hi], (0.5, 1.0, 2.0), (3.0, -2.0, 7.0))  # the IMAGE origin: the slab offset comes from set_slab
        h.set_slab(nz, lo, z0, z1)
        n_pts, n_quads = h.count(p)
        h.set_id_base(pbase, cbase)
        h.emit(4)
        a, b, _ = h.fetch()
        pts.append(a); cells.append(b)
        pbase += n_pts; cbase += 2 * n_quads
        h.close()
    assert_mesh_equal(P.Mesh(np.concatenate(pts), np.concatenate(cells)), ref, "border faces + slabs")


@pytest.mark.parametrize("tri,proj,border", [(False, False, False), (True, True, False), (True, True, True)])
def test_buffered_region_with_a_nonzero_index(tri, proj, border):
    """the buffer's first voxel has image index (4, -3, 10): points are TransformIndexToPhysicalPoint(index + that),
    the interpolators work with image indices (oracle flag region_index)"""
    P, O = pkg(), oracle()
    vol = gyroid((20, 18, 22), 9.0, border=False if border else -2.0)
    geo = dict(spacing=(0.7, 1.1, 1.9), origin=(1.5, -2.25, 3.0))
    ref = O.cuberille(vol, 0.0, triangles=tri, project=proj, thr=0.01, mode=O.CLOSED_FORM, border_faces=border,
                      region_index=(4, -3, 10), **geo)
    img = P.Image(vol, geo["spacing"], geo["origin"])
    img.region_index = (4, -3, 10)
    mesh = run_filter(img, 0.0, triangles=tri, project=proj, thr=0.01, border_faces=border)
    assert_mesh_equal(mesh, ref, "region index")
    # and it is not a no-op
    ref0 = O.cuberille(vol, 0.0, triangles=tri, project=proj, thr=0.01, mode=O.CLOSED_FORM, border_faces=border, **geo)
    assert not np.array_equal(ref0.points, ref.points)


def test_sizes_beyond_the_corner_record_are_refused():
    P = pkg()
    h = P.capi.Handle(0)
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices = 1.0, 0, 0
    for shape in [(1, 1, 65535), (1, 32767, 1)]:
        h.set_volume(np.zeros(shape, np.uint8))
        with pytest.raises(RuntimeError, match="not supported"):
            h.count(p)
    h.close()


def test_noise_volume_literal_lookup_agrees_too():
    O = oracle()
    vol, iso = random_volume((14, 21, 45), np.uint8, seed=3)
    assert (vol >= iso).reshape(vol.shape[0], -1).any(axis=1).all()  # no empty slice: the literal loop is well defined
    ref = O.cuberille(vol, iso, triangles=False, project=False, mode=O.LITERAL)
    assert_mesh_equal(run_filter(vol, iso, triangles=False, project=False), ref, "literal")


@pytest.mark.parametrize("dtype", [np.uint8, np.int16, np.float32])
@pytest.mark.parametrize("tri", [False, True])
def test_smooth_volumes_with_projection(dtype, tri):
    """K4 + K5: projection and the projected-diagonal triangle split, bit-exact against the oracle"""
    O = oracle()
    vol, iso = smooth_volume((40, 37, 70), dtype, seed=11)
    vol[0], vol[-1], vol[:, 0], vol[:, -1], vol[:, :, 0], vol[:, :, -1] = 0, 0, 0, 0, 0, 0
    args = dict(thr=0.05, step=0.3, relax=0.9, max_steps=60)
    ref = O.cuberille(vol, iso, triangles=tri, project=True, **args)
    mesh = run_filter(vol, iso, triangles=tri, project=True, **args)
    assert ref.points.shape[0] > 1000
    assert_mesh_equal(mesh, ref, f"{dtype.__name__} tri={tri}")


def test_anisotropic_spacing_and_origin():
    O = oracle()
    vol = gyroid((30, 26, 44), 11.0)
    sp, og = (0.5, 2.0, 1.25), (-3.0, 10.5, 0.75)
    for proj in (False, True):
        ref = O.cuberille(vol, 0.0, triangles=True, project=proj, thr=0.01, spacing=sp, origin=og)
        mesh = run_filter(vol, 0.0, triangles=True, project=proj, thr=0.01, spacing=sp, origin=og)
        assert_mesh_equal(mesh, ref, f"spacing proj={proj}")


def test_auto_step_length_and_default_parameters():
    """constructor defaults (txx:31-41) incl. step = max spacing * 0.25 (txx:82-85)"""
    O, P = oracle(), pkg()
    img = read_fixture("nucleon")
    f = P.CuberilleImageToMeshFilter.New()
    f.SetInput(img)
    f.SetIsoSurfaceValue(140)
    f.Update()
    assert f.GetProjectVertexStepLength() == 0.25  # sticky
    ref = O.cuberille(img.data, 140)
    assert ref.step_length_used == 0.25
    assert_mesh_equal(f.GetOutput(), ref, "defaults")


@pytest.mark.parametrize("tri,proj", [(False, False), (True, False), (True, True)])
def test_save_pixel_as_cell_data(tri, proj):
    O = oracle()
    vol, iso = smooth_volume((20, 22, 40), np.int16, seed=5)
    ref = O.cuberille(vol, iso, triangles=tri, project=proj, cell_data=True)
    mesh = run_filter(vol, iso, triangles=tri, project=proj, cell_data=True)
    assert_mesh_equal(mesh, ref, "celldata")
    assert mesh.cell_data.dtype == np.int16 and (mesh.cell_data >= iso).all()


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.float32, np.float64])
def test_cell_data_pixel_widths(dtype):
    """1-, 2-, 4- and 8-byte pixels through the typed cell-data stores (quads and fixed-split triangles)"""
    O = oracle()
    vol, iso = random_volume((9, 11, 70), dtype, seed=21, fill=0.45)
    for tri in (False, True):
        ref = O.cuberille(vol, iso, triangles=tri, project=False, cell_data=True, mode=O.CLOSED_FORM)
        mesh = run_filter(vol, iso, triangles=tri, project=False, cell_data=True)
        assert_mesh_equal(mesh, ref, f"celldata {np.dtype(dtype).name} tri={tri}")
        assert mesh.cell_data.dtype == np.dtype(dtype)


def test_64_bit_ids():
    O = oracle()
    vol, iso = random_volume((10, 12, 40), np.uint8, seed=9)
    ref = O.cuberille(vol, iso, triangles=True, project=True, mode=O.CLOSED_FORM)
    mesh = run_filter(vol, iso, triangles=True, project=True, id_bytes=8)
    assert mesh.cells.dtype == np.uint64
    assert_mesh_equal(mesh, ref, "u64")


def test_empty_and_full_volumes():
    for fillv in (0, 200):
        vol = np.full((6, 7, 40), fillv, np.uint8)
        mesh = run_filter(vol, 100, triangles=True, project=True)
        assert mesh.GetNumberOfPoints() == 0 and mesh.GetNumberOfCells() == 0


def test_nan_pixels():
    O = oracle()
    vol = np.zeros((6, 6, 36), np.float32)
    vol[2, 3, 33] = np.nan
    vol[3, 3, 0] = np.nan  # on the border: no face towards the outside
    ref = O.cuberille(vol, 0.5, triangles=False, project=False, mode=O.CLOSED_FORM)
    assert_mesh_equal(run_filter(vol, 0.5, triangles=False, project=False), ref, "nan")


@pytest.mark.parametrize("n_slabs", [2, 3, 5])
@pytest.mark.parametrize("tri,proj", [(False, False), (True, True)])
def test_z_slabs_concatenate_to_the_single_run(n_slabs, tri, proj):
    """§8e on one GPU: each slab runs with its halo, ids are offset by the exclusive scan of the slab
    counts, and the concatenation equals the whole-image mesh (shared boundary vertices belong to the
    first-touch owner, i.e. the lower slab)"""
    P, O = pkg(), oracle()
    vol = gyroid((41, 30, 50), 13.0)
    ref = O.cuberille(vol, 0.0, triangles=tri, project=proj, thr=0.01)
    nz = vol.shape[0]
    bounds = np.linspace(0, nz, n_slabs + 1).astype(int)
    halo = 9 if proj else 2
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices, p.surface_distance_threshold = 0.0, int(tri), int(proj), 0.01
    handles, counts = [], []
    for s in range(n_slabs):
        z0, z1 = int(bounds[s]), int(bounds[s + 1])
        lo, hi = max(0, z0 - halo), min(nz, z1 + halo)
        h = P.capi.Handle(0)
        h.set_volume(vol[lo:hi])
        h.set_slab(nz, lo, z0, z1)
        counts.append(h.count(p))
        if s % 2 == 0:
            h.emit_vertices()  # the vertex stage may be queued before the id base is known (and twice: no-op)
            h.emit_vertices()
        handles.append(h)
    pts, cells, pbase, cbase = [], [], 0, 0
    for h, (np_, nq) in zip(handles, counts):
        h.set_id_base(pbase, cbase)
        h.emit(4)
        a, b, _ = h.fetch()
        pts.append(a)
        cells.append(b)
        pbase += np_
        cbase += nq * (2 if tri else 1)
        h.close()
    mesh = P.Mesh(np.concatenate(pts), np.concatenate(cells))
    assert_mesh_equal(mesh, ref, f"{n_slabs} slabs")


def test_projection_kernel_alone_on_arbitrary_points():
    """K4 on points that are not lattice corners, including points outside the image (clamped reads)"""
    P, O = pkg(), oracle()
    img = read_fixture("neghip")
    rng = np.random.default_rng(0)
    pts = (rng.random((20000, 3)) * (np.array(img.data.shape[::-1]) + 4) - 2).astype(np.float32)
    h = P.capi.Handle(0)
    h.set_volume(img.data)
    p = P.capi.default_params()
    p.iso_value, p.surface_distance_threshold, p.step_length, p.max_steps = 55.0, 0.2, 0.24, 100
    got = h.project_points(p, pts)
    ref = O.project_points(img.data, 55, pts, thr=0.2, step=0.24, relax=0.95, max_steps=100)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    h.close()


def test_device_generated_gyroid_round_trip():
    """bench input path: generate on the device, download the bytes, feed the SAME bytes to the oracle"""
    P, O = pkg(), oracle()
    h = P.capi.Handle(0)
    h.generate(P.capi.GEN_GYROID, (96, 64, 48), p0=24.0)
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices = 0.0, 0, 0
    n_pts, n_cells = h.run(p)
    vol = h.download_volume()
    assert vol.shape == (48, 64, 96) and (vol[0] == -2).all() and (vol[:, :, 0] == -2).all()
    ref = O.cuberille(vol, 0.0, triangles=False, project=False)
    a, b, _ = h.fetch()
    assert_mesh_equal(P.Mesh(a, b), ref, "generated gyroid")
    assert n_pts == ref.points.shape[0] and n_cells == ref.cells.shape[0]
    h.close()


def test_filter_rerun_with_changed_parameters_and_inputs():
    """a filter instance is reused across Update() calls (buffers are recycled, results are not stale)"""
    O, P = oracle(), pkg()
    f = P.CuberilleImageToMeshFilter.New()
    for fixture, iso, tri in [("fuel", 15, True), ("neghip", 55, False), ("blob3", 200, True), ("fuel", 40, False)]:
        img = read_fixture(fixture)
        f.SetInput(img)
        f.SetIsoSurfaceValue(iso)
        f.SetGenerateTriangleFaces(tri)
        f.SetProjectVertexStepLength(0.24)
        f.Update()
        ref = O.cuberille(img.data, iso, triangles=tri, project=True, step=0.24)
        assert_mesh_equal(f.GetOutput(), ref, fixture)


@pytest.mark.parametrize("fixture,iso,tri,proj", [("fuel", 15, True, True), ("neghip", 55, False, False), ("nucleon", 140, True, False),
                                                  ("silicium", 85, False, True), ("blob3", 200, True, True)])
def test_raster_vertex_order_is_a_renumbering_of_the_reference_mesh(fixture, iso, tri, proj):
    """CUB_ORDER_RASTER: bit-exact connectivity, vertex count and positions after canonical ordering"""
    O = oracle()
    img = read_fixture(fixture)
    args = dict(max_steps=100, **KAT_ARGS)
    ref = O.cuberille(img.data, iso, triangles=tri, project=proj, **args)
    ref0 = O.cuberille(img.data, iso, triangles=tri, project=False)
    mesh = run_filter(img, iso, triangles=tri, project=proj, raster_order=True, **args)
    mesh0 = run_filter(img, iso, triangles=tri, project=False, raster_order=True)
    assert_mesh_equal_up_to_vertex_order(mesh, ref, mesh0, ref0, fixture)


@pytest.mark.parametrize("dtype,shape", [(np.uint8, (9, 33, 65)), (np.float32, (6, 7, 8)), (np.int16, (12, 40, 200)), (np.uint8, (1, 1, 1))])
def test_raster_vertex_order_on_noise(dtype, shape):
    O = oracle()
    vol, iso = random_volume(shape, dtype, seed=17)
    ref = O.cuberille(vol, iso, triangles=False, project=False, mode=O.CLOSED_FORM, cell_data=True)
    mesh = run_filter(vol, iso, triangles=False, project=False, raster_order=True, cell_data=True)
    assert_mesh_equal_up_to_vertex_order(mesh, ref, mesh, ref, "noise")


@pytest.mark.parametrize("tri,proj", [(False, False), (True, True)])
def test_raster_vertex_order_z_slabs(tri, proj):
    """slabs in raster order: the corners of a shared plane belong to the lower slab"""
    P, O = pkg(), oracle()
    vol = gyroid((41, 30, 50), 13.0)
    nz, n_slabs = vol.shape[0], 3
    bounds = np.linspace(0, nz, n_slabs + 1).astype(int)

    def run(project):
        p = P.capi.default_params()
        p.iso_value, p.generate_triangles, p.project_vertices, p.surface_distance_threshold = 0.0, int(tri), int(project), 0.01
        p.vertex_order = P.capi.ORDER_RASTER
        hs, counts = [], []
        for s in range(n_slabs):
            z0, z1 = int(bounds[s]), int(bounds[s + 1])
            lo, hi = max(0, z0 - 9), min(nz, z1 + 9)
            h = P.capi.Handle(0)
            h.set_volume(vol[lo:hi])
            h.set_slab(nz, lo, z0, z1)
            counts.append(h.count(p))
            hs.append(h)
        pts, cells, pbase = [], [], 0
        for h, (np_, nq) in zip(hs, counts):
            h.set_id_base(pbase, 0)
            h.emit(4)
            a, b, _ = h.fetch()
            pts.append(a); cells.append(b); pbase += np_
            h.close()
        return P.Mesh(np.concatenate(pts), np.concatenate(cells))

    ref = O.cuberille(vol, 0.0, triangles=tri, project=proj, thr=0.01)
    ref0 = O.cuberille(vol, 0.0, triangles=tri, project=False)
    assert_mesh_equal_up_to_vertex_order(run(proj), ref, run(False), ref0, "raster slabs")


@pytest.mark.parametrize("resident", [False, True])
@pytest.mark.parametrize("n_slabs,n_handles", [(4, 2), (7, 3)])
def test_streamed_slabs_from_host_memory(n_slabs, n_handles, resident):
    """slabs.run_streamed: host volume in, host mesh out through several handles; equals the single run"""
    import torch
    P, O = pkg(), oracle()
    vol = gyroid((45, 28, 40), 11.0)
    ref = O.cuberille(vol, 0.0, triangles=True, project=True, thr=0.01)
    vt = torch.from_numpy(vol).pin_memory()
    pts = torch.zeros((ref.points.shape[0] + 8, 3), dtype=torch.float32).pin_memory()
    cells = torch.zeros((ref.cells.shape[0] + 8, 3), dtype=torch.int32).pin_memory()
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices, p.surface_distance_threshold = 0.0, 1, 1, 0.01
    kw = {}
    if resident:  # the volume is copied once into a device buffer, the handles borrow windows of it
        streams = [torch.cuda.Stream() for _ in range(n_handles)]
        handles = [P.capi.Handle(0, st.cuda_stream) for st in streams]
        kw = dict(device_volume=torch.empty(vol.nbytes, dtype=torch.uint8, device="cuda"), streams=streams)
    else:
        handles = [P.capi.Handle(0) for _ in range(n_handles)]
    n_pts, n_cells = P.slabs.run_streamed(handles, vt.data_ptr(), np.float32, (40, 28, 45), p, n_slabs, pts.data_ptr(),
                                          cells.data_ptr(), halo=9, **kw)
    assert (n_pts, n_cells) == (ref.points.shape[0], ref.cells.shape[0])
    mesh = P.Mesh(pts.numpy()[:n_pts], cells.numpy()[:n_cells].view(np.uint32))
    assert_mesh_equal(mesh, ref, "streamed")
    for h in handles:
        h.close()


# ---- oriented images: direction matrices (SURVEY section 8f-2; cuberille_c.h cub_set_volume `direction`) ------------------
_C30, _S30 = float(np.cos(np.pi / 6)), float(np.sin(np.pi / 6))
DIRECTIONS = {
    "flip_x": (-1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0),
    "flip_yz": (1.0, 0.0, 0.0, 0.0, -1.0, 0.0, 0.0, 0.0, -1.0),
    "permute": (0.0, 1.0, 0.0, 0.0, 0.0, 1.0, 1.0, 0.0, 0.0),
    "rot_z_30": (_C30, -_S30, 0.0, _S30, _C30, 0.0, 0.0, 0.0, 1.0),
    "oblique": tuple(float(v) for v in np.linalg.qr(np.random.default_rng(5).normal(size=(3, 3)))[0].reshape(9)),
}


@pytest.mark.parametrize("name", sorted(DIRECTIONS))
@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
@pytest.mark.parametrize("tri,proj", [(False, False), (True, True)])
def test_direction_matrices(name, dtype, tri, proj):
    """positions through M = D*diag(spacing), continuous indices through M^-1, rotated gradients: bit-exact vs the oracle"""
    O, P = oracle(), pkg()
    vol, iso = smooth_volume((22, 27, 40), dtype, seed=31)
    D, sp, og = DIRECTIONS[name], (0.5, 1.25, 2.0), (3.0, -2.0, 7.0)
    kw = dict(triangles=tri, project=proj, thr=0.02, step=0.24, relax=0.95, max_steps=80)
    ref = O.cuberille(vol, iso, mode=O.CLOSED_FORM, spacing=sp, origin=og, direction=D, **kw)
    mesh = run_filter(P.Image(vol, sp, og, D), iso, **kw)
    assert_mesh_equal(mesh, ref, f"direction {name}")
    if proj:  # the orientation does change the result (the test would pass trivially otherwise)
        plain = O.cuberille(vol, iso, mode=O.CLOSED_FORM, spacing=sp, origin=og, **kw)
        assert not np.array_equal(plain.points, ref.points)


def test_direction_with_slabs_and_projection():
    """z-slabs of an oriented image: the projection halo follows the z row of M^-1"""
    O, P = oracle(), pkg()
    vol, iso = smooth_volume((40, 20, 24), np.float32, seed=33)
    D, sp = DIRECTIONS["rot_z_30"], (1.0, 1.0, 1.0)
    prm = P.capi.default_params()
    prm.iso_value, prm.generate_triangles, prm.project_vertices = float(iso), 1, 1
    prm.surface_distance_threshold, prm.step_length, prm.max_steps = 0.02, 0.24, 80
    ref = O.cuberille(vol, iso, mode=O.CLOSED_FORM, triangles=True, project=True, thr=0.02, step=0.24, relax=0.95, max_steps=80,
                      spacing=sp, direction=D)
    halo = max(P.capi.projection_halo(prm, sp))
    pts, cells, pb, cb = [], [], 0, 0
    for s in P.slabs.plan_slabs(vol.shape[0], 3, halo):
        h = P.capi.Handle(0)
        h.set_volume(vol[s.local_z0:s.local_z1], sp, (0.0, 0.0, 0.0), D)
        h.set_slab(vol.shape[0], s.local_z0, s.own_z0, s.own_z1)
        a, b = h.count(prm)
        h.set_id_base(pb, cb)
        h.emit(4)
        x, y, _ = h.fetch()
        pts.append(x); cells.append(y)
        pb += a; cb += 2 * b
        h.close()
    assert_mesh_equal(P.Mesh(np.concatenate(pts), np.concatenate(cells)), ref, "oriented slabs")


def test_emit_twice_gives_the_same_mesh():
    """a second cub_emit on the same count (new id base, other id width) starts from unprojected points again"""
    O, P = oracle(), pkg()
    img = read_fixture("neghip")
    h = P.capi.Handle(0)
    h.set_volume(img.data)
    p = P.capi.default_params()
    p.iso_value, p.surface_distance_threshold, p.step_length, p.max_steps = 55.0, 0.2, 0.24, 3   # most vertices stop at max_steps
    ref = O.cuberille(img.data, 55, triangles=True, project=True, thr=0.2, step=0.24, relax=0.95, max_steps=3)
    h.count(p)
    h.emit(4)
    a = h.fetch()
    h.emit(4)
    b = h.fetch()
    h.set_id_base(1000, 0)
    h.emit(8)
    c = h.fetch()
    assert_mesh_equal(P.Mesh(a[0], a[1]), ref, "first emit")
    assert_mesh_equal(P.Mesh(b[0], b[1]), ref, "second emit")
    assert np.array_equal(c[0].view(np.uint32), ref.points.view(np.uint32)) and np.array_equal(c[1], ref.cells + 1000)
    h.close()


# the emit modes of the synchronous tests above, each with the volumes and the oracle comparison of its test
ASYNC_MODES = {
    "quads_u32": dict(volume="noise", tri=False, proj=False),
    "quads_u64": dict(volume="noise", tri=False, proj=False, id_bytes=8),
    "triangles_fixed_split": dict(volume="noise", tri=True, proj=False),
    "triangles_projected": dict(volume="smooth", tri=True, proj=True),
    "cell_data": dict(volume="smooth_i16", tri=True, proj=True, cell_data=True),
    "raster_order": dict(volume="noise", tri=False, proj=False, cell_data=True, raster=True),
    "oriented": dict(volume="smooth", tri=True, proj=True, direction="oblique"),
}


def test_async_pipeline_matches_and_survives_a_larger_second_run():
    """cub_count_async / cub_emit_async / cub_finish: buffers sized by a small first run, then a larger volume on the same
    handle overflows them on the device; cub_finish must redo the emission and return the complete mesh"""
    check_async_pipeline("triangles_projected")


@pytest.mark.parametrize("mode", sorted(set(ASYNC_MODES) - {"triangles_projected"}))
def test_async_pipeline_in_the_other_emit_modes(mode):
    """the same small / overflowing / smaller runs through cub_emit_async in every other emit mode"""
    check_async_pipeline(mode)


def check_async_pipeline(mode):
    O, P = oracle(), pkg()
    m = ASYNC_MODES[mode]
    tri, proj, cd, raster, id_bytes = m["tri"], m["proj"], m.get("cell_data", False), m.get("raster", False), m.get("id_bytes", 4)
    kw = dict(triangles=tri, project=proj, cell_data=cd, thr=0.02)
    p = P.capi.default_params()
    p.generate_triangles, p.project_vertices, p.save_pixel_as_cell_data = int(tri), int(proj), int(cd)
    p.surface_distance_threshold = kw["thr"]
    if raster:
        p.vertex_order = P.capi.ORDER_RASTER
    geo = {}
    if "direction" in m:  # the image and projection arguments of test_direction_matrices
        geo = dict(spacing=(0.5, 1.25, 2.0), origin=(3.0, -2.0, 7.0), direction=DIRECTIONS[m["direction"]])
        kw.update(step=0.24, relax=0.95, max_steps=80)
        p.step_length, p.step_relaxation, p.max_steps = kw["step"], kw["relax"], kw["max_steps"]
    h = P.capi.Handle(0)
    for shape, seed in [((10, 12, 33), 1), ((30, 40, 70), 2), ((30, 40, 70), 3), ((12, 9, 20), 4)]:
        if m["volume"] == "noise":
            vol, iso = random_volume(shape, np.uint8, seed=seed)
        else:
            vol, iso = smooth_volume(shape, np.int16 if m["volume"] == "smooth_i16" else np.float32, seed=seed)
        p.iso_value = float(iso)
        h.set_volume(vol, **geo)
        h.count_async(p)
        h.emit_async(id_bytes)
        n_pts, n_cells = h.finish()
        mode_args = dict(mode=O.CLOSED_FORM) if m["volume"] == "noise" or geo else {}
        ref = O.cuberille(vol, iso, **mode_args, **geo, **kw)
        assert (n_pts, n_cells) == (ref.points.shape[0], ref.cells.shape[0])
        a, b, c = h.fetch(want_cell_data=cd)
        mesh = P.Mesh(a, b, c)
        if raster:
            assert_mesh_equal_up_to_vertex_order(mesh, ref, mesh, ref, f"async {mode} {shape}")
        else:
            assert_mesh_equal(mesh, ref, f"async {mode} {shape}")
        assert b.dtype == (np.uint64 if id_bytes == 8 else np.uint32)
        if cd:
            assert c.dtype == vol.dtype
    h.close()


def test_empty_interior_slice_is_reported():
    """SURVEY section 8a row 3: the reference merges vertices across an empty slice; the library does not, and says so"""
    P = pkg()
    vol = np.zeros((9, 5, 5), np.uint8)
    vol[2, 2, 2] = vol[4, 2, 2] = 255   # slice 3 is empty between two occupied ones
    h = P.capi.Handle(0)
    h.set_volume(vol)
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices = 200.0, 0, 0
    assert h.run(p) == (16, 12)
    assert "empty voxel slice" in h.last_warning()
    vol[3, 0, 0] = 255
    h.set_volume(vol)
    h.run(p)
    assert h.last_warning() == ""
    h.close()


def test_slab_without_projection_halo_is_refused():
    P = pkg()
    vol, iso = smooth_volume((40, 16, 16), np.float32, seed=1)
    h = P.capi.Handle(0)
    h.set_volume(vol[8:32])
    h.set_slab(40, 8, 10, 30)   # 2-slice halo: fine without projection, too short with it
    p = P.capi.default_params()
    p.iso_value, p.project_vertices = float(iso), 0
    h.count(p)
    p.project_vertices = 1
    with pytest.raises(P.capi.CuberilleError) as e:
        h.count(p)
    assert "halo" in str(e.value)
    h.close()


def test_generated_slab_without_set_slab_is_refused():
    """ADVICE r1: a generated z-slab (z_offset > 0) used without cub_set_slab wrote before its lattice"""
    P = pkg()
    h = P.capi.Handle(0)
    h.generate(P.capi.GEN_GYROID, (32, 32, 16), (32, 32, 64), 20, 16.0)
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices = 0.0, 0, 0
    with pytest.raises(P.capi.CuberilleError):
        h.count(p)
    h.set_slab(64, 20, 22, 35)
    h.count(p)
    h.close()


# ---- the reference's compile-time alternates of ProjectVertexToIsoSurface (SURVEY section 8f-4) --------------------------
@pytest.mark.parametrize("method", [1, 2], ids=["advanced", "linesearch"])
@pytest.mark.parametrize("fixture,iso,max_steps", [("fuel", 15, 100), ("neghip", 55, 100), ("nucleon", 140, 100), ("marschnerlobb", 55, 40)])
def test_alternate_projections_on_reference_fixtures(method, fixture, iso, max_steps):
    """USE_ADVANCED_PROJECTION (txx:340-397) / USE_LINESEARCH_PROJECTION (txx:398-438) as run-time variants: points and the
    projected triangle split bit-exact against the oracle's restatement of the same branches"""
    O = oracle()
    img = read_fixture(fixture)
    kw = dict(triangles=True, project=True, thr=0.2, step=0.24, relax=0.95, max_steps=max_steps)
    ref = O.cuberille(img.data, iso, method=method, **kw)
    mesh = run_filter(img, iso, method=method, **kw)
    assert_mesh_equal(mesh, ref, f"{fixture} method {method}")
    plain = O.cuberille(img.data, iso, **kw)
    assert not np.array_equal(plain.points, ref.points)   # (the variants do move the vertices differently)


@pytest.mark.parametrize("method", [1, 2], ids=["advanced", "linesearch"])
def test_alternate_projections_float_anisotropic_oriented_and_slabs(method):
    O, P = oracle(), pkg()
    vol, iso = smooth_volume((36, 20, 44), np.float32, seed=77)
    sp, og, D = (0.5, 1.25, 2.0), (3.0, -2.0, 7.0), DIRECTIONS["rot_z_30"]
    kw = dict(triangles=True, project=True, thr=0.02, step=0.3, relax=0.9, max_steps=30)
    ref = O.cuberille(vol, iso, mode=O.CLOSED_FORM, spacing=sp, origin=og, direction=D, method=method, **kw)
    mesh = run_filter(P.Image(vol, sp, og, D), iso, method=method, **kw)
    assert_mesh_equal(mesh, ref, f"oriented method {method}")
    # z-slabs (isotropic, non-oriented): the halo rule of the default branch covers both variants
    ref2 = O.cuberille(vol, iso, mode=O.CLOSED_FORM, method=method, **kw)
    prm = P.capi.default_params()
    prm.iso_value, prm.generate_triangles, prm.project_vertices, prm.projection_method = float(iso), 1, 1, method
    prm.surface_distance_threshold, prm.step_length, prm.step_relaxation, prm.max_steps = 0.02, 0.3, 0.9, 30
    halo = max(P.capi.projection_halo(prm))
    pts, cells, pb, cb = [], [], 0, 0
    for s in P.slabs.plan_slabs(vol.shape[0], 3, halo):
        h = P.capi.Handle(0)
        h.set_volume(vol[s.local_z0:s.local_z1])
        h.set_slab(vol.shape[0], s.local_z0, s.own_z0, s.own_z1)
        a, b = h.count(prm)
        h.set_id_base(pb, cb)
        h.emit(4)
        x, y, _ = h.fetch()
        pts.append(x); cells.append(y)
        pb += a; cb += 2 * b
        h.close()
    assert_mesh_equal(P.Mesh(np.concatenate(pts), np.concatenate(cells)), ref2, f"slabs method {method}")


def test_unknown_projection_method_is_refused():
    P = pkg()
    h = P.capi.Handle(0)
    h.set_volume(np.zeros((4, 4, 4), np.uint8))
    p = P.capi.default_params()
    p.projection_method = 7
    with pytest.raises(P.capi.CuberilleError):
        h.count(p)
    h.close()
