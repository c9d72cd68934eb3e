"""GPU: the fused classification + ownership-sweep kernel (csrc/k_fused.cuh) against the oracle and against the
two-kernel path it replaces, bit for bit.  The two-kernel path runs on the same volume as a device pointer one pixel
past a 16-byte boundary, where the fused kernel cannot run.  The tuning knobs are read once per handle in cub_create,
so several settings can run in one process."""
import os

import numpy as np
import pytest

from test_gpu_pixel_edges import set_route_volume
from util import assert_mesh_equal, gyroid, oracle, pkg, random_volume

pytestmark = pytest.mark.gpu


class _env:
    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        for k, v in self.kv.items():
            os.environ[k] = str(v)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _handle(**env):
    with _env(**env):
        return pkg().capi.Handle(0)


def _run(h, vol, iso, tri=False, two_kernel=False):
    P = pkg()
    buf = set_route_volume(h, vol, misaligned=two_kernel)
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices = float(iso), int(tri), 0
    h.count(p)
    fused = h.count_was_fused()
    bits = h.bitmask().copy()
    h.emit(4)
    pts, cells, _ = h.fetch()
    del buf
    return fused, bits, pts, cells


# rows of whole 16-byte groups (the TMA bulk copies): one / several / ragged tasks per row, rows shorter than a word,
# both sweep tile shapes (<= 8 and > 8 words per row), several z chunks, 4- and 8-byte pixels and unpacked small ones
@pytest.mark.parametrize("dtype,shape", [
    (np.float32, (5, 6, 32)), (np.float32, (9, 33, 64)), (np.float32, (17, 20, 100)), (np.float32, (12, 40, 200)),
    (np.float32, (3, 5, 520)), (np.float32, (7, 3, 1028)), (np.float32, (70, 30, 36)), (np.float32, (2, 2, 4)),
    (np.float32, (1, 1, 8)), (np.float64, (11, 14, 258)), (np.float64, (6, 9, 30)), (np.int32, (13, 21, 300)),
    (np.uint32, (8, 8, 512)), (np.uint8, (9, 10, 48)), (np.int16, (9, 10, 40)), (np.uint16, (5, 4, 1048)),
])
def test_fused_equals_oracle_and_the_unaligned_two_kernel_path(dtype, shape):
    O = oracle()
    vol, iso = random_volume(shape, dtype, seed=shape[2] + shape[0], fill=0.5)
    hf, hu = _handle(), _handle()
    for tri in (False, True):
        ff, bf, pf, cf = _run(hf, vol, iso, tri)
        fu, bu, pu, cu = _run(hu, vol, iso, tri, two_kernel=True)
        assert ff and not fu, (ff, fu)
        assert np.array_equal(bf, bu), "bitmask differs between the fused and the two-kernel path"
        assert np.array_equal(pf.view(np.uint32), pu.view(np.uint32)) and np.array_equal(cf, cu)
        ref = O.cuberille(vol, iso, triangles=tri, project=False, mode=O.CLOSED_FORM)
        assert pf.shape == ref.points.shape and np.array_equal(cf.astype(np.uint64).reshape(ref.cells.shape), ref.cells)
        assert np.array_equal(pf.view(np.uint32), ref.points.view(np.uint32))
    hf.close()
    hu.close()


# rows of 33 voxel words sweep wide tiles, rows of 7 narrow ones (cuberille_capi.cu: choose_count_route)
@pytest.mark.parametrize("shape", [(150, 210, 1040), (400, 420, 200)])
@pytest.mark.parametrize("env", [dict(), dict(CUB_FUSE_TZ=4), dict(CUB_FUSE_TZ=7, CUB_FUSE_CTAS_PER_SM=1)])
def test_fused_large_noise_volume_equals_the_two_kernel_path(env, shape):
    """many tiles, many z chunks, consumers that overtake the producers: everything the count phase leaves behind must
    be identical (mesh, bitmask), on a volume the oracle would need minutes for"""
    vol, iso = random_volume(shape, np.float32, seed=5, fill=0.35)
    hf, hu = _handle(**env), _handle()
    for rep in range(2):  # the second run reuses the control block (tickets, progress counters)
        ff, bf, pf, cf = _run(hf, vol, iso)
        fu, bu, pu, cu = _run(hu, vol, iso, two_kernel=True)
        assert ff and not fu
        assert np.array_equal(bf, bu)
        assert pf.shape == pu.shape and cf.shape == cu.shape
        assert np.array_equal(pf.view(np.uint32), pu.view(np.uint32)) and np.array_equal(cf, cu)
    hf.close()
    hu.close()


def test_fused_z_slabs_concatenate_to_the_single_run():
    """slab handles classify their halo slices too; the sweep range starts above local slice 0"""
    P, O = pkg(), oracle()
    vol = gyroid((41, 30, 52), 13.0)
    ref = O.cuberille(vol, 0.0, triangles=False, project=False)
    nz = vol.shape[0]
    bounds = [0, 13, 14, 30, 41]
    p = P.capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices = 0.0, 0, 0
    pts, cells, pbase, cbase = [], [], 0, 0
    for z0, z1 in zip(bounds[:-1], bounds[1:]):
        lo, hi = max(0, z0 - 2), min(nz, z1 + 2)
        h = _handle()
        h.set_volume(vol[lo:hi])
        h.set_slab(nz, lo, z0, z1)
        n_pts, n_quads = h.count(p)
        assert h.count_was_fused()
        h.set_id_base(pbase, cbase)
        h.emit(4)
        a, b, _ = h.fetch()
        pts.append(a)
        cells.append(b)
        pbase += n_pts
        cbase += n_quads
        h.close()
    got_p, got_c = np.concatenate(pts), np.concatenate(cells)
    assert np.array_equal(got_p.view(np.uint32), ref.points.view(np.uint32))
    assert np.array_equal(got_c.astype(np.uint64).reshape(ref.cells.shape), ref.cells)


def test_fused_falls_back_where_it_does_not_apply():
    """rows that are not whole 16-byte groups, packed 8-bit rows, the padded lattice: two kernels, same results"""
    P = pkg()
    for dtype, shape in ((np.float32, (4, 5, 50)), (np.uint8, (4, 5, 128))):
        vol, iso = random_volume(shape, dtype, seed=1)
        h = _handle()
        fused, *_ = _run(h, vol, iso)
        assert not fused
        h.close()
