"""MetaImage (.mha) reader / writer and legacy-VTK polydata writer.

What Testing/CuberilleTest01.cxx does around the filter with ITK IO
(ImageFileReader Test:113-117, VTKPolyDataWriter Test:180-187), restated without
ITK.  Supports what the reference's fixtures use: NDims 3, ElementDataFile LOCAL,
little-endian, optional zlib compression (CompressedData = True), x-fastest.
"""
from __future__ import annotations

import zlib
from dataclasses import dataclass, field

import numpy as np

_MET_TYPES = {
    "MET_UCHAR": np.uint8, "MET_CHAR": np.int8, "MET_USHORT": np.uint16, "MET_SHORT": np.int16,
    "MET_UINT": np.uint32, "MET_INT": np.int32, "MET_FLOAT": np.float32, "MET_DOUBLE": np.float64,
    "MET_LONG_LONG": np.int64, "MET_ULONG_LONG": np.uint64,
}
_MET_NAMES = {np.dtype(v): k for k, v in _MET_TYPES.items()}


@dataclass
class Image:
    """A 3-D image: `data` indexed [z, y, x]; geometry as in itk::Image."""
    data: np.ndarray
    spacing: tuple = (1.0, 1.0, 1.0)
    origin: tuple = (0.0, 0.0, 0.0)
    direction: tuple = (1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0)   # itk direction cosines, row-major D[i][j]
    meta: dict = field(default_factory=dict)
    region_index: tuple = (0, 0, 0)   # itk::ImageRegion::GetIndex of the buffered region (x, y, z)


def read_mha(path: str) -> Image:
    with open(path, "rb") as f:
        raw = f.read()
    meta = {}
    pos = 0
    while True:
        end = raw.index(b"\n", pos)
        line = raw[pos:end].decode("ascii").strip()
        pos = end + 1
        if not line:
            continue
        key, _, val = line.partition("=")
        meta[key.strip()] = val.strip()
        if key.strip() == "ElementDataFile":
            break
    if meta.get("ElementDataFile") != "LOCAL":
        raise ValueError("only ElementDataFile = LOCAL is supported")
    if int(meta.get("NDims", "3")) != 3:
        raise ValueError("only NDims = 3 is supported")
    if meta.get("BinaryDataByteOrderMSB", meta.get("ElementByteOrderMSB", "False")) == "True":
        raise ValueError("big-endian data not supported")
    nx, ny, nz = (int(v) for v in meta["DimSize"].split())
    dtype = np.dtype(_MET_TYPES[meta["ElementType"]])
    payload = raw[pos:]
    if meta.get("CompressedData", "False") == "True":
        n = int(meta.get("CompressedDataSize", len(payload)))
        payload = zlib.decompress(payload[:n])
    data = np.frombuffer(payload, dtype=dtype, count=nx * ny * nz).reshape(nz, ny, nx).copy()
    spacing = tuple(float(v) for v in meta.get("ElementSpacing", "1 1 1").split())
    origin = tuple(float(v) for v in meta.get("Offset", meta.get("Position", "0 0 0")).split())
    # MetaImage lists the axis direction vectors one after the other, i.e. the COLUMNS of itk's direction
    # matrix (MetaImageIO: TransformMatrix(i, j) = direction[j][i]); Image.direction is row-major D[i][j]
    tm = [float(v) for v in meta.get("TransformMatrix", "1 0 0 0 1 0 0 0 1").split()]
    direction = tuple(tm[3 * j + i] for i in range(3) for j in range(3))
    return Image(data, spacing, origin, direction, meta)


def write_mha(path: str, img: Image, compress: bool = True) -> None:
    data = np.ascontiguousarray(img.data)
    nz, ny, nx = data.shape
    payload = data.tobytes()
    lines = ["ObjectType = Image", "NDims = 3", "BinaryData = True", "BinaryDataByteOrderMSB = False"]
    if compress:
        payload = zlib.compress(payload)
        lines += ["CompressedData = True", f"CompressedDataSize = {len(payload)}"]
    else:
        lines += ["CompressedData = False"]
    lines += [
        "TransformMatrix = " + " ".join(f"{float(img.direction[3 * j + i])!r}" for i in range(3) for j in range(3)),
        "Offset = " + " ".join(f"{float(v)!r}" for v in img.origin),
        "CenterOfRotation = 0 0 0",
        "AnatomicalOrientation = RAI",
        "ElementSpacing = " + " ".join(f"{float(v)!r}" for v in img.spacing),
        f"DimSize = {nx} {ny} {nz}",
        f"ElementType = {_MET_NAMES[data.dtype]}",
        "ElementDataFile = LOCAL",
    ]
    with open(path, "wb") as f:
        f.write(("\n".join(lines) + "\n").encode("ascii"))
        f.write(payload)


def write_vtk_polydata(path: str, points: np.ndarray, cells: np.ndarray, cell_data: np.ndarray | None = None) -> None:
    """Legacy ASCII VTK polydata, the format itk::VTKPolyDataWriter emits (Test:180-187)."""
    n, k = cells.shape if cells.size else (0, 3)
    with open(path, "w") as f:
        f.write("# vtk DataFile Version 2.0\nFile written by cuberille-b200\nASCII\nDATASET POLYDATA\n")
        f.write(f"POINTS {points.shape[0]} float\n")
        np.savetxt(f, points, fmt="%.9g")
        f.write(f"POLYGONS {n} {n * (k + 1)}\n")
        if n:
            np.savetxt(f, np.concatenate([np.full((n, 1), k, np.int64), cells.astype(np.int64)], axis=1), fmt="%d")
        if cell_data is not None:
            f.write(f"CELL_DATA {n}\nSCALARS pixel double 1\nLOOKUP_TABLE default\n")
            np.savetxt(f, cell_data.astype(np.float64), fmt="%.9g")
