"""The device mesh upload's host side, without a GPU: the ctypes descriptor matches include/trace_cuda.h's
trace_mesh_device_desc, and DeviceMeshScene refuses malformed numpy input with ValueError before touching a device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CTYPES = {"int64_t": C.c_int64, "int32_t": C.c_int32, "const void*": C.c_void_p, "const trace_material*": C.c_void_p,
           "const trace_light*": C.c_void_p}


def header_fields():
    """(name, ctypes type) of trace_mesh_device_desc, in declaration order, read from the header"""
    txt = open(os.path.join(ROOT, "include", "trace_cuda.h")).read()
    body = re.search(r"typedef struct trace_mesh_device_desc \{(.*?)\} trace_mesh_device_desc;", txt, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    out = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        m = re.fullmatch(r"((?:const )?\w+\*?) (\w+)", decl)
        assert m, decl
        out.append((m.group(2), _CTYPES[m.group(1)]))
    return out


def test_descriptor_layout_matches_header(T):
    fields = header_fields()
    assert [f for f, _ in fields] == [f for f, _ in T._lib.MeshDeviceDesc._fields_]

    class FromHeader(C.Structure):
        _fields_ = fields

    assert C.sizeof(T._lib.MeshDeviceDesc) == C.sizeof(FromHeader) == 80
    for name, _ in fields:
        assert getattr(T._lib.MeshDeviceDesc, name).offset == getattr(FromHeader, name).offset, name
    sig = T._lib.SIGNATURES["trace_scene_upload_mesh_device"]
    assert sig[0] is C.c_int and len(sig[1]) == 3


def _matte(T):
    return T.MatteMaterial(T.ConstantTexture(T.RGBSpectrum(0.5)), T.ConstantTexture(0.0))


def _tris(n=5):
    return np.arange(n * 9, dtype=np.float32).reshape(n, 3, 3)


@pytest.mark.parametrize("kw, msg", [
    (dict(vertices=_tris().astype(np.float64)), r"vertices must have dtype float32, got float64"),
    (dict(vertices=_tris().reshape(5, 9)), r"vertices must have shape \(n, 3, 3\), got \(5, 9\)"),
    (dict(vertices=_tris().reshape(15, 3)), r"vertices must have shape \(n, 3, 3\)"),
    (dict(vertices=_tris().tolist()), r"vertices must be a numpy array or a CUDA tensor, got list"),
    (dict(vertices=None), r"vertices are required"),
    (dict(vertices=_tris(), normals=_tris(4)), r"normals must have shape \(5, 3, 3\), got \(4, 3, 3\)"),
    (dict(vertices=_tris(), normals=_tris().astype(np.float16)), r"normals must have dtype float32"),
    (dict(vertices=_tris(), flags=np.zeros(5, np.int32)), r"flags must have dtype uint8, got int32"),
    (dict(vertices=_tris(), flags=np.zeros((5, 1), np.uint8)), r"flags must have shape \(5,\), got \(5, 1\)"),
    (dict(vertices=_tris(), material_ids=np.zeros(5, np.float32)), r"material_ids must have dtype integer, got float32"),
    (dict(vertices=_tris(), material_ids=np.zeros(6, np.int64)), r"material_ids must have shape \(5,\)"),
    (dict(vertices=_tris(), material_ids=np.array([0, 1, 0, 2, 0])), r"material_ids must be in \[0, 2\), got values in \[0, 2\]"),
    (dict(vertices=_tris(), material_ids=np.array([0, -1, 0, 1, 0])), r"material_ids must be in \[0, 2\), got values in \[-1, 1\]"),
])
def test_device_mesh_scene_argument_checks(T, kw, msg):
    with pytest.raises(ValueError, match=msg):
        T.DeviceMeshScene([], materials=[_matte(T), _matte(T)], **kw)


def test_device_mesh_scene_needs_materials_and_device_arrays(T):
    with pytest.raises(ValueError, match="at least one material"):
        T.DeviceMeshScene([], _tris(), [])
    with pytest.raises(ValueError, match="materials must be Material objects"):
        T.DeviceMeshScene([], _tris(), ["glass"])
    torch = pytest.importorskip("torch")
    with pytest.raises(ValueError, match="vertices: a CPU tensor"):
        T.DeviceMeshScene([], torch.from_numpy(_tris()), [_matte(T)])
