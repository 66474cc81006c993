"""TEST INFRASTRUCTURE: ctypes binding of tests/mesh_oracle.cpp, the CPU oracle's integrator with per-vertex normals and
texture coordinates of mesh triangles (DESIGN.md §5e).  The shared library is compiled on first use into a temporary
directory keyed by a hash of its sources, so nothing is written into the tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_ROOT = _HERE.parent
_SOURCES = [_HERE / "mesh_oracle.cpp", _HERE / "env_oracle.cpp", _HERE / "light_oracle.cpp", _ROOT / "oracle" / "oracle.cpp",
            _ROOT / "oracle" / "omath.h", _ROOT / "oracle" / "oracle.h", _ROOT / "include" / "rtb.h",
            _ROOT / "include" / "rtb_scene_format.h"]
RNG_PHILOX = 0
ATTR_DTYPE = np.dtype([("n", "<f4", (3, 3)), ("uv", "<f4", (3, 2)), ("flags", "<i4")])   # rtbs_tri_attr
assert ATTR_DTYPE.itemsize == 64
_lib = None


def _build() -> Path:
    h = hashlib.sha1()
    for f in _SOURCES:
        h.update(f.read_bytes())
    out = Path(tempfile.gettempdir()) / f"rtb_mesh_oracle_{h.hexdigest()[:16]}.so"
    if not out.exists():
        tmp = out.with_suffix(f".{os.getpid()}.tmp")
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-Wall", "-pthread", "-shared",
                        "-o", str(tmp), str(_HERE / "mesh_oracle.cpp")], check=True, capture_output=True, text=True)
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is None:
        h = C.CDLL(str(_build()))
        P = C.c_void_p
        h.omesh_scene_load.restype = P; h.omesh_scene_load.argtypes = [P, C.c_size_t]
        h.omesh_scene_free.restype = None; h.omesh_scene_free.argtypes = [P]
        h.orc_last_error.restype = C.c_char_p
        h.omesh_attr_count.restype = C.c_int; h.omesh_attr_count.argtypes = [P]
        h.omesh_attrs.restype = None; h.omesh_attrs.argtypes = [P, P]
        h.omesh_trace_rays.restype = C.c_int; h.omesh_trace_rays.argtypes = [P, P, C.c_size_t, P]
        h.omesh_render.restype = C.c_int
        h.omesh_render.argtypes = [P, P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int, P, P, P]
        _lib = h
    return _lib


class MeshOracleScene:
    """An RTBS v1 - v4 blob on the CPU: the environment-map oracle's integrator, with the triangle attributes of a v4 blob.
    render() has the signature of pyoracle.OracleScene.render; trace() returns rtb_hit records like orc_trace_rays."""

    def __init__(self, blob: bytes):
        self._blob = blob
        self.handle = lib().omesh_scene_load(blob, len(blob))
        if not self.handle:
            raise RuntimeError("omesh_scene_load: " + lib().orc_last_error().decode())

    def __del__(self):
        if getattr(self, "handle", None) and _lib is not None:
            _lib.omesh_scene_free(self.handle); self.handle = None

    def attrs(self) -> np.ndarray:
        n = lib().omesh_attr_count(self.handle)
        out = np.zeros(n, ATTR_DTYPE)
        if n:
            lib().omesh_attrs(self.handle, out.ctypes.data)
        return out

    def trace(self, rays: np.ndarray, hit_dtype) -> np.ndarray:
        rays = np.ascontiguousarray(rays)
        out = np.zeros(len(rays), hit_dtype)
        if lib().omesh_trace_rays(self.handle, rays.ctypes.data, len(rays), out.ctypes.data) != 0:
            raise RuntimeError("omesh_trace_rays: " + lib().orc_last_error().decode())
        return out

    def render(self, cam, width, height, sample_begin, sample_end, max_depth, seed=1984, mode=RNG_PHILOX, threads=0, want_sum2=False):
        """Returns (sum[H,W,4], sum2 or None, rays)."""
        s = np.zeros((height, width, 4), dtype=np.float32)
        s2 = np.zeros_like(s) if want_sum2 else None
        rays = C.c_uint64(0)
        rc = lib().omesh_render(self.handle, C.addressof(cam), width, height, sample_begin, sample_end, max_depth, seed, mode, threads,
                                s.ctypes.data, s2.ctypes.data if want_sum2 else None, C.addressof(rays))
        if rc != 0:
            raise RuntimeError("omesh_render: " + lib().orc_last_error().decode())
        return s, s2, rays.value
