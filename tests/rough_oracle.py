"""TEST INFRASTRUCTURE: ctypes binding of tests/rough_oracle.cpp, the CPU oracle's integrator with the GGX microfacet
materials (DESIGN.md §5f), on top of the triangle-attribute oracle.  The shared library is compiled on first use into a temporary
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
_SOURCES = [_HERE / "rough_oracle.cpp", _HERE / "mesh_oracle.cpp", _HERE / "env_oracle.cpp", _HERE / "light_oracle.cpp", _ROOT / "oracle" / "oracle.cpp",
            _ROOT / "oracle" / "omath.h", _ROOT / "oracle" / "oracle.h", _ROOT / "include" / "rtb.h",
            _ROOT / "include" / "rtb_scene_format.h"]
RNG_PHILOX = 0
_lib = None


def _build() -> Path:
    h = hashlib.sha1()
    for f in _SOURCES:
        h.update(f.read_bytes())
    out = Path(tempfile.gettempdir()) / f"rtb_rough_oracle_{h.hexdigest()[:16]}.so"
    if not out.exists():
        tmp = out.with_suffix(f".{os.getpid()}.tmp")
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-Wall", "-pthread", "-shared",
                        "-o", str(tmp), str(_HERE / "rough_oracle.cpp")], check=True, capture_output=True, text=True)
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is None:
        h = C.CDLL(str(_build()))
        P = C.c_void_p
        h.orough_scene_load.restype = P; h.orough_scene_load.argtypes = [P, C.c_size_t]
        h.orough_scene_free.restype = None; h.orough_scene_free.argtypes = [P]
        h.orc_last_error.restype = C.c_char_p
        h.orough_alpha_count.restype = C.c_int; h.orough_alpha_count.argtypes = [P]
        h.orough_alphas.restype = None; h.orough_alphas.argtypes = [P, P]
        h.orough_render.restype = C.c_int
        h.orough_render.argtypes = [P, P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int, P, P, P]
        _lib = h
    return _lib


class RoughOracleScene:
    """An RTBS v1 - v5 blob on the CPU: the triangle-attribute oracle's integrator, with the GGX widths of a v5 blob.
    render() has the signature of pyoracle.OracleScene.render."""

    def __init__(self, blob: bytes):
        self._blob = blob
        self.handle = lib().orough_scene_load(blob, len(blob))
        if not self.handle:
            raise RuntimeError("orough_scene_load: " + lib().orc_last_error().decode())

    def __del__(self):
        if getattr(self, "handle", None) and _lib is not None:
            _lib.orough_scene_free(self.handle); self.handle = None

    def alphas(self) -> np.ndarray:
        n = lib().orough_alpha_count(self.handle)
        out = np.zeros(n, np.float32)
        if n:
            lib().orough_alphas(self.handle, out.ctypes.data)
        return out

    def render(self, cam, width, height, sample_begin, sample_end, max_depth, seed=1984, mode=RNG_PHILOX, threads=0, want_sum2=False):
        """Returns (sum[H,W,4], sum2 or None, rays)."""
        s = np.zeros((height, width, 4), dtype=np.float32)
        s2 = np.zeros_like(s) if want_sum2 else None
        rays = C.c_uint64(0)
        rc = lib().orough_render(self.handle, C.addressof(cam), width, height, sample_begin, sample_end, max_depth, seed, mode, threads,
                                 s.ctypes.data, s2.ctypes.data if want_sum2 else None, C.addressof(rays))
        if rc != 0:
            raise RuntimeError("orough_render: " + lib().orc_last_error().decode())
        return s, s2, rays.value
