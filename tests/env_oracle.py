"""TEST INFRASTRUCTURE: ctypes binding of tests/env_oracle.cpp, the CPU oracle's integrator with an HDR environment map
(DESIGN.md §5d).  The shared library is compiled on first use into a temporary directory keyed by a hash of its sources,
so nothing is written into the tree."""
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
_SOURCES = [_HERE / "env_oracle.cpp", _HERE / "light_oracle.cpp", _ROOT / "oracle" / "oracle.cpp", _ROOT / "oracle" / "omath.h",
            _ROOT / "oracle" / "oracle.h", _ROOT / "include" / "rtb.h", _ROOT / "include" / "rtb_scene_format.h"]
RNG_PHILOX = 0
_lib = None


def _build() -> Path:
    h = hashlib.sha1()
    for f in _SOURCES:
        h.update(f.read_bytes())
    out = Path(tempfile.gettempdir()) / f"rtb_env_oracle_{h.hexdigest()[:16]}.so"
    if not out.exists():
        tmp = out.with_suffix(f".{os.getpid()}.tmp")
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-Wall", "-pthread", "-shared",
                        "-o", str(tmp), str(_HERE / "env_oracle.cpp")], check=True, capture_output=True, text=True)
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is None:
        h = C.CDLL(str(_build()))
        P = C.c_void_p
        h.oenv_scene_load.restype = P; h.oenv_scene_load.argtypes = [P, C.c_size_t]
        h.oenv_scene_free.restype = None; h.oenv_scene_free.argtypes = [P]
        h.orc_last_error.restype = C.c_char_p
        h.oenv_dims.restype = C.c_int; h.oenv_dims.argtypes = [P, P]
        h.oenv_tables.restype = None; h.oenv_tables.argtypes = [P, P, P, P]
        h.oenv_sample.restype = None; h.oenv_sample.argtypes = [P, P, C.c_int, P, P, P]
        h.oenv_lookup.restype = None; h.oenv_lookup.argtypes = [P, P, C.c_int, P, P]
        h.oenv_render.restype = C.c_int
        h.oenv_render.argtypes = [P, P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int, P, P, P]
        _lib = h
    return _lib


class EnvOracleScene:
    """An RTBS v1 / v2 / v3 blob on the CPU: the light oracle's integrator, with the map of a v3 blob on every miss and, when
    the map is sampled, as one more strategy of the mixture.  render() has the signature of pyoracle.OracleScene.render."""

    def __init__(self, blob: bytes):
        self._blob = blob
        self.handle = lib().oenv_scene_load(blob, len(blob))
        if not self.handle:
            raise RuntimeError("oenv_scene_load: " + lib().orc_last_error().decode())

    def __del__(self):
        if getattr(self, "handle", None) and _lib is not None:
            _lib.oenv_scene_free(self.handle); self.handle = None

    def dims(self) -> tuple[int, int]:
        wh = np.zeros(2, dtype=np.int32)
        if lib().oenv_dims(self.handle, wh.ctypes.data) != 0:
            raise RuntimeError("the scene has no environment map")
        return int(wh[0]), int(wh[1])

    def tables(self):
        """(pdf numerators [H, W], marginal CDF [H + 1], conditional CDFs [H, W + 1])."""
        W, H = self.dims()
        num = np.zeros((H, W), np.float32); cm = np.zeros(H + 1, np.float32); cc = np.zeros((H, W + 1), np.float32)
        lib().oenv_tables(self.handle, num.ctypes.data, cm.ctypes.data, cc.ctypes.data)
        return num, cm, cc

    def sample(self, z: np.ndarray):
        """Directions drawn from the map with the uniforms z[k] = (row, column): (dirs [n, 3], texel [n], pdf [n])."""
        z = np.ascontiguousarray(z, dtype=np.float32).reshape(-1, 2)
        n = len(z)
        d = np.zeros((n, 3), np.float32); t = np.zeros(n, np.int64); p = np.zeros(n, np.float32)
        lib().oenv_sample(self.handle, z.ctypes.data, n, d.ctypes.data, t.ctypes.data, p.ctypes.data)
        return d, t, p

    def lookup(self, dirs: np.ndarray):
        """(texel [n], pdf [n]) of the directions dirs [n, 3]."""
        d = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
        n = len(d)
        t = np.zeros(n, np.int64); p = np.zeros(n, np.float32)
        lib().oenv_lookup(self.handle, d.ctypes.data, n, t.ctypes.data, p.ctypes.data)
        return t, p

    def render(self, cam, width, height, sample_begin, sample_end, max_depth, seed=1984, mode=RNG_PHILOX, threads=0, want_sum2=False):
        """Returns (sum[H,W,4], sum2 or None, rays)."""
        s = np.zeros((height, width, 4), dtype=np.float32)
        s2 = np.zeros_like(s) if want_sum2 else None
        rays = C.c_uint64(0)
        rc = lib().oenv_render(self.handle, C.addressof(cam), width, height, sample_begin, sample_end, max_depth, seed, mode, threads,
                               s.ctypes.data, s2.ctypes.data if want_sum2 else None, C.addressof(rays))
        if rc != 0:
            raise RuntimeError("oenv_render: " + lib().orc_last_error().decode())
        return s, s2, rays.value
