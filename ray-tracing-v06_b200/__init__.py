"""ray-tracing-v06_b200 — Python binding (ctypes) of the C ABI in include/rtb.h.

The product is the CUDA library ``librtb200.so`` (hand-written sm_100a wavefront kernels behind an
``extern "C"`` boundary) and the C++ host mirror of the reference's object model
(``librtb200_scenes.so``).  This module is only glue for tests, the benchmark and multi-GPU
plumbing; it never computes anything itself and there is NO CPU fallback: if the CUDA library is
missing, importing this package raises, and every render/trace call fails when no GPU is present.

The directory name is not a valid identifier; import it with
``importlib.import_module("ray-tracing-v06_b200")`` (repo root on sys.path).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["RTB_LIB"]) if os.environ.get("RTB_LIB") else _HERE / "librtb200.so"   # RTB_LIB: experimental builds only
SCENES_LIB_PATH = _HERE / "librtb200_scenes.so"
DEBUG_LIB_PATH = _HERE / "librtb200_debug.so"     # the same library built with -DRTB_DEBUG_BOUNDS=1 (select it with RTB_LIB)
BOUNDS_CLASSES = ("stack", "node", "primitive", "material", "texture", "queue", "path", "bin")   # (light indices count as "primitive")
MAX_SAMPLED_LIGHTS = 16
ENV_SAMPLE = 1          # rtb_scene_set_environment flag: importance-sample the map in the light mixture

RTB_OK = 0
TEX_SOLID, TEX_CHECKER, TEX_IMAGE, TEX_NOISE = 0, 1, 2, 3
BVH_TOPDOWN_MEDIAN, BVH_TOPDOWN_SAH, BVH_BOTTOMUP = 0, 1, 2
BG_SKY_GRADIENT, BG_CONSTANT = 0, 1
WORLD_BVH_QUALITY, WORLD_BVH_AS_BUILT, WORLD_BVH_GPU_LBVH = 0, 1, 2
BUILDER_NAMES = {0: "host_sah", 1: "as_built", 2: "gpu_lbvh", 3: "host_median_fallback"}
CAM_PINHOLE, CAM_DEFOCUS, CAM_MOTION = 0, 1, 2
RENDER_CLEAR, RENDER_VARIANCE = 1, 2
REDUCE_AUTO, REDUCE_NCCL, REDUCE_P2P = 0, 1, 2
PROFILE_CLASSES = {0: "generate", 1: "traverse", 2: "shade", 3: "accumulate", 4: "tail", 5: "bin", 6: "adaptive_select"}
MISS_DIST = np.float32(3.402823466e38)


class RtbError(RuntimeError):
    pass


def build(verbose: bool = False) -> None:
    """Compile librtb200.so and librtb200_scenes.so in-tree (nvcc cross-compiles without a GPU)."""
    res = subprocess.run(["make", f"-j{os.cpu_count() or 1}", "-C", str(_HERE), "all"], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0:
        raise RtbError("building librtb200.so failed")


class Camera(C.Structure):
    _fields_ = [("kind", C.c_int32), ("o", C.c_float * 3), ("u", C.c_float * 3), ("v", C.c_float * 3), ("w", C.c_float * 3),
                ("viewport_width", C.c_float), ("viewport_height", C.c_float), ("lens_radius", C.c_float), ("focus_dist", C.c_float),
                ("t0", C.c_float), ("t1", C.c_float)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("sample_begin", C.c_uint32), ("sample_end", C.c_uint32),
                ("row_begin", C.c_uint32), ("row_end", C.c_uint32), ("max_depth", C.c_uint32), ("seed", C.c_uint32),
                ("flags", C.c_uint32), ("samples_per_batch", C.c_uint32)]


class Counters(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("launches", C.c_uint64), ("batches", C.c_uint64), ("render_ms", C.c_double)]


class AdaptiveParams(C.Structure):
    _fields_ = [("tolerance", C.c_float), ("min_spp", C.c_uint32), ("max_rounds", C.c_uint32), ("reserved", C.c_uint32)]


class AdaptiveStats(C.Structure):
    _fields_ = [("rounds", C.c_uint32), ("cursor", C.c_uint32), ("active_pixels", C.c_uint32), ("reserved", C.c_uint32), ("samples", C.c_uint64)]


def tolerance_for_db(db: float) -> float:
    """Adaptive-sampling tolerance for a PSNR target (DESIGN.md §5c): 10^(-D/20).  When every pixel meets it, the image is
    about D dB from its converged value; two independent renders at that target are about D - 3 dB apart."""
    return float(10.0 ** (-float(db) / 20.0))


class SceneStats(C.Structure):
    _fields_ = [("primitives", C.c_int32), ("record_slots", C.c_int32), ("inner_nodes", C.c_int32), ("depth", C.c_int32), ("builder", C.c_int32),
                ("flatten_ms", C.c_float), ("bvh_build_ms", C.c_float), ("reserved", C.c_int32)]


class Profile(C.Structure):
    _fields_ = [("generate_ms", C.c_double), ("traverse_ms", C.c_double), ("shade_ms", C.c_double), ("accumulate_ms", C.c_double),
                ("generate_launches", C.c_uint64), ("traverse_launches", C.c_uint64), ("shade_launches", C.c_uint64), ("accumulate_launches", C.c_uint64),
                ("tail_ms", C.c_double), ("tail_launches", C.c_uint64), ("bin_ms", C.c_double), ("bin_launches", C.c_uint64)]


class SceneInfo(C.Structure):
    _fields_ = [("camera", Camera), ("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("max_depth", C.c_int32),
                ("n_lights", C.c_int32), ("lights", C.c_int32 * 8)]

    @property
    def light_ids(self) -> list[int]:
        """The emitters the scene's author names for light sampling (pass them to Scene.sample_lights)."""
        return [int(self.lights[i]) for i in range(self.n_lights)]


RAY_DTYPE = np.dtype([("o", np.float32, 3), ("time", np.float32), ("d", np.float32, 3), ("pad", np.float32)])
HIT_DTYPE = np.dtype([("t", np.float32), ("prim", np.int32), ("object", np.int32), ("material", np.int32), ("p", np.float32, 3),
                      ("n", np.float32, 3), ("front_face", np.int32), ("u", np.float32), ("v", np.float32), ("nodes_visited", np.int32), ("prims_tested", np.int32), ("pad", np.int32)])
BVH_NODE_DTYPE = np.dtype([("bmin", np.float32, 3), ("bmax", np.float32, 3), ("left_child_idx", np.int32), ("right_child_hittable_idx", np.int32)])
assert RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 64 and BVH_NODE_DTYPE.itemsize == 32

# every symbol include/rtb.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_F3 = C.POINTER(C.c_float)
ABI = {
    "rtb_abi_version": (C.c_int, []),
    "rtb_last_error": (C.c_char_p, []),
    "rtb_scene_create": (C.c_int, [C.POINTER(_P)]),
    "rtb_scene_destroy": (None, [_P]),
    "rtb_add_solid_texture": (C.c_int, [_P, _F3]),
    "rtb_add_checker_texture": (C.c_int, [_P, C.c_float, C.c_int, C.c_int]),
    "rtb_add_image_texture": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int]),
    "rtb_add_noise_texture": (C.c_int, [_P, C.c_float, C.c_uint32]),
    "rtb_add_lambertian": (C.c_int, [_P, C.c_int]),
    "rtb_add_lambertian_color": (C.c_int, [_P, _F3]),
    "rtb_add_metal": (C.c_int, [_P, _F3, C.c_float]),
    "rtb_add_dielectric": (C.c_int, [_P, _F3, C.c_float]),
    "rtb_add_diffuse_light": (C.c_int, [_P, C.c_int]),
    "rtb_add_isotropic": (C.c_int, [_P, C.c_int]),
    "rtb_add_rough_metal": (C.c_int, [_P, _F3, C.c_float]),
    "rtb_add_rough_dielectric": (C.c_int, [_P, _F3, C.c_float, C.c_float]),
    "rtb_add_sphere": (C.c_int, [_P, _F3, C.c_float, C.c_int]),
    "rtb_add_moving_sphere": (C.c_int, [_P, _F3, _F3, C.c_float, C.c_int]),
    "rtb_add_quad": (C.c_int, [_P, _F3, _F3, _F3, C.c_int]),
    "rtb_add_triangle": (C.c_int, [_P, _F3, _F3, _F3, C.c_int]),
    "rtb_add_box": (C.c_int, [_P, _F3, _F3, C.c_int]),
    "rtb_add_list": (C.c_int, [_P, C.POINTER(C.c_int), C.c_int]),
    "rtb_add_bvh": (C.c_int, [_P, C.POINTER(C.c_int), C.c_int, C.c_int]),
    "rtb_add_mesh": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int]),
    "rtb_add_mesh_ex": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P, C.c_int]),
    "rtb_add_translate": (C.c_int, [_P, C.c_int, _F3]),
    "rtb_add_rotate_y": (C.c_int, [_P, C.c_int, C.c_float]),
    "rtb_add_constant_medium": (C.c_int, [_P, C.c_int, C.c_float, C.c_int]),
    "rtb_scene_set_root": (C.c_int, [_P, C.c_int]),
    "rtb_scene_set_background": (C.c_int, [_P, C.c_int, _F3]),
    "rtb_scene_set_world_bvh": (C.c_int, [_P, C.c_int]),
    "rtb_scene_set_sampled_lights": (C.c_int, [_P, C.POINTER(C.c_int), C.c_int]),
    "rtb_scene_set_environment": (C.c_int, [_P, _P, C.c_int, C.c_int, _F3, C.c_int]),
    "rtb_scene_num_children": (C.c_int, [_P, C.c_int]),
    "rtb_scene_num_objects": (C.c_int, [_P]),
    "rtb_object_bounds": (C.c_int, [_P, C.c_int, _F3]),
    "rtb_scene_serialize": (C.c_size_t, [_P, _P, C.c_size_t]),
    "rtb_bvh_build": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, C.POINTER(C.c_int)]),
    "rtb_scene_world_bvh": (C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_int)]),
    "rtb_scene_flatten_hash": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "rtb_scene_flatten_stats": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "rtb_camera_pinhole": (C.c_int, [C.POINTER(Camera), _F3, _F3, _F3, C.c_float, C.c_float]),
    "rtb_camera_defocus": (C.c_int, [C.POINTER(Camera), _F3, _F3, _F3, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float]),
    "rtb_camera_motion": (C.c_int, [C.POINTER(Camera), _F3, _F3, _F3, C.c_float, C.c_float, C.c_float, C.c_float]),
    "rtb_device_count": (C.c_int, []),
    "rtb_renderer_create": (C.c_int, [C.POINTER(_P), C.c_int]),
    "rtb_renderer_destroy": (None, [_P]),
    "rtb_renderer_set_scene": (C.c_int, [_P, _P]),
    "rtb_renderer_set_camera": (C.c_int, [_P, C.POINTER(Camera)]),
    "rtb_renderer_scene_bytes": (C.c_size_t, [_P]),
    "rtb_renderer_scene_stats": (C.c_int, [_P, C.POINTER(SceneStats)]),
    "rtb_render": (C.c_int, [_P, C.POINTER(RenderParams), _P]),
    "rtb_synchronize": (C.c_int, [_P]),
    "rtb_renderer_accum_ptr": (_P, [_P]),
    "rtb_renderer_accum2_ptr": (_P, [_P]),
    "rtb_resolve": (C.c_int, [_P, _P, _P]),
    "rtb_download": (C.c_int, [_P, _P]),
    "rtb_download_accum": (C.c_int, [_P, _P, _P]),
    "rtb_get_counters": (C.c_int, [_P, C.POINTER(Counters)]),
    "rtb_render_adaptive": (C.c_int, [_P, C.POINTER(RenderParams), C.POINTER(AdaptiveParams), C.POINTER(AdaptiveStats), _P]),
    "rtb_reset_counters": (C.c_int, [_P]),
    "rtb_queue_lengths": (C.c_int, [_P, _P, C.c_int]),
    "rtb_renderer_set_profiling": (C.c_int, [_P, C.c_int]),
    "rtb_get_profile": (C.c_int, [_P, C.POINTER(Profile)]),
    "rtb_trace_rays": (C.c_int, [_P, _P, C.c_size_t, _P]),
    "rtb_download_rgb8": (C.c_int, [_P, _P, C.c_int]),
    "rtb_renderer_share_scene": (C.c_int, [_P, _P]),
    "rtb_save_accum": (C.c_int, [_P, C.c_char_p]),
    "rtb_load_accum": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "rtb_renderer_sample_cursor": (C.c_uint32, [_P]),
    "rtb_get_profile_launches": (C.c_int, [_P, _P, _P, C.c_int]),
    "rtb_debug_bounds_report": (C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_uint64)]),
    "rtb_multi_renderer_create": (C.c_int, [C.POINTER(_P), C.POINTER(C.c_int), C.c_int, C.c_int]),
    "rtb_multi_renderer_destroy": (None, [_P]),
    "rtb_multi_device_count": (C.c_int, [_P]),
    "rtb_multi_renderer_get": (_P, [_P, C.c_int]),
    "rtb_multi_reduce_mode": (C.c_int, [_P]),
    "rtb_multi_set_scene": (C.c_int, [_P, _P]),
    "rtb_multi_set_camera": (C.c_int, [_P, C.POINTER(Camera)]),
    "rtb_multi_render": (C.c_int, [_P, C.POINTER(RenderParams)]),
    "rtb_multi_synchronize": (C.c_int, [_P]),
    "rtb_multi_download": (C.c_int, [_P, _P]),
    "rtb_multi_download_accum": (C.c_int, [_P, _P, _P]),
    "rtb_multi_download_rgb8": (C.c_int, [_P, _P, C.c_int]),
    "rtb_multi_get_counters": (C.c_int, [_P, C.POINTER(Counters)]),
    "rtb_multi_reset_counters": (C.c_int, [_P]),
}
SCENES_ABI = {
    "rtb_scenes_count": (C.c_int, []),
    "rtb_scenes_name": (C.c_char_p, [C.c_int]),
    "rtb_scenes_build": (_P, [C.c_char_p, C.POINTER(SceneInfo)]),
    "rtb_scenes_last_error": (C.c_char_p, []),
}

_lib = None
_scenes = None


def lib() -> C.CDLL:
    """The CUDA C-ABI library.  Missing library = hard error (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RtbError(f"{LIB_PATH} is missing: run __graft_entry__.build() (make -C {_HERE}); there is no CPU fallback")
        h = C.CDLL(str(LIB_PATH), mode=C.RTLD_GLOBAL)
        for name, (res, args) in ABI.items():
            fn = getattr(h, name)
            fn.restype, fn.argtypes = res, args
        if h.rtb_abi_version() != 1:
            raise RtbError("librtb200.so ABI version mismatch")
        _lib = h
    return _lib


def scenes_lib() -> C.CDLL:
    global _scenes
    if _scenes is None:
        lib()
        if not SCENES_LIB_PATH.exists():
            raise RtbError(f"{SCENES_LIB_PATH} is missing: run __graft_entry__.build()")
        h = C.CDLL(str(SCENES_LIB_PATH), mode=C.RTLD_GLOBAL)
        for name, (res, args) in SCENES_ABI.items():
            fn = getattr(h, name)
            fn.restype, fn.argtypes = res, args
        _scenes = h
    return _scenes


def _check(rc: int, what: str) -> int:
    if rc < 0:
        raise RtbError(f"{what}: {lib().rtb_last_error().decode()} (status {rc})")
    return rc


def _f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


def scene_names() -> list[str]:
    s = scenes_lib()
    return [s.rtb_scenes_name(i).decode() for i in range(s.rtb_scenes_count())]


def make_camera(kind: str, lookfrom, lookat, up=(0, 1, 0), vfov=40.0, aspect=1.0, aperture=0.0, focus_dist=1.0, t0=0.0, t1=0.0) -> Camera:
    cam = Camera()
    if kind == "pinhole":
        _check(lib().rtb_camera_pinhole(C.byref(cam), _f3(lookfrom), _f3(lookat), _f3(up), vfov, aspect), "rtb_camera_pinhole")
    elif kind == "defocus":
        _check(lib().rtb_camera_defocus(C.byref(cam), _f3(lookfrom), _f3(lookat), _f3(up), vfov, aspect, aperture, focus_dist, t0, t1), "rtb_camera_defocus")
    elif kind == "motion":
        _check(lib().rtb_camera_motion(C.byref(cam), _f3(lookfrom), _f3(lookat), _f3(up), vfov, aspect, t0, t1), "rtb_camera_motion")
    else:
        raise ValueError(kind)
    return cam


def sample_range(spp_total: int, rank: int, world: int) -> tuple[int, int]:
    """Sample-range partition of a render job: rank r of `world` renders samples [begin, end) of every pixel.
    Contiguous, covers [0, spp_total) exactly, sizes differ by at most one."""
    return (spp_total * rank) // world, (spp_total * (rank + 1)) // world


def row_range(height: int, rank: int, world: int) -> tuple[int, int]:
    """Image-tile (row band) partition, for renders that are split by tile instead of by sample range."""
    return (height * rank) // world, (height * (rank + 1)) // world


def bvh_build(aabbs: np.ndarray, builder: int = BVH_TOPDOWN_MEDIAN):
    """rtb_bvh_build: (nodes, order, root) exactly as BVH_Handle::Factory produces them."""
    a = np.ascontiguousarray(aabbs, dtype=np.float32).reshape(-1, 6)
    n = a.shape[0]
    nodes = np.zeros(2 * n, dtype=BVH_NODE_DTYPE)
    order = np.zeros(n, dtype=np.int32)
    root = C.c_int(-1)
    cnt = _check(lib().rtb_bvh_build(a.ctypes.data, n, builder, nodes.ctypes.data, order.ctypes.data, C.byref(root)), "rtb_bvh_build")
    return nodes[:cnt].copy(), order, root.value


class Scene:
    """Owns an rtb_scene*.  Build one with Scene.named(<registry name>) or through the add_* calls."""

    def __init__(self, handle=None):
        if handle is None:
            h = _P()
            _check(lib().rtb_scene_create(C.byref(h)), "rtb_scene_create")
            handle = h.value
        self.handle = handle
        self.info: SceneInfo | None = None

    @classmethod
    def named(cls, name: str) -> "Scene":
        info = SceneInfo()
        h = scenes_lib().rtb_scenes_build(name.encode(), C.byref(info))
        if not h:
            raise RtbError(f"rtb_scenes_build({name}): {scenes_lib().rtb_scenes_last_error().decode()}")
        s = cls(h)
        s.info = info
        return s

    def __del__(self):
        if getattr(self, "handle", None) and _lib is not None:
            _lib.rtb_scene_destroy(self.handle)
            self.handle = None

    # -- thin wrappers -------------------------------------------------------------------------
    def solid(self, rgb): return _check(lib().rtb_add_solid_texture(self.handle, _f3(rgb)), "rtb_add_solid_texture")
    def checker(self, scale, even, odd): return _check(lib().rtb_add_checker_texture(self.handle, scale, even, odd), "rtb_add_checker_texture")
    def image(self, pixels: np.ndarray):
        px = np.ascontiguousarray(pixels, dtype=np.uint8)
        h, w = px.shape[:2]
        ch = 1 if px.ndim == 2 else px.shape[2]
        return _check(lib().rtb_add_image_texture(self.handle, px.ctypes.data, w, h, ch), "rtb_add_image_texture")
    def noise(self, scale, seed=1984): return _check(lib().rtb_add_noise_texture(self.handle, scale, seed), "rtb_add_noise_texture")
    def lambertian(self, albedo=None, tex=None):
        if tex is not None:
            return _check(lib().rtb_add_lambertian(self.handle, tex), "rtb_add_lambertian")
        return _check(lib().rtb_add_lambertian_color(self.handle, _f3(albedo)), "rtb_add_lambertian_color")
    def metal(self, albedo, fuzz): return _check(lib().rtb_add_metal(self.handle, _f3(albedo), fuzz), "rtb_add_metal")
    def dielectric(self, ior, albedo=(1, 1, 1)): return _check(lib().rtb_add_dielectric(self.handle, _f3(albedo), ior), "rtb_add_dielectric")
    def diffuse_light(self, tex): return _check(lib().rtb_add_diffuse_light(self.handle, tex), "rtb_add_diffuse_light")
    def isotropic(self, tex): return _check(lib().rtb_add_isotropic(self.handle, tex), "rtb_add_isotropic")
    def rough_metal(self, f0, alpha):
        """GGX conductor: Schlick Fresnel from the per-channel reflectance f0, width alpha in [0.001, 1] (DESIGN.md §5f)."""
        return _check(lib().rtb_add_rough_metal(self.handle, _f3(f0), alpha), "rtb_add_rough_metal")
    def rough_dielectric(self, ior, alpha, albedo=(1, 1, 1)):
        """GGX glass: the dielectric's Schlick reflect / refract choice about a visible normal of width alpha in [0.001, 1]."""
        return _check(lib().rtb_add_rough_dielectric(self.handle, _f3(albedo), ior, alpha), "rtb_add_rough_dielectric")
    def sphere(self, c, r, mat): return _check(lib().rtb_add_sphere(self.handle, _f3(c), r, mat), "rtb_add_sphere")
    def moving_sphere(self, c0, c1, r, mat): return _check(lib().rtb_add_moving_sphere(self.handle, _f3(c0), _f3(c1), r, mat), "rtb_add_moving_sphere")
    def quad(self, Q, u, v, mat): return _check(lib().rtb_add_quad(self.handle, _f3(Q), _f3(u), _f3(v), mat), "rtb_add_quad")
    def triangle(self, Q, u, v, mat): return _check(lib().rtb_add_triangle(self.handle, _f3(Q), _f3(u), _f3(v), mat), "rtb_add_triangle")
    def box(self, a, b, mat): return _check(lib().rtb_add_box(self.handle, _f3(a), _f3(b), mat), "rtb_add_box")
    def list(self, children):
        arr = (C.c_int * len(children))(*children)
        return _check(lib().rtb_add_list(self.handle, arr, len(children)), "rtb_add_list")
    def bvh(self, children, builder=BVH_TOPDOWN_MEDIAN):
        arr = (C.c_int * len(children))(*children)
        return _check(lib().rtb_add_bvh(self.handle, arr, len(children), builder), "rtb_add_bvh")
    def mesh(self, vertices, indices, mat, normals=None, uvs=None):
        """Triangle mesh from (n, 3) float32 vertices and (m, 3) int32 vertex indices: one BVH group of triangles.
        normals (n, 3) and uvs (n, 2), per vertex, make it smooth-shaded and texture-mapped (rtb_add_mesh_ex,
        DESIGN.md §5e)."""
        v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3); i = np.ascontiguousarray(indices, dtype=np.int32).reshape(-1, 3)
        if normals is None and uvs is None:
            return _check(lib().rtb_add_mesh(self.handle, v.ctypes.data, len(v), i.ctypes.data, len(i), mat), "rtb_add_mesh")
        n = None if normals is None else np.ascontiguousarray(normals, dtype=np.float32).reshape(-1, 3)
        t = None if uvs is None else np.ascontiguousarray(uvs, dtype=np.float32).reshape(-1, 2)
        for name, a in (("normals", n), ("uvs", t)):
            if a is not None and len(a) != len(v):
                raise ValueError(f"mesh: {name} has {len(a)} rows for {len(v)} vertices")
        return _check(lib().rtb_add_mesh_ex(self.handle, v.ctypes.data, len(v), i.ctypes.data, len(i),
                                            None if n is None else n.ctypes.data, None if t is None else t.ctypes.data, mat),
                      "rtb_add_mesh_ex")

    def translate(self, child, off): return _check(lib().rtb_add_translate(self.handle, child, _f3(off)), "rtb_add_translate")
    def rotate_y(self, child, deg): return _check(lib().rtb_add_rotate_y(self.handle, child, deg), "rtb_add_rotate_y")
    def constant_medium(self, boundary, density, phase): return _check(lib().rtb_add_constant_medium(self.handle, boundary, density, phase), "rtb_add_constant_medium")
    def set_root(self, obj): _check(lib().rtb_scene_set_root(self.handle, obj), "rtb_scene_set_root")
    def set_background(self, mode, rgb=(0, 0, 0)): _check(lib().rtb_scene_set_background(self.handle, mode, _f3(rgb)), "rtb_scene_set_background")
    def set_world_bvh(self, mode): _check(lib().rtb_scene_set_world_bvh(self.handle, mode), "rtb_scene_set_world_bvh")
    def sample_lights(self, ids):
        """Light importance sampling towards these objects (spheres / quads, optionally under translate / rotate_y);
        an empty list turns it off (rtb_scene_set_sampled_lights)."""
        ids = [int(i) for i in ids]
        arr = (C.c_int * max(len(ids), 1))(*ids)
        _check(lib().rtb_scene_set_sampled_lights(self.handle, arr, len(ids)), "rtb_scene_set_sampled_lights")
    def set_environment(self, rgb, scale=(1.0, 1.0, 1.0), sample=False):
        """HDR environment map (rtb_scene_set_environment): an (H, W, 3) float32 equirectangular map, row 0 at the top
        (+y), multiplied per channel by `scale`; it replaces the background for every ray that leaves the scene.
        sample=True importance-samples it in the light mixture.  None clears it (the background applies again)."""
        if rgb is None:
            _check(lib().rtb_scene_set_environment(self.handle, None, 0, 0, _f3(scale), 0), "rtb_scene_set_environment")
            return
        px = np.asarray(rgb)
        if px.ndim != 3 or px.shape[2] != 3:
            raise ValueError(f"set_environment: expected an (H, W, 3) array, got shape {px.shape}")
        px = np.ascontiguousarray(px, dtype=np.float32)
        h, w = px.shape[:2]
        _check(lib().rtb_scene_set_environment(self.handle, px.ctypes.data, w, h, _f3(scale), ENV_SAMPLE if sample else 0),
               "rtb_scene_set_environment")
    def num_objects(self): return lib().rtb_scene_num_objects(self.handle)

    def bounds(self, obj) -> np.ndarray:
        out = (C.c_float * 6)()
        _check(lib().rtb_object_bounds(self.handle, obj, out), "rtb_object_bounds")
        return np.array(out[:], dtype=np.float32)

    def serialize(self) -> bytes:
        n = lib().rtb_scene_serialize(self.handle, None, 0)
        buf = C.create_string_buffer(n)
        lib().rtb_scene_serialize(self.handle, buf, n)
        return buf.raw

    def flatten_stats(self) -> dict:
        out = (C.c_int32 * 4)()
        _check(lib().rtb_scene_flatten_stats(self.handle, out), "rtb_scene_flatten_stats")
        return {"primitives": out[0], "record_slots": out[1], "inner_nodes": out[2], "depth": out[3]}

    def flatten_hash(self) -> int:
        h = C.c_uint64(0)
        _check(lib().rtb_scene_flatten_hash(self.handle, C.byref(h)), "rtb_scene_flatten_hash")
        return int(h.value)

    def world_bvh(self):
        root = C.c_int(-1)
        n = _check(lib().rtb_scene_world_bvh(self.handle, None, 0, C.byref(root)), "rtb_scene_world_bvh")
        nodes = np.zeros(n, dtype=BVH_NODE_DTYPE)
        _check(lib().rtb_scene_world_bvh(self.handle, nodes.ctypes.data, n, C.byref(root)), "rtb_scene_world_bvh")
        return nodes, root.value


class Renderer:
    """Owns an rtb_renderer* on one CUDA device."""

    def __init__(self, device: int = 0):
        h = _P()
        _check(lib().rtb_renderer_create(C.byref(h), device), "rtb_renderer_create")
        self.handle = h.value
        self.device = device
        self.width = self.height = 0
        self._scene = None

    def __del__(self):
        if getattr(self, "handle", None) and _lib is not None:
            _lib.rtb_renderer_destroy(self.handle)
            self.handle = None

    def set_scene(self, scene: Scene):
        _check(lib().rtb_renderer_set_scene(self.handle, scene.handle), "rtb_renderer_set_scene")
        self._scene = scene

    def scene_bytes(self) -> int:
        return int(lib().rtb_renderer_scene_bytes(self.handle))

    def scene_stats(self) -> dict:
        """Sizes, builder and host build times of the scene last flattened by set_scene (rtb_scene_stats)."""
        st = SceneStats()
        _check(lib().rtb_renderer_scene_stats(self.handle, C.byref(st)), "rtb_renderer_scene_stats")
        return {"primitives": st.primitives, "record_slots": st.record_slots, "inner_nodes": st.inner_nodes, "depth": st.depth,
                "builder": BUILDER_NAMES.get(st.builder, str(st.builder)), "flatten_ms": st.flatten_ms, "bvh_build_ms": st.bvh_build_ms}

    def set_camera(self, cam: Camera):
        _check(lib().rtb_renderer_set_camera(self.handle, C.byref(cam)), "rtb_renderer_set_camera")

    def render(self, width, height, sample_begin, sample_end, max_depth, seed=1984, clear=True, variance=False,
               rows=(0, 0), samples_per_batch=0, stream=None):
        p = RenderParams(width, height, sample_begin, sample_end, rows[0], rows[1], max_depth, seed,
                         (RENDER_CLEAR if clear else 0) | (RENDER_VARIANCE if variance else 0), samples_per_batch)
        _check(lib().rtb_render(self.handle, C.byref(p), stream), "rtb_render")
        self.width, self.height = width, height

    def render_adaptive(self, width, height, max_spp, max_depth, *, tolerance=None, target_db=None, min_spp=64, max_rounds=0,
                        seed=1984, clear=True, rows=(0, 0), samples_per_batch=0, stream=None) -> dict:
        """Adaptive sampling (rtb_render_adaptive, DESIGN.md §5c): rounds of samples for the pixels whose display-space
        standard error (maximum over their 3x3 neighbourhood) is above `tolerance` - or tolerance_for_db(target_db) - after
        at least min_spp samples, up to max_spp.  Blocks.  Without `clear` it continues from what the accumulators hold.
        Returns the call's rounds, sample cursor, active pixels left and camera paths; per-pixel counts are in
        download_accum()[..., 3]."""
        if (tolerance is None) == (target_db is None):
            raise ValueError("render_adaptive: give exactly one of tolerance and target_db")
        tol = float(tolerance) if tolerance is not None else tolerance_for_db(target_db)
        p = RenderParams(width, height, 0, max_spp, rows[0], rows[1], max_depth, seed,
                         (RENDER_CLEAR if clear else 0) | RENDER_VARIANCE, samples_per_batch)
        a = AdaptiveParams(tol, min_spp, max_rounds, 0)
        st = AdaptiveStats()
        _check(lib().rtb_render_adaptive(self.handle, C.byref(p), C.byref(a), C.byref(st), stream), "rtb_render_adaptive")
        self.width, self.height = width, height
        return {"rounds": int(st.rounds), "cursor": int(st.cursor), "active_pixels": int(st.active_pixels), "samples": int(st.samples)}

    def synchronize(self):
        _check(lib().rtb_synchronize(self.handle), "rtb_synchronize")

    def resolve(self, d_out=None, stream=None):
        _check(lib().rtb_resolve(self.handle, d_out, stream), "rtb_resolve")

    def download(self) -> np.ndarray:
        out = np.empty((self.height, self.width, 4), dtype=np.float32)
        _check(lib().rtb_download(self.handle, out.ctypes.data), "rtb_download")
        return out

    def download_into(self, host_ptr: int):
        _check(lib().rtb_download(self.handle, host_ptr), "rtb_download")

    def download_accum(self, want_sum2=False):
        s = np.empty((self.height, self.width, 4), dtype=np.float32)
        s2 = np.empty_like(s) if want_sum2 else None
        _check(lib().rtb_download_accum(self.handle, s.ctypes.data, s2.ctypes.data if want_sum2 else None), "rtb_download_accum")
        return (s, s2) if want_sum2 else s

    def accum_ptr(self) -> int:
        return lib().rtb_renderer_accum_ptr(self.handle)

    def counters(self) -> Counters:
        c = Counters()
        _check(lib().rtb_get_counters(self.handle, C.byref(c)), "rtb_get_counters")
        return c

    def queue_lengths(self, cap: int = 256) -> np.ndarray:
        out = np.zeros(cap, dtype=np.uint32)
        n = _check(lib().rtb_queue_lengths(self.handle, out.ctypes.data, cap), "rtb_queue_lengths")
        return out[:min(n, cap)]

    def set_profiling(self, on: bool):
        _check(lib().rtb_renderer_set_profiling(self.handle, 1 if on else 0), "rtb_renderer_set_profiling")

    def profile(self) -> Profile:
        p = Profile()
        _check(lib().rtb_get_profile(self.handle, C.byref(p)), "rtb_get_profile")
        return p

    def reset_counters(self):
        _check(lib().rtb_reset_counters(self.handle), "rtb_reset_counters")

    def trace_rays(self, rays: np.ndarray) -> np.ndarray:
        r = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.zeros(r.shape[0], dtype=HIT_DTYPE)
        _check(lib().rtb_trace_rays(self.handle, r.ctypes.data, r.shape[0], hits.ctypes.data), "rtb_trace_rays")
        return hits

    def download_rgb8(self, flip_rows: bool = True) -> np.ndarray:
        """The 8-bit image FirstApp::write_renderbuffer writes (x * 255.999, RGB, rows flipped), quantised on the device."""
        out = np.empty((self.height, self.width, 3), dtype=np.uint8)
        _check(lib().rtb_download_rgb8(self.handle, out.ctypes.data, 1 if flip_rows else 0), "rtb_download_rgb8")
        return out

    def share_scene(self, src: "Renderer"):
        _check(lib().rtb_renderer_share_scene(self.handle, src.handle), "rtb_renderer_share_scene")

    def save_accum(self, path):
        _check(lib().rtb_save_accum(self.handle, str(path).encode()), "rtb_save_accum")

    def load_accum(self, path) -> int:
        """Loads a checkpoint; returns the sample cursor (pass it as sample_begin with clear=False to continue)."""
        w, h, cur = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
        _check(lib().rtb_load_accum(self.handle, str(path).encode(), C.byref(w), C.byref(h), C.byref(cur)), "rtb_load_accum")
        self.width, self.height = int(w.value), int(h.value)
        return int(cur.value)

    def sample_cursor(self) -> int:
        return int(lib().rtb_renderer_sample_cursor(self.handle))

    def profile_launches(self, cap: int = 4096):
        """(ms, class) of every launch of the profiled renders since the last profile() call, in launch order."""
        ms = np.zeros(cap, dtype=np.float32); cls = np.zeros(cap, dtype=np.int32)
        n = _check(lib().rtb_get_profile_launches(self.handle, ms.ctypes.data, cls.ctypes.data, cap), "rtb_get_profile_launches")
        n = min(n, cap)
        return ms[:n].copy(), cls[:n].copy()

    def debug_bounds_report(self) -> dict:
        """Out-of-range indices counted by the kernels of the debug build (RTB_LIB=librtb200_debug.so); raises with the release library."""
        v = (C.c_uint64 * 8)(); checks = C.c_uint64(0)
        _check(lib().rtb_debug_bounds_report(self.handle, v, 8, C.byref(checks)), "rtb_debug_bounds_report")
        out = {name: int(v[i]) for i, name in enumerate(BOUNDS_CLASSES)}
        out["rays_checked"] = int(checks.value)
        return out

    def accum_tensor(self):
        """The device accumulator as a torch tensor (H, W, 4) sharing memory — used for the NCCL reduce."""
        import torch

        class _Wrap:
            pass
        w = _Wrap()
        w.__cuda_array_interface__ = {"shape": (self.height, self.width, 4), "typestr": "<f4", "data": (self.accum_ptr(), False), "version": 3}
        return torch.as_tensor(w, device=f"cuda:{self.device}")


class MultiRenderer:
    """Owns an rtb_multi_renderer*: one process, several GPUs of one box (sample-range partition + one reduce)."""

    def __init__(self, devices, reduce=REDUCE_AUTO):
        devs = list(range(devices)) if isinstance(devices, int) else list(devices)
        arr = (C.c_int * len(devs))(*devs)
        h = _P()
        _check(lib().rtb_multi_renderer_create(C.byref(h), arr, len(devs), reduce), "rtb_multi_renderer_create")
        self.handle = h.value
        self.devices = devs
        self.width = self.height = 0
        self._scene = None

    def __del__(self):
        if getattr(self, "handle", None) and _lib is not None:
            _lib.rtb_multi_renderer_destroy(self.handle)
            self.handle = None

    @property
    def reduce_mode(self) -> str:
        return {REDUCE_NCCL: "nccl", REDUCE_P2P: "p2p"}.get(lib().rtb_multi_reduce_mode(self.handle), "?")

    def set_scene(self, scene: Scene):
        _check(lib().rtb_multi_set_scene(self.handle, scene.handle), "rtb_multi_set_scene")
        self._scene = scene

    def set_camera(self, cam: Camera):
        _check(lib().rtb_multi_set_camera(self.handle, C.byref(cam)), "rtb_multi_set_camera")

    def render(self, width, height, sample_begin, sample_end, max_depth, seed=1984, clear=True, variance=False, samples_per_batch=0):
        p = RenderParams(width, height, sample_begin, sample_end, 0, 0, max_depth, seed,
                         (RENDER_CLEAR if clear else 0) | (RENDER_VARIANCE if variance else 0), samples_per_batch)
        _check(lib().rtb_multi_render(self.handle, C.byref(p)), "rtb_multi_render")
        self.width, self.height = width, height

    def synchronize(self):
        _check(lib().rtb_multi_synchronize(self.handle), "rtb_multi_synchronize")

    def download(self) -> np.ndarray:
        out = np.empty((self.height, self.width, 4), dtype=np.float32)
        _check(lib().rtb_multi_download(self.handle, out.ctypes.data), "rtb_multi_download")
        return out

    def download_into(self, host_ptr: int):
        _check(lib().rtb_multi_download(self.handle, host_ptr), "rtb_multi_download")

    def download_accum(self, want_sum2=False):
        s = np.empty((self.height, self.width, 4), dtype=np.float32)
        s2 = np.empty_like(s) if want_sum2 else None
        _check(lib().rtb_multi_download_accum(self.handle, s.ctypes.data, s2.ctypes.data if want_sum2 else None), "rtb_multi_download_accum")
        return (s, s2) if want_sum2 else s

    def download_rgb8(self, flip_rows: bool = True) -> np.ndarray:
        out = np.empty((self.height, self.width, 3), dtype=np.uint8)
        _check(lib().rtb_multi_download_rgb8(self.handle, out.ctypes.data, 1 if flip_rows else 0), "rtb_multi_download_rgb8")
        return out

    def counters(self) -> Counters:
        c = Counters()
        _check(lib().rtb_multi_get_counters(self.handle, C.byref(c)), "rtb_multi_get_counters")
        return c

    def reset_counters(self):
        _check(lib().rtb_multi_reset_counters(self.handle), "rtb_multi_reset_counters")
