"""TEST INFRASTRUCTURE: one scene builder whose switches pick, one by one, the template instantiations the kernel launchers
choose from, and the case list that the schedule tests (tests/test_gpu_schedules.py, tests/test_gpu_adaptive_scale.py) run.
Nothing here renders.  The shade and tail kernels are selected by their feature word (rtb_kernels.h), whose scene bits are
decided in one place, where rtb_render.cu stages the flattened scene (SceneView::launch_flags); launch_traverse and
launch_tail in rtb_kernels.cu add the stack size and media variant.

What selects what, as the launchers read a flattened scene:
  media     none; "pre": one medium, tested before the walk (has_media = 1); "bvh": more media than the eight the
            pre-test list holds, the rest are BVH leaves (has_media = 2).  The tail has one MEDIA flag for both.
  tree      "shallow": depth <= 17, the 16-entry traverse stack; "normal": 18-30, 32 entries; "deep": a GPU linear BVH
            deeper than 30 levels, 64 entries (traverse and tail).
  lights    a sampled quad light.  A sampled environment map alone also selects the LIGHTS kernels.
  env       none, "unsampled" or "sampled" (ENV: any map).
  attr      a smooth, UV-mapped, image-textured mesh (ATTR), or the same mesh plain.
  LIST      not a scene property: adaptive rounds (render_adaptive) run the list-mode kernels, dense renders the others.
Every scene keeps a Perlin-textured ground and an image-textured sphere, so texture_kernel runs in each."""
from __future__ import annotations

import itertools
from dataclasses import dataclass

import numpy as np

import mesh_scenes as ms
from helpers import parse_blob

MEDIA = ("none", "pre", "bvh")
TREES = ("shallow", "normal", "deep")
ENVS = ("none", "unsampled", "sampled")
PRE_LIST_MAX = 8            # media tested before the walk (flatten in rtb_scene.cpp); the rest become BVH leaves
SHALLOW_MAX_DEPTH = 17      # launch_traverse: the 16-entry stack up to this depth
NORMAL_MAX_DEPTH = 30       # STACK_SIZE - 2: deeper trees take the 64-entry stack


@dataclass(frozen=True)
class Case:
    media: str = "none"
    tree: str = "normal"
    lights: bool = False
    env: str = "none"
    attr: bool = False

    @property
    def id(self) -> str:
        return f"{self.media}-{self.tree}-{'lamp' if self.lights else 'nolamp'}-env_{self.env}-{'attr' if self.attr else 'plain'}"

    # ---------------------------------------------------------------- what the launchers select
    @property
    def has_media(self) -> int:
        return MEDIA.index(self.media)

    @property
    def LIGHTS(self) -> bool:
        return self.lights or self.env == "sampled"

    @property
    def ENV(self) -> bool:
        return self.env != "none"

    def traverse_kernel(self, list_mode: bool) -> tuple:
        """(MEDIA, STACK, LIST): only the walks with media have list-mode instantiations."""
        return (self.has_media, {"shallow": 16, "normal": 32, "deep": 64}[self.tree], bool(list_mode and self.has_media))

    def shade_kernel(self, list_mode: bool) -> tuple:
        """(LIGHTS, LIST, ENV, ATTR): bits 0-3 of the feature word."""
        return (self.LIGHTS, bool(list_mode), self.ENV, self.attr)

    def tail_kernel(self, list_mode: bool) -> tuple:
        """(MEDIA, STACK, LIGHTS, LIST, ENV, ATTR): the tail's stack is 32 entries unless the tree is deep."""
        return (self.has_media > 0, 64 if self.tree == "deep" else 32, self.LIGHTS, bool(list_mode), self.ENV, self.attr)


def _cases() -> list[Case]:
    """One case per (media or not, deep or not, LIGHTS, ENV, ATTR): the 32 scene-side keys of the tail.  Within a key the
    variants rotate, so that every traverse instantiation and every way of selecting LIGHTS / ENV is met as well."""
    out = []
    light_env = {(False, False): [(False, "none")], (True, False): [(True, "none")], (False, True): [(False, "unsampled")],
                 (True, True): [(False, "sampled"), (True, "unsampled"), (True, "sampled")]}
    for k, (media_any, deep, LIGHTS, ENV, attr) in enumerate(itertools.product((False, True), repeat=5)):
        media = ("pre", "bvh")[(k // 2) % 2] if media_any else "none"
        tree = "deep" if deep else ("shallow", "normal")[(k // 4 + k) % 2]
        variants = light_env[(LIGHTS, ENV)]
        lights, env = variants[k % len(variants)]
        out.append(Case(media, tree, lights, env, attr))
    return out


CASES = _cases()
# the sizes of the cross products the launchers choose from
ALL_SHADE = set(itertools.product((False, True), repeat=4))
ALL_TAIL = set(itertools.product((False, True), (32, 64), (False, True), (False, True), (False, True), (False, True)))
ALL_TRAVERSE = {(m, s, l) for m in (0, 1, 2) for s in (16, 32, 64) for l in ((False,) if m == 0 else (False, True))}


def coverage(cases=CASES) -> dict:
    """{kind: {instantiation: [case ids (+ ", list")]}} over dense renders and adaptive rounds of every case."""
    table = {"traverse": {}, "shade": {}, "tail": {}}
    for c in cases:
        for list_mode in (False, True):
            tag = c.id + (", list" if list_mode else "")
            table["traverse"].setdefault(c.traverse_kernel(list_mode), []).append(tag)
            table["shade"].setdefault(c.shade_kernel(list_mode), []).append(tag)
            table["tail"].setdefault(c.tail_kernel(list_mode), []).append(tag)
    return table


def check_coverage(cases=CASES) -> dict:
    t = coverage(cases)
    for kind, want in (("shade", ALL_SHADE), ("tail", ALL_TAIL), ("traverse", ALL_TRAVERSE)):
        missing = want - set(t[kind])
        assert not missing, f"no case selects the {kind} instantiations {sorted(missing)}"
        assert set(t[kind]) <= want, f"unknown {kind} instantiations {sorted(set(t[kind]) - want)}"
    return t


check_coverage()
assert len(ALL_SHADE) == 16 and len(ALL_TAIL) == 64 and len(ALL_TRAVERSE) == 15


def format_coverage(table) -> str:
    lines = []
    names = {"traverse": "MEDIA, STACK, LIST", "shade": "LIGHTS, LIST, ENV, ATTR", "tail": "MEDIA, STACK, LIGHTS, LIST, ENV, ATTR"}
    for kind in ("traverse", "shade", "tail"):
        lines.append(f"{kind}<{names[kind]}>: {len(table[kind])} instantiations")
        for key in sorted(table[kind]):
            lines.append(f"  {kind}<{', '.join(str(int(x)) for x in key)}>: {'; '.join(table[kind][key])}")
    return "\n".join(lines)


def sky_map() -> np.ndarray:
    j, i = np.mgrid[0:16, 0:32]
    sky = np.stack([0.3 + 0.02 * i, 0.4 + 0.01 * j, np.where(j < 8, 1.2, 0.2)], -1).astype(np.float32)
    sky[3, 5] = 40.0
    return sky


def _deep_chain(s, mat):
    """The deep-tree construction of test_gpu_lbvh_deep_tree_uses_the_deep_stack, below the ground and out of the picture:
    centres at 1000 * 2^-k peel one Morton bit off per level of a linear BVH, and 4,000 spheres sharing one cell add about
    twelve more.  Grouped in a BVH object, so that the oracle walks it in a few steps."""
    off = np.float32([-40.0, -60.0, -40.0])
    ids = [s.sphere(off + (1000.0 * 2.0 ** -k, 0.0, 0.0), 0.02 * 1000.0 * 2.0 ** -k, mat) for k in range(21)]
    ids += [s.sphere(off, 0.05 * (1 + k / 4000.0), mat) for k in range(4000)]
    return s.bvh(ids, builder=0)


def build(rtb, case: Case):
    """(scene, camera) for a case.  The scene's world BVH is the GPU linear BVH for deep trees, else the default SAH tree."""
    s = rtb.Scene()
    objs = []
    noise_ground = s.quad((-6, -1, -6), (12, 0, 0), (0, 0, 12), s.lambertian(tex=s.noise(2.0)))
    objs.append(noise_ground)
    sub = {"shallow": 1, "normal": 3, "deep": 2}[case.tree]
    v, f = ms.icosphere(sub)
    tex = s.lambertian(tex=s.image(ms.checker_image()))
    if case.attr:
        mesh = s.mesh(v, f, tex, normals=v, uvs=ms.sphere_uvs(v))
    else:
        mesh = s.mesh(v, f, s.lambertian((0.7, 0.6, 0.5)))
    objs.append(s.translate(s.rotate_y(mesh, 20.0), (-0.4, 0.0, 0.0)))
    objs.append(s.sphere((1.45, -0.45, 0.4), 0.55, tex))                                  # image texture through sphere (u, v)
    objs.append(s.sphere((0.9, -0.7, 1.3), 0.3, s.dielectric(1.5)))
    objs.append(s.sphere((-1.9, -0.6, 0.9), 0.4, s.metal((0.8, 0.75, 0.7), 0.1)))
    if case.tree == "normal":
        # a Perlin-textured height field of 2 x 256^2 triangles behind the objects: a SAH tree of about 20 levels
        _, P, tris, _, _ = ms.height_field(rtb, 256, smooth=False)
        objs.append(s.translate(s.mesh(P * np.float32(2.5), tris, s.lambertian(tex=s.noise(4.0))), (0.0, -0.6, -3.5)))
    if case.tree == "deep":
        objs.append(_deep_chain(s, s.lambertian((0.5, 0.5, 0.5))))
    fog = s.isotropic(s.solid((0.9, 0.9, 0.9)))
    if case.media == "pre":
        objs.append(s.constant_medium(s.sphere((1.6, 0.5, -0.6), 0.6, s.lambertian((1, 1, 1))), 1.5, fog))
    elif case.media == "bvh":
        for k in range(PRE_LIST_MAX + 3):
            iso = s.isotropic(s.solid((0.2 + 0.06 * k, 0.9 - 0.05 * k, 0.6)))
            boundary = s.sphere((-2.5 + 0.5 * k, 0.9 + 0.12 * (k % 3), -1.2 - 0.1 * k), 0.22, s.lambertian((1, 1, 1)))
            objs.append(s.constant_medium(boundary, 2.0, iso))
    if case.lights:
        lamp = s.quad((-0.5, 2.5, -0.5), (1, 0, 0), (0, 0, 1), s.diffuse_light(s.solid((8, 8, 8))))
        objs.append(lamp)
    s.set_root(s.list(objs))
    if case.lights:
        s.sample_lights([lamp])
    if case.env == "none":
        s.set_background(rtb.BG_CONSTANT, (0.25, 0.3, 0.4) if not case.lights else (0.05, 0.05, 0.08))
    else:
        s.set_environment(sky_map(), sample=(case.env == "sampled"))
    if case.tree == "deep":
        s.set_world_bvh(rtb.WORLD_BVH_GPU_LBVH)
    cam = rtb.make_camera("pinhole", (0.3, 1.0, 4.2), (0, 0, 0), (0, 1, 0), 45.0, 1.5)
    return s, cam


RTB_OBJ_CONSTANT_MEDIUM = 9


def scene_features(blob: bytes) -> dict:
    """Media, sampled lights, map and triangle attributes of an RTBS blob (include/rtb_scene_format.h), read from the bytes
    the oracle reads."""
    h, _, objs, _ = parse_blob(blob)
    off = 48 + int(h["n_textures"]) * 48 + int(h["n_materials"]) * 24 + int(h["n_objects"]) * 64 + int(h["n_children"]) * 4 + int(h["n_blob_bytes"])
    version = int(h["version"])
    n_lights, env_w, env_flags, n_attr = 0, 0, 0, 0
    if version >= 2:
        n_lights = int(np.frombuffer(blob, np.int32, 1, off)[0]); off += 4 + 4 * n_lights
    if version >= 3:
        env_w, env_h, env_flags = (int(x) for x in np.frombuffer(blob, np.int32, 3, off)); off += 24 + env_w * env_h * 12
    if version >= 4:
        n_attr = int(np.frombuffer(blob, np.uint32, 1, off)[0]); off += 4 + 64 * n_attr
    assert off == len(blob), "unexpected RTBS layout"
    return {"n_media": int((objs["kind"] == RTB_OBJ_CONSTANT_MEDIUM).sum()), "n_lights": n_lights, "env": env_w > 0,
            "env_sample": env_w > 0 and bool(env_flags & 1), "attr": n_attr > 0}


def check_selection(case: Case, scene, stats: dict) -> None:
    """The expectations a flattened scene lets one observe: tree depth and builder (stats: Renderer.scene_stats() or, for
    host-built trees, Scene.flatten_stats()), the light list and map flags, the media count against the pre-test list."""
    d = stats["depth"]
    if case.tree == "shallow":
        assert d <= SHALLOW_MAX_DEPTH, (case.id, stats)
    elif case.tree == "normal":
        assert SHALLOW_MAX_DEPTH < d <= NORMAL_MAX_DEPTH, (case.id, stats)
    else:
        assert d > NORMAL_MAX_DEPTH and stats.get("builder") == "gpu_lbvh", (case.id, stats)
    info = scene_features(scene.serialize())
    assert info["n_media"] == {"none": 0, "pre": 1, "bvh": PRE_LIST_MAX + 3}[case.media], (case.id, info)
    assert (info["n_media"] > PRE_LIST_MAX) == (case.has_media == 2)
    assert info["n_lights"] == (1 if case.lights else 0), (case.id, info)
    assert info["env"] == case.ENV and info["env_sample"] == (case.env == "sampled"), (case.id, info)
    assert info["attr"] == case.attr, (case.id, info)
