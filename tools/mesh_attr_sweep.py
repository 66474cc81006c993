#!/usr/bin/env python
"""What per-vertex shading normals and texture coordinates cost (DESIGN.md §5e).

Two scenes - the 512 x 512 height field of tools/bvh_build_bench.py (524,288 triangles and a glass ball) and a
subdivision-6 icosphere (81,920 triangles) on a ground quad - each in three variants: flat (rtb_add_mesh), smooth (analytic
vertex normals) and smooth + an image texture mapped through vertex UVs.  The tree and the primitive records are the same in
all three, so traverse should not move; shade pays for the attribute lookup and the interpolation.  For each: the device
time of one 800 x 800 frame at 16 spp, depth 20 (best of three after a warm-up), Mrays/s, and the per-class device times of
a profiled render (rtb_get_profile).  Prints one JSON object with the card and its power limit.

    python tools/mesh_attr_sweep.py > profiles/r6_mesh_attr_sweep.json
"""
import importlib
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import mesh_scenes as ms  # noqa: E402

W, H, SPP, D = 800, 800, 16, 20


def icosphere_scene(rtb, variant):
    s = rtb.Scene()
    v, f = ms.icosphere(6)
    mat = s.lambertian(tex=s.image(ms.checker_image(64, 32))) if variant == "textured" else s.lambertian((0.7, 0.6, 0.5))
    m = s.mesh(v, f, mat, normals=None if variant == "flat" else v, uvs=ms.sphere_uvs(v) if variant == "textured" else None)
    ground = s.quad((-6, -1, -6), (12, 0, 0), (0, 0, 12), s.lambertian((0.4, 0.45, 0.35)))
    s.set_root(s.list([ground, m]))
    return s, rtb.make_camera("pinhole", (0.3, 0.9, 3.4), (0, 0, 0), (0, 1, 0), 40.0, 1.0)


def measure(rtb, r, scene, cam):
    r.set_scene(scene); r.set_camera(cam)
    r.render(W, H, 0, SPP, D, seed=3); r.synchronize()
    best, rays = 1e30, 0
    for _ in range(3):
        r.reset_counters()
        t = time.perf_counter(); r.render(W, H, 0, SPP, D, seed=3); r.synchronize(); dt = time.perf_counter() - t
        best = min(best, dt); rays = r.counters().rays
    r.set_profiling(True)
    r.render(W, H, 0, SPP, D, seed=3); r.synchronize()
    p = r.profile()
    r.set_profiling(False)
    return {"render_ms": round(best * 1e3, 2), "mrays_per_s": round(rays / best / 1e6, 1), "rays": int(rays),
            "traverse_ms": round(p.traverse_ms, 2), "shade_ms": round(p.shade_ms, 2), "tail_ms": round(p.tail_ms, 2),
            "bin_ms": round(p.bin_ms, 2), "generate_ms": round(p.generate_ms, 2), "accumulate_ms": round(p.accumulate_ms, 2)}


def main():
    rtb = importlib.import_module("ray-tracing-v06_b200")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    r = rtb.Renderer(0)
    rows = []
    for name, build in (("height_field_512", lambda v: ms.height_field_scene(rtb, 512, v)), ("icosphere_6", lambda v: icosphere_scene(rtb, v))):
        for variant in ("flat", "smooth", "textured"):
            s, cam = build(variant)
            row = {"scene": name, "variant": variant, **measure(rtb, r, s, cam)}
            print(json.dumps(row), file=sys.stderr, flush=True)
            rows.append(row)
    print(json.dumps({"what": f"{W}x{H}, {SPP} spp, depth {D}: render = best of 3 device-synchronised frames; per-class ms from one "
                              "profiled frame (rtb_get_profile; shade includes texture_kernel)", "gpu": gpu, "rows": rows}, indent=1))


if __name__ == "__main__":
    main()
