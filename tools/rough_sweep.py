#!/usr/bin/env python
"""What the GGX microfacet materials cost (DESIGN.md §5f).

A subdivision-6 icosphere (81,920 triangles, smooth: analytic vertex normals) on a ground quad, under the sky gradient and
under the environment sweep's sun-and-sky map (tests/env_scenes.sun_sky_map, 2048 x 1024, 0.5-degree sun, unsampled), in
seven materials: Lambertian, metal (fuzz 0), rough metal at alpha 0.05 and 0.3, dielectric and rough dielectric at alpha
0.05 and 0.3.  For each: the device time of one 800 x 800 frame at 16 spp, depth 20 (best of three after a warm-up),
Mrays/s, and the per-class device times of a profiled render (rtb_get_profile).  Prints one JSON object with the card and
its power limit.

    python tools/rough_sweep.py > profiles/r7_rough_sweep.json
"""
import importlib
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests")); sys.path.insert(0, str(ROOT / "tools"))
import env_scenes as es  # noqa: E402
import mesh_scenes as ms  # noqa: E402
from mesh_attr_sweep import measure  # noqa: E402

MATERIALS = ("lambertian", "metal", "rough_metal_0.05", "rough_metal_0.3", "dielectric", "rough_dielectric_0.05", "rough_dielectric_0.3")


def scene(rtb, material, env):
    s = rtb.Scene()
    v, f = ms.icosphere(6)
    kind, _, a = material.rpartition("_") if material.startswith("rough") else (material, "", "")
    if material == "lambertian":
        mat = s.lambertian((0.7, 0.6, 0.5))
    elif material == "metal":
        mat = s.metal((0.95, 0.64, 0.54), 0.0)
    elif material == "dielectric":
        mat = s.dielectric(1.5)
    elif kind == "rough_metal":
        mat = s.rough_metal((0.95, 0.64, 0.54), float(a))
    else:
        mat = s.rough_dielectric(1.5, float(a))
    ground = s.quad((-6, -1, -6), (12, 0, 0), (0, 0, 12), s.lambertian((0.4, 0.45, 0.35)))
    s.set_root(s.list([ground, s.mesh(v, f, mat, normals=v)]))
    if env is not None:
        s.set_environment(env)
    return s, rtb.make_camera("pinhole", (0.3, 0.9, 3.4), (0, 0, 0), (0, 1, 0), 40.0, 1.0)


def main():
    rtb = importlib.import_module("ray-tracing-v06_b200")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    sun, _ = es.sun_sky_map(2048, 1024, seed=7, sun_deg=0.5)
    r = rtb.Renderer(0)
    rows = []
    for sky, env in (("gradient", None), ("sun_sky", sun)):
        for m in MATERIALS:
            s, cam = scene(rtb, m, env)
            row = {"sky": sky, "material": m, **measure(rtb, r, s, cam)}
            print(json.dumps(row), file=sys.stderr, flush=True)
            rows.append(row)
    print(json.dumps({"what": "subdivision-6 smooth icosphere on a ground quad, 800x800, 16 spp, depth 20: render = best of 3 "
                              "device-synchronised frames; per-class ms from one profiled frame (rtb_get_profile)", "gpu": gpu,
                      "rows": rows}, indent=1))


if __name__ == "__main__":
    main()
