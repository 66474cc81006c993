#!/usr/bin/env python
"""What importance sampling of an HDR environment map buys (DESIGN.md §5d, BASELINE.md §4).

The scene: a procedural sun-and-sky map generated from a seed (tests/env_scenes.sun_sky_map: a gradient sky plus a sun
disc that carries about 90 % of the irradiance), 2048 x 1024 texels, over diffuse, metal and glass spheres on a diffuse
ground quad, 640 x 360, depth 16; a 0.5 degree sun (the real one's size) and a 5 degree one.  For the plain map and the
sampled one:

  - the mean per-pixel variance at 256 spp (sampled / plain = the variance ratio);
  - time to 30, 35 and 40 dB between independent renders: two renders with different seeds, doubling the samples (64 ...
    65,536), the PSNR of their tone-mapped images at every count, and the device time of one render at the first count from
    which the PSNR stays at or above the target.  (It is not monotone: at low counts both renders miss the sun almost
    everywhere and agree on a dark image; as paths that find the sun appear, a pixel saturates in one render and not in
    the other, and the PSNR falls before it rises.)

and the set_scene time (flatten, CDF build, upload) of a 4096 x 2048 map, plain and sampled, next to the same scene
without a map.  Prints one JSON object with the card and its power limit.

    python tools/env_sweep.py > profiles/r5_env_sweep.json
"""
import importlib
import json
import math
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import env_scenes as es  # noqa: E402

W, H, D = 640, 360, 16


def tonemap(a):
    return np.sqrt(np.clip(a[..., :3] / np.maximum(a[..., 3:4], 1.0), 0.0, 1.0))


def psnr(a, b):
    mse = float(np.mean((tonemap(a).astype(np.float64) - tonemap(b).astype(np.float64)) ** 2))
    return 99.0 if mse == 0 else 10.0 * math.log10(1.0 / mse)


def scene(rtb, env, sample):
    s = rtb.Scene()
    ground = s.quad((-40, 0, -40), (80, 0, 0), (0, 0, 80), s.lambertian((0.5, 0.5, 0.5)))
    a = s.sphere((-2.2, 1, 0), 1.0, s.lambertian((0.75, 0.3, 0.2)))
    b = s.sphere((0, 1, 0), 1.0, s.metal((0.85, 0.85, 0.9), 0.05))
    c = s.sphere((2.2, 1, 0), 1.0, s.dielectric(1.5))
    s.set_root(s.list([ground, a, b, c]))
    if env is not None:
        s.set_environment(env, sample=sample)
    return s


def time_to(curve, target):
    """The first point of the curve from which the PSNR stays at or above `target` (None: never within the curve)."""
    for k, c in enumerate(curve):
        if all(x["psnr_db"] >= target for x in curve[k:]):
            return c
    return None


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    rtb = importlib.import_module("ray-tracing-v06_b200")
    cam = rtb.make_camera("pinhole", (0, 2.5, 8), (0, 0.8, 0), (0, 1, 0), 40.0, W / H)
    out = {"what": __doc__.split("\n\n")[1].strip(), "gpu": gpu_info(), "map": [2048, 1024], "width": W, "height": H, "depth": D,
           "suns": []}
    targets = (30.0, 35.0, 40.0)
    for sun_deg in (0.5, 5.0):
        env, sun = es.sun_sky_map(2048, 1024, seed=7, sun_deg=sun_deg)
        row = {"sun_deg": sun_deg, "sun_direction": sun.round(4).tolist(), "estimators": []}
        for sample in (False, True):
            s = scene(rtb, env, sample)
            r = rtb.Renderer(0); r.set_scene(s); r.set_camera(cam)
            r.render(W, H, 0, 16, D, seed=1); r.synchronize()                                # warm-up
            r.render(W, H, 0, 256, D, seed=3, variance=True); r.synchronize()
            a, a2 = r.download_accum(want_sum2=True)
            m = a[..., :3].astype(np.float64) / 256
            var = float(np.maximum(a2[..., :3].astype(np.float64) / 256 - m ** 2, 0).mean())
            r2 = rtb.Renderer(0); r2.set_scene(s); r2.set_camera(cam)
            done, spp, ms, curve = 0, 64, 0.0, []
            while spp <= 65536:
                r.render(W, H, done, spp, D, seed=11, clear=(done == 0)); r.synchronize(); ms += r.counters().render_ms
                r2.render(W, H, done, spp, D, seed=22, clear=(done == 0)); r2.synchronize()
                done = spp
                p = psnr(r.download_accum(), r2.download_accum())
                curve.append({"spp": spp, "psnr_db": round(p, 2), "render_ms": round(ms, 1)})
                spp *= 2
            row["estimators"].append({"sampled": sample, "mean_pixel_variance_256spp": var,
                                      "to_db": {f"{t:g}": time_to(curve, t) for t in targets}, "curve": curve})
        plain, samp = row["estimators"]
        row["variance_ratio_sampled_over_plain"] = samp["mean_pixel_variance_256spp"] / plain["mean_pixel_variance_256spp"]
        row["time_ratio_sampled_over_plain"] = {k: (samp["to_db"][k]["render_ms"] / plain["to_db"][k]["render_ms"])
                                                if plain["to_db"][k] and samp["to_db"][k] else None for k in plain["to_db"]}
        out["suns"].append(row)

    big, _ = es.sun_sky_map(4096, 2048, seed=7, sun_deg=0.5)
    timing = {}
    for label, env_map, sample in (("no_map", None, False), ("map_4096x2048", big, False), ("map_4096x2048_sampled", big, True)):
        rows = []
        for _ in range(3):
            t = time.perf_counter(); s = scene(rtb, env_map, sample); dt_build = (time.perf_counter() - t) * 1e3
            r = rtb.Renderer(0)
            t = time.perf_counter(); r.set_scene(s); r.synchronize(); dt = (time.perf_counter() - t) * 1e3
            rows.append({"scene_and_set_environment_ms": round(dt_build, 1), "set_scene_ms": round(dt, 1),
                         "flatten_ms": round(r.scene_stats()["flatten_ms"], 1), "arena_mb": round(r.scene_bytes() / 2 ** 20, 1)})
        timing[label] = rows
    out["set_scene"] = timing
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
