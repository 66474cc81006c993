#!/usr/bin/env python
"""How PSNR between two independent renders grows with the sample count (BASELINE.md, north_star's ">= 40 dB at 4096 spp").

For the Cornell-smoke (config 4) and Book 2 final (config 5) scenes at their own sizes: two GPU renders with different
seeds at 1k ... 16k spp each, PSNR on the tone-mapped images (clamp, sqrt) - the Monte Carlo noise floor any two correct
renderers see between each other - plus, at 256 spp, the same-stream comparison with the CPU oracle (how far the GPU image
is from the oracle's when both draw the SAME samples).

    python tools/psnr_sweep.py > profiles/r2_psnr_sweep.json
    python tools/psnr_sweep.py --sample-lights > profiles/r3_psnr_sweep_lights.json

--sample-lights renders with light importance sampling towards the emitters each scene lists (Scene.sample_lights,
DESIGN.md §5b).  Every row also carries the render time per sample (device time of the second seed's renders, the
first seed having warmed up graphs and queues) and what it takes to reach 40 dB: spp_for_40_db x ms_per_spp.
"""
import importlib
import json
import math
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "oracle")); sys.path.insert(0, str(ROOT / "tests"))


def tonemap(a):
    return np.sqrt(np.clip(a[..., :3] / np.maximum(a[..., 3:4], 1.0), 0.0, 1.0))


def psnr(a, b):
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    return 99.0 if mse == 0 else 10.0 * math.log10(1.0 / mse)


if __name__ == "__main__":
    rtb = importlib.import_module("ray-tracing-v06_b200")
    orc = importlib.import_module("pyoracle")
    feature_oracle = importlib.import_module("feature_oracle")
    lights = "--sample-lights" in sys.argv[1:]
    out = []
    for cfg, name in (("4", "book2_cornell_smoke"), ("5", "book2_final")):
        s = rtb.Scene.named(name); i = s.info
        if lights:
            s.sample_lights(i.light_ids)
        r = rtb.Renderer(0); r.set_scene(s); r.set_camera(i.camera)
        W, H, D = i.width, i.height, i.max_depth
        row = {"config": cfg, "scene": name, "width": W, "height": H, "depth": D, "sampled_lights": i.light_ids if lights else [],
               "independent_seeds": []}
        acc = {}
        render_ms = 0.0
        for seed in (11, 22):
            acc[seed] = {}
            done = 0
            for spp in (1024, 2048, 4096, 8192, 16384):
                r.render(W, H, done, spp, D, seed=seed, clear=(done == 0)); r.synchronize()      # progressive: add the missing samples
                if seed == 22:
                    render_ms += r.counters().render_ms
                done = spp
                acc[seed][spp] = r.download_accum().copy()
        row["ms_per_spp"] = round(render_ms / 16384, 5)
        for spp in (1024, 2048, 4096, 8192, 16384):
            row["independent_seeds"].append({"spp": spp, "psnr_db": round(psnr(tonemap(acc[11][spp]), tonemap(acc[22][spp])), 2)})
        p = [x["psnr_db"] for x in row["independent_seeds"]]
        row["db_per_doubling"] = round((p[-1] - p[0]) / 4.0, 2)
        row["spp_for_40_db"] = int(round(1024 * 2.0 ** ((40.0 - p[0]) / max(row["db_per_doubling"], 1e-3))))
        row["seconds_to_40_db"] = round(row["spp_for_40_db"] * row["ms_per_spp"] / 1000.0, 3)
        # same streams, GPU vs oracle (256 spp at a quarter of the size to keep the CPU side short)
        w2, h2 = W // 4, H // 4
        r.render(w2, h2, 0, 256, D, seed=1984); g = r.download_accum()
        cpu = feature_oracle.FeatureOracleScene if lights else orc.OracleScene   # (the CPU integrator with the light mixture)
        o, _, _ = cpu(s.serialize()).render(i.camera, w2, h2, 0, 256, D, seed=1984)
        row["same_streams_vs_oracle"] = {"width": w2, "height": h2, "spp": 256, "psnr_db": round(psnr(tonemap(g), tonemap(o)), 2),
                                         "pixels_differing": float((np.abs(g[..., :3] - o[..., :3]).max(axis=2) > 1e-4 * np.maximum(np.abs(o[..., :3]).max(axis=2), 1.0)).mean())}
        out.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    print(json.dumps(out, indent=1))
