#!/usr/bin/env python
"""Adaptive against uniform sampling (DESIGN.md §5c) on the Cornell-smoke (config 4) and Book 2 final (config 5) scenes at
their own sizes, with and without light sampling, on one GPU.

For every (config, light sampling) pair:
  * reference: a 65,536-spp uniform render with an independent seed (light sampling on: the same expected image, less noise);
  * uniform: progressive renders with seed 11 up to 32,768 spp; PSNR against the reference at every doubling and the device
    time per sample, so the uniform time to any PSNR is interpolated (log-linear in spp between doublings);
  * adaptive: rtb_render_adaptive with target_db = 37 / 40 / 43 (min_spp 64, cap 65,536 on config 4 and 32,768 on config 5)
    with seeds 11 and 22: device time of the whole call (select steps and host syncs included), rounds, mean spp, a histogram
    of per-pixel counts (powers of two), PSNR against the reference and between the two seeds (comparable with the
    independent-seed table of BASELINE.md §4), and the image-mean radiance against the reference's (early stopping is
    slightly biased);
  * the uniform time to the PSNR each adaptive render reached, and the ratio.
Per-round overhead (config 4, light sampling off): one round over (nearly) every pixel - tolerance 0, samples [256, 512) after
a 256-spp render - against the same samples rendered densely through rtb_render (CUDA graph), and the select step's own
device time from a profiled run.

    python tools/adaptive_sweep.py OUT_DIR [--configs 4,5] [--no-overhead]
        # writes OUT_DIR/r4_adaptive_cfg{4,5}_{plain,lights}.json and OUT_DIR/r4_adaptive_overhead.json
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
rtb = importlib.import_module("ray-tracing-v06_b200")

TARGETS = (37, 40, 43)
REF_SPP = 65536
UNIFORM_SPP = (256, 512, 1024, 2048, 4096, 8192, 16384, 32768)


def tonemap(a):
    return np.sqrt(np.clip(a[..., :3] / np.maximum(a[..., 3:4], 1.0), 0.0, 1.0))


def psnr(a, b):
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    return 99.0 if mse == 0 else 10.0 * math.log10(1.0 / mse)


def mean_radiance(a):
    return float(np.mean(a[..., :3].astype(np.float64) / np.maximum(a[..., 3:4].astype(np.float64), 1.0)))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make(name, lights):
    s = rtb.Scene.named(name); i = s.info
    if lights:
        s.sample_lights(i.light_ids)
    r = rtb.Renderer(0); r.set_scene(s); r.set_camera(i.camera)
    return r, s, i


def uniform_time_to(db, curve, ms_per_spp):
    """spp and ms for `db` on the uniform curve [(spp, psnr)] (log-linear interpolation, extrapolated past the ends)."""
    pts = sorted(curve)
    for (s0, p0), (s1, p1) in zip(pts[:-1], pts[1:]):
        if p1 >= db or (s1, p1) == pts[-1]:
            slope = (p1 - p0) / math.log2(s1 / s0)
            spp = s0 * 2.0 ** ((db - p0) / max(slope, 1e-6))
            return round(spp), round(spp * ms_per_spp, 1)
    return None, None


def sweep(cfg, name, lights, ref):
    r, s, i = make(name, lights)
    W, H, D = i.width, i.height, i.max_depth
    cap = 65536 if cfg == "4" else 32768
    row = {"config": cfg, "scene": name, "width": W, "height": H, "depth": D, "sampled_lights": i.light_ids if lights else [],
           "reference": {"spp": REF_SPP, "seed": 99, "sampled_lights": True}, "uniform": [], "adaptive": []}
    # uniform, progressive (a first pass at 256 spp warms graphs and queues up and is not timed)
    r.render(W, H, 0, 256, D, seed=5); r.synchronize()
    r.reset_counters()
    done, ms = 0, 0.0
    for spp in UNIFORM_SPP:
        r.render(W, H, done, spp, D, seed=11, clear=(done == 0)); r.synchronize()
        ms += r.counters().render_ms
        done = spp
        a = r.download_accum()
        row["uniform"].append({"spp": spp, "psnr_vs_reference_db": round(psnr(tonemap(a), tonemap(ref)), 2), "device_ms": round(ms, 1)})
    ms_per_spp = ms / UNIFORM_SPP[-1]
    row["uniform_ms_per_spp"] = round(ms_per_spp, 5)
    k = r.counters(); row["uniform_rays_per_path"] = round(k.rays / k.paths, 3); row["uniform_ns_per_camera_path"] = round(ms * 1e6 / k.paths, 4)
    curve = [(u["spp"], u["psnr_vs_reference_db"]) for u in row["uniform"]]
    row["uniform_mean_radiance"] = mean_radiance(a)
    for db in TARGETS:
        spp, t = uniform_time_to(db, curve, ms_per_spp)
        row.setdefault("uniform_to_target", []).append({"db": db, "spp": spp, "device_ms": t})
    ref_mean = mean_radiance(ref)
    for db in TARGETS:
        res = {}
        for seed in (11, 22):
            r.reset_counters()
            t0 = time.perf_counter()
            st = r.render_adaptive(W, H, cap, D, target_db=db, min_spp=64, seed=seed)
            wall = (time.perf_counter() - t0) * 1e3
            a = r.download_accum()
            k = r.counters()
            res[seed] = (st, k.render_ms, wall, a, k.rays / max(k.paths, 1))
        st, dev_ms, wall, a, rpp = res[11]
        counts = a[..., 3].astype(np.int64)
        edges = [64 * 2 ** k for k in range(int(math.log2(cap // 64)) + 1)]
        hist = {str(e): int(((counts >= e) & (counts < 2 * e)).sum()) for e in edges}
        p_ref = psnr(tonemap(a), tonemap(ref))
        u_spp, u_ms = uniform_time_to(p_ref, curve, ms_per_spp)
        m = mean_radiance(a)
        row["adaptive"].append({
            "target_db": db, "tolerance": rtb.tolerance_for_db(db), "min_spp": 64, "cap": cap,
            "rounds": st["rounds"], "final_cursor": st["cursor"], "camera_paths": st["samples"],
            "mean_spp": round(float(counts.mean()), 1), "count_histogram": hist, "pixels_at_cap": int((counts >= cap).sum()),
            "device_ms": round(dev_ms, 1), "host_wall_ms": round(wall, 1), "rays_per_path": round(rpp, 3),
            "ns_per_camera_path": round(dev_ms * 1e6 / st["samples"], 4),
            "psnr_vs_reference_db": round(p_ref, 2),
            "psnr_between_seeds_db": round(psnr(tonemap(a), tonemap(res[22][3])), 2),
            "device_ms_seed22": round(res[22][1], 1),
            "uniform_spp_to_same_psnr": u_spp, "uniform_ms_to_same_psnr": u_ms,
            "speedup_at_same_psnr": round(u_ms / dev_ms, 2) if u_ms else None,
            "mean_radiance": m, "reference_mean_radiance": ref_mean, "mean_radiance_rel_diff": (m - ref_mean) / ref_mean,
            "uniform_mean_radiance_rel_diff": (row["uniform_mean_radiance"] - ref_mean) / ref_mean,
        })
        print(json.dumps(row["adaptive"][-1]), file=sys.stderr, flush=True)
    return row


def overhead():
    """Per-round cost of the adaptive machinery on config 4 (light sampling off)."""
    r, s, i = make("book2_cornell_smoke", False)
    W, H, D = i.width, i.height, i.max_depth
    out = {"config": "4", "round_samples": [256, 512], "runs": []}
    for rep in range(3):
        r.render(W, H, 0, 256, D, seed=3, variance=True); r.synchronize()
        r.render(W, H, 256, 512, D, seed=3, clear=False, variance=True); r.synchronize()
        dense_ms = r.counters().render_ms
        r.render(W, H, 0, 256, D, seed=3, variance=True); r.synchronize()
        t0 = time.perf_counter()
        st = r.render_adaptive(W, H, 512, D, tolerance=0.0, min_spp=256, max_rounds=1, seed=3, clear=False)
        wall = (time.perf_counter() - t0) * 1e3
        ad_ms = r.counters().render_ms
        out["runs"].append({"dense_round_ms": round(dense_ms, 2), "adaptive_round_ms": round(ad_ms, 2), "adaptive_host_wall_ms": round(wall, 2),
                            "active_pixels": int(st["samples"] // 256), "pixels": W * H})
    # the same dense round on one lane without a CUDA graph (RTB_LANES=1 is read when a renderer is made, RTB_NO_GRAPH per call)
    import os
    os.environ["RTB_LANES"] = "1"; os.environ["RTB_NO_GRAPH"] = "1"
    r1, _, _ = make("book2_cornell_smoke", False)
    one = []
    for rep in range(3):
        r1.render(W, H, 0, 256, D, seed=3, variance=True); r1.synchronize()
        r1.render(W, H, 256, 512, D, seed=3, clear=False, variance=True); r1.synchronize()
        one.append(r1.counters().render_ms)
    del os.environ["RTB_LANES"], os.environ["RTB_NO_GRAPH"]
    del r1
    out["dense_round_one_lane_no_graph_ms"] = [round(x, 2) for x in one]
    # the select step alone (profiled: plain launches with events around each)
    r.render(W, H, 0, 256, D, seed=3, variance=True); r.synchronize()
    r.set_profiling(True)
    r.render_adaptive(W, H, 512, D, tolerance=0.0, min_spp=256, max_rounds=1, seed=3, clear=False)
    ms, cls = r.profile_launches(1 << 16)
    r.profile(); r.set_profiling(False)
    sel = [float(x) for x, c in zip(ms, cls) if c == 6]
    out["select_step_ms"] = [round(x, 3) for x in sel]
    d = sorted(x["dense_round_ms"] for x in out["runs"]); a = sorted(x["adaptive_round_ms"] for x in out["runs"])
    out["median_dense_round_ms"], out["median_adaptive_round_ms"] = d[1], a[1]
    # tolerance 0 still stops the pixels whose whole window has zero error (black background, the emitter seen directly):
    # compare time per camera path
    frac = out["runs"][0]["active_pixels"] / out["runs"][0]["pixels"]
    o1 = sorted(one)[1]
    out["ns_per_path"] = {"dense_two_lanes_graph": round(d[1] * 1e6 / (W * H * 256), 4), "dense_one_lane_no_graph": round(o1 * 1e6 / (W * H * 256), 4),
                          "adaptive_round": round(a[1] * 1e6 / (out["runs"][0]["active_pixels"] * 256), 4)}
    out["overhead_vs_dense_per_path"] = round(a[1] / (d[1] * frac) - 1.0, 4)
    out["overhead_vs_one_lane_no_graph_per_path"] = round(a[1] / (o1 * frac) - 1.0, 4)
    out["note"] = ("a one-round call runs the select step twice (before and after the round) and reads the count twice; "
                   "overhead = adaptive round time per camera path against the dense round's")
    return out


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--configs", default="4,5")
    ap.add_argument("--no-overhead", action="store_true")
    args = ap.parse_args()
    od = Path(args.out_dir)
    od.mkdir(parents=True, exist_ok=True)
    info = gpu_info()
    print("gpu:", info, file=sys.stderr, flush=True)
    if not args.no_overhead:
        ov = overhead(); ov["gpu"] = info
        (od / "r4_adaptive_overhead.json").write_text(json.dumps(ov, indent=1))
        print(json.dumps(ov), file=sys.stderr, flush=True)
    for cfg, name in (("4", "book2_cornell_smoke"), ("5", "book2_final")):
        if cfg not in args.configs.split(","):
            continue
        rr, _, ii = make(name, True)
        rr.render(ii.width, ii.height, 0, REF_SPP, ii.max_depth, seed=99); rr.synchronize()
        ref = rr.download_accum()
        del rr
        for lights in (False, True):
            row = sweep(cfg, name, lights, ref)
            row["gpu"] = info
            (od / f"r4_adaptive_cfg{cfg}_{'lights' if lights else 'plain'}.json").write_text(json.dumps(row, indent=1))
