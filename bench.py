#!/usr/bin/env python
"""bench.py — headline benchmark: Book 2 final scene (BASELINE.json configs[4]) through the C ABI.

    python bench.py --gpus N --steps K --warmup W            # the B200 wavefront path tracer
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference on the host cores

A "step" is one pass of the hot path over one batch of synthetic input: `--spp-per-step` samples (1600 by
default) of every pixel of the 800x800 Book 2 final scene, depth 40 - a FIXED total, split over the N ranks
by sample range (strong scaling: rank r renders samples [r S/N, (r+1) S/N) of the step, exactly the
partition of the 10,000 spp job), and the per-rank radiance sums are summed onto rank 0 with one NCCL
reduce per step.  Rank 0 prints ONE JSON line.  `value` is Mrays/s (ray segments submitted to closest-hit
traversal per second, all ranks); Mpaths/s rides along in `paths`.

The oracle (oracle/) is used here only as the checker / CPU baseline, never as the thing measured in
the default arm.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))

SCENE = "book2_final"
ALG_BYTES_PER_RAY_TRAVERSE = 40      # traverse kernel: 32 B ray record read + 8 B hit record written (DESIGN.md)
ALG_BYTES_PER_RAY_STEP = 152         # SURVEY.md 8(d): whole wavefront, per ray segment
ALG_BYTES_PER_PATH_STEP = 32         # SURVEY.md 8(d): accumulate, per path


def measured_peak_hbm():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index          # one index, or "0,1,2,..." (one poller for all the GPUs of the run)
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_golden_scene():
    """The headline scene as a committed RTBS blob + camera (tests/golden/book2_final.rtbs.xz, .json - written by
    tests/golden/make_golden.py scenes): the reference arm maps only oracle/, never the product's libraries."""
    import lzma
    orc = importlib.import_module("pyoracle")
    blob = lzma.decompress((ROOT / "tests" / "golden" / f"{SCENE}.rtbs.xz").read_bytes())
    meta = json.loads((ROOT / "tests" / "golden" / f"{SCENE}.json").read_text())
    return orc, orc.OracleScene(blob), orc.camera_from_dict(meta["camera"]), meta


def run_reference_arm(args, rank, world):
    """The reference's own implementation of the path on the host cores.  The reference has no CPU
    renderer (its integrator is __device__-only), so this is the CPU restatement of it (oracle/, kind
    "port") on all host threads, on a bounded sample of the same workload."""
    if rank != 0:
        return
    orc, o, cam, meta = load_golden_scene()
    threads = os.cpu_count() or 1
    W, H, depth = meta["width"], meta["height"], meta["max_depth"]
    spp = args.ref_spp
    for i in range(args.warmup):
        o.render(cam, W, H, i * spp, (i + 1) * spp, depth, seed=1984, threads=threads)
    t0 = time.perf_counter(); rays = 0
    for i in range(args.steps):
        s0 = (args.warmup + i) * spp
        _, _, r = o.render(cam, W, H, s0, s0 + spp, depth, seed=1984, threads=threads)
        rays += r
    dt = time.perf_counter() - t0
    mrays = rays / dt / 1e6
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": mrays, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"Book 2 final scene {W}x{H} depth {depth} (BASELINE.json configs[4]), step = {spp} spp of every pixel (bounded sample of the 10000 spp job; a rate, "
                               f"so comparable with the GPU arm's {args.spp_per_step}-spp steps)", "scene": SCENE, "rng": "philox4x32-10 keyed (seed,pixel)x(sample,bounce,stream)"},
        "paths": {"value": W * H * spp * args.steps / dt / 1e6, "unit": "Mpaths/s"},
        "cpu_baseline": {"value": mrays, "unit": "Mrays/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} steps x {W}x{H}x{spp} spp, std::thread over image rows, -O2, no fast-math; the reference has no CPU renderer, this is oracle/ (CPU restatement)"},
        "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_JSON_OUT, flush=True)


def load_ncu_profile():
    """Counters of the dominant kernel from the committed ncu capture (profiles/r2_ncu.json, written by
    tools/ncu_summary.py json): nothing profiler-derived is typed into this script.  `stale` says the capture was taken
    at another commit of the kernel sources."""
    p = ROOT / "profiles" / "r2_ncu.json"
    if not p.exists():
        return None
    j = json.loads(p.read_text())
    import hashlib
    h = hashlib.sha1()
    for f in sorted((ROOT / "ray-tracing-v06_b200" / "csrc").glob("*")):
        if f.suffix in (".cu", ".h", ".cpp"):
            h.update(f.name.encode()); h.update(f.read_bytes())
    j["stale"] = (h.hexdigest() != j.get("kernel_sources_sha1")) if j.get("kernel_sources_sha1") else None
    return j


_JSON_OUT = sys.stdout


def camera_rays_for(pkg, cam, width, height):
    """Primary rays through pixel centres (Renderer.cu:192) as rtb_ray records, for the traversal-statistics hook."""
    import numpy as np
    xs = (np.arange(width, dtype=np.float32) + np.float32(0.5)) * (np.float32(1) / np.float32(width)) * np.float32(2) - np.float32(1)
    ys = (np.arange(height, dtype=np.float32) + np.float32(0.5)) * (np.float32(1) / np.float32(height)) * np.float32(2) - np.float32(1)
    U, V = np.meshgrid(xs, ys)
    o = np.array(cam.o[:], dtype=np.float32); cu = np.array(cam.u[:], dtype=np.float32); cv = np.array(cam.v[:], dtype=np.float32); cw = np.array(cam.w[:], dtype=np.float32)
    d = cw[None, None, :] + cu[None, None, :] * U[..., None] + cv[None, None, :] * V[..., None]
    rays = np.zeros(width * height, dtype=pkg.RAY_DTYPE)
    rays["o"] = o; rays["d"] = d.reshape(-1, 3).astype(np.float32); rays["time"] = 0.0
    return rays


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--spp-per-step", type=int, default=1600, help="samples per pixel per step, ALL GPUs together (split by sample range)")
    ap.add_argument("--cpu-spp", type=int, default=128, help="samples per pixel of the cpu_baseline sample (rank 0, N=1)")
    ap.add_argument("--ref-spp", type=int, default=16, help="samples per pixel per step of the --impl reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip the reference megakernel run beside ours (A/B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the framebuffer of the last timed step "
                    "(radiance sums + sample count, float32, 800x800x4; rank 0 after the reduce) to DIR/accum.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun (the driver launches torchrun itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ.get("MASTER_PORT", "29533"), __file__] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    # Exactly ONE line goes to stdout (the JSON line, rank 0): everything libraries print on fd 1 meanwhile (NCCL's
    # version banner, subprocess chatter) is sent to stderr, and the line is written to the saved descriptor at the end.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    pkg = importlib.import_module("ray-tracing-v06_b200")
    pkg.lib()                                   # fails loudly if librtb200.so is missing: no fallback
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"), timeout=datetime.timedelta(seconds=180))

    scene = pkg.Scene.named(SCENE)
    info = scene.info
    W, H, depth, S = info.width, info.height, info.max_depth, args.spp_per_step
    if S < world:
        raise SystemExit("bench.py: --spp-per-step must be at least the number of GPUs")
    r = pkg.Renderer(local_rank)
    r.set_scene(scene); r.set_camera(info.camera)
    stream = torch.cuda.current_stream().cuda_stream

    def step(i, clear=True):
        a, b = pkg.sample_range(S, rank, world)   # this rank's share of the step's S samples (strong scaling)
        r.render(W, H, i * S + a, i * S + b, depth, seed=1984, clear=clear, stream=stream)
        if world > 1:
            dist.reduce(r.accum_tensor(), dst=0)  # the only collective: framebuffer sum over NVLink

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(",".join(str(g) for g in range(world)) if world > 1 else local_rank)
    if rank == 0:                                                # ONE nvidia-smi poller for all the GPUs of the run (a poller per rank only loads the driver)
        sampler.start()                                          # sampled from the warm-up on, through the timed region
    for i in range(args.warmup):
        step(i)
    barrier()
    r.reset_counters()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    ev1.record()
    barrier()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    cnt = r.counters()
    if args.dump_outputs and rank == 0:
        # what rtb_render left in the accumulator after the last timed step (inputs are fixed by seed and sample range)
        Path(args.dump_outputs).mkdir(parents=True, exist_ok=True)
        np.save(Path(args.dump_outputs) / "accum.npy", r.download_accum())
    rank_ms = [ms]
    if world > 1:
        gathered = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([ms], dtype=torch.float64, device="cuda"))
        rank_ms = [float(x.item()) for x in gathered]
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(cnt.rays), float(cnt.paths), float(cnt.launches)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms = float(t.item()); rays, paths, launches = [float(x) for x in tot.tolist()]
    mrays = rays / ms / 1e3; mpaths = paths / ms / 1e3

    # ---- e2e: the call a user makes, HOST buffers: scene upload (H2D) + render + framebuffer download (D2H), every step
    host_fb = torch.empty((H, W, 4), dtype=torch.float32, pin_memory=True)
    e2e_steps = max(1, min(args.steps, 5))
    r.set_scene(scene); step(0); r.download_into(host_fb.data_ptr())   # warm
    barrier(); r.reset_counters()
    flatten_ms = []
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        scene.set_world_bvh(pkg.WORLD_BVH_QUALITY)  # bumps the scene's version: the renderer must flatten it again (graph walk, SAH build, wide layout)
        r.set_scene(scene)                        # flatten + H2D of the scene arena
        flatten_ms.append(r.scene_stats()["flatten_ms"])
        step(args.warmup + args.steps + i)
        if rank == 0:
            r.download_into(host_fb.data_ptr())   # resolve + D2H into pinned memory
    barrier()
    e2e_s = time.perf_counter() - t0
    c2 = r.counters()
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda"); re_ = torch.tensor([float(c2.rays)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX); dist.all_reduce(re_, op=dist.ReduceOp.SUM)
    e2e_mrays = float(re_.item()) / float(te.item()) / 1e6

    # ---- roofline of the dominant kernel (traverse): one profiled step, CUDA events around every launch on its stream
    roof = None; split = None
    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        r.reset_counters(); r.set_profiling(True)
        a, b = pkg.sample_range(S, rank, world)
        s0p = (args.warmup + args.steps + e2e_steps) * S
        r.render(W, H, s0p + a, s0p + b, depth, seed=1984, clear=True, stream=stream)   # rank-local: no collective here
        prof = r.profile(); pc = r.counters(); r.set_profiling(False)
        total_ms = prof.generate_ms + prof.traverse_ms + prof.shade_ms + prof.accumulate_ms + prof.tail_ms + prof.bin_ms
        trav_s = prof.traverse_ms * 1e-3
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        ncu = load_ncu_profile()
        nt = (ncu or {}).get("traverse") or {}
        # The kernel is bound by instruction issue and SIMT lane occupancy (the scene is L1/L2 resident; HBM carries only the
        # queues).  Work per unit = thread-instructions per ray, from the committed ncu capture of this kernel; time = this
        # run's CUDA events.  Peak = every lane of every scheduler issuing every cycle at the clock seen during the run.
        issue_peak = 148 * 4 * 32 * sm_mhz * 1e6 / 1e12
        tipr = nt.get("thread_inst_per_ray")
        ach_issue = tipr * pc.rays / trav_s / 1e12 if (tipr and trav_s > 0) else None
        ach_hbm = ALG_BYTES_PER_RAY_TRAVERSE * pc.rays / trav_s / 1e9 if trav_s > 0 else 0.0
        roof = {"bound": "issue", "kernel": "traverse_kernel", "achieved": ach_issue, "peak": issue_peak, "unit": "T thread-instructions/s",
                "frac": ach_issue / issue_peak if ach_issue else None,
                "traffic": nt.get("dram_bytes_per_ray") * pc.rays / max(1, prof.traverse_launches) if nt.get("dram_bytes_per_ray") else None,
                "traffic_note": "DRAM bytes per launch = dram__bytes_read+write per ray of the committed ncu capture x this run's rays per launch; algorithmic 40 B/ray",
                "per_unit": {"thread_instructions_per_ray": tipr, "source": "profiles/r2_ncu.json (sm__inst_executed x smsp__thread_inst_executed_per_inst_executed over every traverse launch of a step / rays)"},
                "peak_note": f"148 SMs x 4 schedulers x 32 lanes x {sm_mhz:.0f} MHz (clock sampled during the timed region)",
                "avg_launch_ms": prof.traverse_ms / max(1, prof.traverse_launches), "launches": int(prof.traverse_launches),
                "ncu": {k: nt.get(k) for k in ("issue_busy_pct", "active_lanes", "warp_inst_per_ray", "l1_hit_pct", "dram_bytes_per_ray")} | {"stale": (ncu or {}).get("stale"), "kernel_sources_sha1": (ncu or {}).get("kernel_sources_sha1")},
                "hbm": {"achieved": ach_hbm, "peak": peak, "unit": "GB/s", "frac": ach_hbm / peak, "peak_source": peak_src, "algorithmic_bytes_per_ray": ALG_BYTES_PER_RAY_TRAVERSE,
                        "note": "the same kernel against the HBM roofline: 32 B ray record read + 8 B hit record written per ray"},
                "note": "traversal is instruction-issue bound with SIMT divergence: frac = issue-slot utilisation x active lanes / 32"}
        # FP32 work in SURVEY 8(d)'s accounting: 24 flop per box test, 30 per primitive test, 150 per shaded segment, with
        # the box / primitive tests per ray counted live through the rtb_trace_rays hook on this scene's primary rays and
        # one generation of diffuse secondary rays (the mix of a depth-40 path is dominated by the latter).
        try:
            cam_rays = camera_rays_for(pkg, info.camera, 200, 200)
            h1 = r.trace_rays(cam_rays); hit1 = h1["object"] >= 0
            rng = np.random.default_rng(0)
            v = rng.normal(size=(int(hit1.sum()), 3)).astype(np.float32); v /= np.linalg.norm(v, axis=1, keepdims=True)
            sec = np.zeros(int(hit1.sum()), dtype=pkg.RAY_DTYPE); dsec = h1["n"][hit1] + v
            sec["o"] = h1["p"][hit1] + dsec * np.float32(0.001); sec["d"] = dsec; sec["time"] = 0.5
            h2 = r.trace_rays(sec)
            w_sec = 1.0 - paths / rays                                   # share of ray segments that are not camera rays
            boxes = 2.0 * ((1 - w_sec) * float(h1["nodes_visited"].mean()) + w_sec * float(h2["nodes_visited"].mean()))
            prims = (1 - w_sec) * float(h1["prims_tested"].mean()) + w_sec * float(h2["prims_tested"].mean())
            flop_per_ray = 24.0 * boxes + 30.0 * prims + 150.0
            fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
            roof["fp32"] = {"achieved_tflops": flop_per_ray * (rays / world) / (ms * 1e-3) / 1e12, "peak_tflops": fp32_peak, "peak_note": f"148 SMs x 128 lanes x 2 x {sm_mhz:.0f} MHz (non-tensor FP32)",
                            "frac": flop_per_ray * (rays / world) / (ms * 1e-3) / 1e12 / fp32_peak, "box_tests_per_ray": boxes, "prim_tests_per_ray": prims, "flop_per_ray": flop_per_ray,
                            "model": "24 flop / box test + 30 / primitive test + 150 / shaded segment (SURVEY 8d); tests per ray measured through rtb_trace_rays"}
        except Exception as e:   # the counters are diagnostics: never fail the bench line over them
            roof["fp32"] = {"error": str(e)}
        step_bytes = ALG_BYTES_PER_RAY_STEP * rays + ALG_BYTES_PER_PATH_STEP * paths
        split = {"traverse_ms": prof.traverse_ms, "shade_ms": prof.shade_ms, "generate_ms": prof.generate_ms, "accumulate_ms": prof.accumulate_ms, "tail_ms": prof.tail_ms, "bin_ms": prof.bin_ms,
                 "traverse_share": prof.traverse_ms / total_ms if total_ms else None,
                 "step_hbm": {"achieved": step_bytes / (ms * 1e-3) / 1e9 / max(1, world), "peak": peak, "unit": "GB/s per GPU", "frac": step_bytes / (ms * 1e-3) / 1e9 / peak / max(1, world),
                              "accounting": "SURVEY 8(d): 152 B per ray segment + 32 B per path, whole wavefront, over the timed region"}}

    # ---- once per run: the reduced image of N ranks == one GPU rendering the same sample range (96x96, 16 spp, depth 40)
    multi_check = None
    if world > 1:
        cw = ch = 96; cs = 16
        a, b = pkg.sample_range(cs, rank, world)
        r.render(cw, ch, a, b, depth, seed=7, clear=True, stream=stream)
        red = r.accum_tensor().clone()
        dist.reduce(red, dst=0)
        torch.cuda.synchronize()
        if rank == 0:
            r.render(cw, ch, 0, cs, depth, seed=7, clear=True, stream=stream); r.synchronize()
            one = r.download_accum()
            got = red.cpu().numpy()
            err = float(np.abs(got[..., :3] - one[..., :3]).max() / max(1.0, float(np.abs(one[..., :3]).max())))
            multi_check = {"what": f"{cw}x{ch}x{cs} spp split over {world} ranks + NCCL reduce vs the same range on rank 0 alone", "max_rel_err": err,
                           "sample_counts_equal": bool(np.array_equal(got[..., 3], one[..., 3])), "ok": bool(err < 1e-5 and np.array_equal(got[..., 3], one[..., 3]))}
        r.render(W, H, 0, 1, depth, seed=1984, clear=True, stream=stream); r.synchronize()      # back to the headline framebuffer size

    # ---- CPU baseline + same-stream image check (rank 0, N=1 only)
    cpu = None; psnr_db = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        orc = importlib.import_module("pyoracle")
        o = orc.OracleScene(scene.serialize())
        threads = os.cpu_count() or 1
        t0 = time.perf_counter()
        osum, _, orays = o.render(info.camera, W, H, 0, args.cpu_spp, depth, seed=1984, threads=threads)
        dt = time.perf_counter() - t0
        cpu = {"value": orays / dt / 1e6, "unit": "Mrays/s", "cores": threads, "kind": "port",
               "sample": f"{W}x{H}x{args.cpu_spp} spp of the same scene ({dt:.1f} s); oracle/ = CPU restatement (the reference has no CPU renderer)"}
        r.render(W, H, 0, args.cpu_spp, depth, seed=1984, clear=True, stream=stream); r.synchronize()
        g = r.download_accum()
        tm = lambda a: np.sqrt(np.clip(a[..., :3] / np.maximum(a[..., 3:4], 1.0), 0.0, 1.0))
        mse = float(np.mean((tm(g).astype(np.float64) - tm(osum).astype(np.float64)) ** 2))
        psnr_db = 99.0 if mse == 0 else float(10.0 * np.log10(1.0 / mse))

    # ---- the reference's own GPU megakernel on the one config it can express (cfg 2), beside ours
    refgpu = None
    ref_bin = ROOT / "oracle" / "_ref" / "ref_render"
    if rank == 0 and world == 1 and ref_bin.exists() and not args.no_reference_gpu:
        try:
            out = subprocess.run([str(ref_bin), "render", "400", "225", "100", "50", "/tmp/ref_cfg2.bin"], capture_output=True, text=True, timeout=120).stdout
            js = [l for l in out.splitlines() if l.startswith("REF_JSON")]
            s2 = pkg.Scene.named("book2_bouncing"); r2 = pkg.Renderer(local_rank); r2.set_scene(s2); r2.set_camera(s2.info.camera)
            for _ in range(3):
                r2.render(400, 225, 0, 100, 50, seed=1984); r2.synchronize()
            r2.reset_counters(); r2.render(400, 225, 0, 100, 50, seed=1984); r2.synchronize(); k2 = r2.counters()
            refgpu = {"config": "Book 2 bouncing spheres 400x225, 100 spp, depth 50 (configs[1])",
                      "reference_megakernel": json.loads(js[-1][len("REF_JSON"):]) if js else None,
                      "ours": {"render_ms": k2.render_ms, "mpaths_per_s": 400 * 225 * 100 / k2.render_ms / 1e3, "mrays_per_s": k2.rays / k2.render_ms / 1e3}}
        except Exception as e:  # the checker binary is optional
            refgpu = {"error": str(e)}

    if rank == 0:
        line = {
            "metric": "Mrays/s", "value": mrays, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"Book 2 final scene {W}x{H} depth {depth} (BASELINE.json configs[4]); step = {S} spp of every pixel in total, split over the "
                                   f"{world} GPU(s) by sample range (the partition of the 10000 spp job)", "scene": SCENE, "spp_per_step": S,
                       "l2": "per-step wavefront queue traffic (~0.15 GB per Mray) is far larger than the 126 MB L2; no flush needed",
                       "rng": "philox4x32-10 keyed (seed,pixel)x(sample,bounce,stream)", "collective": "one NCCL reduce(sum) of the 10.24 MB framebuffer per step" if world > 1 else "none"},
            "paths": {"value": mpaths, "unit": "Mpaths/s"},
            "rays_per_path": rays / paths if paths else None,
            "e2e": {"value": e2e_mrays, "unit": "Mrays/s", "h2d_bytes_per_step": r.scene_bytes(), "d2h_bytes_per_step": W * H * 16,
                    "flatten_ms_per_step": sum(flatten_ms) / len(flatten_ms),
                    "what": "per step, wall clock: rtb_renderer_set_scene of a CHANGED scene (full flatten: graph walk, SAH build, wide layout; then H2D of the arena) "
                            "+ rtb_render + rtb_download (resolve + D2H into pinned host memory)"},
            "gpu_launches": int(launches), "rank_ms_per_step": [x / args.steps for x in rank_ms], "render_ms_per_step_rank0": cnt.render_ms,
            "clocks": clocks,
            "roofline": roof, "kernel_split": split, "multi_gpu_check": multi_check,
            "cpu_baseline": cpu, "psnr_vs_oracle_db": psnr_db,
            "reference_gpu": refgpu,
        }
    else:
        line = None
    if world > 1:
        dist.destroy_process_group()
    if line is not None:                       # last thing this process writes anywhere
        sys.stderr.flush()
        print(json.dumps(line), file=_JSON_OUT, flush=True)


if __name__ == "__main__":
    main()
