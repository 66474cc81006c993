#!/usr/bin/env python
"""Regenerates the golden fixtures in this directory from the REFERENCE itself.

Needs a checkout of the reference for `make -C oracle ref REF=<checkout>`, and a GPU for the megakernel part:

  # CPU part: the reference's own BVH_Handle::Factory on the bouncing-spheres boxes
  python tests/golden/make_golden.py bvh

  # GPU part (on a B200; oracle/_ref/ref_render is the reference's Renderer.cu/BVH.cu/
  # SphereHittable.cu/Scenes.cu/cuHostRND.cpp compiled unmodified for sm_100a), into a directory OUT:
  python tests/golden/make_golden.py trace_rays      # writes oracle/_ref/trace_rays.bin
  oracle/_ref/ref_render rng OUT/ref_rng.bin
  oracle/_ref/ref_render scene OUT/ref_scene.bin
  oracle/_ref/ref_render render 200 112 4 50 OUT/ref_img_200x112_4spp_d50.bin
  oracle/_ref/ref_render render 400 225 100 50 OUT/ref_img_400x225_100spp_d50.bin
  oracle/_ref/ref_render trace oracle/_ref/trace_rays.bin OUT/ref_trace.bin
  python tests/golden/make_golden.py collect OUT          # copies / converts OUT/* into tests/golden/
  python tests/golden/make_golden.py collect_trace OUT

Fixtures:
  ref_rng.bin                              4608 uniforms of the reference's cuHostRND(512,1984) + 4 x 64 device XORWOW uniforms
  ref_scene_book2_bouncing.bin             the 488 spheres + material bytes the reference's Scenes.cu built on the GPU box
  ref_megakernel_200x112_4spp_d50.bin      raw float4 framebuffer of the reference's render_kernel (first Render call)
  ref_megakernel_400x225_100spp_d50_f16.npy  same at config 2's size, stored as float16 RGB
  ref_trace_book2_bouncing.npz             hit records (t, normal, point, sphere index) of the reference's own
                                           world->ClosestIntersection + getNormal on the rays of helpers.reference_trace_rays
                                           (point and normal stored losslessly as residuals: helpers.encode_reference_trace)
  ref_sphere_index_host_1280x720.npz       (`python tests/golden/make_golden.py sphere_index`, CPU) the ground truth of the reference's
                                           own unit test (google_testing/test.cpp:87-106) computed by the reference's
                                           _sphere_closest_intersection + PinholeCamera (oracle/_ref/ref_sphere_index host)
  book2_final.rtbs.xz / .json              (`python tests/golden/make_golden.py scenes`) the headline scene serialised by the host mirror
                                           (RTBS blob, camera as hex floats, sizes): what `bench.py --impl reference` renders, so
                                           that arm loads nothing of the product
  ref_bvh_book2_bouncing.bin               node array + primitive order of the reference's BuildBVH_TopDown
  oracle_images_32x18.npz                  (`python tests/golden/make_golden.py oracle`) the ORACLE's own Philox renders of every
                                           registered scene at 32x18, 2 spp, depth 8 - not a reference fixture: a tripwire that
                                           the oracle (the checker of every GPU test) has not drifted
"""
import importlib
import shutil
import struct
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
GOLD = ROOT / "tests" / "golden"
sys.path.insert(0, str(ROOT))


def oracle_images():
    rtb = importlib.import_module("ray-tracing-v06_b200")
    sys.path.insert(0, str(ROOT / "oracle")); orc = importlib.import_module("pyoracle")
    out = {}
    for name in rtb.scene_names():
        s = rtb.Scene.named(name)
        acc, _, rays = orc.OracleScene(s.serialize()).render(s.info.camera, 32, 18, 0, 2, 8, seed=1984)
        out[name] = acc.astype(np.float32); out[name + "__rays"] = np.array([rays], dtype=np.int64)
    np.savez_compressed(GOLD / "oracle_images_32x18.npz", **out)
    print("wrote", GOLD / "oracle_images_32x18.npz", len(out) // 2, "scenes")


def bvh():
    rtb = importlib.import_module("ray-tracing-v06_b200")
    s = rtb.Scene.named("book2_bouncing")
    boxes = np.array([s.bounds(i) for i in range(488)], dtype=np.float32)
    tmp_in, tmp_out = "/tmp/ref_bvh_in.bin", "/tmp/ref_bvh_out.bin"
    open(tmp_in, "wb").write(struct.pack("i", len(boxes)) + boxes.tobytes())
    subprocess.run([str(ROOT / "oracle" / "_ref" / "ref_bvh"), tmp_in, tmp_out, "0"], check=True)
    shutil.copy(tmp_out, GOLD / "ref_bvh_book2_bouncing.bin")
    print("wrote", GOLD / "ref_bvh_book2_bouncing.bin")


def scenes():
    """The headline scene as the oracle-side fixture of bench.py --impl reference: RTBS blob + camera + sizes."""
    import json
    import lzma
    rtb = importlib.import_module("ray-tracing-v06_b200")
    sys.path.insert(0, str(ROOT / "oracle")); orc = importlib.import_module("pyoracle")
    for name in ("book2_final",):
        s = rtb.Scene.named(name)
        (GOLD / f"{name}.rtbs.xz").write_bytes(lzma.compress(s.serialize(), preset=9 | lzma.PRESET_EXTREME))
        meta = {"scene": name, "width": int(s.info.width), "height": int(s.info.height), "spp": int(s.info.spp), "max_depth": int(s.info.max_depth),
                "camera": orc.camera_to_dict(s.info.camera)}
        (GOLD / f"{name}.json").write_text(json.dumps(meta, indent=1) + "\n")
        print("wrote", GOLD / f"{name}.rtbs.xz", (GOLD / f"{name}.rtbs.xz").stat().st_size, "bytes")


def sphere_index():
    rtb = importlib.import_module("ray-tracing-v06_b200")
    sys.path.insert(0, str(ROOT / "tests")); import helpers
    idx, cam, _ = helpers.reference_sphere_index(rtb, "host", "/tmp")
    np.savez_compressed(GOLD / "ref_sphere_index_host_1280x720.npz", index=idx.astype(np.int16).reshape(720, 1280), camera=cam)
    print("wrote", GOLD / "ref_sphere_index_host_1280x720.npz")


def trace_rays():
    rtb = importlib.import_module("ray-tracing-v06_b200")
    sys.path.insert(0, str(ROOT / "tests")); import helpers
    rays = helpers.reference_trace_rays(rtb)
    (ROOT / "oracle" / "_ref").mkdir(exist_ok=True)
    rays.tofile(ROOT / "oracle" / "_ref" / "trace_rays.bin")
    print("wrote", len(rays), "rays")


def collect_trace(out_dir):
    rtb = importlib.import_module("ray-tracing-v06_b200")
    sys.path.insert(0, str(ROOT / "tests")); import helpers
    rec = np.fromfile(Path(out_dir) / "ref_trace.bin", dtype=helpers.REF_TRACE_DTYPE)
    np.savez_compressed(GOLD / "ref_trace_book2_bouncing.npz", **helpers.encode_reference_trace(helpers.reference_trace_rays(rtb), rec))
    print("wrote", len(rec), "records,", int((rec["index"] >= 0).sum()), "hits")


def collect(out_dir):
    out = Path(out_dir)
    shutil.copy(out / "ref_rng.bin", GOLD / "ref_rng.bin")
    shutil.copy(out / "ref_scene.bin", GOLD / "ref_scene_book2_bouncing.bin")
    shutil.copy(out / "ref_img_200x112_4spp_d50.bin", GOLD / "ref_megakernel_200x112_4spp_d50.bin")
    a = np.fromfile(out / "ref_img_400x225_100spp_d50.bin", dtype=np.float32).reshape(225, 400, 4)[..., :3]
    np.save(GOLD / "ref_megakernel_400x225_100spp_d50_f16.npy", a.astype(np.float16))


if __name__ == "__main__":
    {"bvh": bvh, "collect": collect, "oracle": oracle_images, "trace_rays": trace_rays, "sphere_index": sphere_index, "scenes": scenes, "collect_trace": collect_trace}[sys.argv[1]](*sys.argv[2:])
