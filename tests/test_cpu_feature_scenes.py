"""CPU checks of the feature-scene builder (tests/feature_scenes.py) that the schedule tests rely on: its cases cover every
traverse, shade and tail instantiation, every scene loads into the oracle with the features its case asks for, and the
host-built trees have the depths that pick the 16- and 32-entry stacks."""
import numpy as np
import pytest

import feature_scenes as fs
from mesh_oracle import MeshOracleScene


def test_cases_cover_every_instantiation():
    table = fs.check_coverage()
    print(fs.format_coverage(table))
    assert len(table["shade"]) == 16 and len(table["tail"]) == 64 and len(table["traverse"]) == 15
    assert len({c.id for c in fs.CASES}) == len(fs.CASES)
    # dropping any one case loses at least one tail instantiation: the list has no passengers
    for k in range(len(fs.CASES)):
        with pytest.raises(AssertionError):
            fs.check_coverage(fs.CASES[:k] + fs.CASES[k + 1:])


@pytest.mark.parametrize("case", fs.CASES, ids=lambda c: c.id)
def test_scene_selects_what_its_case_says(rtb, case):
    scene, cam = fs.build(rtb, case)
    if case.tree == "deep":
        # (the GPU linear BVH is built on a device: its depth is asserted by the GPU tests)
        stats = {"depth": fs.NORMAL_MAX_DEPTH + 1, "builder": "gpu_lbvh"}
    else:
        stats = scene.flatten_stats()
    fs.check_selection(case, scene, stats)
    MeshOracleScene(scene.serialize())


def test_oracle_renders_a_case(rtb):
    """The oracle half of one parity case of tests/test_gpu_schedules.py (every switch on, at a smaller size)."""
    case = fs.Case("bvh", "normal", True, "sampled", True)
    scene, cam = fs.build(rtb, case)
    ref, _, rays = MeshOracleScene(scene.serialize()).render(cam, 48, 32, 0, 4, 24, seed=1984)
    assert rays > 48 * 32 * 4 and np.isfinite(ref).all() and (ref[..., 3] == 4).all() and ref[..., :3].sum() > 0
