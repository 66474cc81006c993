"""The loader of the feature oracle (tests/feature_oracle.cpp) section by section: valid RTBS v2 - v5 blobs load, and each one
damaged in one place is refused with the message of the check that section's reader makes.  A render comparison cannot
pin these: a refused blob renders nothing."""
import re
import struct

import numpy as np
import pytest

from feature_oracle import FeatureOracleScene
from helpers import RTBS_OBJECT, parse_blob

MAX_SAMPLED_LIGHTS, ENV_MAX_SIZE = 16, 16384


def _blob(rtb, version):
    """A lit floor with one sampled quad light; v3 adds a sampled 4 x 2 map, v4 a smooth-shaded triangle, v5 a rough metal
    sphere."""
    s = rtb.Scene()
    white = s.lambertian((0.7, 0.7, 0.7)); lamp = s.diffuse_light(s.solid((4, 4, 4)))
    light = s.quad((-0.5, 2, -0.5), (1, 0, 0), (0, 0, 1), lamp)
    parts = [s.quad((-2, 0, -2), (4, 0, 0), (0, 0, 4), white), light]
    if version >= 4:
        v = np.float32([[-1, 0.5, 0], [1, 0.5, 0], [-1, 1.5, 0]])
        parts.append(s.mesh(v, np.int32([[0, 1, 2]]), white, normals=np.float32([[0.2, 0, 1], [0, 0.2, 1], [0, 0, 1]])))
    if version >= 5:
        parts.append(s.sphere((1, 0.5, 1), 0.5, s.rough_metal((0.9, 0.8, 0.7), 0.3)))
    s.set_root(s.list(parts))
    s.sample_lights([light])
    if version >= 3:
        s.set_environment(np.linspace(0.1, 2.0, 24, dtype=np.float32).reshape(2, 4, 3), sample=True)
    blob = s.serialize()
    assert parse_blob(blob)[0]["version"] == version
    return blob


def _sections(blob):
    """Offsets of the light list, map record, attribute table and width table (those the blob has), and of the objects."""
    h = parse_blob(blob)[0]
    ver = int(h["version"])
    objs = 48 + int(h["n_textures"]) * 48 + int(h["n_materials"]) * 24
    off = objs + int(h["n_objects"]) * 64 + int(h["n_children"]) * 4 + int(h["n_blob_bytes"])
    sec = {"objects": objs, "v1": off}
    if ver >= 2:
        sec["lights"] = off
        off += 4 + 4 * struct.unpack_from("<i", blob, off)[0]
    if ver >= 3:
        sec["env"] = off
        w, hh = struct.unpack_from("<ii", blob, off)
        off += 24 + 12 * w * hh
    if ver >= 4:
        sec["attrs"] = off
        off += 4 + 64 * struct.unpack_from("<I", blob, off)[0]
    if ver >= 5:
        sec["widths"] = off
    return sec


def _put(blob, off, fmt, *values):
    b = bytearray(blob)
    struct.pack_into(fmt, b, off, *values)
    return bytes(b)


def _triangle_aux(blob, value):
    """The blob with the attribute index of its (one) attributed triangle set to value."""
    objs = np.frombuffer(blob, RTBS_OBJECT, count=int(parse_blob(blob)[0]["n_objects"]), offset=_sections(blob)["objects"])
    k = int(np.flatnonzero((objs["kind"] == 3) & (objs["aux"] > 0))[0])   # RTB_OBJ_TRIANGLE
    return _put(blob, _sections(blob)["objects"] + 64 * k + 16, "<i", value)


def _rough_alpha(blob, value):
    mats = parse_blob(blob)[1]
    k = int(np.flatnonzero(mats["kind"] == 5)[0])   # RTB_MAT_ROUGH_METAL
    return _put(blob, _sections(blob)["widths"] + 4 + 4 * k, "<f", value)


# (name, lowest version, damage(blob, sections) -> blob, the whole message for every version or {version: message})
DAMAGE = [
    ("short header", 2, lambda b, s: b[:40], "blob too small"),
    ("bad magic", 2, lambda b, s: _put(b, 0, "<I", 0), "bad magic/version"),
    ("version 6", 2, lambda b, s: _put(b, 4, "<I", 6), "bad magic/version"),
    ("v1 body cut", 2, lambda b, s: b[:s["v1"] - 4], {2: "blob truncated", 3: "blob truncated", 4: "blob truncated",
                                                        5: "blob truncated (light list)"}),
    ("bad root", 2, lambda b, s: _put(b, 28, "<i", 9999), "bad object id / graph too deep"),
    ("light count cut", 2, lambda b, s: b[:s["lights"] + 2], "blob truncated (light list)"),
    ("too many lights", 2, lambda b, s: _put(b, s["lights"], "<i", MAX_SAMPLED_LIGHTS + 1), "bad light list"),
    ("negative light count", 2, lambda b, s: _put(b, s["lights"], "<i", -1), "bad light list"),
    ("no light in v2", 2, lambda b, s: _put(b, s["lights"], "<i", 0), {2: "bad light list"}),
    ("light ids cut", 2, lambda b, s: b[:s["lights"] + 6], {2: "bad light list", 3: "blob truncated (environment map)",
                                                           4: "blob truncated (environment map)", 5: "blob truncated (environment map)"}),
    ("light id out of range", 2, lambda b, s: _put(b, s["lights"] + 4, "<i", 9999), "sampled light: bad object id"),
    ("light is the root list", 2, lambda b, s: _put(b, s["lights"] + 4, "<i", int(parse_blob(b)[0]["root_object"])),
     "sampled light: only spheres and quads (under translate / rotate_y) can be sampled"),
    ("map record cut", 3, lambda b, s: b[:s["env"] + 10], "blob truncated (environment map)"),
    # v5 refuses an N x 0 map only after its width table, whose reader here finds the texels where the attribute count was
    ("map width 0", 3, lambda b, s: _put(b, s["env"], "<i", 0), {3: "bad environment map", 4: "bad environment map",
                                                                  5: "blob truncated (GGX widths)"}),
    ("map too wide", 3, lambda b, s: _put(b, s["env"], "<i", ENV_MAX_SIZE + 1), "bad environment map"),
    ("negative map height", 3, lambda b, s: _put(b, s["env"] + 4, "<i", -2), "bad environment map"),
    ("map texels cut", 3, lambda b, s: b[:s["env"] + 24 + 12], {3: "bad environment map", 4: "blob truncated (triangle attributes)",
                                                               5: "blob truncated (triangle attributes)"}),
    ("attribute count cut", 4, lambda b, s: b[:s["attrs"] + 2], "blob truncated (triangle attributes)"),
    ("attribute records cut", 4, lambda b, s: b[:s["attrs"] + 4 + 10], {4: "blob truncated (triangle attributes)",
                                                                       5: "blob truncated (GGX widths)"}),
    ("attribute index beyond the table", 4, lambda b, s: _triangle_aux(b, 2), "bad triangle attribute index"),
    ("negative attribute index", 4, lambda b, s: _triangle_aux(b, -1), "bad triangle attribute index"),
    ("width count cut", 5, lambda b, s: b[:s["widths"] + 2], "blob truncated (GGX widths)"),
    ("width count off by one", 5, lambda b, s: _put(b, s["widths"], "<I", struct.unpack_from("<I", b, s["widths"])[0] + 1),
     "bad GGX width table"),
    ("widths cut", 5, lambda b, s: b[:-2], "bad GGX width table"),
    ("bytes after the widths", 5, lambda b, s: b + bytes(4), "bad GGX width table"),
    ("rough width too small", 5, lambda b, s: _rough_alpha(b, 0.0005), "bad GGX width"),
    ("rough width too large", 5, lambda b, s: _rough_alpha(b, 1.5), "bad GGX width"),
]

CASES = [pytest.param(v, name, damage, msg if isinstance(msg, str) else msg[v], id=f"v{v}-{name.replace(' ', '_')}")
         for name, lowest, damage, msg in DAMAGE for v in range(lowest, 6) if isinstance(msg, str) or v in msg]


@pytest.fixture(scope="module")
def blobs(rtb):
    return {v: _blob(rtb, v) for v in range(2, 6)}


def test_valid_blobs_load(blobs):
    for v, blob in blobs.items():
        o = FeatureOracleScene(blob)
        assert o.num_lights == 1, v
        assert len(o.alphas()) == len(parse_blob(blob)[1]), v
        assert len(o.attrs()) == (1 if v >= 4 else 0), v
        if v >= 3:
            assert o.dims() == (4, 2), v


@pytest.mark.parametrize("version,name,damage,msg", CASES)
def test_damaged_section_is_refused(blobs, version, name, damage, msg):
    blob = blobs[version]
    with pytest.raises(RuntimeError, match="load: " + re.escape(msg) + "$"):
        FeatureOracleScene(damage(blob, _sections(blob)))


def test_empty_map_record_is_no_map(blobs):
    """v4 and v5 write a 0 x 0 map record for a scene without a map, and v3 and later may list no light."""
    for v in (4, 5):
        blob = blobs[v]
        s = _sections(blob)
        w = struct.unpack_from("<i", blob, s["env"])[0]
        empty = blob[:s["lights"]] + struct.pack("<i", 0) + struct.pack("<iii3f", 0, 0, 0, 1, 1, 1) + blob[s["attrs"]:]
        o = FeatureOracleScene(empty)
        assert o.num_lights == 0
        with pytest.raises(RuntimeError, match="no environment map"):
            o.dims()
        # one dimension zero is a damaged record, not an empty one
        with pytest.raises(RuntimeError, match="bad environment map"):
            FeatureOracleScene(_put(empty, s["lights"] + 4, "<i", w))
