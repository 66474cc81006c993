"""CPU tests of per-vertex shading normals and texture coordinates of mesh triangles (DESIGN.md §5e): the rtb_add_mesh_ex
API, the RTBS v4 blob, the flattener, MeshHandle::LoadObjShaded, rtb_app's --smooth / --obj-texture, and hand-derived
answers on the CPU restatement (tests/feature_oracle.cpp): interpolated normals and UVs on one triangle, plain and instanced,
canonical UVs reproducing the plain mesh bit for bit, and the white furnace on a smooth icosphere."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

import mesh_scenes as ms
from feature_oracle import FeatureOracleScene
from helpers import parse_blob

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "ray-tracing-v06_b200"
ERR_INVALID = -1


def _mesh_ex(rtb, s, v, f, n, uv, mat):
    ptr = lambda a: None if a is None else np.ascontiguousarray(a, np.float32).ctypes.data
    v = np.ascontiguousarray(v, np.float32); f = np.ascontiguousarray(f, np.int32)
    return rtb.lib().rtb_add_mesh_ex(s.handle, v.ctypes.data, len(v), f.ctypes.data, len(f), ptr(n), ptr(uv), mat)


def _two_meshes(rtb, v, f, normals=None, uvs=None):
    """The same mesh, once plain and once with the given attributes, in two scenes."""
    out = []
    for attrs in (False, True):
        s = rtb.Scene()
        mat = s.lambertian((0.5, 0.5, 0.5))
        m = s.mesh(v, f, mat, normals=normals if attrs else None, uvs=uvs if attrs else None)
        s.set_root(s.list([m, s.sphere((0, -101, 0), 100, mat)]))
        out.append(s)
    return out


def test_api_refusals_leave_the_scene_unchanged(rtb):
    s = rtb.Scene()
    mat = s.lambertian((0.5, 0.5, 0.5))
    s.set_root(s.sphere((0, 0, 0), 1, mat))
    before, h0 = s.serialize(), s.flatten_hash()
    v = ms.TRI_V; f = np.int32([[0, 1, 2]]); n = ms.TRI_N; uv = ms.TRI_UV
    refused = [
        (v, np.int32([[0, 1, 3]]), n, uv, mat),                              # index out of range
        (v, np.int32([[0, -1, 2]]), n, uv, mat),
        (v, f, n, uv, mat + 7),                                              # bad material
        (np.float32([[0, 0, 0], [1, 0, 0], [2, 0, 0]]), f, n, uv, mat),      # no face has an area
    ]
    for bad in (np.nan, np.inf, -np.inf):
        nn = n.copy(); nn[1, 2] = bad; refused.append((v, f, nn, uv, mat))
        uu = uv.copy(); uu[2, 0] = bad; refused.append((v, f, None, uu, mat))
    for args in refused:
        assert _mesh_ex(rtb, s, *args) == ERR_INVALID
        assert s.serialize() == before and s.flatten_hash() == h0
    assert rtb.lib().rtb_add_mesh_ex(s.handle, None, 3, f.ctypes.data, 1, None, None, mat) == ERR_INVALID
    assert rtb.lib().rtb_add_mesh_ex(s.handle, np.ascontiguousarray(v).ctypes.data, 2, f.ctypes.data, 1, None, None, mat) == ERR_INVALID
    assert s.serialize() == before
    with pytest.raises(ValueError):
        s.mesh(v, f, mat, normals=n[:2])


def test_null_attributes_are_the_plain_mesh(rtb):
    """rtb_add_mesh_ex(..., NULL, NULL, ...) makes rtb_add_mesh's ids, blob and flatten hash (the degenerate face dropped
    by both)."""
    v = np.float32([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0], [2, 2, 2]])
    f = np.int32([[0, 1, 2], [0, 2, 3], [0, 0, 4]])
    blobs, hashes, ids = [], [], []
    for ex in (False, True):
        s = rtb.Scene()
        mat = s.lambertian((0.5, 0.5, 0.5))
        g = _mesh_ex(rtb, s, v, f, None, None, mat) if ex else s.mesh(v, f, mat)
        s.set_root(g)
        blobs.append(s.serialize()); hashes.append(s.flatten_hash()); ids.append(g)
    assert blobs[0] == blobs[1] and hashes[0] == hashes[1] and ids[0] == ids[1]
    assert parse_blob(blobs[0])[0]["version"] == 1


def test_v4_blob_round_trip(rtb, orc):
    """With attributes: v4 = the v1 body with each attributed triangle's aux = record + 1, an empty light list, an empty
    map record, n and the records (normals normalised in double, zero kept).  The plain oracle refuses v4; the feature oracle
    reads back what was given."""
    v, f = ms.icosphere(1)
    n = v * np.float32(3.0)
    n[5] = 0.0                                                   # a zero normal stays zero
    uv = ms.sphere_uvs(v)
    s = rtb.Scene()
    s.set_root(s.mesh(v, f, s.lambertian((0.5, 0.5, 0.5)), normals=n, uvs=uv))
    blob = s.serialize()
    h, _, objs, _ = parse_blob(blob)
    assert h["version"] == 4
    tris = [o for o in objs if o["kind"] == 3]
    assert [int(o["aux"]) for o in tris] == list(range(1, len(f) + 1))
    s2 = rtb.Scene(); s2.set_root(s2.mesh(v, f, s2.lambertian((0.5, 0.5, 0.5))))
    v1 = s2.serialize()
    assert len(blob) == len(v1) + 4 + 24 + 4 + 64 * len(f)
    tail = blob[len(v1):]
    assert np.frombuffer(tail[:4], np.int32)[0] == 0
    assert list(np.frombuffer(tail[4:16], np.int32)) == [0, 0, 0]
    assert np.frombuffer(tail[28:32], np.uint32)[0] == len(f)
    got = FeatureOracleScene(blob).attrs()
    assert len(got) == len(f) and np.all(got["flags"] == 3)
    n64 = n.astype(np.float64); ln = np.linalg.norm(n64, axis=1, keepdims=True)
    unit = np.where(ln > 0, n64 / np.where(ln > 0, ln, 1), 0).astype(np.float32)
    assert np.array_equal(got["n"], unit[f]) and np.array_equal(got["uv"], uv[f])
    with pytest.raises(RuntimeError, match="version"):
        orc.OracleScene(blob)
    # with a light list and a map too: the list, the map, then the attributes
    s.set_environment(np.ones((2, 4, 3), np.float32))
    blob3 = s.serialize()
    assert parse_blob(blob3)[0]["version"] == 4 and len(blob3) == len(blob) + 4 * 2 * 3 * 4
    assert len(FeatureOracleScene(blob3).attrs()) == len(f)


def test_scenes_without_attributes_keep_their_format(rtb):
    """Registry scenes through the feature oracle's loader, and a mesh without attributes: unchanged versions and hashes."""
    for name in ("mesh_icospheres", "book2_final"):
        s = rtb.Scene.named(name)
        blob = s.serialize()
        assert parse_blob(blob)[0]["version"] == 1
        FeatureOracleScene(blob)


@pytest.mark.parametrize("attrs", ["normals", "uvs", "both"])
def test_same_tree_and_records_with_and_without_attributes(rtb, attrs):
    v, f = ms.icosphere(2)
    plain, ex = _two_meshes(rtb, v, f, normals=v if attrs != "uvs" else None, uvs=ms.sphere_uvs(v) if attrs != "normals" else None)
    assert plain.flatten_stats() == ex.flatten_stats()
    (a, ra), (b, rb) = plain.world_bvh(), ex.world_bvh()
    assert ra == rb and a.tobytes() == b.tobytes()
    assert plain.flatten_hash() != ex.flatten_hash()


# ------------------------------------------------------------------------------------------------ LoadObjShaded

_LOADER = r'''
#include <cstdio>
#include "rt_engine/geometry/Mesh.cuh"
int main(int, char** argv) {
	Mesh m = MeshHandle::LoadObjShaded(argv[1]);
	printf("%zu %zu %zu %zu\n", m.vertices.size(), m.indices.size() / 3, m.normals.size(), m.uvs.size());
	for (size_t i = 0; i < m.vertices.size(); ++i)
		printf("%.9g %.9g %.9g %.9g %.9g %.9g %.9g %.9g\n", m.vertices[i].x, m.vertices[i].y, m.vertices[i].z,
		       m.normals[i].x, m.normals[i].y, m.normals[i].z, m.uvs.empty() ? -1.0f : m.uvs[i].x, m.uvs.empty() ? -1.0f : m.uvs[i].y);
	for (int i : m.indices) printf("%d ", i);
	printf("\n");
	return 0;
}'''


@pytest.fixture(scope="module")
def loader(tmp_path_factory):
    d = tmp_path_factory.mktemp("loader")
    (d / "l.cpp").write_text(_LOADER)
    subprocess.run(["g++", "-std=c++20", "-O1", f"-I{PKG / 'host'}", f"-I{PKG / 'host' / 'glm_compat'}", f"-I{ROOT / 'include'}", "-I/usr/local/cuda/include",
                    "-o", str(d / "l"), str(d / "l.cpp"), f"-L{PKG}", "-lrtb200", f"-Wl,-rpath,{PKG}"], check=True, capture_output=True)

    def run(text):
        (d / "m.obj").write_text(text)
        out = subprocess.run([str(d / "l"), str(d / "m.obj")], check=True, capture_output=True, text=True).stdout.splitlines()
        nv, nf, nn, nt = map(int, out[0].split())
        rows = np.array([list(map(float, r.split())) for r in out[1:1 + nv]], np.float64).reshape(nv, 8)
        idx = np.array(out[1 + nv].split(), np.int32).reshape(nf, 3)
        return nv, nf, nn, nt, rows, idx
    return run


def test_obj_shaded_corners_and_file_normals(loader):
    """v/vt/vn corners: one vertex per distinct (v, vt, vn); a polygon is fanned; normals and UVs from the file."""
    nv, nf, nn, nt, rows, idx = loader(
        "v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\n"
        "vt 0 0\nvt 1 0\nvt 1 1\nvt 0 1\nvt 0.5 0.5\n"
        "vn 0 0 2\nvn 0 1 1\n"
        "f 1/1/1 2/2/1 3/3/1 4/4/1\n"              # quad -> 2 triangles over 4 corners
        "f 1/5/2 -3/-4/-1 -2/3/1\n")               # (1, 5, 2) and (2, 2, 2) are new triples, (3, 3, 1) is not
    assert (nv, nf, nn, nt) == (6, 3, 6, 6)
    assert idx.tolist() == [[0, 1, 2], [0, 2, 3], [4, 5, 2]]
    assert np.allclose(rows[:, 3:6], [[0, 0, 2], [0, 0, 2], [0, 0, 2], [0, 0, 2], [0, 1, 1], [0, 1, 1]])   # as written (the ABI normalises)
    assert np.allclose(rows[:, 6:8], [[0, 0], [1, 0], [1, 1], [0, 1], [0.5, 0.5], [1, 0]])


def test_obj_shaded_computed_normals(loader):
    """Without vn on every corner: area-weighted face normals summed per position in double, normalised; no vt on every
    corner: no UVs; v//vn corners with missing vn records (the registry's icosphere file) load with computed normals."""
    v, f = ms.icosphere(1)
    v = v * np.float32([1.0, 0.7, 1.3])                       # an ellipsoid: the weights matter
    text = "".join(f"v {x:.9g} {y:.9g} {z:.9g}\n" for x, y, z in v) + "vt 0.5 0.5\n"
    text += "".join(f"f {a + 1}//{a + 1} {b + 1}/1/{b + 1} {c + 1}//{c + 1}\n" for a, b, c in f)   # vn indices, no vn records
    nv, nf, nn, nt, rows, idx = loader(text)
    assert (nv, nf, nn, nt) == (len(v), len(f), len(v), 0)
    order = np.array(list(dict.fromkeys(f.reshape(-1).tolist())))        # positions in order of first appearance
    assert np.array_equal(order[idx], f) and np.array_equal(rows[:, :3].astype(np.float32), v[order])
    p = v.astype(np.float64)
    cr = np.cross(p[f[:, 1]] - p[f[:, 0]], p[f[:, 2]] - p[f[:, 0]])
    acc = np.zeros_like(p)
    for k in range(3):
        np.add.at(acc, f[:, k], cr)
    want = (acc / np.linalg.norm(acc, axis=1, keepdims=True)).astype(np.float32)
    assert np.allclose(rows[:, 3:6], want[order], rtol=0, atol=1e-7)
    # a lone degenerate face keeps zero normals; an isolated position is not a vertex
    nv, nf, nn, nt, rows, idx = loader("v 0 0 0\nv 1 0 0\nv 2 0 0\nv 5 5 5\nf 1 2 3\n")
    assert (nv, nf) == (3, 1) and np.all(rows[:, 3:6] == 0)


def test_registry_icosphere_file_loads_shaded(rtb, tmp_path):
    """The registry writes its icosphere as `f a//a b//b c//c` without vn records: LoadObjShaded reads it with computed
    normals, and the mirror hands it to rtb_add_mesh_ex."""
    v, f = ms.icosphere(3)
    text = "".join(f"v {x:.9g} {y:.9g} {z:.9g}\n" for x, y, z in v)
    text += "".join(f"f {a + 1}//{a + 1} {b + 1}//{b + 1} {c + 1}//{c + 1}\n" for a, b, c in f)
    (tmp_path / "ico.obj").write_text(text)
    (tmp_path / "m.cpp").write_text(r'''
#include <cstdio>
#include <vector>
#include "rt_engine/geometry/Mesh.cuh"
#include "rt_engine/shaders/cu_materials.cuh"
int main(int, char** argv) {
	Mesh m = MeshHandle::LoadObjShaded(argv[1]);
	Lambertian grey(glm::vec3(0.5f));
	MeshHandle h = MeshHandle::MakeMesh(m, &grey);
	rtb_scene_set_root(rtb_host::scene(), h.getHittablePtr()->rtb_object);
	size_t n = rtb_scene_serialize(rtb_host::scene(), nullptr, 0);
	std::vector<unsigned char> blob(n); rtb_scene_serialize(rtb_host::scene(), blob.data(), n);
	FILE* f = fopen(argv[2], "wb"); fwrite(blob.data(), 1, n, f); fclose(f);
	printf("%zu %d\n", m.vertices.size(), h.triangleCount());
	return 0;
}''')
    subprocess.run(["g++", "-std=c++20", "-O1", f"-I{PKG / 'host'}", f"-I{PKG / 'host' / 'glm_compat'}", f"-I{ROOT / 'include'}", "-I/usr/local/cuda/include",
                    "-o", str(tmp_path / "m"), str(tmp_path / "m.cpp"), f"-L{PKG}", "-lrtb200", f"-Wl,-rpath,{PKG}"], check=True, capture_output=True)
    out = subprocess.run([str(tmp_path / "m"), str(tmp_path / "ico.obj"), str(tmp_path / "m.rtbs")], check=True, capture_output=True, text=True).stdout.split()
    assert out == [str(len(v)), str(len(f))]
    at = FeatureOracleScene((tmp_path / "m.rtbs").read_bytes()).attrs()
    assert len(at) == len(f) and np.all(at["flags"] == 1)
    # on a unit icosphere the computed normals are close to the positions
    assert np.allclose(at["n"], v[f], atol=0.02)


def test_app_refuses_obj_texture_without_uvs(rtb, tmp_path):
    app = str(PKG / "rtb_app")
    (tmp_path / "m.obj").write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    (tmp_path / "t.ppm").write_bytes(b"P6\n2 1\n255\n" + bytes(6))
    no_uv = subprocess.run([app, "--obj", str(tmp_path / "m.obj"), "--smooth", "--obj-texture", str(tmp_path / "t.ppm")], capture_output=True, text=True)
    assert no_uv.returncode == 1 and "texture coordinates" in no_uv.stderr
    no_smooth = subprocess.run([app, "--obj", str(tmp_path / "m.obj"), "--obj-texture", str(tmp_path / "t.ppm")], capture_output=True, text=True)
    assert no_smooth.returncode == 1 and "--smooth" in no_smooth.stderr
    no_obj = subprocess.run([app, "--smooth"], capture_output=True, text=True)
    assert no_obj.returncode == 1


# ------------------------------------------------------------------------------------------------ known answers (oracle)

def _check_hits(got, rays, ab, back, normals, uvs, instanced):
    ns, uv = ms.expected_attributes(ab, back, normals=normals, uvs=uvs, instanced=instanced)
    assert np.all(got["t"] < 1e30), "every ray hits the triangle"
    assert np.allclose(got["n"], ns, rtol=0, atol=1e-6)
    assert np.allclose(np.stack([got["u"], got["v"]], -1), uv, rtol=0, atol=1e-6)
    assert np.array_equal(got["front_face"], (~back).astype(np.int32))


@pytest.mark.parametrize("instanced", [False, True])
@pytest.mark.parametrize("flip", [False, True])
@pytest.mark.parametrize("normals,uvs", [(True, True), (True, False), (False, True)])
def test_triangle_known_answers_oracle(rtb, instanced, flip, normals, uvs):
    """The interpolated normal and UV at the vertices, edge midpoints and centroid, from both sides, with vertex normals
    that agree and that disagree with the winding, plain and under rotate_y(90) + translate: float64 within 1e-6."""
    if flip and not normals:
        pytest.skip("flip negates normals")
    s = ms.triangle_scene(rtb, normals=normals, flip=flip, uvs=uvs, instanced=instanced)
    rays, ab, back = ms.triangle_rays(rtb, instanced=instanced, inset=1e-4)
    got = FeatureOracleScene(s.serialize()).trace(rays, rtb.HIT_DTYPE)
    _check_hits(got, rays, ab, back, normals, uvs, instanced)


def test_canonical_uvs_reproduce_the_plain_mesh_oracle(rtb):
    """Canonical UVs (0,0), (1,0), (0,1) on unshared faces, UVs only: (u, v) = (alpha, beta) exactly, so the image-textured
    accumulators equal the plain mesh's bit for bit."""
    (a, cam), (b, _) = ms.canonical_uv_scene(rtb, False), ms.canonical_uv_scene(rtb, True)
    assert parse_blob(b.serialize())[0]["version"] == 4
    ra = FeatureOracleScene(a.serialize()).render(cam, 48, 32, 0, 4, 8)
    rb = FeatureOracleScene(b.serialize()).render(cam, 48, 32, 0, 4, 8)
    assert ra[2] == rb[2] and np.array_equal(ra[0], rb[0])


@pytest.mark.parametrize("smooth", [True, False])
def test_white_furnace_on_an_icosphere_oracle(rtb, smooth):
    """White Lambertian under a white sky: every path that leaves returns exactly 1 and every other path 0, so each
    pixel's sum is spp minus the paths that ran out of depth (below the geometric surface a smooth normal can send a path
    into the closed mesh), and no pixel exceeds spp."""
    s, cam = ms.furnace_scene(rtb, smooth=smooth)
    spp = 16
    acc, _, _ = FeatureOracleScene(s.serialize()).render(cam, 32, 32, 0, spp, 20)
    rgb = acc[..., :3]
    assert np.all(rgb == np.round(rgb)) and np.all(rgb <= spp) and np.all(rgb >= 0)
    assert np.all(rgb[..., 0] == rgb[..., 1]) and np.all(rgb[..., 1] == rgb[..., 2])
    lost = spp * rgb[..., 0].size - rgb[..., 0].sum()
    assert lost <= 0.05 * spp * rgb[..., 0].size
