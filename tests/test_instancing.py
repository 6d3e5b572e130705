"""EXT_mesh_gpu_instancing and meshes shared by several nodes (DESIGN.md "Loader contract").

The oracle's glTF driver does not read the extension, so parity is stated through the twin: an instanced file flattens, builds,
traces and renders to the same bits as the same scene written with one plain child node per instance (tests/instancing_scenes.py
instanced_scene).  C5 rewritten with one-instance extension nodes must still match the oracle's committed C5 digests.

CPU part: the host-compiled kernel bodies.  GPU part: the same through the CUDA library, plus the full-size scenes."""
import json
import os

import numpy as np
import pytest

import parity_checks as pc
import instancing_scenes
import scenes
from golden import make_golden_c4c5 as MG
from sailor_b200.capi import ERR_FORMAT, ERR_LIMIT, Params, SailorPtError

HERE = os.path.dirname(os.path.abspath(__file__))

SMALL_HITS = Params(height=54, width_override=96)
SMALL_RENDER = dict(height=18, width_override=32, num_samples=2, num_ambient_samples=2, max_bounces=3, msaa=2, ambient=(0.6, 0.7, 0.9), seed=7)


@pytest.fixture(scope="module")
def D4():
    return json.load(open(os.path.join(HERE, "golden", "digests_c4c5.json")))


def _scene_pair(d, tag, **kw):
    a = instancing_scenes.instanced_scene(os.path.join(d, "inst_%s_ext.glb" % tag), form="ext", **kw)
    b = instancing_scenes.instanced_scene(os.path.join(d, "inst_%s_nodes.glb" % tag), form="nodes", **kw)
    return a, b


def _u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


def check_same_scene(lib, a, b, hits=SMALL_HITS, render=SMALL_RENDER):
    """Everything the C-ABI reports about the two files is bit-identical."""
    with lib.load_scene(a) as s, lib.load_scene(b) as t:
        assert s.counts() == t.counts()
        ta, ma = s.triangles()
        tb, mb = t.triangles()
        assert len(ta) == s.counts()["triangles"]
        assert np.array_equal(_u32(ta), _u32(tb)), "flattened triangles differ from the twin's"
        assert np.array_equal(ma, mb), "material indices differ from the twin's"
        assert np.array_equal(s.materials(), t.materials())
        na, pa = s.bvh()
        nb, pb = t.bvh()
        assert na.tobytes() == nb.tobytes() and np.array_equal(pa, pb), "BVH differs from the twin's"
        ha, hb = s.primary_hits(hits), t.primary_hits(hits)
        assert int((ha["triId"] != pc.NOHIT).sum()) > 0
        assert ha.tobytes() == hb.tobytes(), "primary hits differ from the twin's"
        if render is not None:
            la, sa = s.render(Params(**render))
            lb, sb = t.render(Params(**render))
            assert np.isfinite(la).all() and la.max() > 0
            assert np.array_equal(_u32(la), _u32(lb)) and np.array_equal(sa, sb), "rendered frame differs from the twin's"
        return s.counts()["triangles"]


def _check_small_twins(lib, d):
    for rotation in ("f32", "i8", "i16"):
        a, b = _scene_pair(d, rotation, rotation=rotation)
        assert check_same_scene(lib, a, b) == 2 * 8 * 8 * 7 + 2
    # missing attributes are the identity; "_ID" is ignored
    a, b = _scene_pair(d, "tr", attributes=("TRANSLATION", "ROTATION"), instances=5)
    assert check_same_scene(lib, a, b) == 2 * 8 * 8 * 5 + 2
    # many draws per flatten span: 2,000 instances of a 12-triangle mesh
    a, b = _scene_pair(d, "many", nx=2, nz=3, instances=2000)
    assert check_same_scene(lib, a, b) == 2000 * 12 + 2


def _check_c5_small_as_extension(lib, d, D4):
    path = instancing_scenes.c5_as_instancing_extension(scenes.ensure(d, "instanced", **MG.C5_SMALL_KW), os.path.join(d, "c5_small_ext.glb"))
    with lib.load_scene(path) as s:
        tris, mat = s.triangles()
        assert len(tris) == D4["c5_small_tris"]["count"]
        assert pc.sha(tris) == D4["c5_small_tris"]["sha256"] and pc.sha(mat) == D4["c5_small_tris"]["mat"], "instanced flatten differs"
        nodes, mapping = s.bvh()
        dg = D4["c5_small_bvh"]
        assert len(nodes) == dg["nodes"] and pc.sha(mapping) == dg["mapping"]
        assert pc.sha(nodes["leftFirst"]) == dg["leftFirst"] and pc.sha(nodes["triCount"]) == dg["triCount"]
        assert pc.sha(nodes["aabbMin"] + np.float32(0)) == dg["aabbMin"] and pc.sha(nodes["aabbMax"] + np.float32(0)) == dg["aabbMax"]
        hits = s.primary_hits(Params(height=270, width_override=480))
        assert pc.sha(hits) == D4["c5_small_hits"]["sha256"]


def _check_shared_mesh_upload(lib, d):
    """C5-small places one mesh's streams under 10 nodes: they cross to the device once."""
    n = MG.C5_SMALL_KW["n"]
    one_instance = (n + 1) * (n + 1) * 3 * 4 + n * n * 6 * 4          # float3 positions + uint32 indices = 84,108 B
    with lib.load_scene(scenes.ensure(d, "instanced", **MG.C5_SMALL_KW)) as s:
        h2d = lib.stats()["h2dBytes"]
        assert s.counts()["triangles"] == 10 * 2 * n * n
    assert one_instance <= h2d <= 1.2 * one_instance, "h2dBytes = %d for streams of %d B" % (h2d, one_instance)


def _check_refusals(lib, d):
    for kind in ("missing_accessor", "vec2_translation", "unequal_counts", "no_attributes"):
        path = instancing_scenes.broken_instancing_scene(os.path.join(d, "broken_%s.glb" % kind), kind)
        with pytest.raises(SailorPtError) as e:
            lib.load_scene(path)
        assert e.value.code == ERR_FORMAT and "node[1]" in str(e.value), (kind, str(e.value))
    path = instancing_scenes.instancing_limit_scene(os.path.join(d, "limit_2p32.glb"))
    assert os.path.getsize(path) < 2 << 20
    with pytest.raises(SailorPtError) as e:
        lib.load_scene(path)
    assert e.value.code == ERR_LIMIT and "node[0]" in str(e.value)
    # the smallest instance count above floor((2^32 - 1) / 3) triangles, a count that still fits in 32 bits
    path = instancing_scenes.instancing_limit_scene(os.path.join(d, "limit_bound.glb"), instances=21846)
    with pytest.raises(SailorPtError) as e:
        lib.load_scene(path)
    assert e.value.code == ERR_LIMIT


def test_instanced_scene_equals_its_twin_cpu(emu, tmp_path):
    _check_small_twins(emu, str(tmp_path))


def test_c5_small_as_one_instance_extensions_matches_the_digests_cpu(emu, D4, tmp_path):
    _check_c5_small_as_extension(emu, str(tmp_path), D4)


def test_a_shared_mesh_is_uploaded_once_cpu(emu, scene_dir):
    _check_shared_mesh_upload(emu, scene_dir)


def test_malformed_and_oversized_instancing_is_refused_cpu(emu, tmp_path):
    _check_refusals(emu, str(tmp_path))


def test_extension_on_a_node_without_mesh_is_ignored_cpu(emu, tmp_path):
    d = str(tmp_path)
    path = instancing_scenes.instanced_scene(os.path.join(d, "plain.glb"), form="nodes", instances=3)
    j, b = instancing_scenes.read_glb(path)
    # the parent of the instances (no mesh) gets an extension object, which must change nothing
    parent = next(n for n in j["nodes"] if "children" in n and "mesh" not in n and len(n["children"]) == 4)
    parent["extensions"] = {"EXT_mesh_gpu_instancing": {"attributes": {"TRANSLATION": 999}}}
    g = scenes.GlbBuilder()
    g.j, g.bin = j, bytearray(b)
    other = g.write(os.path.join(d, "plain_ext_on_empty.glb"))
    check_same_scene(emu, path, other, render=None)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_instanced_scene_equals_its_twin_gpu(gpu, tmp_path):
    _check_small_twins(gpu, str(tmp_path))


@pytest.mark.gpu
def test_c5_small_as_one_instance_extensions_matches_the_digests_gpu(gpu, D4, tmp_path):
    _check_c5_small_as_extension(gpu, str(tmp_path), D4)


@pytest.mark.gpu
def test_a_shared_mesh_is_uploaded_once_gpu(gpu, scene_dir):
    _check_shared_mesh_upload(gpu, scene_dir)


@pytest.mark.gpu
def test_malformed_and_oversized_instancing_is_refused_gpu(gpu, tmp_path):
    _check_refusals(gpu, str(tmp_path))


@pytest.mark.gpu
def test_c5_as_one_instance_extensions_matches_the_digests_gpu(gpu, D4, scene_dir, tmp_path):
    """Full-size C5 (9,996,980 triangles) written as one-instance extension nodes: the oracle's C5 digests."""
    path = instancing_scenes.c5_as_instancing_extension(scenes.ensure(scene_dir, "instanced", **MG.C5_KW), os.path.join(str(tmp_path), "c5_ext.glb"))
    with gpu.load_scene(path) as s:
        assert s.counts()["triangles"] == D4["c5_counts"]["triangles"]
        nodes, mapping = s.bvh()
        dg = D4["c5_bvh"]
        assert len(nodes) == dg["nodes"] and pc.sha(mapping) == dg["mapping"]
        assert pc.sha(nodes["leftFirst"]) == dg["leftFirst"] and pc.sha(nodes["triCount"]) == dg["triCount"]
        assert pc.sha(nodes["aabbMin"] + np.float32(0)) == dg["aabbMin"] and pc.sha(nodes["aabbMax"] + np.float32(0)) == dg["aabbMax"]
        hits = s.primary_hits(Params(height=2160, width_override=3840))
        assert list(hits.shape) == D4["c5_hits_4k"]["shape"] and pc.sha(hits) == D4["c5_hits_4k"]["sha256"]


@pytest.mark.gpu
def test_ten_million_triangle_instanced_scene_equals_its_twin_gpu(gpu, tmp_path):
    a, b = _scene_pair(str(tmp_path), "10m", nx=707, nz=707, instances=10)
    render = dict(height=135, width_override=240, num_samples=2, num_ambient_samples=2, max_bounces=6, msaa=2, ambient=(1, 1, 1), seed=3)
    assert check_same_scene(gpu, a, b, hits=Params(height=1080, width_override=1920), render=render) == 10 * 2 * 707 * 707 + 2


@pytest.mark.gpu
def test_many_small_instances_equal_their_twin_gpu(gpu, tmp_path):
    """100,000 instances of a 120-triangle mesh (12 M triangles): 10^5 draws in the flatten pass."""
    a, b = _scene_pair(str(tmp_path), "100k", nx=6, nz=10, instances=100000)
    render = dict(height=135, width_override=240, num_samples=2, num_ambient_samples=2, max_bounces=6, msaa=2, ambient=(1, 1, 1), seed=3)
    assert check_same_scene(gpu, a, b, hits=Params(height=1080, width_override=1920), render=render) == 100000 * 120 + 2


@pytest.mark.gpu
def test_instanced_multi_device_frame_equals_single_device_frame_gpu(gpu, tmp_path, monkeypatch):
    monkeypatch.setenv("SAILOR_PT_MULTI_SAME_DEVICE", "1")
    a = instancing_scenes.instanced_scene(os.path.join(str(tmp_path), "inst_multi.glb"), nx=64, nz=64, instances=50, rotation="i16")
    assert pc.check_multi_device_frame(gpu, a, devices=3, height=40) == 3
