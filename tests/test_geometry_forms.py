"""glTF triangle strips and fans, sparse accessors and quantized streams, assembled and decoded on the device (DESIGN.md "Loader
contract").

The oracle's glTF driver reads only TRIANGLES and no sparse data, so parity is stated through the twin (tests/geometry_scenes.py):
each file flattens, builds, traces and renders to the same bits as the same triangles written as a float32 TRIANGLES list with
u32 indices.  CPU part: the host-compiled kernel bodies.  GPU part: the same through the CUDA library, plus the full-size C5 forms."""
import json
import os

import numpy as np
import pytest

import geometry_scenes as gs
import parity_checks as pc
import scenes
from golden import make_golden_c4c5 as MG
from sailor_b200.capi import ERR_FORMAT, ERR_LIMIT, Params, SailorPtError
from test_instancing import check_same_scene

HERE = os.path.dirname(os.path.abspath(__file__))


def _pair(d, tag, **kw):
    return (gs.forms_scene(os.path.join(d, "%s.glb" % tag), **kw), gs.forms_scene(os.path.join(d, "%s_twin.glb" % tag), twin=True, **kw))


def _corners(lib, path):
    """Vertex numbers of every flattened triangle of a literal_scene (vertex k sits at x = k)."""
    with lib.load_scene(path) as s:
        tris, _ = s.triangles()
    return [tuple(int(round(x)) for x in t[3:12:3]) for t in tris]


def _check_literals(lib, d):
    strip, fan = [(0, 1, 2), (1, 3, 2), (2, 3, 4)], [(1, 2, 0), (2, 3, 0), (3, 4, 0)]
    for it in (None, np.uint8, np.uint16, np.uint32):
        name = "none" if it is None else np.dtype(it).name
        assert _corners(lib, gs.literal_scene(os.path.join(d, "strip_%s.glb" % name), 5, it)) == strip
        assert _corners(lib, gs.literal_scene(os.path.join(d, "fan_%s.glb" % name), 6, it)) == fan
        assert _corners(lib, gs.literal_scene(os.path.join(d, "list_%s.glb" % name), 4, it, n=7)) == [(0, 1, 2), (3, 4, 5)]
        for mode in (5, 6):
            for n in (1, 2):                      # fewer than 3: no faces (the file's other primitive still draws)
                path = gs.literal_scene(os.path.join(d, "short_%d_%d_%s.glb" % (mode, n, name)), mode, it, n=n, extra_primitive=True)
                assert len(_corners(lib, path)) == 1
    # modes 0-3 (points, lines) stay ignored
    for mode in (0, 1, 2, 3):
        assert len(_corners(lib, gs.literal_scene(os.path.join(d, "mode%d.glb" % mode), mode, None, extra_primitive=True))) == 1


def _check_form_twins(lib, d):
    cases = []
    for mode in (5, 6, 4):
        for it in (None, np.uint8, np.uint16, np.uint32):
            cases.append(dict(mode=mode, index_type=it))
    for enc in ("i16n", "i8n", "u16n", "u8n", "i16", "u8", "u16", "interleaved"):
        cases.append(dict(mode=5, index_type=np.uint16, encoding=enc))
        cases.append(dict(mode=4, index_type=np.uint8, encoding=enc))
    cases.append(dict(mode=6, index_type=None, encoding="i8n"))
    cases.append(dict(mode=5, index_type=np.uint16, shared_list=True))               # same accessors, two modes: two sources
    cases.append(dict(mode=5, index_type=np.uint8, encoding="i16n", shared_list=True))
    cases.append(dict(mode=5, index_type=np.uint16, instances=5))                   # a strip mesh under EXT_mesh_gpu_instancing
    cases.append(dict(mode=5, index_type=None, encoding="i8n", instances=3))
    for k, kw in enumerate(cases):
        a, b = _pair(d, "case%d" % k, **kw)
        render = gs_render if k % 4 == 0 else None
        assert check_same_scene(lib, a, b, render=render) > 0, kw


gs_render = dict(height=18, width_override=32, num_samples=2, num_ambient_samples=2, max_bounces=3, msaa=2, ambient=(0.6, 0.7, 0.9), seed=7)


# ---------------------------------------------------------------------------------------------------------------- sparse
def _sparse_scene(path, target, kind="ok", twin=False, base=True):
    """A strip mesh (u16 indices, float streams) whose `target` accessor (POSITION, NORMAL, indices, TRANSLATION) carries a sparse block.
    kind: "ok", or a malformed block: "count0", "count_big", "index_type", "view", "index_big", "not_increasing".  base=False: the
    accessor has no bufferView (its base is zeros).  twin=True: the dense result, or what the loader does with a malformed block."""
    w = gs.Writer()
    g = w.g
    m = gs._material(g, 0)
    pos, nrm, uv, _, _ = gs._mesh_streams(5, 4, 6)
    idx = gs._strip_indices(5, 4).astype(np.uint16)
    arrays = {"POSITION": pos, "NORMAL": nrm}
    at = np.array([1, 4, 7, 11, 17], np.uint32)
    count = {"POSITION": len(pos), "NORMAL": len(nrm), "indices": len(idx), "TRANSLATION": 4}[target]
    if target in arrays:
        vals = (arrays[target][at] * np.float32(1.25) + np.float32(0.125)).astype(np.float32)
    elif target == "indices":
        at = np.array([0, 3, 8, 20, 21], np.uint8)
        vals = np.array([5, 13, 2, 29, 7], np.uint16)
    else:
        at = np.array([1, 3], np.uint16)
        vals = np.array([[0.5, 0.25, -0.5], [1.0, 0.0, 0.75]], np.float32)
    dense_base = {"POSITION": pos, "NORMAL": nrm, "indices": idx, "TRANSLATION": np.stack([np.arange(4) * 1.5, np.zeros(4), np.zeros(4)], -1).astype(np.float32)}[target]
    if not base:
        dense_base = np.zeros_like(dense_base)
    dense = dense_base.copy()
    dense[at.astype(np.int64)] = vals
    if kind == "index_big":
        at = at.copy()
        at[-1] = count
    elif kind == "not_increasing":
        at = at.copy()
        at[-1] = at[-2]
    typ = {"POSITION": "VEC3", "NORMAL": "VEC3", "indices": "SCALAR", "TRANSLATION": "VEC3"}[target]

    def acc(name, arr):
        if name != target:
            return w.accessor(arr, typ if name == target else {"POSITION": "VEC3", "NORMAL": "VEC3", "indices": "SCALAR", "TEXCOORD_0": "VEC2", "TRANSLATION": "VEC3"}[name])
        if twin:
            if kind == "ok":
                return w.accessor(dense, typ)
            return None                          # the documented fallback: the accessor is unreadable
        a = w.accessor(dense_base, typ, sparse=(at, vals), view=base)
        sp = g.j["accessors"][a]["sparse"]
        if kind == "index_type":
            sp["indices"]["componentType"] = 5126
        elif kind == "count0":
            sp["count"] = 0
        elif kind == "count_big":
            sp["count"] = count + 1
        elif kind == "view":
            sp["values"]["byteOffset"] = 10 ** 6
        return a

    attrs = {"POSITION": acc("POSITION", pos), "NORMAL": acc("NORMAL", nrm), "TEXCOORD_0": w.accessor(uv, "VEC2")}
    attrs = {k: v for k, v in attrs.items() if v is not None}
    prim = {"attributes": attrs, "mode": 5, "material": m}
    ia = acc("indices", idx)
    if ia is not None:
        prim["indices"] = ia
    if "POSITION" not in attrs:
        prim = None
    other = {"attributes": {"POSITION": w.accessor(np.array([[0, 0, -1], [1, 0, -1], [0, 1, -1]], np.float32), "VEC3")}, "material": m}
    g.j["meshes"].append({"primitives": ([prim] if prim else []) + [other]})
    if target == "TRANSLATION":
        ta = acc("TRANSLATION", dense_base)
        if twin:
            kids = [g.node(root=False, mesh=0, translation=[float(x) for x in t]) for t in dense]
            g.node(children=kids)
        else:
            g.j["extensionsUsed"] = ["EXT_mesh_gpu_instancing"]
            g.node(mesh=0, extensions={"EXT_mesh_gpu_instancing": {"attributes": {"TRANSLATION": ta}}})
    else:
        g.node(mesh=0)
    gs._camera_and_sun(g, eye=(0.0, 0.9, 1.4), forward=(0.0, -0.6, -0.9))
    return g.write(path)


MALFORMED = ("count0", "count_big", "index_type", "view", "index_big", "not_increasing")


def _check_sparse(lib, d):
    for target in ("POSITION", "NORMAL", "indices", "TRANSLATION"):
        for base in ((True, False) if target == "POSITION" else (True,)):
            a = _sparse_scene(os.path.join(d, "sp_%s_%d.glb" % (target, base)), target, base=base)
            b = _sparse_scene(os.path.join(d, "sp_%s_%d_twin.glb" % (target, base)), target, base=base, twin=True)
            check_same_scene(lib, a, b, render=gs_render if target == "POSITION" and base else None)
    for target in ("POSITION", "NORMAL", "indices"):
        for kind in MALFORMED:
            a = _sparse_scene(os.path.join(d, "bad_%s_%s.glb" % (target, kind)), target, kind)
            b = _sparse_scene(os.path.join(d, "bad_%s_%s_twin.glb" % (target, kind)), target, kind, twin=True)
            check_same_scene(lib, a, b, render=None)
    for kind in MALFORMED:
        path = _sparse_scene(os.path.join(d, "bad_T_%s.glb" % kind), "TRANSLATION", kind)
        with pytest.raises(SailorPtError) as e:
            lib.load_scene(path)
        assert e.value.code == ERR_FORMAT and "node[0]" in str(e.value), (kind, str(e.value))


def _oversized(path, what):
    """A small file asking for a bufferView-less sparse POSITION of 2^31 elements, or a strip of 2^33 indices."""
    w = gs.Writer()
    g = w.g
    m = gs._material(g, 0)
    pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    if what == "position":
        pa = w.accessor(np.zeros((1, 3), np.float32), "VEC3", sparse=(np.array([5], np.uint32), np.ones((1, 3), np.float32)), view=False)
        g.j["accessors"][pa]["count"] = 2 ** 31
        prim = {"attributes": {"POSITION": pa}, "mode": 4, "material": m}
    else:
        ia = w.accessor(np.zeros(1, np.uint32), "SCALAR", sparse=(np.array([7], np.uint32), np.ones(1, np.uint32)), view=False)
        g.j["accessors"][ia]["count"] = 2 ** 33
        prim = {"attributes": {"POSITION": w.accessor(pos, "VEC3")}, "mode": 5, "indices": ia, "material": m}
    g.j["bin_pad"] = "x" * (1 << 20)                            # about 1 MB, like a real file
    g.j["meshes"].append({"primitives": [prim]})
    g.node(mesh=0)
    return g.write(path)


def _check_oversized(lib, d):
    for what in ("position", "strip"):
        path = _oversized(os.path.join(d, "over_%s.glb" % what), what)
        assert os.path.getsize(path) < 2 << 20
        with pytest.raises(SailorPtError) as e:
            lib.load_scene(path)
        assert e.value.code == ERR_LIMIT and "node[0]" in str(e.value), str(e.value)
    # EXT_mesh_gpu_instancing with a bufferView-less sparse TRANSLATION of 2^40 instances: a mesh that draws nothing (a points
    # primitive) gets no per-instance data and the file loads; a mesh with a triangle is above the triangle limit
    for faces in (0, 1):
        path = _sparse_instances(os.path.join(d, "over_instances_%d.glb" % faces), faces)
        if faces:
            with pytest.raises(SailorPtError) as e:
                lib.load_scene(path)
            assert e.value.code == ERR_LIMIT and "node[0]" in str(e.value), str(e.value)
        else:
            with lib.load_scene(path) as s:
                assert s.counts()["triangles"] == 1


def _sparse_instances(path, faces, count=2 ** 40):
    """Node 0 instances a mesh (one points primitive, or one triangle) by a bufferView-less sparse TRANSLATION of `count` entries;
    node 1 draws one plain triangle."""
    w = gs.Writer()
    g = w.g
    m = gs._material(g, 0)
    tri = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    g.j["meshes"].append({"primitives": [{"attributes": {"POSITION": w.accessor(tri, "VEC3")}, "mode": 4 if faces else 0, "material": m}]})
    g.j["meshes"].append({"primitives": [{"attributes": {"POSITION": w.accessor(tri + np.float32(2), "VEC3")}, "mode": 4, "material": m}]})
    ta = w.accessor(np.zeros((1, 3), np.float32), "VEC3", sparse=(np.array([3], np.uint32), np.ones((1, 3), np.float32)), view=False)
    g.j["accessors"][ta]["count"] = count
    g.j["extensionsUsed"] = ["EXT_mesh_gpu_instancing"]
    g.node(mesh=0, extensions={"EXT_mesh_gpu_instancing": {"attributes": {"TRANSLATION": ta}}})
    g.node(mesh=1)
    return g.write(path)


# ---------------------------------------------------------------------------------------------------------------- upload bytes
def stored_bytes(n):
    """Stream bytes of the quantized C5-small form as the loader keeps them: int16 x3, int8 x3, u16 x2 per vertex, u16 indices."""
    return (n + 1) ** 2 * (6 + 3 + 4) + n * n * 6 * 2


def _check_upload_bytes(lib, d):
    kw = MG.C5_SMALL_KW
    q = gs.heightfield_forms(os.path.join(d, "c5s_q.glb"), "quantized", **kw)
    f = gs.heightfield_forms(os.path.join(d, "c5s_q_twin.glb"), "quantized", twin=True, **kw)
    with lib.load_scene(q):
        hq = lib.stats()["h2dBytes"]
    with lib.load_scene(f):
        hf = lib.stats()["h2dBytes"]
    assert hq <= 1.1 * stored_bytes(kw["n"]), (hq, stored_bytes(kw["n"]))
    assert hq < 0.6 * hf, (hq, hf)
    check_same_scene(lib, q, f, render=None)


def _check_c5_small_forms(lib, d):
    kw = MG.C5_SMALL_KW
    for form in ("quantized", "strips"):
        a = gs.heightfield_forms(os.path.join(d, "c5s_%s.glb" % form), form, **kw)
        b = gs.heightfield_forms(os.path.join(d, "c5s_%s_twin.glb" % form), form, twin=True, **kw)
        assert check_same_scene(lib, a, b, hits=Params(height=90, width_override=160)) == 10 * 2 * kw["n"] ** 2


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_strip_and_fan_corners_cpu(emu, tmp_path):
    _check_literals(emu, str(tmp_path))


def test_strips_fans_and_quantized_streams_equal_their_twins_cpu(emu, tmp_path):
    _check_form_twins(emu, str(tmp_path))


def test_sparse_accessors_cpu(emu, tmp_path):
    _check_sparse(emu, str(tmp_path))


def test_oversized_counts_are_refused_cpu(emu, tmp_path):
    _check_oversized(emu, str(tmp_path))


def test_quantized_streams_upload_as_stored_cpu(emu, tmp_path):
    _check_upload_bytes(emu, str(tmp_path))


def test_c5_small_forms_equal_their_twins_cpu(emu, tmp_path):
    _check_c5_small_forms(emu, str(tmp_path))


def test_multi_device_frame_of_strips_and_quantized_streams_cpu(emu, tmp_path):
    a = gs.forms_scene(os.path.join(str(tmp_path), "multi.glb"), mode=5, index_type=np.uint16, encoding="i16n", instances=3)
    assert pc.check_multi_device_frame(emu, a, devices=3, height=40) >= 1


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_strip_and_fan_corners_gpu(gpu, tmp_path):
    _check_literals(gpu, str(tmp_path))


@pytest.mark.gpu
def test_strips_fans_and_quantized_streams_equal_their_twins_gpu(gpu, tmp_path):
    _check_form_twins(gpu, str(tmp_path))


@pytest.mark.gpu
def test_sparse_accessors_gpu(gpu, tmp_path):
    _check_sparse(gpu, str(tmp_path))


@pytest.mark.gpu
def test_oversized_counts_are_refused_gpu(gpu, tmp_path):
    _check_oversized(gpu, str(tmp_path))


@pytest.mark.gpu
def test_quantized_streams_upload_as_stored_gpu(gpu, tmp_path):
    _check_upload_bytes(gpu, str(tmp_path))


@pytest.mark.gpu
def test_c5_small_forms_equal_their_twins_gpu(gpu, tmp_path):
    _check_c5_small_forms(gpu, str(tmp_path))


@pytest.mark.gpu
def test_multi_device_frame_of_strips_and_quantized_streams_gpu(gpu, tmp_path, monkeypatch):
    monkeypatch.setenv("SAILOR_PT_MULTI_SAME_DEVICE", "1")
    a = gs.forms_scene(os.path.join(str(tmp_path), "multi.glb"), mode=5, index_type=np.uint16, encoding="i16n", instances=3)
    assert pc.check_multi_device_frame(gpu, a, devices=3, height=40) == 3


@pytest.mark.gpu
def test_c5_row_strips_equal_their_float_list_twin_gpu(gpu, tmp_path):
    """Full-size C5 (9,996,980 triangles) as int16 / int8 / u16 row strips against its float-list twin."""
    d = str(tmp_path)
    a = gs.heightfield_forms(os.path.join(d, "c5_strips.glb"), "strips", **MG.C5_KW)
    b = gs.heightfield_forms(os.path.join(d, "c5_strips_twin.glb"), "strips", twin=True, **MG.C5_KW)
    render = dict(height=135, width_override=240, num_samples=2, num_ambient_samples=2, max_bounces=6, msaa=2, ambient=(1, 1, 1), seed=3)
    assert check_same_scene(gpu, a, b, hits=Params(height=1080, width_override=1920), render=render) == 9996980


@pytest.mark.gpu
def test_c5_float_lists_match_the_digests_gpu(gpu, scene_dir):
    D4 = json.load(open(os.path.join(HERE, "golden", "digests_c4c5.json")))
    with gpu.load_scene(gs.heightfield_forms(os.path.join(scene_dir, "c5_list.glb"), "list", **MG.C5_KW)) as s:
        assert s.counts()["triangles"] == D4["c5_counts"]["triangles"]
        nodes, mapping = s.bvh()
        dg = D4["c5_bvh"]
        assert len(nodes) == dg["nodes"] and pc.sha(mapping) == dg["mapping"]
        hits = s.primary_hits(Params(height=2160, width_override=3840))
        assert pc.sha(hits) == D4["c5_hits_4k"]["sha256"]
