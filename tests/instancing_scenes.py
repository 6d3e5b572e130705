"""Scenes for EXT_mesh_gpu_instancing (tests/test_instancing.py, tools/instancing_bench.py), written with tests/scenes.py's GLB writer.

* instanced_scene()    — a two-primitive grid mesh drawn K times by one node (form="ext") or the same scene written with one child
                        node per instance (form="nodes", the twin that needs no extension).
* c5_as_instancing_extension() — a scene (BASELINE C5) rewritten so that every mesh node carries its TRS as a one-instance extension.
* instancing_limit_scene(), broken_instancing_scene() — files the loader must refuse.
"""
import json
import math
import struct

import numpy as np

from scenes import GlbBuilder, _cube_arrays, _quad, lcg_uniform_fast, look_at_quat, quat_from_to_neg_z


def _raw_accessor(g, arr, typ, component_type, normalized=False):
    """Accessor of any component type (GlbBuilder.accessor writes only the unsigned and float ones)."""
    a = {"bufferView": g._view(np.ascontiguousarray(arr).tobytes()), "componentType": component_type, "count": int(arr.shape[0]), "type": typ}
    if normalized:
        a["normalized"] = True
    g.j["accessors"].append(a)
    return len(g.j["accessors"]) - 1


def _f32_list(v):
    """float32 values as JSON numbers that parse back to the same float32."""
    return [float(x) for x in np.asarray(v, np.float32)]


def instance_trs(instances, rotation="f32"):
    """TRS of K instances on a centred grid inside the unit square: (translation f32 [K,3], stored rotation [K,4], decoded rotation
    f32 [K,4], scale f32 [K,3]).  rotation: "f32", or "i8" / "i16" normalized integers (KHR_mesh_quantization), decoded the way glTF
    says: max(v / 127, -1) and max(v / 32767, -1) in float32."""
    k = np.arange(instances)
    cols = int(math.ceil(math.sqrt(instances)))
    rows = (instances + cols - 1) // cols
    sp = 1.0 / cols
    cx, cz = k % cols, k // cols
    t = np.stack([(cx - (cols - 1) / 2) * sp, 0.004 * (k % 5), (cz - (rows - 1) / 2) * sp], -1).astype(np.float32)
    axis = np.array([0.1, 1.0, 0.05]) / np.linalg.norm([0.1, 1.0, 0.05])
    ang = 0.35 * k
    q = np.concatenate([np.sin(ang / 2)[:, None] * axis[None, :], np.cos(ang / 2)[:, None]], -1)
    s = np.stack([0.95 * sp * (1 + 0.1 * (k % 3)), 1.0 + 0.2 * (k % 3), 0.95 * sp * (1 + 0.05 * (k % 2))], -1).astype(np.float32)
    if rotation == "f32":
        stored = q.astype(np.float32)
        dec = stored
    else:
        lim = {"i8": 127, "i16": 32767}[rotation]
        stored = np.round(q * lim).astype(np.int8 if rotation == "i8" else np.int16)
        dec = np.maximum(stored.astype(np.float32) / np.float32(lim), np.float32(-1.0))
    return t, stored, dec, s


def _grid_mesh_streams(nx, nz, seed):
    nvx, nvz = nx + 1, nz + 1
    u = lcg_uniform_fast(nvx * nvz, seed)
    jj, ii = np.meshgrid(np.arange(nvz), np.arange(nvx), indexing="ij")
    pos = np.stack([-0.5 + ii / nx, 0.05 * u.reshape(nvz, nvx), -0.5 + jj / nz], axis=-1).reshape(-1, 3).astype(np.float32)
    q = (jj[:-1, :-1] * nvx + ii[:-1, :-1]).reshape(-1)
    idx = np.stack([q, q + nvx, q + 1, q + 1, q + nvx, q + nvx + 1], axis=-1).reshape(-1).astype(np.uint32)
    return pos, idx


def instanced_scene(path, form="ext", rotation="f32", nx=8, nz=8, instances=7, attributes=("TRANSLATION", "ROTATION", "SCALE"), seed=3):
    """One (nx x nz)-quad grid mesh with TWO primitives (the first half of its rows and the rest, two materials), drawn once per
    instance by a node below a parent with its own TRS; the instancing node has a child (a quad) and the scene a camera and a
    directional light.  form="ext": EXT_mesh_gpu_instancing with the listed attributes (a missing one is the identity) plus an
    application-specific "_ID" attribute that readers ignore; form="nodes": the twin, one child node per instance carrying the
    decoded TRS, inserted before the quad child.  Flattened, both are the same 2 * nx * nz * instances + 2 triangles."""
    assert form in ("ext", "nodes")
    g = GlbBuilder()
    pos, idx = _grid_mesh_streams(nx, nz, seed)
    half = (nz // 2) * nx * 6
    m0 = g.material(pbrMetallicRoughness={"baseColorFactor": [0.75, 0.55, 0.3, 1.0], "metallicFactor": 0.0, "roughnessFactor": 0.8})
    m1 = g.material(pbrMetallicRoughness={"baseColorFactor": [0.3, 0.6, 0.8, 1.0], "metallicFactor": 0.5, "roughnessFactor": 0.3})
    pa = g.accessor(pos, "VEC3", 34962, True)
    prims = [{"attributes": {"POSITION": pa}, "mode": 4, "material": m, "indices": g.accessor(part, "SCALAR", 34963)}
             for m, part in ((m0, idx[:half]), (m1, idx[half:]))]
    g.j["meshes"].append({"primitives": prims})
    mesh = len(g.j["meshes"]) - 1
    p, n, uv, i = _quad((0, 0, 0), (0.05, 0, 0), (0, 0.05, 0))
    quad = g.mesh(p, i, m1, nrm=n, uv=uv)
    t, stored, dec, s = instance_trs(instances, rotation)
    child = g.node(root=False, mesh=quad, translation=[0.0, 0.12, 0.0])
    if form == "ext":
        acc = {}
        if "TRANSLATION" in attributes:
            acc["TRANSLATION"] = g.accessor(t, "VEC3")
        if "ROTATION" in attributes:
            ct = {"f32": 5126, "i8": 5120, "i16": 5122}[rotation]
            acc["ROTATION"] = _raw_accessor(g, stored, "VEC4", ct, normalized=rotation != "f32")
        if "SCALE" in attributes:
            acc["SCALE"] = g.accessor(s, "VEC3")
        acc["_ID"] = g.accessor(np.arange(instances, dtype=np.float32), "SCALAR")
        g.j["extensionsUsed"] = ["EXT_mesh_gpu_instancing"]
        inst = g.node(root=False, mesh=mesh, children=[child], rotation=_f32_list([0.0, 0.0998334, 0.0, 0.9950042]),
                      extensions={"EXT_mesh_gpu_instancing": {"attributes": acc}})
    else:
        kids = []
        for k in range(instances):
            kw = {}
            if "TRANSLATION" in attributes:
                kw["translation"] = _f32_list(t[k])
            if "ROTATION" in attributes:
                kw["rotation"] = _f32_list(dec[k])
            if "SCALE" in attributes:
                kw["scale"] = _f32_list(s[k])
            kids.append(g.node(root=False, mesh=mesh, **kw))
        inst = g.node(root=False, children=kids + [child], rotation=_f32_list([0.0, 0.0998334, 0.0, 0.9950042]))
    g.node(children=[inst], translation=[0.05, -0.02, 0.1], rotation=_f32_list([0.0499792, 0.0, 0.0, 0.9987503]), scale=[1.1, 0.9, 1.1])
    g.j["cameras"] = [{"type": "perspective", "perspective": {"yfov": 0.8, "aspectRatio": 16.0 / 9.0, "znear": 0.01, "zfar": 100.0}}]
    g.node(camera=0, name="main", translation=[0.0, 0.8, 1.1], rotation=look_at_quat((0.0, -0.6, -0.9)))
    g.j.setdefault("extensionsUsed", []).append("KHR_lights_punctual")
    g.j["extensions"] = {"KHR_lights_punctual": {"lights": [{"type": "directional", "color": [1.0, 1.0, 1.0], "intensity": 2049.0}]}}
    g.node(name="sun", rotation=quat_from_to_neg_z((0.3, -1.0, 0.2)), extensions={"KHR_lights_punctual": {"light": 0}})
    return g.write(path)


def read_glb(path):
    """(json dict, BIN chunk bytes) of a GLB written by GlbBuilder."""
    with open(path, "rb") as f:
        data = f.read()
    jlen = struct.unpack_from("<I", data, 12)[0]
    j = json.loads(data[20:20 + jlen])
    blen = struct.unpack_from("<I", data, 20 + jlen)[0]
    return j, bytes(data[28 + jlen:28 + jlen + blen])


def c5_as_instancing_extension(src, path):
    """The scene at `src` with every mesh node's translation / rotation / scale moved into a one-instance EXT_mesh_gpu_instancing
    (float32 accessors holding the values the node's JSON numbers parse to); the nodes keep the identity transform."""
    j, b = read_glb(src)
    g = GlbBuilder()
    g.j = j
    g.bin = bytearray(b)
    for node in j["nodes"]:
        if "mesh" not in node:
            continue
        acc = {}
        for key, attr, typ, identity in (("translation", "TRANSLATION", "VEC3", [0, 0, 0]), ("rotation", "ROTATION", "VEC4", [0, 0, 0, 1]),
                                         ("scale", "SCALE", "VEC3", [1, 1, 1])):
            acc[attr] = g.accessor(np.asarray([node.pop(key, identity)], np.float32), typ)
        node.setdefault("extensions", {})["EXT_mesh_gpu_instancing"] = {"attributes": acc}
    j.setdefault("extensionsUsed", []).append("EXT_mesh_gpu_instancing")
    return g.write(path)


def instancing_limit_scene(path, faces=65536, instances=65536):
    """A file of about 1 MB that asks for faces * instances triangles (2^32 by default): a mesh of `faces` copies of one triangle
    (uint16 indices), instanced by a TRANSLATION accessor of `instances` entries."""
    g = GlbBuilder()
    m = g.material(pbrMetallicRoughness={"baseColorFactor": [0.5, 0.5, 0.5, 1.0]})
    pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    mesh = g.mesh(pos, np.tile(np.array([0, 1, 2], np.uint16), faces), m)
    t = np.zeros((instances, 3), np.float32)
    g.node(mesh=mesh, extensions={"EXT_mesh_gpu_instancing": {"attributes": {"TRANSLATION": g.accessor(t, "VEC3")}}})
    return g.write(path)


def broken_instancing_scene(path, kind):
    """Malformed EXT_mesh_gpu_instancing objects: "missing_accessor" (TRANSLATION names no accessor), "vec2_translation",
    "unequal_counts" (3 translations, 2 scales) and "no_attributes"."""
    g = GlbBuilder()
    m = g.material(pbrMetallicRoughness={"baseColorFactor": [0.5, 0.5, 0.5, 1.0]})
    pos, nrm, idx = _cube_arrays(0.3)
    mesh = g.mesh(pos, idx, m, nrm=nrm)
    if kind == "missing_accessor":
        attrs = {"TRANSLATION": 999}
    elif kind == "vec2_translation":
        attrs = {"TRANSLATION": g.accessor(np.zeros((3, 2), np.float32), "VEC2")}
    elif kind == "unequal_counts":
        attrs = {"TRANSLATION": g.accessor(np.zeros((3, 3), np.float32), "VEC3"), "SCALE": g.accessor(np.ones((2, 3), np.float32), "VEC3")}
    elif kind == "no_attributes":
        attrs = {"_ID": g.accessor(np.zeros(3, np.float32), "SCALAR")}
    else:
        raise KeyError(kind)
    g.node(mesh=mesh)
    g.node(mesh=mesh, name="broken", extensions={"EXT_mesh_gpu_instancing": {"attributes": attrs}})
    return g.write(path)
