"""Scenes for glTF primitive assembly and stream decoding (tests/test_geometry_forms.py, tools/geometry_bench.py), written with
tests/scenes.py's GLB writer.

Each generator writes a file and, with twin=True, its twin: the same triangles stated as a float32 TRIANGLES list with u32 indices
(strips and fans expanded by glTF 2.0 section 3.7.2.1, quantized streams decoded as the specification says, sparse accessors applied).
A file and its twin flatten, build, trace and render to the same bits.
"""
import math

import numpy as np

from scenes import GlbBuilder, lcg_uniform_fast, look_at_quat, quat_from_to_neg_z

CT = {np.dtype("float32"): 5126, np.dtype("uint32"): 5125, np.dtype("uint16"): 5123, np.dtype("uint8"): 5121,
      np.dtype("int16"): 5122, np.dtype("int8"): 5120}


def decode(stored, normalized):
    """float32 values of a stored attribute, as the glTF specification (and KHR_mesh_quantization) decodes them."""
    v = np.asarray(stored)
    f = v.astype(np.float32)
    if not normalized or v.dtype == np.float32:
        return f
    lim = {np.dtype("uint8"): 255, np.dtype("uint16"): 65535, np.dtype("int8"): 127, np.dtype("int16"): 32767}[v.dtype]
    f = f / np.float32(lim)
    return np.maximum(f, np.float32(-1.0)) if v.dtype.kind == "i" else f


def corners(mode, n):
    """Vertex slots of every face of a primitive with n indices (or n vertices without indices): [faces, 3]."""
    if mode == 4:
        return np.arange(n // 3 * 3, dtype=np.int64).reshape(-1, 3)
    i = np.arange(max(n - 2, 0), dtype=np.int64)
    if mode == 5:
        return np.stack([i, i + 1 + i % 2, i + 2 - i % 2], -1)
    return np.stack([i + 1, i + 2, np.zeros_like(i)], -1)


def expand(mode, indices, num_verts):
    """The u32 TRIANGLES list of a primitive (out-of-range indices read vertex 0)."""
    n = num_verts if indices is None else len(indices)
    c = corners(mode, n)
    v = c if indices is None else np.asarray(indices, np.int64)[c]
    v = np.where(v < num_verts, v, 0)
    return v.reshape(-1).astype(np.uint32)


class Writer:
    """GlbBuilder with accessors of any component type, padded or interleaved views and sparse blocks."""

    def __init__(self):
        self.g = GlbBuilder()

    def view(self, data, stride=None):
        v = self.g._view(bytes(data))
        if stride:
            self.g.j["bufferViews"][v]["byteStride"] = stride
        return v

    def accessor(self, arr, typ, normalized=False, stride=None, sparse=None, view=True):
        """arr [count, comps] (or [count]); stride: pad every element to that many bytes; sparse: (indices, values) to substitute;
        view=False: no bufferView (the base is zeros, sparse is required)."""
        arr = np.ascontiguousarray(arr)
        count = arr.shape[0]
        a = {"componentType": CT[arr.dtype], "count": int(count), "type": typ}
        if view:
            raw = arr.reshape(count, -1).view(np.uint8)
            if stride:
                pad = np.zeros((count, stride), np.uint8)
                pad[:, :raw.shape[1]] = raw
                raw = pad
            a["bufferView"] = self.view(raw.tobytes(), stride)
        if normalized:
            a["normalized"] = True
        if sparse is not None:
            idx, val = sparse
            idx, val = np.ascontiguousarray(idx), np.ascontiguousarray(val, arr.dtype)
            a["sparse"] = {"count": int(len(idx)), "indices": {"bufferView": self.view(idx.tobytes()), "componentType": CT[idx.dtype]},
                           "values": {"bufferView": self.view(val.tobytes())}}
        self.g.j["accessors"].append(a)
        return len(self.g.j["accessors"]) - 1

    def interleaved(self, arrays, typs, normalized):
        """One bufferView holding every array's element i side by side, each padded to 4 bytes: one accessor per array."""
        count = arrays[0].shape[0]
        parts = [np.ascontiguousarray(a).reshape(count, -1).view(np.uint8) for a in arrays]
        widths = [(p.shape[1] + 3) // 4 * 4 for p in parts]
        stride = sum(widths)
        buf = np.zeros((count, stride), np.uint8)
        off = 0
        for p, w in zip(parts, widths):
            buf[:, off:off + p.shape[1]] = p
            off += w
        v = self.view(buf.tobytes(), stride)
        out, off = [], 0
        for a, t, n, w in zip(arrays, typs, normalized, widths):
            acc = {"bufferView": v, "byteOffset": off, "componentType": CT[a.dtype], "count": int(count), "type": t}
            if n:
                acc["normalized"] = True
            self.g.j["accessors"].append(acc)
            out.append(len(self.g.j["accessors"]) - 1)
            off += w
        return out


def _material(g, k):
    return g.material(pbrMetallicRoughness={"baseColorFactor": [0.4 + 0.1 * k, 0.7 - 0.1 * k, 0.5, 1.0], "metallicFactor": 0.2 * k, "roughnessFactor": 0.6})


def _camera_and_sun(g, eye=(0.0, 1.1, 1.6), forward=(0.0, -0.5, -0.9)):
    g.j["cameras"] = [{"type": "perspective", "perspective": {"yfov": 0.8, "aspectRatio": 16.0 / 9.0, "znear": 0.01, "zfar": 100.0}}]
    g.node(camera=0, name="main", translation=list(eye), rotation=look_at_quat(forward))
    g.j.setdefault("extensionsUsed", []).append("KHR_lights_punctual")
    g.j["extensions"] = {"KHR_lights_punctual": {"lights": [{"type": "directional", "color": [1.0, 1.0, 1.0], "intensity": 2049.0}]}}
    g.node(name="sun", rotation=quat_from_to_neg_z((0.3, -1.0, 0.2)), extensions={"KHR_lights_punctual": {"light": 0}})


# ------------------------------------------------------------------------------------------------------------ grid meshes
def grid(n, seed=2, extent=1.0):
    """The vertices of an n x n heightfield grid (BASELINE C5's, by default): float32 positions [(n+1)^2, 3], normals, uvs."""
    nv = n + 1
    u = lcg_uniform_fast(nv * nv, seed)
    jj, ii = np.meshgrid(np.arange(nv), np.arange(nv), indexing="ij")
    pos = np.stack([(-0.5 + ii / n) * extent, 0.05 * u.reshape(nv, nv), (-0.5 + jj / n) * extent], axis=-1).reshape(-1, 3).astype(np.float32)
    h = u.reshape(nv, nv)
    gx, gz = np.gradient(0.05 * h * n)
    nrm = np.stack([-gz, np.ones_like(gx), -gx], -1).reshape(-1, 3)
    nrm = (nrm / np.linalg.norm(nrm, axis=-1, keepdims=True)).astype(np.float32)
    uv = np.stack([ii / n, jj / n], -1).reshape(-1, 2).astype(np.float32)
    return pos, nrm, uv


def grid_list(n):
    nv = n + 1
    jj, ii = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    q = (jj * nv + ii).reshape(-1)
    return np.stack([q, q + nv, q + 1, q + 1, q + nv, q + nv + 1], axis=-1).reshape(-1).astype(np.uint32)


def grid_row_strip(n, row):
    """Strip indices of one row of quads: a_0 b_0 a_1 b_1 ... (a on row `row`, b on the next); faces (a_i, b_i, a_i+1), (b_i, b_i+1, a_i+1)."""
    nv = n + 1
    a = row * nv + np.arange(nv)
    return np.stack([a, a + nv], -1).reshape(-1).astype(np.uint32)


def quantize(values, dtype):
    """(stored values, decoded float32) of values in [-1, 1] (signed) or [0, 1] (unsigned) as normalized integers."""
    info = np.iinfo(dtype)
    q = np.clip(np.round(values * info.max), info.min, info.max).astype(dtype)
    return q, decode(q, True)


def heightfield_forms(path, form, n=48, instances=10, twin=False, seed=2):
    """BASELINE C5's layout (an n x n grid mesh drawn by `instances` nodes through 4 meshes that share its accessors) in one of the
    forms a glTF exporter writes:
      "list"       float32 positions, u32 / u16 TRIANGLES list: tests/scenes.py instanced_heightfield itself (twin: the same file);
      "quantized"  int16 normalized positions under a dequantizing child node, int8 normalized normals (VEC3 padded to 4 bytes), u16
                   normalized UVs, the index list as GlbBuilder stores it (u16 below 65,536 vertices, else u32);
      "strips"     the quantized streams drawn as one unindexed TRIANGLE_STRIP per row of quads (each row's vertices in strip order).
    twin=True writes the float32 / u32-list twin of that form."""
    assert form in ("list", "quantized", "strips")
    if form == "list":
        import scenes
        return scenes.instanced_heightfield(path, n=n, instances=instances, seed=seed)
    pos, nrm, uv = grid(n, seed)
    scale = np.float32(0.5)                     # positions within [-0.5, 0.5] x [0, 0.05]: int16 of pos / scale, the node scales back
    qpos, dpos = quantize(pos / scale, np.int16)
    qnrm, dnrm = quantize(nrm, np.int8)
    quv, duv = quantize(uv, np.uint16)
    if form == "quantized":
        prims = [(4, grid_list(n), None)]
    else:                                       # each row's vertices gathered in strip order, no indices
        prims = [(5, None, grid_row_strip(n, r)) for r in range(n)]
    w = Writer()
    g = w.g
    mats = [_material(g, k) for k in range(min(instances, 4))]

    def attrs_of(sel):
        if twin:
            return {"POSITION": w.accessor(dpos[sel], "VEC3"), "NORMAL": w.accessor(dnrm[sel], "VEC3"), "TEXCOORD_0": w.accessor(duv[sel], "VEC2")}
        return {"POSITION": w.accessor(qpos[sel], "VEC3", True, stride=8), "NORMAL": w.accessor(qnrm[sel], "VEC3", True, stride=4),
                "TEXCOORD_0": w.accessor(quv[sel], "VEC2", True)}

    primitives = []
    for mode, idx, sel in prims:
        if sel is None:
            sel = np.arange(len(pos))
        a = attrs_of(sel)
        nverts = len(sel)
        if twin:
            lst = expand(mode, idx, nverts)
            primitives.append({"attributes": a, "mode": 4, "indices": w.accessor(lst, "SCALAR")})
        elif idx is not None:
            primitives.append({"attributes": a, "mode": mode, "indices": w.accessor(idx if idx.max() >= 65536 else idx.astype(np.uint16), "SCALAR")})
        else:
            primitives.append({"attributes": a, "mode": mode})
    meshes = []
    for m in mats:
        g.j["meshes"].append({"primitives": [dict(p, material=m) for p in primitives]})
        meshes.append(len(g.j["meshes"]) - 1)
    cols = int(math.ceil(math.sqrt(instances)))
    for k in range(instances):
        cx, cz = k % cols, k // cols
        ang = 0.35 * k
        child = g.node(root=False, mesh=meshes[k % len(meshes)], scale=[float(scale)] * 3)
        g.node(children=[child], translation=[(cx - (cols - 1) / 2) * 0.98, 0.01 * k, -(cz * 0.98)],
               rotation=[0.0, math.sin(ang / 2), 0.0, math.cos(ang / 2)], scale=[1.0, 1.0 + 0.2 * (k % 3), 1.0])
    _camera_and_sun(g)
    return g.write(path)


# ------------------------------------------------------------------------------------------------------------ small cases
def literal_scene(path, mode, index_type=None, n=5, extra_primitive=False):
    """One primitive of n vertices at (k, k % 2, 0.1 k): TRIANGLE_STRIP / FAN / list, with u8 / u16 / u32 identity indices or none.
    extra_primitive: a second primitive (one list triangle) so that the file has triangles when the first has none."""
    w = Writer()
    g = w.g
    m = _material(g, 0)
    k = np.arange(n)
    pos = np.stack([k, k % 2, 0.1 * k], -1).astype(np.float32)
    prim = {"attributes": {"POSITION": w.accessor(pos, "VEC3")}, "mode": mode, "material": m}
    if index_type is not None:
        prim["indices"] = w.accessor(k.astype(index_type), "SCALAR")
    prims = [prim]
    if extra_primitive:
        prims.append({"attributes": {"POSITION": w.accessor(np.array([[0, 0, 5], [1, 0, 5], [0, 1, 5]], np.float32), "VEC3")}, "material": m})
    g.j["meshes"].append({"primitives": prims})
    g.node(mesh=0)
    return g.write(path)


def _mesh_streams(nx=6, nz=5, seed=4):
    pos, nrm, uv = grid(max(nx, nz), seed)
    nv = max(nx, nz) + 1
    sel = np.array([j * nv + i for j in range(nz + 1) for i in range(nx + 1)])
    pos, nrm, uv = pos[sel], nrm[sel], uv[sel]
    tan = np.concatenate([np.tile([[1.0, 0.0, 0.0]], (len(pos), 1)), np.where(np.arange(len(pos))[:, None] % 3 == 0, -1.0, 1.0)], -1).astype(np.float32)
    uv1 = (uv * np.float32(0.5) + np.float32(0.25)).astype(np.float32)
    return pos, nrm, uv, uv1, tan


def _strip_indices(nx, nz):
    """One strip over all rows, rows joined by two repeated indices (degenerate faces, kept as in a list)."""
    out = []
    for r in range(nz):
        a = r * (nx + 1) + np.arange(nx + 1)
        row = np.stack([a, a + nx + 1], -1).reshape(-1)
        if out:
            out += [out[-1], row[0]]
        out += list(row)
    return np.array(out, np.int64)


def _fan_indices(nx, nz):
    """A fan around the centre vertex over the boundary loop of the grid, with one index out of range."""
    c = (nz // 2) * (nx + 1) + nx // 2
    ring = [i for i in range(nx + 1)] + [j * (nx + 1) + nx for j in range(1, nz + 1)] + [nz * (nx + 1) + i for i in range(nx - 1, -1, -1)] \
        + [j * (nx + 1) for j in range(nz - 1, 0, -1)]
    return np.array([c] + ring + [ring[0], 250], np.int64)


ENCODINGS = {
    # name: {stream: (dtype, normalized, stride)}; positions under a node scale when not float
    "f32": {},
    "i16n": {"POSITION": (np.int16, True, 8), "NORMAL": (np.int16, True, 8), "TEXCOORD_0": (np.int16, True, None), "TANGENT": (np.int8, True, None)},
    "i8n": {"POSITION": (np.int8, True, 4), "NORMAL": (np.int8, True, 4), "TEXCOORD_0": (np.int8, True, None), "TEXCOORD_1": (np.uint8, True, None), "TANGENT": (np.int8, True, None)},
    "u16n": {"POSITION": (np.uint16, True, 8), "TEXCOORD_0": (np.uint16, True, None), "TEXCOORD_1": (np.uint16, True, None)},
    "u8n": {"POSITION": (np.uint8, True, 4), "TEXCOORD_0": (np.uint8, True, None)},
    "i16": {"POSITION": (np.int16, False, 8), "TEXCOORD_0": (np.int16, False, None)},
    "u8": {"POSITION": (np.uint8, False, 4), "TEXCOORD_1": (np.uint8, False, None)},
    "u16": {"POSITION": (np.uint16, False, 8), "NORMAL": (np.int8, False, 4)},
    "interleaved": "interleaved",
}


def position_node(dtype, normalized):
    """The node transform that turns stored positions back into the mesh's (as gltfpack writes it), and the inverse for encoding."""
    unsigned = np.iinfo(dtype).min == 0
    scale = 0.5 if normalized and not unsigned else (1.0 if normalized else 1.0 / 64)
    offset = -0.5 if unsigned else 0.0
    kw = {"scale": [scale] * 3}
    if offset:
        kw["translation"] = [offset] * 3
    return kw, (lambda p: (p - np.float32(offset)) / np.float32(scale))


def _encode(w, name, values, typ, enc, twin):
    """(accessor, decoded float32 values) of one stream in encoding `enc` of ENCODINGS."""
    spec = enc.get(name)
    if spec is None:
        return w.accessor(values, typ), values
    dtype, normalized, stride = spec
    info = np.iinfo(dtype)
    if name == "POSITION":
        values = position_node(dtype, normalized)[1](values)
    elif info.min == 0:
        values = np.abs(values)
    q = np.round(values * (info.max if normalized else 1)).clip(info.min, info.max).astype(dtype)
    if info.min < 0 and name != "POSITION":
        q.reshape(len(q), -1)[::7, 0] = info.min          # -128 / -32768: decodes to -1 through the clamp when normalized
    d = decode(q, normalized)
    if twin:
        return w.accessor(d, typ), d
    return w.accessor(q, typ, normalized, stride=stride), d


def forms_scene(path, mode, index_type, encoding="f32", twin=False, nx=6, nz=5, shared_list=False, instances=0, seed=4):
    """A small grid mesh as a strip (mode 5), a fan (6) or a list (4); index_type None (unindexed: the vertices gathered in primitive
    order), uint8 / uint16 / uint32.  encoding: a key of ENCODINGS.  shared_list: a second primitive, a list, reading the same
    accessors (both draw).  instances > 0: the mesh drawn by EXT_mesh_gpu_instancing (twin: one child node per instance)."""
    w = Writer()
    g = w.g
    m0, m1 = _material(g, 0), _material(g, 1)
    pos, nrm, uv, uv1, tan = _mesh_streams(nx, nz, seed)
    idx = {5: _strip_indices(nx, nz), 6: _fan_indices(nx, nz), 4: grid_list(max(nx, nz))[:0]}[mode]
    if mode == 4:
        nv = nx + 1
        jj, ii = np.meshgrid(np.arange(nz), np.arange(nx), indexing="ij")
        q = (jj * nv + ii).reshape(-1)
        idx = np.stack([q, q + nv, q + 1, q + 1, q + nv, q + nv + 1], -1).reshape(-1)
        idx = np.concatenate([idx, [0, 1]])                     # a trailing partial triangle: dropped
    if index_type is None:                                      # unindexed: gather the vertices in primitive order
        sel = np.where(idx < len(pos), idx, 0)
        pos, nrm, uv, uv1, tan = pos[sel], nrm[sel], uv[sel], uv1[sel], tan[sel]
    streams = {"POSITION": (pos, "VEC3"), "NORMAL": (nrm, "VEC3"), "TEXCOORD_0": (uv, "VEC2"), "TEXCOORD_1": (uv1, "VEC2"), "TANGENT": (tan, "VEC4")}
    attrs, dec = {}, {}
    if encoding == "interleaved":
        if twin:
            for k, (v, t) in streams.items():
                attrs[k] = w.accessor(v, t)
        else:
            names = list(streams)
            accs = w.interleaved([streams[k][0] for k in names], [streams[k][1] for k in names], [False] * len(names))
            attrs = dict(zip(names, accs))
    else:
        for k, (v, t) in streams.items():
            attrs[k], dec[k] = _encode(w, k, v, t, ENCODINGS[encoding], twin)
    nverts = len(pos)
    if twin:
        lst = expand(mode, None if index_type is None else idx, nverts)
        prim = {"attributes": attrs, "mode": 4, "indices": w.accessor(lst, "SCALAR"), "material": m0}
        prims = [prim]
        if shared_list:
            prims.append({"attributes": attrs, "mode": 4, "indices": w.accessor(expand(4, None if index_type is None else idx, nverts), "SCALAR"), "material": m1})
    else:
        prim = {"attributes": attrs, "mode": mode, "material": m0}
        if index_type is not None:
            prim["indices"] = w.accessor(idx.astype(index_type), "SCALAR")
        prims = [prim]
        if shared_list:
            prims.append(dict(prim, mode=4, material=m1))
    g.j["meshes"].append({"primitives": prims})
    pspec = ENCODINGS[encoding].get("POSITION") if encoding != "interleaved" else None
    node_kw = position_node(pspec[0], pspec[1])[0] if pspec else {}
    if instances:
        t = np.stack([np.arange(instances) * 1.1 - 0.5 * instances, np.zeros(instances), 0.2 * (np.arange(instances) % 2)], -1).astype(np.float32)
        if twin:
            inst = g.node(root=False, children=[g.node(root=False, mesh=0, translation=[float(x) for x in t[k]]) for k in range(instances)], **node_kw)
        else:
            g.j["extensionsUsed"] = ["EXT_mesh_gpu_instancing"]
            inst = g.node(root=False, mesh=0, extensions={"EXT_mesh_gpu_instancing": {"attributes": {"TRANSLATION": w.accessor(t, "VEC3")}}}, **node_kw)
        g.node(children=[inst], scale=[0.3, 0.3, 0.3])
    else:
        g.node(mesh=0, **node_kw)
    _camera_and_sun(g, eye=(0.0, 0.9, 1.4), forward=(0.0, -0.6, -0.9))
    return g.write(path)
