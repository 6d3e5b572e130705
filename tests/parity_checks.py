"""Parity checks shared by the CPU-side tests (kernel bodies compiled for the host, tests/emu) and the GPU tests
(the product library through its C-ABI).  `lib` is the library under test, `oracle` the reference build, `G` the
golden vectors minted from the oracle by tests/golden/make_golden.py.

Bars: bit-exact for flattened triangles, BVH topology / leaf order, hit triangle ids, hit distance and barycentrics,
texel fetch + bilinear blend, and the 8-bit output; relative
1e-4 for the BSDF function table (libm transcendentals differ in the last ulps); a stated mean relative error for
converged images.
"""
import hashlib
import os

import numpy as np

from sailor_b200.capi import Params

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))

NOHIT = 0xFFFFFFFF


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_hits_equal(a, b):
    assert a.shape == b.shape
    assert np.array_equal(a["triId"], b["triId"]), "hit triangle ids differ at %d rays" % int((a["triId"] != b["triId"]).sum())
    for k in ("t", "baryU", "baryV"):
        assert np.array_equal(bits(a[k]), bits(b[k])), "%s differs (bitwise) at %d rays" % (k, int((bits(a[k]) != bits(b[k])).sum()))


def check_flatten(lib, path, tris_ref, mat_ref):
    with lib.load_scene(path) as s:
        tris, mat = s.triangles()
    assert tris.shape == tris_ref.shape
    assert np.array_equal(bits(tris), bits(tris_ref)), "flattened triangles differ"
    assert np.array_equal(mat, mat_ref)


def check_bvh(lib, path, nodes_ref, mapping_ref):
    with lib.load_scene(path) as s:
        nodes, mapping = s.bvh()
    assert len(nodes) == len(nodes_ref), "node count %d vs %d" % (len(nodes), len(nodes_ref))
    assert np.array_equal(nodes["leftFirst"], nodes_ref["leftFirst"])
    assert np.array_equal(nodes["triCount"], nodes_ref["triCount"])
    assert np.array_equal(mapping, mapping_ref), "m_triIdxMapping differs"
    assert np.array_equal(nodes["aabbMin"], nodes_ref["aabbMin"]) and np.array_equal(nodes["aabbMax"], nodes_ref["aabbMax"])


def check_primary_hits(lib, path, height, width_override, camera, cam_ref, hits_ref):
    with lib.load_scene(path) as s:
        p = Params(height=height, width_override=width_override, camera=camera)
        w, h, cam = s.camera(p)
        hits = s.primary_hits(p)
    assert np.array_equal(bits(cam), bits(cam_ref)), "camera vectors differ"
    assert_hits_equal(hits, hits_ref)


def random_rays(n, seed, scale=1.5):
    r = np.random.RandomState(seed)
    o = r.uniform(-scale, scale, (n, 3)).astype(np.float32)
    d = r.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True).astype(np.float32)
    # edge cases the reference's slab test is sensitive to: axis-aligned directions (1/0 = inf, 0*inf = NaN), rays
    # starting exactly on box planes / vertices, un-normalised and zero directions
    k = n // 8
    d[:k] = 0; d[np.arange(k), r.randint(0, 3, k)] = r.choice([-1.0, 1.0], k)
    o[:k // 2] = np.round(o[:k // 2] * 2) / 2
    d[k:k + 8] *= 1e-3
    d[k + 8:k + 12] = 0.0
    d[k + 12:k + 16, 1] = -0.0
    return o, d


def surface_rays(tris, n, seed, far_corner=False):
    """Rays as the integrator emits them: origins ON random triangles (offset 1e-6 along the face normal, like
    PathTracer.cpp:667), random directions, the origin's triangle as `ignore`.  tris: (N, 51) flattened triangles."""
    r = np.random.RandomState(seed)
    k = r.randint(0, len(tris), n)
    v = tris[k, 3:12].reshape(n, 3, 3).astype(np.float64)
    b = r.dirichlet((1.0, 1.0, 1.0), n)
    p = (v * b[:, :, None]).sum(axis=1)
    fn = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])
    fn /= np.maximum(np.linalg.norm(fn, axis=1, keepdims=True), 1e-30)
    d = r.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = p + 1e-6 * fn * np.where(r.uniform(size=(n, 1)) < 0.5, -1.0, 1.0)
    # rays aimed exactly at the far corner (+M, -M, +M) that stands in for the missing second level of the root's climb nodes
    # (trace_fast.cuh, FastClimbKernel): an unnormalised (1, -1, 1) "hits" that point box and walks the tree once more from the root
    if far_corner and n >= 64:
        d[-16:-8] = (1.0, -1.0, 1.0)
        d[-8:] = np.array((1.0, -1.0, 1.0)) / np.sqrt(3.0)
    return o.astype(np.float32), d.astype(np.float32), k.astype(np.uint32)


def check_random_rays(lib, oracle, path, n=20000, seed=1, far_corner=False):
    """BVH::IntersectBVH on random, degenerate and secondary-ray shaped queries: the exact kernel, and the two traversal variants
    the integrator uses for secondary rays (origin-local walk, wide layout) with their exact replay of ambiguous rays -- all bit
    for bit the oracle's closest hit; hit-or-miss queries give the same boolean."""
    o, d = random_rays(n, seed)
    replayed = {}
    with lib.load_scene(path) as a, oracle.load_scene(path) as b:
        nt = a.counts()["triangles"]
        ignore = np.random.RandomState(seed + 1).randint(0, nt, n).astype(np.uint32)
        so, sd, sk = surface_rays(b.triangles()[0], n, seed + 2, far_corner)
        cases = [("surface", so, sd, sk, b.intersect_rays(so, sd, sk)), ("random", o, d, None, b.intersect_rays(o, d)), ("random+ignore", o, d, ignore, b.intersect_rays(o, d, ignore))]
        for tag, ro, rd, ig, ref in cases:
            assert_hits_equal(a.intersect_rays(ro, rd, ig), ref)
            for mode in ("local", "wide"):      # origin-local walk, wide layout
                kw = {mode: True}
                assert_hits_equal(a.intersect_rays(ro, rd, ig, **kw), ref)
                replayed[(tag, mode)] = lib.stats()["replayedRays"]
                any_hits = a.intersect_rays(ro, rd, ig, any_hit=True, **kw)
                got = any_hits["triId"] != NOHIT
                assert np.array_equal(got, ref["triId"] != NOHIT), "%s/%s: hit-or-miss differs at %d rays" % (tag, mode, int((got != (ref["triId"] != NOHIT)).sum()))
                # a reachable hit, so not nearer than the closest one -- except by rounding: among (nearly) coplanar triangles the reference's
                # shrinking ray length can cull the truly nearest one (those are the rays a closest-hit query replays exactly)
                assert np.all(any_hits["t"][got] >= ref["t"][got] * np.float32(1.0 - 2.0 ** -15) - np.float32(1e-6)), "%s/%s: a hit-or-miss query reported a hit nearer than the closest hit" % (tag, mode)
    return replayed


def check_default_material(lib, oracle, path, own_materials):
    """A primitive without a material (or with an index outside the array) uses the glTF default material, appended after the
    file's own (ADVICE r1: such a file used to fault the device).  Product and oracle import identically and the frame renders."""
    with lib.load_scene(path) as a, oracle.load_scene(path) as b:
        assert a.counts()["materials"] == b.counts()["materials"] == own_materials + 1
        ta, ma = a.triangles()
        tb, mb = b.triangles()
        assert np.array_equal(bits(ta), bits(tb)) and np.array_equal(ma, mb)
        assert ma.max() == own_materials and (ma == own_materials).sum() >= 12
        assert np.array_equal(a.materials(), b.materials())
        d = a.materials()[own_materials].view(np.float32)
        assert list(d[9:13]) == [1.0, 1.0, 1.0, 1.0] and d[19] == 1.0 and d[20] == 1.0      # baseColor 1, metallic 1, roughness 1
        p = Params(height=48, num_samples=2, num_ambient_samples=2, max_bounces=2, msaa=2, ambient=(0.7, 0.7, 0.7), seed=3)
        lin, _ = a.render(p, want_srgb=False)
        assert np.isfinite(lin).all()
        ref = np.mean([b.render(Params(height=48, num_samples=2, num_ambient_samples=2, max_bounces=2, msaa=2, ambient=(0.7, 0.7, 0.7), seed=k), want_srgb=False)[0] for k in range(6)], axis=0)
        assert abs(float(lin.mean()) - float(ref.mean())) / float(ref.mean()) < 0.05


def check_textures(lib, path, uv, expected):
    with lib.load_scene(path) as s:
        for t, exp in enumerate(expected):
            got = s.sample_texture(t, uv)
            assert np.array_equal(bits(got), bits(exp)), "texture %d: %d samples differ" % (t, int((bits(got) != bits(exp)).any(axis=1).sum()))


def check_output_stage(lib, acc, expected):
    """Byte-exact: the sRGB power is glibc's powf restated (csrc/glibc_powf.h), everything else is IEEE fp32 in the reference's order."""
    got = lib.output_stage(acc)
    assert np.array_equal(got, expected), "output stage: %d of %d bytes differ" % (int((got != expected).sum()), got.size)


def check_lighting(lib, rec, expected, rtol=2e-4):
    got = lib.eval_lighting(rec)
    both_nan = np.isnan(got) & np.isnan(expected)
    scale = np.maximum(np.abs(expected), 1e-3)
    err = np.where(both_nan, 0.0, np.abs(got - expected) / scale)
    assert not np.isnan(err).any(), "NaN pattern differs"
    assert err.max() <= rtol, "BSDF table max relative error %.3g (column %d)" % (err.max(), int(np.argmax(err.max(axis=0))))


def mean_rel_error(img, ref):
    """Mean |a-b| over pixels / mean(b): the converged-image metric north_star names."""
    return float(np.abs(img.astype(np.float64) - ref).mean() / np.abs(ref).mean())


def render_mean(lib, path, params, seeds):
    acc = None
    with lib.load_scene(path) as s:
        for seed in seeds:
            params.seed = seed
            lin, _ = s.render(params, want_srgb=False)
            acc = lin.astype(np.float64) if acc is None else acc + lin
    return acc / len(seeds)


def read_pfm(path):
    with open(path, "rb") as f:
        assert f.readline().strip() == b"PF"
        w, h = (int(v) for v in f.readline().split())
        assert float(f.readline()) < 0              # little endian
        data = np.frombuffer(f.read(), dtype="<f4").reshape(h, w, 3)
    return data[::-1]                               # PFM stores the bottom row first


def read_hdr(path):
    with open(path, "rb") as f:
        assert f.readline().startswith(b"#?RADIANCE")
        while f.readline().strip():
            pass
        dims = f.readline().split()
        h, w = int(dims[1]), int(dims[3])
        rgbe = np.frombuffer(f.read(), np.uint8).reshape(h, w, 4).astype(np.float32)
    scale = np.where(rgbe[..., 3:] > 0, np.exp2(rgbe[..., 3:] - 136.0), 0.0)
    return rgbe[..., :3] * scale


def check_progressive_and_image_io(lib, path, tmpdir):
    """SURVEY 8f ranks 3 and 4: a progressive render (in passes, interrupted, resumed from its checkpoint in a NEW scene object)
    has the same bits as the one-shot render; .pfm keeps the exact bits, .hdr is within RGBE precision; the comparison report
    equals numpy's."""
    import os
    from sailor_b200.capi import Params, SailorPtError
    base = dict(height=40, num_samples=2, num_ambient_samples=2, max_bounces=2, msaa=5, ambient=(0.9, 0.8, 0.7), seed=11)
    ck = os.path.join(str(tmpdir), "frame.ckpt")
    with lib.load_scene(path) as s:
        full, srgb_full = s.render(Params(**base))
        # 1. all passes in one call
        lin, srgb, done = s.render_progressive(Params(**base), 2)
        assert done == 5 and np.array_equal(bits(lin), bits(full)) and np.array_equal(srgb, srgb_full)
        # 2. interrupted after one pass of 2 samples: the partial estimate is normalised by the samples done
        part, _, done = s.render_progressive(Params(**base), 2, max_passes=1, checkpoint=ck)
        assert done == 2 and os.path.exists(ck)
        two = s.render(Params(msaa_range=(0, 2), **base))[0].astype(np.float64) * 5 / 2
        assert np.allclose(part, two, rtol=1e-5, atol=1e-6)
    with lib.load_scene(path) as s2:                # a new process would start here
        # 3. resume: 2 + 2 + 1 samples, checkpoint after every pass
        lin2, srgb2, done = s2.render_progressive(Params(**base), 2, checkpoint=ck, resume=True, checkpoint_every_pass=True)
        assert done == 5 and np.array_equal(bits(lin2), bits(full)) and np.array_equal(srgb2, srgb_full)
        # 4. resuming a finished checkpoint renders nothing and returns the same frame
        lin3, _, done = s2.render_progressive(Params(**base), 2, checkpoint=ck, resume=True)
        assert done == 5 and np.array_equal(bits(lin3), bits(full))
        # 5. a checkpoint of another parameter set is refused
        other = dict(base); other["max_bounces"] = 3
        with pytest_raises(SailorPtError):
            s2.render_progressive(Params(**other), 2, checkpoint=ck, resume=True)
        # 6. a damaged checkpoint is an error, not a silent restart
        blob = bytearray(open(ck, "rb").read()); blob[200] ^= 0x40
        bad = os.path.join(str(tmpdir), "bad.ckpt"); open(bad, "wb").write(bytes(blob))
        with pytest_raises(SailorPtError):
            s2.render_progressive(Params(**base), 2, checkpoint=bad, resume=True)
    # image files
    pfm, hdr, png = (os.path.join(str(tmpdir), "f." + e) for e in ("pfm", "hdr", "png"))
    lib.write_image(pfm, full); lib.write_image(hdr, full); lib.write_image(png, full)
    assert np.array_equal(bits(read_pfm(pfm)), bits(full))
    back = read_hdr(hdr)
    assert np.all(np.abs(back - full) <= full.max(axis=2, keepdims=True) / 128.0 + 1e-6)
    assert open(png, "rb").read(8) == b"\x89PNG\r\n\x1a\n"
    # comparison report
    noisy = (full * 1.01 + 0.001).astype(np.float32)
    m = lib.compare_images(noisy, full)
    d = np.abs(noisy.astype(np.float64) - full.astype(np.float64))
    assert np.isclose(m["mean_rel_error"], d.sum() / np.abs(full.astype(np.float64)).sum(), rtol=1e-9)
    assert np.isclose(m["rmse"], np.sqrt((d * d).mean()), rtol=1e-9) and np.isclose(m["max_abs"], d.max(), rtol=1e-9)
    assert lib.compare_images(full, full)["psnr_db"] == 1e30


def pytest_raises(exc):
    import pytest
    return pytest.raises(exc)


def check_multi_device_frame(lib, path, devices=3, **base):
    """SailorPtParams::deviceCount: the frame spread over several devices (one host thread per device inside the library, dynamic row
    bands, peer copies into the scene's own device, output stage there) has the bit pattern of the single-device frame, for the
    float accumulator AND the sRGB8 image, with a row shard and with a second frame that reuses the replicas (PathTracer.cpp:418-487)."""
    kw = dict(height=23, num_samples=2, num_ambient_samples=2, max_bounces=3, msaa=4, ambient=(1, 1, 1), seed=9)
    kw.update(base)
    with lib.load_scene(path) as s:
        one_lin, one_srgb = s.render(Params(**kw))
        for n in (2, devices):
            lin, srgb = s.render(Params(device_count=n, **kw))
            st = lib.stats()
            assert np.array_equal(lin.view(np.uint32), one_lin.view(np.uint32)) and np.array_equal(srgb, one_srgb)
            assert 1 <= st["devicesUsed"] <= n and st["rays"] > 0
        h = one_lin.shape[0]
        part, _ = s.render(Params(rows=(3, h - 5), **kw))
        part_n, _ = s.render(Params(rows=(3, h - 5), device_count=devices, **kw))
        assert np.array_equal(part.view(np.uint32), part_n.view(np.uint32))
        # a second frame with other parameters through the same replicas
        kw2 = dict(kw, seed=10, msaa=2)
        a, _ = s.render(Params(**kw2)); b, _ = s.render(Params(device_count=devices, **kw2))
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    return st["devicesUsed"]


def check_shade_hits(lib, oracle, path, n=4000, seed=5, num_samples=7, num_ambient=5):
    """Rows a13/a15: the shading context of a hit -- interpolated frame, flipped face normal, uvTransform, every field of
    GetMaterialData (factors x bilinear texture samples, MASK cut-off), world normal, alpha-scaled sample counts -- is BIT-IDENTICAL to
    the reference's own GetMaterialData / Raytrace head (PathTracer.cpp:636-661, 881-927) at random points of random triangles,
    including triangle corners and edges."""
    r = np.random.RandomState(seed)
    with lib.load_scene(path) as a, oracle.load_scene(path) as b:
        nt = a.counts()["triangles"]
        tri = r.randint(0, nt, n).astype(np.uint32)
        bary = r.dirichlet((1.0, 1.0, 1.0), n).astype(np.float32)[:, 1:]
        bary[:16] = [[0, 0], [1, 0], [0, 1], [0.5, 0.5], [0.5, 0], [0, 0.5], [0.25, 0.25], [1.0 / 3, 1.0 / 3]] * 2
        tri[n - 1] = nt + 7                                   # out of range: all zeros from both
        d = r.normal(size=(n, 3)).astype(np.float32)
        got = a.shade_hits(tri, bary, d, num_samples, num_ambient)
        ref = b.shade_hits(tri, bary, d, num_samples, num_ambient)
    bad = np.argwhere(bits(got) != bits(ref))
    assert bad.size == 0, "shading context differs at %d of %d values, first (hit, field) %s: %r vs %r" % (len(bad), got.size, bad[0], got[tuple(bad[0])], ref[tuple(bad[0])])
    return got


def check_sample_generators(lib):
    """Row a17: the counter-based generators have the distributions of the reference's (glm::linearRand on rand() % 255 bytes,
    glm/gtc/random.inl:19-27,66-85,176-183; NextVec2_BlueNoise table walk, PathTracer.cpp:934-1077)."""
    n = 1 << 18
    u = lib.sample_generators(12345, 0, n)
    by = u.view(np.uint8).reshape(n, 4)
    assert by.max() == 254, "a byte is rand() % 255: never 255"
    for k in range(4):
        h = np.bincount(by[:, k], minlength=255)[:255]
        assert h.min() > 0 and abs(h - n / 255.0).max() < 6.0 * np.sqrt(n / 255.0), "byte %d is not uniform over 0..254" % k
    assert not np.array_equal(u[:1000], lib.sample_generators(12346, 0, 1000)), "streams of different keys differ"
    assert np.array_equal(u[:1000], lib.sample_generators(12345, 0, 1000)), "a stream is a pure function of its key"
    f = lib.sample_generators(99, 1, n)
    raw = lib.sample_generators(99, 0, n)
    # linearRand(0.f, 1.f) = float(u32) / float(UINT32_MAX) * (Max - Min) + Min (random.inl:176-183), bit for bit
    expect = (raw.astype(np.float32) / np.float32(4294967296.0)) * np.float32(1.0) + np.float32(0.0)
    assert np.array_equal(bits(f), bits(expect))
    assert f.min() >= 0.0 and f.max() < 1.0 and abs(float(f.mean()) - 0.498) < 0.003      # top byte <= 254: mean = 127/255 + ...
    # blue-noise walk: values are table[k] / 1024, indices advance by one up to 687 and restart at linearRand(0, 680)
    table = blue_noise_table()
    for key in (1, 2, 77):
        w = lib.sample_generators(key, 2, 3000)
        ix, iy = w[:, 2].astype(np.int64), w[:, 3].astype(np.int64)
        assert np.array_equal(w[:, 0], table[ix].astype(np.float32) / np.float32(1024)) and np.array_equal(w[:, 1], table[iy].astype(np.float32) / np.float32(1024))
        for idx in (ix, iy):
            assert idx.min() >= 0 and idx.max() <= 687
            step = np.diff(idx)
            restart = step != 1
            assert np.all(idx[:-1][restart] == 687) and np.all(idx[1:][restart] <= 680) and restart.sum() >= 3
        assert ix[0] <= 680 and iy[0] <= 680


def blue_noise_table():
    """The integers of sailor_b200/csrc/blue_noise_table.h (value = k / 1024)."""
    import re
    src = open(os.path.join(ROOT, "sailor_b200", "csrc", "blue_noise_table.h")).read()
    body = src[src.index("kBlueNoiseK[kBlueNoiseCount] = {") :]
    body = body[body.index("{") + 1:body.index("};")]
    t = np.array([int(x) for x in re.findall(r"\d+", body)], np.int64)
    assert len(t) == 688
    return t


def check_batching_and_overflow_retry(lib, path, monkeypatch, **base):
    """The wavefront works on batches of first hits sized by a memory budget, and redoes a batch smaller when an arena overflows
    (render.cuh).  Results are keyed per activation, so the frame must not depend on either: a 1 MiB budget (many batches) and a forced
    overflow of every first attempt (SAILOR_PT_TEST_OVERFLOW) give the bits of the default frame."""
    kw = dict(height=72, num_samples=3, num_ambient_samples=3, max_bounces=3, msaa=3, ambient=(1, 1, 1), seed=4)
    kw.update(base)
    with lib.load_scene(path) as s:
        ref, _ = s.render(Params(**kw)); b0 = lib.stats()["batches"]
        monkeypatch.setenv("SAILOR_PT_BATCH_MB", "1")
        many, _ = s.render(Params(**kw)); b1 = lib.stats()["batches"]
        monkeypatch.delenv("SAILOR_PT_BATCH_MB")
        monkeypatch.setenv("SAILOR_PT_TEST_OVERFLOW", "1")
        redo, _ = s.render(Params(**kw)); b2 = lib.stats()["batches"]
        monkeypatch.delenv("SAILOR_PT_TEST_OVERFLOW")
    assert b1 > b0, (b0, b1, b2)          # (a forced overflow redoes the batch; whether it also splits it depends on the budget)
    assert np.array_equal(bits(ref), bits(many)) and np.array_equal(bits(ref), bits(redo))
