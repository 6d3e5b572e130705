#!/usr/bin/env python3
"""Scene load and flatten cost of glTF geometry forms, this tree's library against an earlier build, on one GPU.

    python tools/geometry_bench.py --baseline-lib OTHER.so [--reps 3] [--out FILE.json]

Scenes (generated into a temporary directory by tests/geometry_scenes.py): BASELINE C5 (one 1 M-triangle mesh under 10 nodes) as
  list       float32 positions and a u32 TRIANGLES list (C5 itself)
  quantized  int16 positions, int8 normals, u16 UVs, u32 TRIANGLES list
  strips     the quantized streams as one unindexed TRIANGLE_STRIP per row of quads
For each library and scene: SailorPt_SceneLoad wall time with the parsed-scene cache off (parse + upload + decode + flatten, ending in
a device synchronise), h2dBytes and secondsFlatten (CUDA events around the decode, assembly and flatten launches), medians over
--reps repetitions that alternate the two libraries scene by scene.  A SHA-256 of the flattened triangles is recorded for every
load; the two libraries must agree on every file both can load (the earlier build draws no strips: 0 triangles).  Card name and power limit are
read in the same run.
"""
import argparse
import hashlib
import json
import os
import statistics
import sys
import tempfile
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import geometry_scenes as gs  # noqa: E402
from golden import make_golden_c4c5 as MG  # noqa: E402
from instancing_bench import card  # noqa: E402
from sailor_b200.capi import Library, SailorPtError  # noqa: E402


def load_once(lib, path):
    t0 = time.perf_counter()
    try:
        s = lib.load_scene(path)
    except SailorPtError as e:
        return {"error": str(e)}
    wall = time.perf_counter() - t0
    st = lib.stats()
    tris, mat = s.triangles()
    digest = hashlib.sha256(tris.tobytes() + mat.tobytes()).hexdigest()
    s.close()
    return {"load_s": wall, "h2d_bytes": st["h2dBytes"], "flatten_s": st["secondsFlatten"], "triangles": len(tris), "sha256": digest}


def summarise(runs):
    if "error" in runs[0]:
        return {"error": runs[0]["error"]}
    assert len({r["sha256"] for r in runs}) == 1, "a library flattened one file two ways"
    return {"triangles": runs[0]["triangles"], "h2d_bytes": runs[0]["h2d_bytes"], "sha256": runs[0]["sha256"],
            "load_s_median": statistics.median(r["load_s"] for r in runs), "load_s": [round(r["load_s"], 4) for r in runs],
            "flatten_s_median": statistics.median(r["flatten_s"] for r in runs), "flatten_s": [r["flatten_s"] for r in runs]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--baseline-lib", required=True)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    os.environ["SAILOR_PT_SCENE_CACHE"] = "0"
    import sailor_b200
    from sailor_b200 import build as product_build
    product_build.build()
    libs = {"this": sailor_b200.library(), "baseline": Library(a.baseline_lib)}
    with tempfile.TemporaryDirectory() as d:
        paths = {form: gs.heightfield_forms(os.path.join(d, "c5_%s.glb" % form), form, **MG.C5_KW) for form in ("list", "quantized", "strips")}
        plan = [(name, which) for name in paths for which in ("baseline", "this")]
        for name, which in plan:                 # warm-up: module load, first allocations, page cache
            load_once(libs[which], paths[name])
        runs = {key: [] for key in plan}
        for _ in range(a.reps):
            for key in plan:
                runs[key].append(load_once(libs[key[1]], paths[key[0]]))
    scenes = {"%s/%s" % key: summarise(r) for key, r in runs.items()}
    for name in paths:
        base, this = scenes["%s/baseline" % name], scenes["%s/this" % name]
        assert "error" not in this, this
        if "error" not in base and base["triangles"]:
            assert base["sha256"] == this["sha256"], "%s: the two libraries flatten it differently" % name
    result = {"card": card(), "reps": a.reps, "scene": "BASELINE C5 (%d triangles) in three forms" % scenes["list/this"]["triangles"],
              "scenes": scenes}
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
