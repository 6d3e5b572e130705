#!/usr/bin/env python3
"""Scene load and flatten cost of shared meshes and EXT_mesh_gpu_instancing, on one GPU.

    python tools/instancing_bench.py [--reps 3] [--baseline-lib OTHER.so] [--out FILE.json]

Scenes (generated into a temporary directory by tests/scenes.py and tests/instancing_scenes.py):
  c5_nodes       BASELINE C5: one 1 M-triangle mesh under 10 nodes (node-level instancing)
  c5_ext         the same scene with every node's TRS in a one-instance EXT_mesh_gpu_instancing
  inst10m_ext    one node instancing a two-primitive 707 x 707 grid 10 times (10 M triangles)
  inst100k_ext   100,000 instances of a 120-triangle mesh (12 M triangles)
  inst100k_nodes the same written with one node per instance
For each: SailorPt_SceneLoad wall time with the parsed-scene cache off (parse + upload + flatten, ending in a device
synchronise), h2dBytes, secondsFlatten (CUDA events around the flatten launches), and flatten's achieved bytes/s over the 232 B
it writes per triangle (vtx 48 + centroid 16 + shade 144 + uv2 24) against the HBM figure bench.py uses.

--baseline-lib: another build of the library (e.g. an earlier commit's) measured on the node-level scenes in the same process,
alternating with this tree's build, repetition by repetition.  Card name and power limit are recorded with the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
import instancing_scenes  # noqa: E402
import scenes  # noqa: E402
from golden import make_golden_c4c5 as MG  # noqa: E402
from sailor_b200.capi import Library  # noqa: E402

BYTES_PER_TRIANGLE = 48 + 16 + 144 + 24


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:      # the numbers stay, marked as measured on an unidentified card
        return {"error": repr(e)}


def make_scenes(d):
    c5 = scenes.ensure(d, "instanced", **MG.C5_KW)
    return {
        "c5_nodes": c5,
        "c5_ext": instancing_scenes.c5_as_instancing_extension(c5, os.path.join(d, "c5_ext.glb")),
        "inst10m_ext": instancing_scenes.instanced_scene(os.path.join(d, "inst10m_ext.glb"), form="ext", nx=707, nz=707, instances=10),
        "inst100k_ext": instancing_scenes.instanced_scene(os.path.join(d, "inst100k_ext.glb"), form="ext", nx=6, nz=10, instances=100000),
        "inst100k_nodes": instancing_scenes.instanced_scene(os.path.join(d, "inst100k_nodes.glb"), form="nodes", nx=6, nz=10, instances=100000),
    }


def load_once(lib, path):
    t0 = time.perf_counter()
    s = lib.load_scene(path)
    wall = time.perf_counter() - t0
    st = lib.stats()
    tris = s.counts()["triangles"]
    s.close()
    return {"load_s": wall, "h2d_bytes": st["h2dBytes"], "flatten_s": st["secondsFlatten"], "triangles": tris}


def summarise(runs, hbm_gbs):
    flat = statistics.median(r["flatten_s"] for r in runs)
    tris = runs[0]["triangles"]
    gbs = tris * BYTES_PER_TRIANGLE / flat / 1e9 if flat > 0 else float("nan")
    return {"triangles": tris, "h2d_bytes": runs[0]["h2d_bytes"],
            "load_s_median": statistics.median(r["load_s"] for r in runs), "load_s": [round(r["load_s"], 4) for r in runs],
            "flatten_s_median": flat, "flatten_s": [r["flatten_s"] for r in runs],
            "flatten_written_gbs": gbs, "flatten_frac_of_hbm": gbs / hbm_gbs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--baseline-lib", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    os.environ["SAILOR_PT_SCENE_CACHE"] = "0"
    import sailor_b200
    from sailor_b200 import build as product_build
    product_build.build()
    libs = {"this": sailor_b200.library()}
    if a.baseline_lib:
        libs["baseline"] = Library(a.baseline_lib)
    hbm, hbm_src = bench.peaks()
    with tempfile.TemporaryDirectory() as d:
        paths = make_scenes(d)
        plan = [(name, "this") for name in paths]
        if "baseline" in libs:
            plan += [(name, "baseline") for name in paths if name.endswith("_nodes")]
        for name, which in plan:                 # warm-up: module load, first allocations, page cache
            load_once(libs[which], paths[name])
        runs = {key: [] for key in plan}
        for _ in range(a.reps):
            for key in plan:
                runs[key].append(load_once(libs[key[1]], paths[key[0]]))
    result = {"card": card(), "hbm_gbs": hbm, "hbm_source": hbm_src, "bytes_per_triangle_written": BYTES_PER_TRIANGLE, "reps": a.reps,
              "scenes": {"%s/%s" % key: summarise(r, hbm) for key, r in runs.items()}}
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
