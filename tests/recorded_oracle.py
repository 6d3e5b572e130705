"""Recorded answers for the oracle where the oracle library cannot be built.

The oracle (oracle/_ref/libsailor_pt_ref.so) is compiled from the reference path tracer's own sources, which are not
part of this repository.  Without it, `RecordedOracle` stands in: every call runs on a build of this project (`inner`:
the CUDA library in GPU tests, the host-compiled kernel bodies otherwise), its result must have the SHA-256 digest
recorded for the same call in tests/golden/oracle_calls.json, and is then handed to the test.  A call is identified by
its name, its arguments (Params by the fields that differ from their defaults) and, for scene methods, the bytes of the
scene file.

The file has two sections, and a failure message names the one the recorded result came from:

  "oracle"   the oracle's results.  Recorded from this project's libraries at commit 85c2190, whose compiled code equals
             that of the two runs against the oracle library committed under profiles/: all 55 GPU tests at 8fd1808
             (r03z_pytest.txt; later commits change comments only), and the CPU tests of test_host_logic,
             test_multi_device and test_gltf_containers at c5c43cd (r03z_asan_host_compiled_bodies.txt).  Calls of
             those tests, plus those of test_oracle_golden, whose every recorded result the same recording run checked
             against the goldens minted from the oracle (make_golden.py).
  "project"  this project's own results at commit 85c2190, for the remaining calls (image decoding, command-line
             parsing, the C4 material tables, the oracle-only glTF variants).  No committed run shows them equal to the
             oracle's -- for damaged image files test_image_codecs even allows 2 % to differ -- so there they pin this
             project's behaviour, not the reference's.

Not recorded: renders (the reference draws its own random numbers, so only the statistics of its images compare); the
BSDF table is answered from the oracle's own table in tests/golden/golden.npz.

SAILOR_ORACLE_RECORD=<file.json> python -m pytest tests ...  records the digests of every oracle call into the "oracle"
section of that file.  It runs only where the oracle library is built: recording anything else would store this
project's results as the oracle's.
"""
import atexit
import hashlib
import json
import os

import numpy as np
import pytest

from sailor_b200.capi import Params, SailorPtError

HERE = os.path.dirname(os.path.abspath(__file__))
CALLS = os.path.join(HERE, "golden", "oracle_calls.json")
RECORD = os.environ.get("SAILOR_ORACLE_RECORD")
ORIGIN = {"oracle": "the oracle's recorded result",
          "project": "this project's recorded result at commit 85c2190 (not shown equal to the oracle's)"}
NOT_RECORDED = {
    "render": "compares with the oracle's renders, which are not recorded: they use the reference's own random numbers",
    "render_progressive": "compares with the oracle's renders, which are not recorded: they use the reference's own random numbers",
    "eval_lighting": None,           # answered from golden.npz
    "lib": "checks the oracle library itself, which is built from the reference's sources",
    "backend": "checks the oracle library itself, which is built from the reference's sources",
}
_DEFAULTS = vars(Params())
_recorded = None
_new = {}


def _feed(h, v):
    if isinstance(v, np.ndarray):
        h.update(("array %s %s;" % (v.dtype.str if v.dtype.names is None else v.dtype.descr, v.shape)).encode())
        h.update(np.ascontiguousarray(v).tobytes())
    elif isinstance(v, (tuple, list)):
        h.update(b"(")
        for e in v:
            _feed(h, e)
        h.update(b")")
    elif isinstance(v, dict):
        _feed(h, sorted(v.items()))
    elif isinstance(v, Params):
        _feed(h, sorted((k, e) for k, e in vars(v).items() if not k.startswith("_") and (k not in _DEFAULTS or e != _DEFAULTS[k])))
    elif isinstance(v, (bytes, bytearray)):
        h.update(b"bytes %d;" % len(v) + bytes(v))
    elif isinstance(v, (np.generic, int, float)):
        h.update(repr(v.item() if isinstance(v, np.generic) else v).encode())
    else:
        h.update(repr(v).encode())
    h.update(b";")


def digest(*values):
    h = hashlib.sha256()
    for v in values:
        _feed(h, v)
    return h.hexdigest()[:16]


def _file(path):
    with open(path, "rb") as f:
        return digest(f.read())


def _lookup(key):
    global _recorded
    if _recorded is None:
        _recorded = json.load(open(CALLS))
    for section in ("oracle", "project"):
        if key in _recorded[section]:
            return _recorded[section][key], section
    return None, None


def _save():
    if not _new:
        return
    out =json.load(open(RECORD)) if os.path.exists(RECORD) else {"oracle": {}, "project": {}}
    out["oracle"].update(_new)
    for k in _new:
        out["project"].pop(k, None)
    with open(RECORD, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")


if RECORD:
    atexit.register(_save)


def _bsdf_table(records):
    """The oracle's BSDF table for the records it was minted with (golden.npz); this project's differs in the last bits."""
    G = np.load(os.path.join(HERE, "golden", "golden.npz"))
    rec = np.ascontiguousarray(records, dtype=np.float32)
    assert rec.shape == G["lighting_in"].shape and np.array_equal(rec.view(np.uint32), G["lighting_in"].view(np.uint32)), \
        "no recorded oracle result for eval_lighting of these records (golden.npz holds the table for lighting_in only)"
    return G["lighting_out"]


class RecordedOracle:
    """Library (or, from load_scene, Scene) interface of the oracle: `inner`'s results, checked against the recorded ones.
    recording=True (the oracle library itself as `inner`): record instead of checking."""

    def __init__(self, inner, scope="library", recording=False):
        self._inner = inner
        self._scope = scope
        self._recording = recording

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self._inner.close()

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        f = getattr(self._inner, name)
        if name in NOT_RECORDED and not self._recording:
            if name == "eval_lighting":
                return _bsdf_table
            pytest.skip(NOT_RECORDED[name])
        if name in NOT_RECORDED or not callable(f):
            return f

        def call(*args, **kw):
            if name == "load_scene":
                key = digest(self._scope, name, _file(args[0]))
            else:
                key = digest(self._scope, name, args, kw)
            try:
                out = f(*args, **kw)
                got = "loaded" if name == "load_scene" else digest(out)
            except SailorPtError as e:
                out, got = e, "error %d" % e.code
            if self._recording:
                if _new.get(key, got) != got:
                    raise AssertionError("%s: two different results for one oracle call while recording" % name)
                _new[key] = got
            else:
                want, section = _lookup(key)
                assert want is not None, ("no recorded oracle result for this %s call: its inputs differ from the recorded ones (another "
                                          "encoder build, or new Params fields with non-default values); record with the oracle library" % name)
                assert got == want, "%s: result differs from %s (digest %s, got %s)" % (name, ORIGIN[section], want, got)
            if isinstance(out, Exception):
                raise out
            return RecordedOracle(out, key, self._recording) if name == "load_scene" else out
        return call


def for_tests(oracle_library, inner):
    """The `oracle` fixture's value: the oracle library (recording its calls under SAILOR_ORACLE_RECORD), or else the
    recorded answers computed by `inner`."""
    if oracle_library is not None:
        return RecordedOracle(oracle_library, recording=True) if RECORD else oracle_library
    if RECORD:
        pytest.fail("SAILOR_ORACLE_RECORD records the oracle library's results, and it is not built here")
    return RecordedOracle(inner())
