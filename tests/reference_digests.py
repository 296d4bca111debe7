"""What the reference's own code (oracle/_ref: its templates compiled from its sources) returned on the tests' seeded inputs, kept in
tests/golden/reference_digests.json, per compared output: a SHA-256 digest of all its values, the shapes of its arrays and a seeded
sample of SAMPLE values.  Every comparison with the reference thereby also runs where the reference was never built, at full size, for
a few hundred bytes of fixture (all compared outputs are exact integers); when one fails, the shapes and the sample say where to start.

Recording needs oracle/_ref:  NVB_RECORD_REFERENCE=<out.json> pytest <tests> -- every check then also runs the reference, compares
with it and stores its record; <out.json> receives the committed records with those updated (copy it over the fixture)."""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
RECORD = os.environ.get("NVB_RECORD_REFERENCE")
SAMPLE = 8
_saved = {}
if os.path.exists(PATH):
    with open(PATH) as f:
        _saved = json.load(f)


def _arrays(v):
    if isinstance(v, dict):
        return [a for k in sorted(v) for a in _arrays(v[k])]
    if isinstance(v, (tuple, list)):
        return [a for x in v for a in _arrays(x)]
    return [np.ascontiguousarray(v, dtype=np.int64)]


def record(v):
    """digest, shapes and a seeded sample of the values of a (nested tuple / list / dict of) integer array(s); the dtype does not enter,
    as in np.array_equal.  The sample is [flat index, value] pairs over the arrays' values laid end to end."""
    arrays = _arrays(v)
    h = hashlib.sha256()
    for a in arrays:
        h.update(repr(a.shape).encode())
        h.update(a.tobytes())
    flat = np.concatenate([a.reshape(-1) for a in arrays])
    idx = np.unique(np.random.default_rng(0).integers(0, len(flat), SAMPLE)) if len(flat) else []
    return {"sha256": h.hexdigest(), "shapes": [list(a.shape) for a in arrays], "sample": [[int(i), int(flat[i])] for i in idx]}


def _difference(arrays, want):
    shapes = [list(a.shape) for a in arrays]
    if shapes != want["shapes"]:
        return "array shapes %s, the reference's %s" % (shapes, want["shapes"])
    flat = np.concatenate([a.reshape(-1) for a in arrays])
    bad = ["[%d] = %d, the reference's %d" % (i, flat[i], w) for i, w in want["sample"] if flat[i] != w]
    return "%d of %d sampled values differ%s" % (len(bad), len(want["sample"]), (": " + "; ".join(bad)) if bad else "")


class Reference:
    """One test's view of the reference: `live` is the reference library while recording (else None); same(got, want) asserts that
    `got` equals the reference's output -- want(), which calls `live`, while recording, else the record stored for this call."""

    def __init__(self, request, make_live):
        self.key = "%s::%s" % (os.path.splitext(os.path.basename(str(request.node.fspath)))[0], request.node.name)
        self.n = 0
        self.live = make_live() if RECORD else None

    def same(self, got, want):
        key = "%s#%d" % (self.key, self.n)
        self.n += 1
        if RECORD:
            _saved[key] = record(want())
            with open(RECORD, "w") as f:                 # one output per line
                f.write("{\n" + ",\n".join("%s: %s" % (json.dumps(k), json.dumps(_saved[k])) for k in sorted(_saved)) + "\n}\n")
        assert key in _saved, "no recorded reference output for " + key
        if record(got)["sha256"] != _saved[key]["sha256"]:
            raise AssertionError("%s differs from the reference: %s" % (key, _difference(_arrays(got), _saved[key])))
