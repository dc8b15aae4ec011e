"""Recorded answers of the reference's own sources for the tests that compare the oracle with them.

Those sources (the Eagle package's src/, compiled through oracle/refshim into oracle/_ref/libeagle_ref.so) are not part
of the repository.  tests/golden/reference_calls.json keeps, per test and in call order, a fingerprint of every answer
they gave: arrays and file contents as dtype, shape and (64 bits of) sha256; messages, verdicts and counts as they are, with the
pytest temporary directory written as "<tmp>"; and, for arrays that a test compares within a tolerance, a fixed
seeded sample of values and the largest magnitude.  A test compares the oracle's own answer with the record.  When the
compiled reference is present, each answer is also computed live and must match its record.  Long fuzz loops record
one digest of each whole answer instead.

EAGLE_RECORD_REFERENCE=reference rewrites the records from the compiled reference.  EAGLE_RECORD_REFERENCE=oracle
writes them from the C oracle instead; the file's "source" field says which one produced them.
"""
import hashlib
import json
import os
import re

import numpy as np
import pytest

from oracle import eagle_oracle as eo

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.json")
SAMPLE = 256
SOURCES = {
    "reference": "the reference's own sources compiled through oracle/refshim",
    "oracle": "oracle/eagle_oracle.c standing in for the reference's own sources: the tests that use these records "
              "had found the two identical call for call (bit for bit, or within their stated tolerance for the "
              "scan and reduced-a products), and the oracle's arithmetic has not changed since",
}


class Approx:
    """An array that the test compares within a tolerance: recorded as a seeded sample of its values."""

    def __init__(self, x, keep=()):
        self.x = np.asarray(x, dtype=np.float64).reshape(-1)
        self.keep = [int(i) for i in keep]


def _sha(b):
    return hashlib.sha256(b).hexdigest()[:16]


def fingerprint(x, tmp):
    if isinstance(x, Approx):
        v = x.x
        idx = np.random.default_rng(0).choice(v.size, min(v.size, SAMPLE), replace=False)
        idx = sorted(set(idx.tolist()) | set(x.keep))
        return {"approx": True, "size": int(v.size), "absmax": float(np.abs(v).max()) if v.size else 0.0,
                "idx": idx, "values": [float(v[i]) for i in idx]}
    if isinstance(x, np.ndarray):
        return {"dtype": str(x.dtype), "shape": list(x.shape), "sha256": _sha(np.ascontiguousarray(x).tobytes())}
    if isinstance(x, (bytes, bytearray)):
        return {"bytes": len(x), "sha256": _sha(bytes(x))}
    if isinstance(x, str):
        return re.sub(re.escape(tmp) + r"/[^/]+", "<tmp>", x)
    if isinstance(x, (list, tuple)):
        return [fingerprint(v, tmp) for v in x]
    if isinstance(x, dict):
        return {str(k): fingerprint(v, tmp) for k, v in x.items()}
    if isinstance(x, (bool, np.bool_)):
        return bool(x)
    if isinstance(x, (int, np.integer)):
        return int(x)
    if isinstance(x, (float, np.floating)):
        return float(x)
    if x is None:
        return None
    raise TypeError(f"no fingerprint for {type(x).__name__}")


def error_message(fn, *a):
    """The OracleError message fn(*a) raises (the reference's Rcpp::stop text), or None."""
    try:
        fn(*a)
    except eo.OracleError as ex:
        return str(ex)
    return None


def close(mine, rec, rtol, atol):
    """mine (the whole array) against a recorded Approx sample: |mine - ref| <= rtol |ref| + atol at every sampled index."""
    m = np.asarray(mine, dtype=np.float64).reshape(-1)
    assert rec["approx"] and m.size == rec["size"]
    np.testing.assert_allclose(m[rec["idx"]], rec["values"], rtol=rtol, atol=atol)


def _same(live, rec):
    if isinstance(rec, dict) and rec.get("approx"):
        return live["size"] == rec["size"] and live["idx"] == rec["idx"] and np.allclose(
            live["values"], rec["values"], rtol=1e-12, atol=1e-10 * rec["absmax"])
    if isinstance(rec, dict):
        return isinstance(live, dict) and live.keys() == rec.keys() and all(_same(live[k], rec[k]) for k in rec)
    if isinstance(rec, list):
        return isinstance(live, list) and len(live) == len(rec) and all(_same(a, b) for a, b in zip(live, rec))
    return live == rec


class Reference:
    """ref(f) -> fingerprint of what f() returns with the oracle's calls routed to the reference's sources."""

    def __init__(self, name, tmp):
        self.name, self.tmp, self.calls = name, tmp, 0
        self.mode = os.environ.get("EAGLE_RECORD_REFERENCE")
        if self.mode not in (None, "reference", "oracle"):
            raise ValueError("EAGLE_RECORD_REFERENCE must be 'reference' or 'oracle'")
        if self.mode == "reference" and not eo.reference_available():
            raise RuntimeError("EAGLE_RECORD_REFERENCE=reference needs oracle/_ref/libeagle_ref.so")
        self.data = json.load(open(PATH)) if os.path.exists(PATH) else {"source": None, "tests": {}}
        self.rec = [] if self.mode else self.data["tests"].get(name)
        if self.rec is None:
            pytest.fail(f"{os.path.basename(PATH)} has no record for {name}")

    def fp(self, x, digest=False):
        x = fingerprint(x, self.tmp)
        return _sha(json.dumps(x, sort_keys=True).encode()) if digest else x

    def __call__(self, f, digest=False):
        i, self.calls = self.calls, self.calls + 1
        if self.mode == "oracle":
            self.rec.append(self.fp(f(), digest))
            return self.rec[i]
        if eo.reference_available():
            with eo.use_reference():
                live = self.fp(f(), digest)
            if self.mode:
                self.rec.append(live)
            else:
                assert i < len(self.rec) and _same(live, self.rec[i]), f"{self.name}: reference answer {i} differs from its record"
            return live
        assert i < len(self.rec), f"{self.name}: more calls than recorded"
        return self.rec[i]

    def finish(self):
        if self.mode:
            self.data["source"] = SOURCES[self.mode]
            self.data["tests"][self.name] = self.rec
            with open(PATH, "w") as fh:
                json.dump(self.data, fh, separators=(",", ":"), sort_keys=True)
        else:
            assert self.calls == len(self.rec), f"{self.name}: {self.calls} calls, {len(self.rec)} recorded"


@pytest.fixture
def reference(request, tmp_path_factory):
    r = Reference(request.node.name, str(tmp_path_factory.getbasetemp()))
    yield r
    r.finish()
