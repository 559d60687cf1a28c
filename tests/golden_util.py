"""Shared helpers for the golden-vector tests (tests/golden/golden.json, generated from the unmodified reference by
tests/golden/make_golden.py) and for the tests that compare with the reference through stored results
(tests/golden/ref_results.json, see reference())."""
import hashlib
import json
import os

import numpy as np

import aissynth as S

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "golden.json")

FMT_CF32, FMT_CU8 = 0, 1


def load():
    with open(GOLDEN) as f:
        return json.load(f)["cases"]


def case_input(case):
    """(raw numpy array, elements per complex sample).  Seeded cases verify the generator against input_sha256."""
    if "file" in case:
        return np.fromfile(os.path.join(HERE, "golden", case["file"]), dtype=np.uint8), 2
    x = S.random_stream(case["fs"], case["N"] * case["nchunks"], case["seed"], multi_sentence=case["multi"])[0]
    raw, per = (S.to_cu8(x), 2) if case["fmt"] == FMT_CU8 else (x, 1)
    got = hashlib.sha256(np.ascontiguousarray(raw).tobytes()).hexdigest()
    assert got == case["input_sha256"], "seeded generator no longer reproduces the golden input (numpy RNG change?)"
    return raw, per


def fbits(v):
    return int(np.float32(v).view(np.uint32))


def msg_record(ch, nbits, payload, nmea, start, end, level, ppm):
    return {"ch": ch, "nbits": nbits, "payload": payload.hex(), "nmea": list(nmea), "start": start, "end": end,
            "level": fbits(level), "ppm": fbits(ppm)}


REF_RESULTS = os.path.join(HERE, "golden", "ref_results.json")
RECORD = None  # a dict while tests/golden/make_ref_results.py records
_stored = None


class Digest:
    """sha256 + element count of byte blocks fed in order (block lengths are part of the digest)."""

    def __init__(self):
        self.h, self.n = hashlib.sha256(), 0

    def add(self, a, n=None):
        b = a if isinstance(a, bytes) else np.ascontiguousarray(a).tobytes()
        self.h.update(len(b).to_bytes(8, "little") + b)
        self.n += len(a) if n is None else n
        return self

    def value(self):
        return [self.n, self.h.hexdigest()]


def msgs_digest(msgs):
    """[count, sha256] of a message list in order: key, start/end counters, level and ppm bit patterns.  Takes the
    messages of the oracle (oracle.Msg) and of the engine (aisgpu.Msg) alike."""
    d = Digest()
    for m in msgs:
        d.add(repr((m.channel, m.nbits, m.payload.hex(), list(m.nmea), m.start_idx, m.end_idx, fbits(m.level), fbits(m.ppm))).encode(), 1)
    return d.value()


def reference(key, compute):
    """What the unmodified reference computed for the test case `key` (digests and small values, JSON-shaped).
    Where oracle/_ref was built, compute() runs it live and the result must equal the stored one; elsewhere the result
    stored in tests/golden/ref_results.json (written by tests/golden/make_ref_results.py) stands in for it."""
    global _stored
    import oracle as O
    if _stored is None:
        _stored = {}
        if os.path.exists(REF_RESULTS):
            with open(REF_RESULTS) as f:
                _stored = json.load(f)
    want = _stored.get(key)
    if not O.have_ref():
        assert want is not None, "%s: no stored reference result" % key
        return want
    got = json.loads(json.dumps(compute()))
    if RECORD is not None:
        RECORD[key] = got
    else:
        assert want is not None, "%s: no stored reference result (run tests/golden/make_ref_results.py)" % key
        assert got == want, "%s: the reference no longer computes the stored result" % key
    return got
