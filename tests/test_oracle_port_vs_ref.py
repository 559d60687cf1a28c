"""CPU (-m "not gpu"): pins the plain-C restatement oracle/ais_oracle.c against the UNMODIFIED reference
(oracle/_ref/libaisref.so, strict IEEE flags) -- every tap and every message bit for bit, through digests.
The reference holds no golden vectors for the IQ path (SURVEY.md 4, 8c), so outputs of the reference itself are the
pin: computed live where oracle/_ref was built, else the digests stored in tests/golden/ref_results.json.
"""
import numpy as np
import pytest

import aissynth as S
import golden_util as G
import oracle as O


def digests(Model, model, fs, N, nchunks, fmt, flags, seed, multi):
    """Every tap and every message of one model over the seeded stimulus, as digests (per-chunk block lengths included)."""
    x = S.random_stream(fs, N * nchunks, seed, multi_sentence=multi)[0]
    per = 1
    if fmt == O.FMT_CU8:
        x, per = S.to_cu8(x), 2
    elif fmt == O.FMT_CS8:
        x, per = (S.to_cu8(x).astype(np.int16) - 128).astype(np.int8), 2
    elif fmt == O.FMT_CS16:
        v = np.empty(2 * len(x), dtype=np.float32)
        v[0::2], v[1::2] = x.real, x.imag
        x, per = np.clip(np.round(v * 32767.0), -32768, 32767).astype(np.int16), 2
    m = Model(model=model, sample_rate=fs, fmt=fmt, flags=flags, taps=True)
    d = {"complex tap %d" % t: G.Digest() for t in range(9)}
    d.update({"float tap %d" % t: G.Digest() for t in range(14)})
    d.update({"ppm tap %d" % t: G.Digest() for t in (O.TAP_CGF_A, O.TAP_CGF_B)})
    d["messages"] = G.Digest()
    for c in range(nchunks):
        m.push(x[c * N * per:(c + 1) * N * per])
        for t in range(9):
            d["complex tap %d" % t].add(m.tap_c(t))
        for t in range(14):
            d["float tap %d" % t].add(m.tap_f(t))
        for t in (O.TAP_CGF_A, O.TAP_CGF_B):
            d["ppm tap %d" % t].add(m.tap_ppm(t))
        ms = m.messages()
        d["messages"].add(repr(G.msgs_digest(ms)).encode(), len(ms))
    return {k: v.value() for k, v in d.items()}


def compare(model, fs, N, nchunks, fmt=O.FMT_CF32, flags=O.DEFAULT_FLAGS, seed=0, multi=False):
    args = (model, fs, N, nchunks, fmt, flags, seed, multi)
    want = G.reference("port_vs_ref %r" % (args,), lambda: digests(O.RefModel, *args))
    got = digests(O.PortModel, *args)
    for k in want:
        assert got[k] == want[k], "%s differs from the reference's" % k
    return got["messages"][0]


@pytest.mark.parametrize("model", [O.MODEL_DEFAULT, O.MODEL_STANDARD, O.MODEL_BASE])
def test_models_1536k(built, model):
    assert compare(model, 1536000, 65536, 4) >= (1 if model == O.MODEL_BASE else 3)


@pytest.mark.parametrize("fs,N", [(96000, 4096), (192000, 8192), (288000, 12288), (384000, 16384), (768000, 32768),
                                  (3072000, 131072), (6000000, 262144), (6144000, 262144), (12288000, 524288),
                                  (2000000, 65536), (250000, 16384)])
def test_rates_default(built, fs, N):
    # includes the /3 DownsampleKFilter path (288k) and interpolated non-bucket rates (6 MSPS AirSpy shape, 2 M, 250 k)
    assert compare(O.MODEL_DEFAULT, fs, N, 3, seed=23) >= 1


@pytest.mark.parametrize("fmt", [O.FMT_CU8, O.FMT_CS8, O.FMT_CS16])
def test_integer_formats(built, fmt):
    assert compare(O.MODEL_DEFAULT, 1536000, 65536, 3, fmt=fmt, seed=17) >= 2


@pytest.mark.parametrize("flags", [O.FLAG_AFC_WIDE | O.FLAG_DROOP, O.FLAG_PS_EMA, O.FLAG_PS_EMA | O.FLAG_DROOP, 0])
def test_flag_variants(built, flags):
    compare(O.MODEL_DEFAULT, 1536000, 32768, 6, flags=flags, seed=11)


def test_small_chunks(built):
    # 48 kHz count per chunk (128) below one CGF block (512): re-blocking paths
    assert compare(O.MODEL_DEFAULT, 1536000, 4096, 48, seed=7) >= 1
    compare(O.MODEL_STANDARD, 1536000, 4096, 48, seed=7)


def test_multi_sentence(built):
    # 424-bit messages -> two sentences with the sequence id of Message.cpp:28-39
    n = compare(O.MODEL_DEFAULT, 1536000, 65536, 6, seed=31, multi=True)
    assert n >= 2
