"""Randomised configuration matrix: model x sample rate (exact buckets, interpolated rates, the /3 path, DSK buckets) x sample
format x -go options, frames + tags against the compiled reference (live where oracle/_ref was built, else its stored
digests).  The engines run WITHOUT taps, i.e. on the production stream layout (two back-end streams where the chain pipelines), half of the cases without any poll between the submits."""
import numpy as np
import pytest

import aisgpu
import aissynth as S
import golden_util as G
import oracle as O

pytestmark = pytest.mark.gpu

MODELS = [aisgpu.MODEL_STANDARD, aisgpu.MODEL_BASE, aisgpu.MODEL_DEFAULT, aisgpu.MODEL_CHALLENGER, aisgpu.MODEL_V2]
RATES = [96000, 192000, 240000, 288000, 384000, 576000, 768000, 1000000, 1152000, 1536000, 1920000, 2304000, 2400000, 3072000, 6000000, 6144000]
DSK_ONLY = {576000, 1152000, 2304000}


def to_format(x, fmt):
    if fmt == aisgpu.FMT_CF32:
        return x, 1
    if fmt == aisgpu.FMT_CU8:
        return S.to_cu8(x), 2
    if fmt == aisgpu.FMT_CS8:
        return (S.to_cu8(x).astype(np.int16) - 128).astype(np.int8), 2
    v = np.empty(2 * len(x), dtype=np.float32)
    v[0::2], v[1::2] = x.real, x.imag
    return np.clip(np.round(v * 32767.0), -32768, 32767).astype(np.int16), 2


def draw_case(rng):
    model = MODELS[int(rng.integers(0, len(MODELS)))]
    fs = RATES[int(rng.integers(0, len(RATES)))]
    fmt = int(rng.choice([aisgpu.FMT_CF32, aisgpu.FMT_CF32, aisgpu.FMT_CU8, aisgpu.FMT_CS8, aisgpu.FMT_CS16]))
    dsk = fs in DSK_ONLY or bool(rng.integers(0, 4) == 0)
    fp_ds = fs == 1536000 and fmt == aisgpu.FMT_CU8 and bool(rng.integers(0, 2))
    ps_ema = bool(rng.integers(0, 4) != 0) or model == aisgpu.MODEL_CHALLENGER
    afc_wide = bool(rng.integers(0, 4) != 0)
    droop = bool(rng.integers(0, 4) != 0)
    g = aisgpu.chunk_granule(fs, model=model, dsk=dsk, fp_ds=fp_ds, fmt=fmt)
    target = int(fs * float(rng.choice([0.02, 0.043, 0.085])))  # 20 .. 85 ms per submit
    N = max(g, (target // g) * g)
    nchunks = int(rng.integers(3, 7))
    return dict(model=model, fs=fs, fmt=fmt, dsk=dsk, fp_ds=fp_ds, ps_ema=ps_ema, afc_wide=afc_wide, droop=droop, N=N, nchunks=nchunks,
                poll_each=bool(rng.integers(0, 2)), B=int(rng.integers(2, 5)))


@pytest.mark.parametrize("seed", range(36))
def test_random_configuration(built, seed):
    c = draw_case(np.random.default_rng(9000 + seed))
    flags = (O.FLAG_PS_EMA if c["ps_ema"] else 0) | (O.FLAG_AFC_WIDE if c["afc_wide"] else 0) | (O.FLAG_DROOP if c["droop"] else 0)
    flags |= (O.FLAG_DSK if c["dsk"] else 0) | (O.FLAG_FP_DS if c["fp_ds"] else 0)
    N, B = c["N"], c["B"]
    raws = []
    for s in range(B):
        x = S.random_stream(c["fs"], N * c["nchunks"], 9100 + 10 * seed + s, bursts_per_sec=(8, 16))[0]
        raw, per = to_format(x, c["fmt"])
        raws.append(raw)

    def reference():
        refs = [O.RefModel(model=c["model"], sample_rate=c["fs"], fmt=c["fmt"], flags=flags) for _ in range(B)]
        for k in range(c["nchunks"]):
            for s in range(B):
                refs[s].push(raws[s][k * N * per:(k + 1) * N * per])
        return [G.msgs_digest(r.messages()) for r in refs]

    want = G.reference("gpu_matrix %d" % seed, reference)
    eng = aisgpu.Engine(model=c["model"], sample_rate=c["fs"], fmt=c["fmt"], n_streams=B, max_chunk=N, ps_ema=c["ps_ema"], afc_wide=c["afc_wide"],
                        droop=c["droop"], dsk=c["dsk"], fp_ds=c["fp_ds"])
    got = [[] for _ in range(B)]
    for k in range(c["nchunks"]):
        eng.submit(np.stack([r[k * N * per:(k + 1) * N * per] for r in raws]), N)
        if c["poll_each"]:
            for m in eng.poll():
                got[m.stream].append(m)
    for m in eng.poll():
        got[m.stream].append(m)
    assert eng.overflows == 0
    # messages (key, start/end idx) and their tags (level, ppm bit patterns), in order, per stream
    problems = [("MSG", s, len(got[s]), want[s][0]) for s in range(B) if G.msgs_digest(got[s]) != want[s]]
    eng.close()
    assert not problems, "%r: %r" % (c, problems[:6])
