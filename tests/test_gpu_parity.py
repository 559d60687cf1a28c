"""-m gpu parity tests: the CUDA path (through the C ABI) against the oracle, bit for bit.

Oracle = oracle/_ref/libaisref.so (the unmodified reference, strict IEEE flags) when it was built, else the
pinned C restatement oracle/libaisoracle.so; where the C restatement does not cover a case (-go DSK / FP_DS, the V2 and
Challenger models), the reference's results stored in tests/golden/ref_results.json.  Integer/byte outputs (frames, NMEA) and -- because every kernel
replays the reference's operation order -- all float taps are required to be BIT-IDENTICAL (tolerance 0);
the north_star tolerance for floats (1e-5 rel) is therefore met with margin.
"""
import numpy as np
import pytest

import aisgpu
import aissynth as S
import golden_util as G
import oracle as O

pytestmark = pytest.mark.gpu


def oracle_model(**kw):
    return (O.RefModel if O.have_ref() else O.PortModel)(**kw)


def bits_equal(a, b):
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def first_diff(a, b):
    n = min(len(a), len(b))
    av = a[:n].view(np.uint32).reshape(n, -1)
    bv = b[:n].view(np.uint32).reshape(n, -1)
    d = np.nonzero((av != bv).any(axis=1))[0]
    return (int(d[0]), int(len(d))) if len(d) else (-1, 0)


def tap_table(model):
    """(name, engine tap, oracle tap) for every tap compared per stream and channel."""
    t = [("C", lambda e, s, ch: e.tap(aisgpu.TAP_C, s, ch), lambda r, ch: r.tap_c(O.TAP_CA + ch))]
    if model == aisgpu.MODEL_DEFAULT:
        t += [("CGF", lambda e, s, ch: e.tap(aisgpu.TAP_CGF, s, ch), lambda r, ch: r.tap_c(O.TAP_CGF_A + ch)),
              ("FIR17", lambda e, s, ch: e.tap(aisgpu.TAP_FIR, s, ch), lambda r, ch: r.tap_c(O.TAP_FC_A + ch))]
    else:
        t += [("FM", lambda e, s, ch: e.tap(aisgpu.TAP_FM, s, ch, dtype=np.float32), lambda r, ch: r.tap_f(O.TAP_FM_A + ch)),
              ("FIR37", lambda e, s, ch: e.tap(aisgpu.TAP_FIR, s, ch, dtype=np.float32), lambda r, ch: r.tap_f(O.TAP_FR_A + ch))]
    for ph in range(1 if model == aisgpu.MODEL_BASE else 5):
        t.append(("DEC%d" % ph, lambda e, s, ch, ph=ph: e.tap(aisgpu.TAP_DEC, s, ch + 2 * ph, dtype=np.float32), lambda r, ch, ph=ph: r.tap_f(ch * 5 + ph)))
    return t


def run_case(built, model, fs, N, nchunks, B, ps_ema=True, afc_wide=True, droop=True, fmt=aisgpu.FMT_CF32, check_taps=True, seed0=0, dsk=False,
             fp_ds=False):
    xs = [S.random_stream(fs, N * nchunks, seed0 + s)[0] for s in range(B)]
    if fmt == aisgpu.FMT_CU8:
        raw = [S.to_cu8(x) for x in xs]
        per = 2
    elif fmt == aisgpu.FMT_CS8:
        raw = [(S.to_cu8(x).astype(np.int16) - 128).astype(np.int8) for x in xs]
        per = 2
    elif fmt == aisgpu.FMT_CS16:
        raw = []
        for x in xs:
            v = np.empty(2 * len(x), dtype=np.float32)
            v[0::2], v[1::2] = x.real, x.imag
            raw.append(np.clip(np.round(v * 32767.0), -32768, 32767).astype(np.int16))
        per = 2
    else:
        raw = xs
        per = 1
    flags = (O.FLAG_PS_EMA if ps_ema else 0) | (O.FLAG_AFC_WIDE if afc_wide else 0) | (O.FLAG_DROOP if droop else 0)
    flags |= (O.FLAG_DSK if dsk else 0) | (O.FLAG_FP_DS if fp_ds else 0)
    taps = tap_table(model) if check_taps else []

    def oracle_side(Model):
        """Digests of every tap (per stream, channel; per-submit block lengths included) and of every stream's messages."""
        refs = [Model(model=model, sample_rate=fs, fmt=fmt, flags=flags, taps=True) for _ in range(B)]
        d = {"%s %d %d" % (t[0], s, ch): G.Digest() for t in taps for s in range(B) for ch in range(2)}
        msgs = [[] for _ in range(B)]
        for c in range(nchunks):
            for s in range(B):
                refs[s].push(raw[s][c * N * per:(c + 1) * N * per])
                for ch in range(2):
                    for name, _, ref_tap in taps:
                        d["%s %d %d" % (name, s, ch)].add(ref_tap(refs[s], ch))
                msgs[s] += refs[s].messages()
        return {"taps": {k: v.value() for k, v in d.items()}, "messages": [G.msgs_digest(m) for m in msgs]}

    if dsk or fp_ds:  # the C port has no -go DSK / FP_DS: the reference, or its stored digests
        want = G.reference("parity %r" % ((model, fs, N, nchunks, B, ps_ema, afc_wide, droop, fmt, check_taps, seed0, dsk, fp_ds),),
                           lambda: oracle_side(O.RefModel))
    else:
        want = oracle_side(oracle_model)
    eng = aisgpu.Engine(model=model, sample_rate=fs, fmt=fmt, n_streams=B, max_chunk=N, ps_ema=ps_ema, afc_wide=afc_wide,
                        droop=droop, taps=check_taps, dsk=dsk, fp_ds=fp_ds)
    d = {k: G.Digest() for k in want["taps"]}
    got_msgs = [[] for _ in range(B)]
    for c in range(nchunks):
        batch = np.stack([r[c * N * per:(c + 1) * N * per] for r in raw])
        eng.submit(batch, N)
        for s in range(B):
            for ch in range(2):
                for name, eng_tap, _ in taps:
                    d["%s %d %d" % (name, s, ch)].add(eng_tap(eng, s, ch))
        for m in eng.poll():
            got_msgs[m.stream].append(m)
    eng.close()
    # taps bit for bit; messages (key, start/end idx) and tags (level, ppm bit patterns) in order, per stream
    problems = [(k, d[k].value()[0], want["taps"][k][0]) for k in d if d[k].value() != want["taps"][k]]
    problems += [("MSG", s, len(got_msgs[s]), want["messages"][s][0]) for s in range(B) if G.msgs_digest(got_msgs[s]) != want["messages"][s]]
    assert not problems, "parity problems (first 12): %r" % (problems[:12],)
    return sum(w[0] for w in want["messages"])


def test_default_1536k(built):
    n = run_case(built, aisgpu.MODEL_DEFAULT, 1536000, 65536, 4, 3)
    assert n >= 6


def test_standard_1536k(built):
    n = run_case(built, aisgpu.MODEL_STANDARD, 1536000, 65536, 4, 3)
    assert n >= 6


def test_base_1536k(built):
    run_case(built, aisgpu.MODEL_BASE, 1536000, 65536, 4, 3)


def test_default_small_chunks(built):
    # chunks smaller than a CGF block (48 kHz count 128 < 512): exercises the unconsumed-sample carry
    n = run_case(built, aisgpu.MODEL_DEFAULT, 1536000, 4096, 48, 2, seed0=7)
    assert n >= 1


def test_standard_small_chunks(built):
    run_case(built, aisgpu.MODEL_STANDARD, 1536000, 4096, 48, 2, seed0=7)


def test_default_phasesearch(built):
    n = run_case(built, aisgpu.MODEL_DEFAULT, 1536000, 32768, 8, 2, ps_ema=False, seed0=11)
    assert n >= 4


def test_default_narrow_nodroop(built):
    run_case(built, aisgpu.MODEL_DEFAULT, 1536000, 32768, 8, 2, afc_wide=False, droop=False, seed0=13)


def test_default_cu8(built):
    n = run_case(built, aisgpu.MODEL_DEFAULT, 1536000, 65536, 4, 2, fmt=aisgpu.FMT_CU8, seed0=17)
    assert n >= 4


@pytest.mark.parametrize("fs,N", [(96000, 4096), (192000, 8192), (384000, 16384), (768000, 32768), (3072000, 131072),
                                  (6144000, 262144), (12288000, 524288)])
def test_default_rates(built, fs, N):
    n = run_case(built, aisgpu.MODEL_DEFAULT, fs, N, 4, 2, seed0=23)
    assert n >= 2


@pytest.mark.parametrize("fs,N,model", [(288000, 12288, aisgpu.MODEL_DEFAULT), (288000, 49152, aisgpu.MODEL_STANDARD),
                                        (6000000, 262144, aisgpu.MODEL_DEFAULT), (6000000, 65536, aisgpu.MODEL_STANDARD),
                                        (2000000, 65536, aisgpu.MODEL_DEFAULT), (250000, 16384, aisgpu.MODEL_DEFAULT), (300000, 16384, aisgpu.MODEL_DEFAULT),
                                        (1000000, 32768, aisgpu.MODEL_BASE)])
def test_resampled_rates(built, fs, N, model):
    # DownsampleKFilter (/3, 288 kS/s) and Upsample (non-bucket rates; 6 MSPS is the AirSpy shape of BASELINE configs[2]).
    # The reference re-blocks behind the resampler, so per-submit taps do not line up; frames are compared bit for bit.
    n = run_case(built, model, fs, N, 6, 2, check_taps=False, seed0=29)
    assert n >= 2
    if O.have_ref():
        resampler_taps(fs, N, 6, model)


def resampler_taps(fs, N, nchunks, model, dsk=False):
    """The resampler outputs themselves (DSP::Upsample, DownsampleKFilter) against taps on the reference's US.out / DSK.out:
    the sample streams must be bit-identical (the reference emits whole blocks, so the common prefix is compared)."""
    x = S.random_stream(fs, N * nchunks, 91)[0]
    eng = aisgpu.Engine(model=model, sample_rate=fs, n_streams=1, max_chunk=N, taps=True, dsk=dsk)
    ref = O.RefModel(model=model, sample_rate=fs, flags=O.DEFAULT_FLAGS | (O.FLAG_DSK if dsk else 0), taps=True)
    got = {aisgpu.TAP_PRE: [], aisgpu.TAP_PRE2: []}
    want = {O.TAP_US: [], O.TAP_DSK: []}
    for c in range(nchunks):
        eng.submit(x[None, c * N:(c + 1) * N], N)
        ref.push(x[c * N:(c + 1) * N])
        for t in got:
            try:
                got[t].append(eng.tap(t))
            except aisgpu.AisGpuError:
                pass
        for t in want:
            want[t].append(ref.tap_c(t))
    eng.close()
    us, dsk_ = np.concatenate(want[O.TAP_US]), np.concatenate(want[O.TAP_DSK])
    pre = np.concatenate(got[aisgpu.TAP_PRE]) if got[aisgpu.TAP_PRE] else np.zeros(0, np.complex64)
    pre2 = np.concatenate(got[aisgpu.TAP_PRE2]) if got[aisgpu.TAP_PRE2] else np.zeros(0, np.complex64)
    pairs = []
    if len(us) and len(dsk_):
        pairs = [("US", pre, us), ("DSK", pre2, dsk_)]
    elif len(us):
        pairs = [("US", pre, us)]
    elif len(dsk_):
        pairs = [("DSK", pre, dsk_)]
    assert pairs, "no resampler at this rate"
    for name, g, w in pairs:
        n = min(len(g), len(w))
        assert n > 1000 and bits_equal(g[:n], w[:n]), "%s output differs: %r" % (name, first_diff(g[:n], w[:n]))


def test_resampled_cu8(built):
    n = run_case(built, aisgpu.MODEL_DEFAULT, 6000000, 262144, 3, 2, fmt=aisgpu.FMT_CU8, check_taps=False, seed0=31)
    assert n >= 2


@pytest.mark.parametrize("model", [aisgpu.MODEL_DEFAULT, aisgpu.MODEL_STANDARD])
def test_pipelined_backend(built, model):
    # without taps the back-end stages of consecutive submits overlap on two streams (per-stage events, double-buffered
    # hand-off buffers): many short submits, frames only
    n = run_case(built, model, 1536000, 32768, 16, 4, check_taps=False, seed0=41)
    assert n >= 8


def test_pipelined_backend_tiny_chunks(built):
    # chunks below one CGF block: several submits share a 512-block, Ec / Cbuf leftovers hop between the streams
    run_case(built, aisgpu.MODEL_DEFAULT, 1536000, 4096, 64, 2, check_taps=False, seed0=43)


@pytest.mark.parametrize("fmt", [aisgpu.FMT_CS8, aisgpu.FMT_CS16])
@pytest.mark.parametrize("fs,N", [(1536000, 65536), (384000, 16384)])
def test_signed_integer_formats(built, fmt, fs, N):
    # Convert::toFloat(CS8) / (CS16) (reference Utilities/Convert.cpp:266-286) through the streaming (1536k) and the tiled
    # (384k) front end
    n = run_case(built, aisgpu.MODEL_DEFAULT, fs, N, 3, 2, fmt=fmt, seed0=37)
    assert n >= 2


@pytest.mark.parametrize("fs,N,model", [(576000, 24576, aisgpu.MODEL_DEFAULT), (1152000, 49152, aisgpu.MODEL_STANDARD), (2304000, 98304, aisgpu.MODEL_DEFAULT),
                                        (500000, 16384, aisgpu.MODEL_DEFAULT), (1000000, 32768, aisgpu.MODEL_DEFAULT), (2000000, 65536, aisgpu.MODEL_STANDARD),
                                        (288000, 12288, aisgpu.MODEL_DEFAULT), (1536000, 65536, aisgpu.MODEL_DEFAULT)])
def test_dsk_buckets(built, fs, N, model):
    # -go DSK on (reference Model.cpp:130, 208-218, 248-258, 278-288): the 576K / 1152K / 2304K buckets = CIC stages ->
    # DownsampleKFilter /3, exact and interpolated (CIC -> Upsample -> /3); rates outside those buckets keep their chain
    n = run_case(built, model, fs, N, 6, 2, check_taps=False, seed0=51, dsk=True)
    assert n >= 2
    if fs != 1536000 and O.have_ref():
        resampler_taps(fs, N, 6, model, dsk=True)


def test_dsk_cu8(built):
    n = run_case(built, aisgpu.MODEL_DEFAULT, 1152000, 49152, 4, 2, fmt=aisgpu.FMT_CU8, check_taps=False, seed0=53, dsk=True)
    assert n >= 2


@pytest.mark.parametrize("model", [aisgpu.MODEL_DEFAULT, aisgpu.MODEL_STANDARD])
def test_fp_ds_integer_frontend(built, model):
    # -go FP_DS on (Model.cpp:233-236; DSP.cpp:499-665): CU8 @1536K through four packed-uint16 CIC stages; the 48 kHz taps and
    # everything behind them are compared bit for bit
    n = run_case(built, model, 1536000, 65536, 4, 3, fmt=aisgpu.FMT_CU8, seed0=57, fp_ds=True)
    assert n >= 4


def test_fp_ds_small_blocks(built):
    # the shortest block the integer front end takes (32 lane sub-segments of 512 samples)
    run_case(built, aisgpu.MODEL_DEFAULT, 1536000, 16384, 12, 2, fmt=aisgpu.FMT_CU8, seed0=59, fp_ds=True)


def test_fp_ds_needs_cu8(built):
    with pytest.raises(aisgpu.AisGpuError, match="needs CU8"):
        aisgpu.Engine(sample_rate=1536000, fmt=aisgpu.FMT_CF32, fp_ds=True)


def run_v2_case(fs, N, nchunks, B, check_taps, seed0, fmt=aisgpu.FMT_CF32):
    """Model 11 "v2_base" (reference DSP/Decoder/V2/V2Engine.cpp, Model.cpp:440-460) against the compiled reference
    (its stored digests where oracle/_ref was not built)."""
    xs = [S.random_stream(fs, N * nchunks, seed0 + s, bursts_per_sec=(6, 12))[0] for s in range(B)]
    per = 1
    if fmt == aisgpu.FMT_CU8:
        xs = [S.to_cu8(x) for x in xs]
        per = 2
    N_el = N * per  # array elements per chunk
    names = ("V2.CGF", "V2.FIR17", "V2.FIR37")

    def reference():
        refs = [O.RefModel(model=O.MODEL_V2, sample_rate=fs, fmt=fmt, taps=check_taps) for _ in range(B)]
        taps = {"%s %d %d" % (n, s, ch): G.Digest() for n in names for s in range(B) for ch in range(2)}
        want = [[] for _ in range(B)]
        for c in range(nchunks):
            for s in range(B):
                refs[s].push(xs[s][c * N_el:(c + 1) * N_el])
                if check_taps:
                    for ch in range(2):
                        for n, w in zip(names, (refs[s].tap_c(O.TAP_CGF_A + ch), refs[s].tap_c(O.TAP_FC_A + ch), refs[s].tap_f(O.TAP_FR_A + ch))):
                            taps["%s %d %d" % (n, s, ch)].add(w)
                want[s] += refs[s].messages()
        return {"taps": {k: d.value() for k, d in taps.items()} if check_taps else {}, "messages": [G.msgs_digest(w) for w in want]}

    want = G.reference("v2 %r" % ((fs, N, nchunks, B, check_taps, seed0, fmt),), reference)
    eng = aisgpu.Engine(model=aisgpu.MODEL_V2, sample_rate=fs, fmt=fmt, n_streams=B, max_chunk=N, taps=check_taps)
    taps = {k: G.Digest() for k in want["taps"]}
    got = [[] for _ in range(B)]
    for c in range(nchunks):
        eng.submit(np.stack([x[c * N_el:(c + 1) * N_el] for x in xs]), N)
        if check_taps:
            for s in range(B):
                for ch in range(2):
                    for n, g in zip(names, (eng.tap(aisgpu.TAP_CGF, s, ch), eng.tap(aisgpu.TAP_FIR, s, ch), eng.tap(aisgpu.TAP_FM, s, ch, dtype=np.float32))):
                        taps["%s %d %d" % (n, s, ch)].add(g)
        for m in eng.poll():
            got[m.stream].append(m)
    eng.close()
    # every block's taps bit for bit; messages (key, start/end idx) and tags (level, ppm bit patterns) in order, per stream
    problems = [k for k in taps if taps[k].value() != want["taps"][k]]
    problems += [("MSG", s, len(got[s]), want["messages"][s][0]) for s in range(B) if G.msgs_digest(got[s]) != want["messages"][s]]
    assert not problems, "parity problems (first 12): %r" % (problems[:12],)
    return sum(w[0] for w in want["messages"])


def test_v2_engine_blockwise_taps(built):
    # one 512-sample block per submit: every block's derotated samples, FIR17 and FIR37 outputs are compared bit for bit
    n = run_v2_case(1536000, 16384, 40, 2, True, 61)
    assert n >= 4


@pytest.mark.parametrize("fs,N", [(1536000, 65536), (1536000, 36864), (384000, 16384), (6144000, 262144)])
def test_v2_engine_messages(built, fs, N):
    # several blocks per submit (and submits that are not whole blocks: 36864 / 32 = 1152 samples at 48 kHz)
    n = run_v2_case(fs, N, 8, 3, False, 67)
    assert n >= 6


def test_v2_engine_cu8(built):
    n = run_v2_case(1536000, 65536, 16, 2, False, 71, fmt=aisgpu.FMT_CU8)
    assert n >= 8


def run_msg_case(model, fs, N, nchunks, B, seed0, fmt=aisgpu.FMT_CF32, bursts=(6, 12)):
    """Frames + tags of a model the oracle has no taps for, against the compiled reference (its stored digests where
    oracle/_ref was not built)."""
    xs = [S.random_stream(fs, N * nchunks, seed0 + s, bursts_per_sec=bursts)[0] for s in range(B)]

    def reference():
        refs = [O.RefModel(model=model, sample_rate=fs, fmt=fmt) for _ in range(B)]
        want = [[] for _ in range(B)]
        for c in range(nchunks):
            for s in range(B):
                refs[s].push(xs[s][c * N:(c + 1) * N])
                want[s] += refs[s].messages()
        return [G.msgs_digest(w) for w in want]

    want = G.reference("msgs %r" % ((model, fs, N, nchunks, B, seed0, fmt, bursts),), reference)
    eng = aisgpu.Engine(model=model, sample_rate=fs, fmt=fmt, n_streams=B, max_chunk=N)
    got = [[] for _ in range(B)]
    for c in range(nchunks):
        eng.submit(np.stack([x[c * N:(c + 1) * N] for x in xs]), N)
        for m in eng.poll():
            got[m.stream].append(m)
    eng.close()
    # messages (key, start/end idx) and tags (level, ppm bit patterns) in order, per stream
    problems = [("MSG", s, len(got[s]), want[s][0]) for s in range(B) if G.msgs_digest(got[s]) != want[s]]
    assert not problems, "parity problems (first 12): %r" % (problems[:12],)
    return sum(w[0] for w in want)


@pytest.mark.parametrize("fs,N", [(1536000, 65536), (1536000, 16384), (1536000, 4096), (384000, 16384), (3072000, 131072)])
def test_challenger(built, fs, N):
    # model 4 "v1_high" (Model.cpp:601-678): coherent and FM decoders side by side behind one CGF, ten cross-reset decoders per channel
    n = run_msg_case(aisgpu.MODEL_CHALLENGER, fs, N, 8 if N >= 16384 else 64, 3, 81)
    assert n >= 4


def test_challenger_dense(built):
    # many overlapping / back-to-back bursts: frames complete in both branches close together, the Reset crosses branches
    xs = [S.fuzz_stream(96000, 262144, 300 + s)[0] for s in range(6)]
    want = G.reference("challenger_dense", lambda: [G.msgs_digest(O.RefModel(model=O.MODEL_CHALLENGER, sample_rate=96000).run(x, 8192).messages())
                                                    for x in xs])
    eng = aisgpu.Engine(model=aisgpu.MODEL_CHALLENGER, sample_rate=96000, n_streams=6, max_chunk=8192)
    got = [[] for _ in range(6)]
    for c in range(32):
        eng.submit(np.stack([x[c * 8192:(c + 1) * 8192] for x in xs]), 8192)
    for m in eng.poll():
        got[m.stream].append(m)
    for s in range(6):
        assert G.msgs_digest(got[s]) == want[s], "stream %d" % s
    eng.close()


@pytest.mark.parametrize("amp,exact", [(0.0, True), (1e-30, True), (3e-39, False)])
def test_tiny_and_zero_inputs(built, amp, exact):
    """All-zero and tiny inputs through the front end.  Zero and small NORMAL values are bit-exact.  With SUBNORMAL values the
    streaming kernel is allowed a deviation: ptxas contracts the exact x 1/32 scaling of a CIC stage with the next stage's
    first add into one FFMA2, which rounds once where the reference rounds twice -- identical for normal numbers (a power-of-two
    scaling is exact), not when the scaled value is subnormal.  Bounded here to a few denormal ulps (1.4e-45); no SDR delivers
    such samples (CU8/CS16 inputs have 8/16-bit granularity)."""
    fs, N, B = 1536000, 65536, 2
    rng = np.random.default_rng(5)
    xs = [((rng.standard_normal(N * 2) + 1j * rng.standard_normal(N * 2)) * amp).astype(np.complex64) for _ in range(B)]
    eng = aisgpu.Engine(model=aisgpu.MODEL_DEFAULT, sample_rate=fs, n_streams=B, max_chunk=N, taps=True)
    refs = [oracle_model(model=aisgpu.MODEL_DEFAULT, sample_rate=fs, taps=True) for _ in range(B)]
    for c in range(2):
        eng.submit(np.stack([x[c * N:(c + 1) * N] for x in xs]), N)
        for s in range(B):
            refs[s].push(xs[s][c * N:(c + 1) * N])
            for ch in range(2):
                w = refs[s].tap_c(O.TAP_CA + ch)
                g = eng.tap(aisgpu.TAP_C, s, ch)
                if exact:
                    assert bits_equal(g, w), (amp, c, s, ch, first_diff(g, w))
                else:
                    assert len(g) == len(w) and np.max(np.abs(g - w)) <= 8 * 1.4e-45, (amp, float(np.max(np.abs(g - w))))
    eng.close()


@pytest.mark.parametrize("lanes", ["0", "1", "3", "7", "18", "33", "100"])
def test_streaming_frontend_lane_split(built, monkeypatch, lanes):
    """The streaming front end splits a stream's super-steps over L lanes, L not dividing the block (uneven q / q + 1 split,
    warps spanning streams, spare lanes in the last warp): AISGPU_ST_L forces L, "0" lets the launcher plan it.
    N = 64 * 1017 has no power-of-two lane split at all."""
    monkeypatch.setenv("AISGPU_ST_L", lanes)
    n = run_case(built, aisgpu.MODEL_STANDARD, 1536000, 64 * 1017, 4, 5, seed0=41)
    assert n >= 6


@pytest.mark.parametrize("fmt,fs,N", [(aisgpu.FMT_CU8, 1536000, 64 * 1017), (aisgpu.FMT_CS16, 768000, 32 * 999), (aisgpu.FMT_CF32, 3072000, 128 * 613)])
def test_streaming_frontend_lane_split_formats(built, monkeypatch, fmt, fs, N):
    for lanes in ("5", "19"):
        monkeypatch.setenv("AISGPU_ST_L", lanes)
        run_case(built, aisgpu.MODEL_DEFAULT, fs, N, 3, 3, fmt=fmt, seed0=43)
