"""SURVEY.md 8f rank 4 (egress): aisgpu_msg_json / aisgpu_msg_binary against the reference's own Message::getNMEAJSON /
getBinaryNMEA (oracle/_ref, ref_harness.cpp aisref_format; stored as a digest in tests/golden/ref_results.json) on the same
message fields.  Host-only formatters: no GPU needed."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ais-catcher_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import aisgpu  # noqa: E402
import golden_util as G  # noqa: E402
import oracle  # noqa: E402

needs_lib = pytest.mark.skipif(not os.path.exists(aisgpu.LIB_PATH), reason="libaisgpu.so not built")

HARDWARE = ["", "RTL2838UHIDIR", 'quo"te\\back', "tab\there\nnl", "ctl\x01\x1f", "caf\xe9"]


def random_fields(rng):
    nbits = int(rng.choice([0, 38, 72, 168, 168, 168, 256, 424, 1064, 1064]))
    payload = bytes(rng.integers(0, 256, (nbits + 7) // 8, dtype=np.uint8))
    if rng.random() < 0.3 and payload:  # plenty of bytes the binary framing has to escape
        b = bytearray(payload)
        for i in rng.integers(0, len(b), 6):
            b[i] = int(rng.choice([0x0a, 0x0d, 0xad]))
        payload = bytes(b)
    f32 = lambda lo, hi: float(np.float32(rng.uniform(lo, hi)))
    return dict(
        payload=payload, nbits=nbits, channel=str(rng.choice(list("AB12"))), station=int(rng.choice([0, 0, 7, 12345])),
        start_idx=int(rng.integers(0, 1 << 40)), end_idx=int(rng.integers(0, 1 << 40)),
        rxtime_us=int(rng.choice([0, 1758600000000000, int(rng.integers(1, 1 << 52)), 1758600000500000, 2573 * 1000000 + 0x0a0d00ad])),
        toa_us=int(rng.choice([0, 0, 1758600000000000, int(rng.integers(1, 1 << 50))])),
        level=float(rng.choice([1024.0, 0.0, -0.5, f32(-90, 10), f32(-90, 10), -12.3456785, 2.5e-7, 1.0000005])),
        ppm=float(rng.choice([1024.0, 0.0, f32(-60, 60), f32(-60, 60), 12.75, -12.85])),
        version=int(rng.choice([0, 163, 70])), driver=int(rng.integers(0, 20)), hardware=str(rng.choice(HARDWARE)),
        mode=int(rng.integers(0, 4)), status=int(rng.choice([0, 0, 1, 6])), ipv4=int(rng.choice([0, 0, 0xC0A80001, 0xFFFFFFFF])),
        uuid=str(rng.choice(["", "9c0b1e5e-0000-4d6f-8a55-1f2a3b4c5d6e"])), include_ssl=bool(rng.integers(0, 2)),
        suffix=[None, "\r\n", "\n"][int(rng.integers(0, 3))])


def product(kind, f, sentences):
    m = aisgpu.make_msg(f["payload"], f["nbits"], f["channel"], f["start_idx"], f["end_idx"], f["level"], f["ppm"], sentences)
    t = aisgpu.make_tag(f["version"], f["driver"], f["hardware"], f["mode"], f["status"], f["ipv4"], f["rxtime_us"], f["toa_us"],
                        f["station"], f["include_ssl"], f["uuid"] or None, f["suffix"])
    return aisgpu.msg_json(m, t) if kind == 0 else aisgpu.msg_binary(m, t, kind == 2)


def restart_reference_seq():
    """The reference numbers multi-sentence messages with a process-global id (0-9, Message.cpp:28-39), so what it formats
    depends on how many such messages the process formatted before.  Advance that id until the next one is 0."""
    payload = bytes(53)  # 424 bits: two sentences
    q = int(oracle.ref_format(0, payload, 424)[1][0].split(b",")[3])
    for _ in range(9 - q):
        oracle.ref_format(0, payload, 424)


def reference_outputs(kind):
    """A digest of the reference's formatter outputs over the seeded field sets, its sequence ids starting at 0."""
    restart_reference_seq()
    rng = np.random.default_rng(4100 + kind)
    d = G.Digest()
    for it in range(1500):
        f = random_fields(rng)
        kw = {k: v for k, v in f.items() if k not in ("payload", "nbits")}
        d.add(oracle.ref_format(kind, f["payload"], f["nbits"], **kw)[0], 1)
    return d.value()


@needs_lib
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_egress_matches_reference(kind):
    """The product's NMEA builder (sequence ids from 0, chained like the reference's counter) and formatters on the same
    field sets give byte for byte what the reference gives."""
    want = G.reference("egress %d" % kind, lambda: reference_outputs(kind))
    rng = np.random.default_rng(4100 + kind)
    d, seq = G.Digest(), 0
    for it in range(1500):
        f = random_fields(rng)
        sentences, seq = aisgpu.build_nmea(f["payload"], f["nbits"], f["channel"], seq=seq)
        d.add(product(kind, f, sentences), 1)
    assert d.value() == want


@needs_lib
def test_egress_known_line_and_errors():
    # SAMPLE_A of the reference's python tests (python/tests/test_decode.py:12): type 1, mmsi 366730000
    sent = "!AIVDM,1,1,,A,15MgK45P3@G?fl0E`JbR0OwT0@MS,0*4E"
    bits = "".join(format((ord(c) - 48 - (8 if ord(c) - 48 > 40 else 0)) & 63, "06b") for c in sent.split(",")[5])
    payload = int(bits, 2).to_bytes(len(bits) // 8, "big")
    m = aisgpu.make_msg(payload, 168, "A", 100, 1380, -20.5, 1.25, [sent])
    t = aisgpu.make_tag(version=163, driver=1, hardware="bench", mode=1, station=3, include_ssl=True)
    line = aisgpu.msg_json(m, t).decode()
    assert line == ('{"class":"AIS","device":"AIS-catcher","version":163,"driver":1,"hardware":"bench","channel":"A","repeat":0,'
                    '"ssc":100,"sl":1280,"signalpower":-20.5,"ppm":1.25,"station_id":3,"mmsi":366730000,"type":1,"nmea":["%s"]}' % sent)
    b = aisgpu.msg_binary(m, t, True)
    assert b[:2] == b"\xac\x00" and b[2] == 3 and b[-1:] == b"\n"
    with pytest.raises(aisgpu.AisGpuError):  # AISGPU_EOVERFLOW: the caller's buffer is too small
        aisgpu.msg_json(m, t, cap=40)
    with pytest.raises(aisgpu.AisGpuError):
        aisgpu.msg_binary(m, t, True, cap=10)
