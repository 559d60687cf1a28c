#!/usr/bin/env python
"""bench.py -- IQ MSamples/s through the full two-channel AIS demodulation chain on B200.

Contract: `python bench.py --gpus N --steps K --warmup W` (under torchrun for N>1) prints ONE JSON line on rank 0.
A "step" is one submit of one batch: B streams x N complex samples (BASELINE.json configs[1]: batch=1024 synthetic
CF32 streams @1536 kSPS, FM path = ModelStandard semantics, SURVEY.md 8d "Config 2"), inputs already resident in HBM.
  value     : whole-job complex samples/s (all ranks) with inputs resident in HBM, device-timed on the launch stream:
              the K timed steps run back to back in `--blocks` blocks (default one per 20 steps), the MEDIAN block's
              time per step is the value, min/max go to `spread`, every rank's median to `per_rank_ms`
  e2e       : the same metric through aisgpu_submit_async()/aisgpu_poll_upto() with pinned HOST buffers (H2D and the
              frame D2H inside the timed region); e2e_cu8 = the same with CU8 host input (2 B/sample)
  roofline  : front-end kernel (reads every input byte): 8 B/sample x samples per launch / its CUDA-event duration,
              against MEASURED_PEAKS.json hbm_gbs
  parity    : after the timed region, sampled streams of this rank's slice are re-run through the strict-flags build
              of the unmodified reference (oracle/_ref/libaisref.so) on the exact inputs the engine saw, with the same
              chunking; NMEA sentences, their order and start/end sample counters must be identical
  also      : ModelDefault on the same data, and BASELINE.json configs[2] (batch 4096 @6 MSPS, coherent chain)
  cpu_baseline : the reference's own CPU implementation (oracle/_ref fast build, shipping flags) on this box's cores
`--impl reference` times that CPU implementation alone on the same workload shape (steady state).
`--dump-outputs DIR` writes the frames the timed path delivered in its last step as .npy arrays (see dump_outputs); the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "ais-catcher_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))  # aissynth: the seeded stimulus generator shared with the parity tests

FS = 1536000
N_CHUNK = 131072
BATCH = 1024
RESIDENT = 8
UNIQUE = 32
ALGO_BYTES_PER_SAMPLE = 8  # CF32 in; SURVEY.md 8d


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Exactly ONE line may reach stdout (the JSON result): libraries that print there (NCCL's version banner, ...) are
# diverted to stderr by pointing fd 1 at fd 2 for the lifetime of the process; emit() writes to the saved stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def make_unique_streams(n_unique, n_samples, seed0=0, fs=FS):
    import numpy as np
    import aissynth
    out = np.empty((n_unique, n_samples), dtype=np.complex64)
    for u in range(n_unique):
        out[u] = aissynth.random_stream(fs, n_samples, seed0 + u)[0]
    return out


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def host_cpus():
    try:
        return sorted(os.sched_getaffinity(0))
    except Exception:
        return list(range(os.cpu_count() or 1))


class CpuReference:
    """The reference's CPU implementation of the path in steady state: `n_streams` model instances (one per stream, as the
    reference runs one model per receiver) are created ONCE and spread over one pinned OS thread per host core
    (Device/FileRAW.cpp:205-206: one thread per device); a step = every instance processes one chunk."""

    def __init__(self, uniq, model, n_streams, n_chunk=N_CHUNK, fs=FS):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as O
        fast = O.have_ref(fast=True)
        self.kind = "reference" if fast else "port"
        Model = (lambda **kw: O.RefModel(fast=True, **kw)) if fast else O.PortModel
        omodel = model
        self.cpus = host_cpus()
        self.T = min(len(self.cpus), n_streams)
        self.n_streams = n_streams
        self.n_chunk = n_chunk
        self.uniq = uniq
        self.models = [[] for _ in range(self.T)]
        for s in range(n_streams):
            self.models[s % self.T].append((s, Model(model=omodel, sample_rate=fs)))
        self.go = threading.Barrier(self.T + 1)
        self.done = threading.Barrier(self.T + 1)
        self.chunk = 0
        self.stop = False
        self.threads = [threading.Thread(target=self._work, args=(t,), daemon=True) for t in range(self.T)]
        for th in self.threads:
            th.start()

    def _work(self, t):
        try:
            os.sched_setaffinity(0, {self.cpus[t % len(self.cpus)]})  # pid 0 = the calling thread
        except Exception:
            pass
        nres = self.uniq.shape[1] // self.n_chunk
        while True:
            self.go.wait()
            if self.stop:
                return
            cc = self.chunk % nres
            for s, m in self.models[t]:
                m.push(self.uniq[s % len(self.uniq)][cc * self.n_chunk:(cc + 1) * self.n_chunk])
            self.done.wait()

    def step(self):
        """One chunk through every instance; returns the wall time in seconds."""
        t0 = time.perf_counter()
        self.go.wait()
        self.done.wait()
        dt = time.perf_counter() - t0
        self.chunk += 1
        return dt

    def msg_count(self):
        return sum(m.msg_count() for ms in self.models for _, m in ms)

    def close(self):
        self.stop = True
        self.go.wait()
        for th in self.threads:
            th.join()


def workload_name(args):
    m = {0: "ModelStandard (FM path)", 1: "ModelBase (FM+PLL)", 2: "ModelDefault (coherent PhaseSearchEMA)"}[args.model]
    return "batch=%d synthetic CF32 IQ streams @%d kSPS, %s, chunk %d samples/stream/launch, 1 GPU slice per rank" % (
        args.batch, FS // 1000, m, N_CHUNK)


def config_dict(args, world):
    """Identical for the CUDA arm and the reference arm (the driver compares the two `config` objects key by key)."""
    return {"workload": workload_name(args), "model": args.model, "sample_rate": FS, "batch_per_gpu": args.batch,
            "chunk_samples": N_CHUNK, "resident_chunks": RESIDENT, "bytes_per_step_per_gpu": args.batch * N_CHUNK * 8,
            "l2": "inputs_larger_than_L2 (1.07 GB per step vs 126 MB L2)", "parallelism": "streams sharded, %d rank(s)" % world}


def run_reference_arm(args, rank, world):
    """`--impl reference`: the unmodified reference (oracle/_ref, shipping flags) on the host cores, steady state: the
    batch's model instances are created once, warmed with `--warmup` chunks, then `--steps` chunks are timed."""
    if rank != 0:
        return
    uniq = make_unique_streams(8, N_CHUNK * 2)
    ref = CpuReference(uniq, args.model, args.batch)
    for _ in range(max(1, args.warmup)):
        ref.step()
    dts = [ref.step() for _ in range(args.steps)]
    kind, T = ref.kind, ref.T
    ref.close()
    tot_t = sum(dts)
    samples_per_step = args.batch * N_CHUNK
    v = samples_per_step * len(dts) / tot_t / 1e6
    line = {
        "impl": "reference", "metric": "IQ MSamples/s through full 2-ch demod chain", "value": v, "unit": "MSamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, len(dts)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, args.gpus),
        "cpu_baseline": {"value": v, "unit": "MSamples/s", "cores": T, "kind": kind,
                         "sample": "%d model instances (one per stream) on %d pinned threads, 1 chunk of %d samples each per step, %d timed steps after %d warm-up chunks"
                                   % (args.batch, T, N_CHUNK, len(dts), max(1, args.warmup))},
        "spread": {"min_ms": 1e3 * min(dts), "max_ms": 1e3 * max(dts)},
        "e2e": {"value": v, "unit": "MSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def median(v):
    s = sorted(v)
    return s[len(s) // 2]


def poll_streams(eng, wanted, out, last_chunk=None, last=None):
    """Drains the engine's frame queue; keeps (key, start_idx, end_idx) only for the streams in `wanted` (a set) -- the
    ctypes structs of the other streams are never turned into Python objects -- and, when `last` is a list, every frame
    completed by the submit with ordinal `last_chunk`.  Returns the number of frames drained."""
    import aisgpu
    batch = 8192
    buf = (aisgpu.MsgStruct * batch)()
    n = ctypes.c_int(0)
    total = 0
    while True:
        eng._chk(eng.lib.aisgpu_poll(eng.h, buf, batch, ctypes.byref(n)))
        if n.value == 0:
            break
        total += n.value
        for i in range(n.value):
            if buf[i].stream in wanted:
                m = aisgpu.Msg(buf[i])
                out[m.stream].append((m.key(), m.start_idx, m.end_idx))
            if last is not None and buf[i].chunk == last_chunk:
                last.append(aisgpu.Msg(buf[i]))
    return total


DUMP_LIMIT = 64 << 20


def dump_outputs(path, msgs, n_streams):
    """The frames of one step as the arrays a caller reads out of aisgpu_msg, sorted by (stream, start_idx, end_idx,
    channel): frames.npy float64 [n, 8] = stream, channel (ASCII), nbits, start_idx, end_idx, level, ppm, n_sentences;
    payload.npy float32 [n, 140] = payload bytes; nmea.npy float32 [n, 4, 100] = sentence characters, zero-padded.
    Above 64 MB in all, only the frames of a fixed seeded sample of the streams are written."""
    import numpy as np
    per_frame = 8 * 8 + 140 * 4 + 4 * 100 * 4
    if len(msgs) * per_frame > DUMP_LIMIT:
        count = np.bincount([m.stream for m in msgs], minlength=n_streams)
        keep, size = set(), 0
        for s in np.random.default_rng(0).permutation(n_streams):
            if (size + count[s]) * per_frame > DUMP_LIMIT:
                break
            keep.add(int(s))
            size += count[s]
        msgs = [m for m in msgs if m.stream in keep]
    msgs = sorted(msgs, key=lambda m: (m.stream, m.start_idx, m.end_idx, m.channel, m.nbits, m.payload))
    frames = np.array([[m.stream, ord(m.channel), m.nbits, m.start_idx, m.end_idx, m.level, m.ppm, len(m.nmea)] for m in msgs],
                      dtype=np.float64).reshape(-1, 8)
    payload = np.zeros((len(msgs), 140), dtype=np.float32)
    nmea = np.zeros((len(msgs), 4, 100), dtype=np.float32)
    for i, m in enumerate(msgs):
        payload[i, :len(m.payload)] = np.frombuffer(m.payload, dtype=np.uint8)
        for j, t in enumerate(m.nmea):
            b = t.encode("latin-1")
            nmea[i, j, :len(b)] = np.frombuffer(b, dtype=np.uint8)
    os.makedirs(path, exist_ok=True)
    for name, a in (("frames", frames), ("payload", payload), ("nmea", nmea)):
        np.save(os.path.join(path, name + ".npy"), a)
    return len(msgs)


def oracle_check(streams, fetch_chunk, n_chunks, got, model, fs, fmt=0, ps_ema=True):
    """Runs every sampled stream through the strict-flags reference (or the pinned C port when it was not built) with the
    engine's chunking and compares message lists incl. order and start/end counters.  fetch_chunk(c) -> {stream: array}."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    if not O.have_ref() and model not in (O.MODEL_STANDARD, O.MODEL_BASE, O.MODEL_DEFAULT):
        return {"skipped": "the C port has no model %d: checked against the compiled reference (oracle/_ref) only" % model}
    Model = O.RefModel if O.have_ref() else O.PortModel
    flags = (O.FLAG_PS_EMA if ps_ema else 0) | O.FLAG_AFC_WIDE | O.FLAG_DROOP
    refs = {s: Model(model=model, sample_rate=fs, fmt=fmt, flags=flags) for s in streams}
    want = {s: [] for s in streams}
    cpus = host_cpus()

    def run(sub, chunks):
        for s in sub:
            refs[s].push(chunks[s])

    for c in range(n_chunks):
        chunks = fetch_chunk(c)
        T = min(len(cpus), len(streams))
        ths = [threading.Thread(target=run, args=(streams[t::T], chunks)) for t in range(T)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
    mism, nmsg = 0, 0
    first = None
    for s in streams:
        want[s] = [(m.key(), m.start_idx, m.end_idx) for m in refs[s].messages()]
        nmsg += len(want[s])
        if want[s] != got[s]:
            mism += 1
            if first is None:
                first = {"stream": int(s), "got": len(got[s]), "want": len(want[s])}
    return {"streams_checked": len(streams), "msgs_checked": nmsg, "mismatches": mism, "first_mismatch": first,
            "oracle": "libaisref.so (unmodified reference, strict IEEE flags)" if O.have_ref() else "C port (pinned to the reference)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--model", type=int, default=0, help="0 ModelStandard (FM path, configs[1]), 2 ModelDefault, 1 ModelBase")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--blocks", type=int, default=0,
                    help="the K timed steps run as this many back-to-back blocks (0: one per 20 steps); the median block's ms per step is reported")
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--parity-streams", type=int, default=32)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the ModelDefault / configs[2] side measurements")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frames of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.blocks = min(args.blocks or max(1, args.steps // 20), args.steps)
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import aisgpu
    import shard

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B, N, R = args.batch, N_CHUNK, RESIDENT
    t_gen = time.time()
    uniq = make_unique_streams(UNIQUE, N * R, seed0=1000 * rank)
    log("[rank %d] generated %d unique streams x %d samples in %.1fs" % (rank, UNIQUE, N * R, time.time() - t_gen))
    uniq_pin = torch.from_numpy(uniq.view(np.float32)).pin_memory()
    uniq_dev = torch.view_as_complex(uniq_pin.to(dev, non_blocking=True).view(UNIQUE, N * R, 2))
    # resident input: R chunks of [B][N]; stream b = unique[b % U] + its own AWGN realisation (so all streams differ)
    x = torch.empty((R, B, N), dtype=torch.complex64, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    for b0 in range(0, B, UNIQUE):
        nb = min(UNIQUE, B - b0)
        blk = uniq_dev[:nb].view(nb, R, N).permute(1, 0, 2)
        x[:, b0:b0 + nb, :] = blk
    noise = torch.empty((B, N), dtype=torch.complex64, device=dev)
    for r in range(R):
        torch.view_as_real(noise).normal_(0.0, 0.005, generator=g)
        x[r] += noise
    del noise
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_blocks(eng, xin, n, warmup, steps, blocks, first=0):
        """`steps` submits in `blocks` back-to-back blocks (sizes differ by at most one), each block bracketed by CUDA
        events on the engine's stream (aisgpu_join makes that stream wait for every internal stream).  Returns the
        per-block ms per step, the total ms and the submit count."""
        est = torch.cuda.ExternalStream(eng.cuda_stream(), device=dev)
        nres = xin.shape[0]
        i = first
        for _ in range(warmup):
            eng.submit_device(xin[i % nres].data_ptr(), n, n)
            i += 1
        eng.sync()
        sizes = [steps // blocks + (b < steps % blocks) for b in range(blocks)]
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(blocks + 1)]
        eng.join()
        evs[0].record(est)
        for b in range(blocks):
            for _ in range(sizes[b]):
                eng.submit_device(xin[i % nres].data_ptr(), n, n)
                i += 1
            eng.join()
            evs[b + 1].record(est)
        evs[-1].synchronize()
        ms = [evs[b].elapsed_time(evs[b + 1]) for b in range(blocks)]
        return [t / k for t, k in zip(ms, sizes)], sum(ms), i

    # ---- the timed engine; the sampled streams' frames are kept for the parity check ----
    eng = aisgpu.Engine(model=args.model, sample_rate=FS, n_streams=B, max_chunk=N, device=local_rank, max_frames=1 << 20)
    rng = np.random.default_rng(99 + rank)
    sample_streams = sorted(int(s) for s in rng.choice(B, size=min(args.parity_streams, B), replace=False))
    wanted = set(sample_streams)
    got = {s: [] for s in sample_streams}
    for i in range(args.warmup):
        eng.submit_device(x[i % R].data_ptr(), N, N)
    eng.sync()
    poll_streams(eng, wanted, got)
    c0 = eng.counters()
    sampler = ClockSampler(local_rank)
    if world > 1:  # NCCL set-up (lazy communicator, first-collective kernels) must not bleed into the timed region
        t = torch.ones(1, device=dev)
        dist.all_reduce(t)
    barrier()
    sampler.start()
    blk_ms, tot_ms, n_sub = timed_blocks(eng, x, N, 0, args.steps, args.blocks, first=args.warmup)
    barrier()
    sampler.stop_flag = True
    ms = median(blk_ms)
    launches = eng.last_launches() * args.steps
    fe_times = eng.frontend_times(min(128, args.steps))
    last = [] if args.dump_outputs else None
    n_frames = poll_streams(eng, wanted, got, eng.counters()[3] - 1, last)
    if last is not None:
        n_dumped = dump_outputs(os.path.join(args.dump_outputs, "rank%d" % rank) if world > 1 else args.dump_outputs, last, B)
        log("[rank %d] --dump-outputs: %d of the %d frames of the last timed step written to %s" % (rank, n_dumped, len(last), args.dump_outputs))
    c1 = eng.counters()
    # the only collectives of the job: MAX of the device time, SUM of a few counters (NCCL over NVLink; SURVEY.md 8e)
    ms_max = shard.max_over_ranks(ms, device=dev)
    per_rank = [ms]
    if world > 1:
        t = torch.zeros(world, dtype=torch.float64, device=dev)
        t[rank] = ms
        dist.all_reduce(t)
        per_rank = [float(v) for v in t.tolist()]
    delta = [a - b for a, b in zip(c1, c0)]
    delta[2] = B * N * args.steps  # samples of this rank's slice (the engine counts samples per stream)
    tot = shard.gather_counts(delta, device=dev)
    # the same reduction inside the C library (aisgpu_comm_init / aisgpu_allreduce_counts: NCCL resolved with dlopen, no
    # torch on that path): the counters since engine creation, summed over the ranks -- what a C++ host would call
    c_totals = None
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(aisgpu.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        eng.comm_init(bytes(uid.cpu().numpy().tobytes()), world, rank)
        c_totals = eng.allreduce_counts()
        local_all = shard.gather_counts(c1, device=dev)
        assert c_totals[0] == local_all[0] and c_totals[1] == local_all[1], "C-side NCCL all-reduce disagrees with torch.distributed"
    value = world * B * N / (ms_max * 1e-3) / 1e6
    region_ms = shard.max_over_ranks(tot_ms, device=dev)
    msgs_per_s = float(tot[1]) / (region_ms * 1e-3)

    # ---- parity: the sampled streams through the unmodified reference, same inputs, same chunking ----
    parity = None
    if not args.no_parity:
        idx = torch.tensor(sample_streams, device=dev)

        cache = {}

        def fetch(c):  # the resident chunks cycle with period R: copy each of them back once
            if c % R not in cache:
                blk = x[c % R].index_select(0, idx).cpu().numpy()
                cache[c % R] = {s: blk[j] for j, s in enumerate(sample_streams)}
            return cache[c % R]

        t0 = time.time()
        parity = oracle_check(sample_streams, fetch, n_sub, got, args.model, FS)
        parity["chunks"] = n_sub
        parity["frames_dropped"] = int(c1[4])
        log("[rank %d] parity: %r (%.1fs)" % (rank, parity, time.time() - t0))
        pm = shard.gather_counts([parity["streams_checked"], parity["msgs_checked"], parity["mismatches"], int(c1[4]), 0, 0, 0, 0], device=dev)
        parity.update({"streams_checked": pm[0], "msgs_checked": pm[1], "mismatches": pm[2], "frames_dropped": pm[3]})

    # ---- end to end: pinned host buffers -> aisgpu_submit_async (H2D inside) -> aisgpu_poll_upto (frame D2H inside) ----
    def e2e_run(engine, hosts, n, steps):
        """Double-buffered: the copy + kernels of step c are enqueued, then the frames of step c-1 are drained on the host
        while that copy is in flight.  Every step's input crosses PCIe and every step's frames come back."""
        nfr_total = 0
        t_prev = engine.submit_async_ptr(hosts[0].data_ptr(), n)
        engine.poll_upto_count(t_prev)
        barrier()
        t0 = time.perf_counter()
        prev = None
        for i in range(steps):
            tk = engine.submit_async_ptr(hosts[i & 1].data_ptr(), n)
            if prev is not None:
                nfr_total += engine.poll_upto_count(prev)[0]
            prev = tk
        nfr_total += engine.poll_upto_count(prev)[0]
        torch.cuda.synchronize()
        return time.perf_counter() - t0, nfr_total

    host = [torch.empty((B, N, 2), dtype=torch.float32).pin_memory() for _ in range(2)]
    host[0].copy_(torch.view_as_real(x[0]).cpu())
    host[1].copy_(torch.view_as_real(x[1]).cpu())
    e2e_dt, nfr = e2e_run(eng, host, N, args.e2e_steps)
    e2e_value = world * B * N * args.e2e_steps / shard.max_over_ranks(e2e_dt, device=dev) / 1e6
    d2h = 4 + 184 * nfr // max(1, args.e2e_steps)
    del host
    # the same with CU8 host input (what RTL-SDR class receivers deliver: 2 B per complex sample)
    e2e_cu8 = None
    try:
        eng8 = aisgpu.Engine(model=args.model, sample_rate=FS, fmt=aisgpu.FMT_CU8, n_streams=B, max_chunk=N, device=local_rank, max_frames=1 << 20)
        host8 = []
        for j in range(2):
            q = torch.clamp(torch.round(torch.view_as_real(x[j]) * 127.0 + 128.0), 0, 255).to(torch.uint8)
            host8.append(q.cpu().pin_memory())
            del q
        dt8, nfr8 = e2e_run(eng8, host8, N, args.e2e_steps)
        e2e_cu8 = {"value": world * B * N * args.e2e_steps / shard.max_over_ranks(dt8, device=dev) / 1e6, "unit": "MSamples/s",
                   "h2d_bytes_per_step": B * N * 2, "d2h_bytes_per_step": 4 + 184 * nfr8 // max(1, args.e2e_steps), "steps": args.e2e_steps,
                   "format": "CU8 host input, same streams quantised to 8 bit"}
        eng8.close()
        del host8
    except Exception as e:  # pragma: no cover
        e2e_cu8 = {"error": str(e)}

    # the same kernel timed alone (a sync after every submit), for the record next to the live number
    iso = []
    for i in range(6):
        eng.submit_device(x[i % R].data_ptr(), N, N)
        eng.sync()
        iso.append(eng.last_frontend_ms())
    eng.poll_upto_count(-1)

    # ---- side measurements the driver should record too: ModelDefault, and configs[2] ----
    also = None
    if not args.no_also:
        also = []
        if args.model != 2:
            eng2 = aisgpu.Engine(model=2, sample_rate=FS, n_streams=B, max_chunk=N, device=local_rank, max_frames=1 << 20)
            got2 = {s: [] for s in sample_streams}
            b2, _, n2 = timed_blocks(eng2, x, N, 3, args.steps, max(1, min(3, args.blocks)))
            fe2 = eng2.frontend_times(args.steps)
            nm2 = poll_streams(eng2, wanted, got2)
            par2 = None
            if not args.no_parity:
                par2 = oracle_check(sample_streams[:8], lambda c: {s: x[c % R][s].cpu().numpy() for s in sample_streams[:8]}, n2,
                                    {s: got2[s] for s in sample_streams[:8]}, 2, FS)
            m2 = median(b2)
            also.append({"workload": "same data and batch, ModelDefault (coherent PhaseSearchEMA chain, the reference's default model)",
                         "value": B * N / (m2 * 1e-3) / 1e6, "unit": "MSamples/s (this rank)", "ms_per_step": m2,
                         "whole_chain_frac": ALGO_BYTES_PER_SAMPLE * B * N / (m2 * 1e-3) / 1e9 / peaks()[0],
                         "frontend_ms": sum(fe2) / len(fe2), "frames": nm2, "parity": par2,
                         "blocks_ms_per_step": [round(b, 4) for b in b2]})
            eng2.close()
        # SURVEY.md 8f rank 1: the V2 engine (model 11) on the same data
        engv = aisgpu.Engine(model=aisgpu.MODEL_V2, sample_rate=FS, n_streams=B, max_chunk=N, device=local_rank, max_frames=1 << 20, host_staging=False)
        gotv = {s: [] for s in sample_streams[:8]}
        bv, _, nv = timed_blocks(engv, x, N, 2, 24, 3)
        nmv = poll_streams(engv, set(sample_streams[:8]), gotv)
        parv = None
        if not args.no_parity:
            parv = oracle_check(sample_streams[:8], lambda c: {s: x[c % R][s].cpu().numpy() for s in sample_streams[:8]}, nv, gotv, 11, FS)
        mv = median(bv)
        also.append({"workload": "same data and batch, V2::Engine (model 11)", "value": B * N / (mv * 1e-3) / 1e6, "unit": "MSamples/s (this rank)",
                     "ms_per_step": mv, "frames": nmv, "parity": parv, "blocks_ms_per_step": [round(b, 4) for b in bv]})
        engv.close()
        # SURVEY.md 8f rank 3: ModelChallenger (model 4) on the same data
        engc = aisgpu.Engine(model=aisgpu.MODEL_CHALLENGER, sample_rate=FS, n_streams=B, max_chunk=N, device=local_rank, max_frames=1 << 20, host_staging=False)
        gotc = {s: [] for s in sample_streams[:8]}
        bc, _, nc = timed_blocks(engc, x, N, 2, 36, 3)  # long enough blocks to show the steady state
        nmc = poll_streams(engc, set(sample_streams[:8]), gotc)
        parc = None
        if not args.no_parity:
            parc = oracle_check(sample_streams[:8], lambda c: {s: x[c % R][s].cpu().numpy() for s in sample_streams[:8]}, nc, gotc, 4, FS)
        mc = median(bc)
        also.append({"workload": "same data and batch, ModelChallenger (model 4)", "value": B * N / (mc * 1e-3) / 1e6, "unit": "MSamples/s (this rank)",
                     "ms_per_step": mc, "frames": nmc, "parity": parc, "blocks_ms_per_step": [round(b, 4) for b in bc]})
        engc.close()
        del x
        torch.cuda.empty_cache()
        # BASELINE.json configs[2]: batch 4096 CF32 @6 MSPS (AirSpy shape: 4 CIC stages -> Upsample 125/128 -> 2 CIC stages), coherent chain
        fs3, B3, N3, R3 = 6000000, 4096, 65536, 3
        u3 = make_unique_streams(8, N3 * R3, seed0=5000 + rank, fs=fs3)
        u3d = torch.view_as_complex(torch.from_numpy(u3.view(np.float32)).to(dev).view(8, N3 * R3, 2))
        x3 = torch.empty((R3, B3, N3), dtype=torch.complex64, device=dev)
        for b0 in range(0, B3, 8):
            x3[:, b0:b0 + 8, :] = u3d.view(8, R3, N3).permute(1, 0, 2)
        noise = torch.empty((B3, N3), dtype=torch.complex64, device=dev)
        for r in range(R3):
            torch.view_as_real(noise).normal_(0.0, 0.005, generator=g)
            x3[r] += noise
        del noise
        s3 = sorted(int(s) for s in rng.choice(B3, size=8, replace=False))
        for ps_ema in (True, False):
            eng3 = aisgpu.Engine(model=2, sample_rate=fs3, n_streams=B3, max_chunk=N3, ps_ema=ps_ema, device=local_rank, max_frames=1 << 20)
            got3 = {s: [] for s in s3}
            b3, _, n3 = timed_blocks(eng3, x3, N3, 3, 30, 5)
            nm3 = poll_streams(eng3, set(s3), got3)
            par3 = None
            if not args.no_parity:
                par3 = oracle_check(s3, lambda c: {s: x3[c % R3][s].cpu().numpy() for s in s3}, n3, got3, 2, fs3, ps_ema=ps_ema)
            m3 = median(b3)
            also.append({"workload": "BASELINE configs[2]: batch=4096 CF32 @6 MSPS, ModelDefault, %s, chunk %d" % (
                "PhaseSearchEMA" if ps_ema else "PS_EMA off (Demod::PhaseSearch)", N3),
                "value": B3 * N3 / (m3 * 1e-3) / 1e6, "unit": "MSamples/s (this rank)", "ms_per_step": m3,
                "whole_chain_frac": 8.0 * B3 * N3 / (m3 * 1e-3) / 1e9 / peaks()[0], "frames": nm3, "parity": par3,
                "blocks_ms_per_step": [round(b, 4) for b in b3]})
            eng3.close()
        del x3

    if rank == 0:
        peak, peak_src = peaks()
        fe_ms = sum(fe_times) / max(1, len(fe_times))
        achieved = ALGO_BYTES_PER_SAMPLE * B * N / (fe_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "frontend_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        cpu = None
        if not args.no_cpu:
            ref = CpuReference(uniq, args.model, B)
            for _ in range(2):
                ref.step()
            dts = [ref.step() for _ in range(6)]
            cpu = {"value": B * N * len(dts) / sum(dts) / 1e6, "unit": "MSamples/s", "cores": ref.T, "kind": ref.kind,
                   "sample": "%d model instances on %d pinned threads, %d timed chunks of %d samples each after 2 warm-up chunks (%.1f s wall), %s flags" % (
                       B, ref.T, len(dts), N, sum(dts), "-O3 -ffast-math (reference shipping)" if ref.kind == "reference" else "strict C port")}
            ref.close()
        step_ms = ms_max
        line = {
            "metric": "IQ MSamples/s through full 2-ch demod chain", "value": value, "unit": "MSamples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, world),
            "blocks": args.blocks, "timed_region_ms": region_ms,
            "spread": {"min_ms_per_step": min(blk_ms), "max_ms_per_step": max(blk_ms),
                       "note": "median of %d blocks over %d timed steps (this rank); value uses the max over ranks of the per-rank medians" % (args.blocks, args.steps)},
            "per_rank_ms": per_rank,
            "msgs_per_s": msgs_per_s,
            "counters_allreduce_c": c_totals,
            "parity": parity,
            "e2e": {"value": e2e_value, "unit": "MSamples/s", "h2d_bytes_per_step": B * N * 8,
                    "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
                    "api": "aisgpu_submit_async + aisgpu_poll_upto, two caller-owned pinned buffers"},
            "e2e_cu8": e2e_cu8,
            "gpu_launches": launches,
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "kernel": "k_frontend_st", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "frontend_ms_per_launch": fe_ms, "frontend_share_of_step": fe_ms / step_ms,
                         "isolated_ms_per_launch": min(iso), "isolated_frac": ALGO_BYTES_PER_SAMPLE * B * N / (min(iso) * 1e-3) / 1e9 / peak,
                         "note": "achieved = 8 B/sample x samples per launch / live CUDA-event duration of the front-end kernel (mean of the last %d launches of the timed region) while the back end of the previous submit shares the GPU; isolated_* = the same launch alone" % len(fe_times),
                         "whole_chain_frac": ALGO_BYTES_PER_SAMPLE * B * N / (step_ms * 1e-3) / 1e9 / peak},
            "cpu_baseline": cpu,
        }
        if also:
            line["also"] = also
        emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
