#!/usr/bin/env python
"""bench.py -- throughput of the analyzer hot path (main PSD + FFT channeliser + inspectors).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the CPU restatement on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

Workload (BASELINE.json configs[1], "cfg2"): complex64 IQ at a nominal 100 MS/s, 65536-point
Blackman-Harris main spectrum over every frame + one QPSK inspector (1 MBd, RRC 0.35, Costas + Gardner,
3 MHz channel at +12.5 MHz -> 2048-point IFFT, decimation 32).  `--workload cfg3` selects the 64-inspector
mix of configs[2].  One "step" = one pass over a batch of `streams` independent IQ streams of
`hops * 32768` samples each (the serial carrier/clock loops bound a single stream, so the engine batches
independent sources; config.streams says how many).  Metric: complex MSamples/s ingested, whole job.

Prints ONE JSON line (see README / DESIGN.md section "Measurement").
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree (it may be read-only)

N_FFT = 65536
FS_BY = {"cfg2": 100e6, "cfg3": 200e6, "cfg4": 50e6, "cfg5": 100e6}
NFFT_BY = {"cfg2": 65536, "cfg3": 65536, "cfg4": 32768, "cfg5": 65536}
FS = 100e6     # replaced per workload in main()
B_ALG = {"cfg2": 12.09, "cfg3": 14.41, "cfg4": 12.06, "cfg5": 12.0}     # SURVEY 8(d), bytes per input sample


# --------------------------------------------------------------------------------------------------
# workload definition (shared by both arms)
# --------------------------------------------------------------------------------------------------
def workload_channels(name):
    """-> list of (kind, f_hz, baud, bw_hz)."""
    if name == "cfg2":
        return [("qpsk", 12.5e6 + 300.0, 1e6, 3e6)]
    if name == "cfg3":
        out = []
        for k in range(64):
            f = (k - 31.5) * 3e6
            kind = ("fsk", "qpsk", "ask")[k % 3]
            baud = 0.5e6 if kind == "ask" else 1e6
            out.append((kind, f + 300.0, baud, 2.5e6))
        return out
    if name == "cfg4":      # 8 audio channels, 200 kHz wide (Default/Audio/AudioProcessor.cpp:118-121)
        return [(d, (k - 3.5) * 2.0e6 + 300.0, 0.0, 200e3) for k, d in enumerate(["am"] * 3 + ["fm"] * 3 + ["usb"] * 2)]
    if name == "cfg5":
        return []
    raise ValueError(name)


def insp_kwargs(kind, baud, fs_ch):
    if kind == "qpsk":
        return "psk", dict(baud=baud, costas_order=2, bits_per_symbol=2, loop_bw=fs_ch * 2e-3, mf_type=1,
                           mf_rolloff=0.35, clock_type=1, clock_gain=0.1)
    if kind == "fsk":
        return "fsk", dict(baud=baud, bits_per_symbol=1, mf_type=1, mf_rolloff=0.35, clock_type=1, clock_gain=0.2)
    if kind == "ask":
        return "ask", dict(baud=baud, bits_per_symbol=1, ask_use_pll=1, ask_channel=0, loop_bw=fs_ch * 5e-3,
                           mf_type=1, mf_rolloff=0.35, clock_type=1, clock_gain=0.2)
    if kind in ("am", "fm", "usb"):
        return "audio", dict(audio_demod={"am": 1, "fm": 2, "usb": 3}[kind], audio_cutoff=5000.0,
                             audio_sample_rate=44100, agc_enabled=1, agc_ts=0.0005, offset=1300.0, audio_squelch=0,
                             audio_volume=1.0)
    raise ValueError(kind)


def chan_angular(f_hz, bw_hz):
    f0 = 2 * np.pi * ((f_hz - 300.0) / FS % 1.0)
    return float(np.float32(f0)), float(np.float32(2 * np.pi * bw_hz / FS))


def make_base_signal(name, n, seed):
    from sigdigger_b200 import synth
    if name == "cfg4":      # 3 AM (m = 0.5), 3 FM (5 kHz deviation), 2 USB two-tone, 1 kHz programme tone
        t = np.arange(n) / FS
        tone = np.cos(2 * np.pi * 1000 * t)
        x = synth.awgn(n, 10 ** (-60 / 20), np.random.default_rng(seed))
        for kind, f, _, _ in workload_channels(name):
            if kind == "am":
                sg = (1 + 0.5 * tone) * 0.2
            elif kind == "fm":
                sg = 0.2 * np.exp(1j * 2 * np.pi * 5000 * np.cumsum(tone) / FS)
            else:
                sg = 0.1 * (np.exp(2j * np.pi * 700 * t) + 0.5 * np.exp(2j * np.pi * 1900 * t))
            x = x + sg * np.exp(2j * np.pi * (f - 300.0) * t)
        return x.astype(np.complex64)
    carriers = []
    for kind, f, baud, _ in workload_channels(name):
        kw = {"levels": 2} if kind == "ask" else {}
        carriers.append((kind, f, baud, -20.0 if name == "cfg3" else -12.0, kw))
    x, _ = synth.multi_carrier(n, FS, carriers, noise_db=-80.0, seed=seed)
    return x


# --------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.t = threading.Thread(target=self.run, daemon=True)

    def run_nvml(self):
        """In-process NVML polling (~every 5 ms): a 40 ms timed region still gets several samples."""
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        bits = ((0x8, 2), (0x40, 3), (0x20, 4), (0x4, 5))   # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        while not self.stop:
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            row = [str(sm), str(mx), "", "", "", ""]
            for bit, col in bits:
                row[col] = "Active" if r & bit else "Not Active"
            self.rows.append(row)
            time.sleep(0.005)

    def run(self):
        try:
            self.run_nvml()
            return
        except Exception:
            pass
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if o.returncode == 0 and o.stdout.strip():
                    self.rows.append([c.strip() for c in o.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        t0 = time.time()
        while not self.rows and time.time() - t0 < 3.0:      # NVML / nvidia-smi start-up stays outside the timed region
            time.sleep(0.002)
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle restatement on the host cores
# --------------------------------------------------------------------------------------------------
def oracle_params(name):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    chans = []
    for kind, f, baud, bw in workload_channels(name):
        f0, bwa = chan_angular(f, bw)
        _, size, _ = O.channel_geometry(N_FFT, f0, bwa, 1.0)
        fs_ch = FS * size / N_FFT
        cls, kw = insp_kwargs(kind, baud, fs_ch)
        chans.append((f0, bwa, 1.0, 0, O.insp_config(cls, fs_ch, **kw)))
    return O, O.make_an_params(N_FFT, "blackmann_harris", chans)


def usable_cores():
    """Host threads the CPU legs may really use: the affinity mask, capped by the cgroup CPU quota (a container
    that reports 128 CPUs but is throttled to 16 runs 128 OpenMP threads slower than 16).  SDB_CPU_THREADS overrides.
    Returns (threads, description)."""
    if os.environ.get("SDB_CPU_THREADS"):
        t = max(1, int(os.environ["SDB_CPU_THREADS"]))
        return t, "SDB_CPU_THREADS=%d" % t
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                      # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()
            if q != "max":
                quota = float(q) / float(p)
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:     # cgroup v1
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0 and p > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    t = aff
    if quota is not None:
        t = max(1, min(aff, int(quota + 0.999)))
    return t, "cpu_count %d, affinity %d, cgroup quota %s" % (os.cpu_count() or 1, aff,
                                                               "none" if quota is None else "%.1f CPUs" % quota)


_CPU_LIBS = {}


def cpu_lib(kind):
    """CPU legs run the SPEED build of the oracle sources (oracle/Makefile: -O3, AVX2+FMA or the box's native ISA,
    contraction on) with the vectorisable transforms of oracle/fft_fast.c; the parity build (-O2 -ffp-contract=off,
    SPEC transforms) is for tests.  kind: "fast" (shipped, x86-64-v3), "native" (built here if gcc is present),
    "parity".  Returns a ctypes library or None."""
    import ctypes as C
    if kind in _CPU_LIBS:
        return _CPU_LIBS[kind]
    odir = os.path.join(ROOT, "oracle")
    path = {"fast": "libsdoracle_fast.so", "native": "libsdoracle_native.so", "parity": "libsdoracle.so"}[kind]
    path = os.path.join(odir, "_build", path)
    tmp = None
    if kind in ("native", "fast") and not os.path.exists(path):
        # built in a temporary directory, not in the tree (which may be read-only); removed once loaded
        tmp = tempfile.mkdtemp(prefix="sdb_oracle_")
        path = os.path.join(tmp, os.path.basename(path))
        subprocess.run(["make", "-C", odir, path, "%s=%s" % (kind.upper(), path)], capture_output=True)
    L = None
    if os.path.exists(path):
        try:
            L = C.CDLL(path)
            L.sdo_baseline_run.restype = C.c_double
            L.sdo_baseline_run.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int,
                                           C.POINTER(C.c_uint64)]
            L.sdo_set_fast_transforms(0 if kind == "parity" else 1)
        except OSError:
            L = None
    if tmp:
        shutil.rmtree(tmp, ignore_errors=True)
    _CPU_LIBS[kind] = L
    return L


CPU_FLAGS = {"fast": "gcc -O3 -march=x86-64-v3 -ffp-contract=fast + fft_fast.c (Stockham radix-4, vectorised)",
             "native": "gcc -O3 -march=native -ffp-contract=fast + fft_fast.c (Stockham radix-4, vectorised)",
             "parity": "gcc -O2 -ffp-contract=off, SPEC transforms (the build the parity tests use)"}


def cpu_run(name, n_streams, n, threads, reps=1, warm=0, kind="fast"):
    import ctypes as C
    O, p = oracle_params(name)
    L = cpu_lib(kind) or cpu_lib("fast") or O.lib()
    base = make_base_signal(name, n, seed=1)
    x = np.ascontiguousarray(np.tile(base, (n_streams, 1)))
    rng = np.random.default_rng(0)
    x += (1e-3 * (rng.standard_normal(x.shape) + 1j * rng.standard_normal(x.shape))).astype(np.complex64)
    chk = C.c_uint64()
    times = []
    for i in range(warm + reps):
        t = L.sdo_baseline_run(C.byref(p), O.ptr(x), n_streams, n, threads, C.byref(chk))
        if i >= warm:
            times.append(t)
    return times, n_streams * n


def pick_threads(name):
    """Thread count and build for the CPU legs: the usable cores, or a fraction of them when a short probe of the
    same workload (4 frames per stream, one stream per thread, best of 2) runs faster that way (SMT siblings,
    throttled containers); the native-ISA build when it beats the shipped AVX2 one on the same probe.
    Returns (threads, build kind, description)."""
    cores, how = usable_cores()
    kinds = ["fast"] + (["native"] if cpu_lib("native") is not None and not os.environ.get("SDB_CPU_NO_NATIVE") else [])
    if os.environ.get("SDB_CPU_THREADS"):
        return cores, kinds[0], how
    best, table = (0.0, cores, kinds[0]), []
    for t in sorted({cores, max(1, cores // 2), max(1, cores // 4), max(1, cores // 8)}, reverse=True):
        for kd in kinds:
            times, samples = cpu_run(name, t, 4 * N_FFT, t, reps=2, warm=1, kind=kd)
            rate = samples / min(times) / 1e6
            table.append("%d/%s:%.0f" % (t, kd, rate))
            if rate > best[0] * 1.05:                      # prefer more threads unless fewer are clearly faster
                best = (rate, t, kd)
    return best[1], best[2], "%s; probe threads/build:MS/s %s" % (how, " ".join(table))


def fft_comparators():
    """Single-thread time of one 65536-point complex64 transform: the oracle's parity (SPEC) transform, its speed
    transform, numpy (pocketfft) and torch (MKL) -- shows the CPU arm's transform is not a straw man."""
    import ctypes as C
    out = {}
    x = (np.random.default_rng(3).standard_normal(2 * N_FFT).astype(np.float32)).view(np.complex64)
    y = np.empty_like(x)

    def best(fn, reps=5):
        fn()
        t = []
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); t.append(time.perf_counter() - t0)
        return round(min(t) * 1e3, 3)
    for kd in ("fast", "native"):
        L = cpu_lib(kd)
        if L is not None:
            L.sdo_fast_fft.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint, C.c_int]
            out["oracle_" + kd + "_ms"] = best(lambda: L.sdo_fast_fft(x.ctypes.data, None, y.ctypes.data, N_FFT, -1))
    Lp = cpu_lib("parity")
    if Lp is not None:
        # the parity build's SPEC transform through the same entry point (fast transforms are off in that library)
        try:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as O
            x8 = np.tile(x, 8)          # 8 frames per call: plan set-up amortised
            out["oracle_spec_ms"] = round(best(lambda: O.psd_frames(x8, N_FFT, "none"), 2) / 8, 3)
        except Exception:
            pass
    try:
        out["numpy_pocketfft_ms"] = best(lambda: np.fft.fft(x))
    except Exception:
        pass
    try:
        import torch
        nt = torch.get_num_threads()
        torch.set_num_threads(1)
        xt = torch.from_numpy(x)
        out["torch_mkl_ms"] = best(lambda: torch.fft.fft(xt))
        torch.set_num_threads(nt)
    except Exception:
        pass
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "cfg5":
        t0 = time.perf_counter()
        reps = []
        for _ in range(max(1, args.warmup) + args.steps):
            reps.append(cfg5_cpu(min(128, CFG5_HOPS)))
        reps = reps[max(1, args.warmup):]
        v = float(np.mean([r["value"] for r in reps]))
        cb = dict(reps[-1], value=v)
        print(json.dumps({"impl": "reference", "metric": "complex MSamples/s ingested (65536-pt PSD per tuner hop, stitched)",
                          "value": v, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 * 128 * N_FFT / (v * 1e6), "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg5_config(),
                          "cpu_baseline": cb,
                          "e2e": {"value": v, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    cores, kind, how = pick_threads(args.workload)
    n = N_FFT // 2 * 16                      # 2^19 samples per stream: one stream per host thread
    streams = cores
    times, samples = cpu_run(args.workload, streams, n, cores, reps=args.steps, warm=args.warmup, kind=kind)
    total = sum(times)
    v = samples * len(times) / total / 1e6
    sample = "%d streams x %d samples per step, %d OpenMP threads (%s)" % (streams, n, cores, how)
    # the round-1 arm (parity build, SPEC transforms) on a shorter sample, for the record
    tp, sp = cpu_run(args.workload, streams, N_FFT * 2, cores, reps=1, warm=0, kind="parity")
    out = {"impl": "reference", "metric": "complex MSamples/s ingested (%d-pt PSD + N inspectors)" % N_FFT,
           "value": v, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           # the CUDA arm's own configuration (the workload this arm is a bounded sample of; the sample itself is
           # described in cpu_baseline.sample)
           "config": workload_config(args, streams=args.streams, hops=args.hops),
           "cpu_baseline": {"value": v, "unit": "MS/s", "cores": cores, "kind": "port", "sample": sample,
                            "build": CPU_FLAGS[kind], "per_thread_msps": v / cores,
                            "parity_build_msps": sp / sum(tp) / 1e6,
                            "fft_65536_single_thread": fft_comparators()},
           "e2e": {"value": v, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def workload_config(args, streams, hops):
    k = len(workload_channels(args.workload))
    what = {"cfg2": "QPSK 1 MBd, Costas + RRC + Gardner + decision",
            "cfg3": "2-FSK / QPSK / ASK mix on a 3 MHz raster, Costas / PLL + RRC + Gardner + decision",
            "cfg4": "3 AM + 3 FM + 2 USB audio channels, AGC + demodulator + LPF + resampler to 44.1 kS/s"}[args.workload]
    return {"workload": "%s: fs %g MS/s nominal, %d-pt Blackman-Harris PSD every frame + %d-pt "
                        "50%%-overlap FFT channeliser + %d inspector(s) (%s)"
                        % (args.workload, FS / 1e6, N_FFT, N_FFT, k, what),
            "streams_per_gpu": streams, "samples_per_stream_per_step": hops * N_FFT // 2,
            "inputs": "larger than L2 (no flush needed)", "parallelism": "independent streams per GPU"}


# --------------------------------------------------------------------------------------------------
# cfg5: panoramic sweep (BASELINE.json configs[4]): 1024 tuner hops x 65536-pt PSD, per-GPU channel detector,
# stitched on rank 0 -- the one workload with a collective (NCCL gather of the contribution lists)
# --------------------------------------------------------------------------------------------------
CFG5_HOPS = 1024


def cfg5_geometry():
    rel_bw = 0.5
    fmin = 1.0e9
    fmax = fmin + CFG5_HOPS * FS * rel_bw
    centers = fmin + FS * rel_bw * (0.5 + np.arange(CFG5_HOPS))
    return fmin, fmax, rel_bw, centers


def cfg5_hops(lo, hi, seed=17):
    """hops [lo, hi): noise + 3 carriers per hop at seeded offsets (the same bits on every rank layout)."""
    out = np.empty((hi - lo, N_FFT), np.complex64)
    t = np.arange(N_FFT)
    for h in range(lo, hi):
        rng = np.random.default_rng(seed * 100003 + h)
        x = 0.02 * (rng.standard_normal(N_FFT) + 1j * rng.standard_normal(N_FFT))
        for _ in range(3):
            x = x + 0.3 * np.exp(2j * np.pi * rng.uniform(-0.2, 0.2) * t)
        out[h - lo] = x.astype(np.complex64)
    return out


def cfg5_config():
    return {"workload": "cfg5: panoramic sweep, %d tuner hops x %d-pt Blackman-Harris PSD at %g MS/s per hop, relBw 0.5, "
                        "per-hop channel detector on the owning GPU, SpectrumView (65536 bins) stitched on rank 0"
                        % (CFG5_HOPS, N_FFT, FS / 1e6),
            "hops": CFG5_HOPS, "samples_per_hop": N_FFT,
            "inputs": "hop buffers larger than L2 at 1-2 GPUs (537 MB in total); L2 flushed between steps otherwise",
            "parallelism": "hops sharded contiguously over ranks; one NCCL gather of the contribution lists per sweep"}


def bind_to_gpu_numa_node(local):
    """Run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA node its GPU hangs off, so that the
    H2D / D2H copies of N ranks do not all cross the socket interconnect.  Returns a description for the JSON line;
    never fatal (containers without /sys topology just keep their affinity)."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = local
        if vis:
            toks = [t for t in vis.split(",") if t.strip()]
            if local < len(toks) and toks[local].strip().isdigit():
                idx = int(toks[local])
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        bus = nv.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bdf = bus.lower()
        if len(bdf.split(":")[0]) == 8:                      # NVML prints an 8-digit domain, sysfs a 4-digit one
            bdf = bdf[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA information for " + bdf}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return {"numa_node": node, "note": "node CPUs outside this process's affinity mask"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as ex:                                   # noqa: BLE001
        return {"numa_node": None, "note": "not bound: %s" % type(ex).__name__}


def run_cuda_cfg5(args):
    import torch
    import sigdigger_b200 as sdb
    from sigdigger_b200 import panoramic
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if sdb.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    affinity0 = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    fmin, fmax, rel_bw, centers = cfg5_geometry()
    lo, hi = panoramic.shard(CFG5_HOPS, world, rank)
    xh = torch.from_numpy(cfg5_hops(lo, hi)).pin_memory()
    x = xh.cuda()
    det = dict(alpha=1.0, gamma=0.5, snr=6.0, min_bins=2)
    p = sdb.Panoramic(N_FFT, "blackmann_harris", FS, (fmin, fmax), rel_bw, device=local, rank=rank, world=world,
                      unique_id=panoramic.exchange_unique_id(sdb, torch, dist), detect=det)
    flush = torch.empty(160 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run(fn, steps, do_flush):
        tot = 0.0
        for _ in range(steps):
            if do_flush:
                flush.fill_(1)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        if dist is not None:
            t = torch.tensor([tot], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            tot = float(t.item())
        return tot

    small = x.numel() * 8 < (256 << 20)
    step_dev = lambda: (p.reset(), p.sweep(x, centers))
    for _ in range(max(3, args.warmup)):
        step_dev()
    with Clocks(local) as clk:
        ms = run(step_dev, args.steps, small)
    if args.dump_outputs and rank == 0:
        psd, accum, count = p.read()                # the stitched SpectrumView of the last sweep
        write_dump(args.dump_outputs, {"view_psd": psd, "view_psd_accum": accum, "view_psd_count": count})
    samples = CFG5_HOPS * N_FFT
    value = samples * args.steps / (ms * 1e-3) / 1e6
    tm = p.timing()
    # end to end: pinned host hop buffers -> H2D -> sweep -> D2H of the stitched view (+ channel lists) on rank 0
    def step_e2e():
        p.reset()
        p.sweep(xh.numpy(), centers)
        if rank == 0:
            p.read()
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    dt = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    e2e_v = samples * args.steps / dt / 1e6
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # dominant kernels: the two passes of the hop PSDs (inside psd_project_ms); B_alg = 8 B in + 4 B out per sample
    ach = B_ALG["cfg5"] * (hi - lo) * N_FFT / (tm["psd_project_ms"] * 1e-3) / 1e9 if tm["psd_project_ms"] > 0 else 0.0
    try:
        os.sched_setaffinity(0, affinity0)
    except OSError:
        pass
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cfg5_cpu(min(128, CFG5_HOPS))
    if rank == 0:
        out = {"metric": "complex MSamples/s ingested (65536-pt PSD per tuner hop, stitched)", "value": value,
               "unit": "MS/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
               "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f32", "data": "synthetic", "config": cfg5_config(), "host_binding": numa, "clocks": clk.summary(),
               "gpu_launches": None,
               "e2e": {"value": e2e_v, "unit": "MS/s", "h2d_bytes_per_step": int(samples * 8),
                       "d2h_bytes_per_step": int(3 * 65536 * 4)},
               "roofline": {"bound": "hbm", "kernel": "hop PSD passes + projection (rank 0's shard)", "achieved": ach,
                            "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                            "phases_ms": {k: round(v, 4) for k, v in tm.items() if k.endswith("_ms")},
                            "gather_bytes": tm["gather_bytes"],
                            "note": "phase times of the LAST sweep on rank 0 (CUDA events inside sdb_panoramic_sweep)"},
               "cpu_baseline": cpu}
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def cfg5_cpu(n_hops):
    """CPU arm of cfg5 on a bounded sample: hop PSDs (speed build, one hop per thread) + the sequential stitch."""
    import ctypes as C
    from concurrent.futures import ThreadPoolExecutor
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    cores, how = usable_cores()
    L = cpu_lib("fast") or O.lib()
    L.sdo_fast_fft.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint, C.c_int]
    fmin, fmax, rel_bw, centers = cfg5_geometry()
    x = cfg5_hops(0, n_hops)
    w = O.window(N_FFT, "blackmann_harris")
    psd = np.empty((n_hops, N_FFT), np.float32)

    def one(h):
        y = np.empty(N_FFT, np.complex64)
        L.sdo_fast_fft(x[h].ctypes.data, w.ctypes.data, y.ctypes.data, N_FFT, -1)
        p_ = ((y.real * y.real + y.imag * y.imag) / np.float32(N_FFT)).astype(np.float32)
        O.lib().sdo_psd_shift_db(O.ptr(p_), N_FFT)
        psd[h] = p_
    t0 = time.perf_counter()
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(one, range(n_hops)))
    v = O.SpectrumView()
    Lo = O.lib()
    assert Lo.sdo_sview_init(C.byref(v)) == 0
    Lo.sdo_sview_set_range(C.byref(v), fmin, fmin + n_hops * FS * rel_bw)
    v.fft_bandwidth = FS
    v.fft_rel_bw = rel_bw
    for h in range(n_hops):
        Lo.sdo_sview_feed(C.byref(v), O.ptr(psd[h]), None, N_FFT, float(centers[h]), 1)
    dt = time.perf_counter() - t0
    val = n_hops * N_FFT / dt / 1e6
    return {"value": val, "unit": "MS/s", "cores": cores, "kind": "port", "build": CPU_FLAGS["fast"],
            "sample": "%d of the %d hops: windowed PSD per hop (one hop per thread, %d threads; %s) + sequential "
                      "SpectrumView feed, no detector" % (n_hops, CFG5_HOPS, cores, how)}


# --------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path handed back in its last step, so that two builds can be compared output for
# output (inputs are seeded: the same arguments give the same inputs)
# --------------------------------------------------------------------------------------------------
DUMP_LIMIT = 64 << 20         # bytes written in all
DUMP_STREAMS_BUDGET = 48 << 20


def write_dump(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte bound" % (total, DUMP_LIMIT))
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def dump_engine_outputs(out_dir, e, hs):
    """PSD frames [streams, frames, N] and every inspector's soft / hard symbols of the last feed, for a fixed seeded
    sample of the streams (all of them when they fit the budget); the sampled stream indices go with them."""
    psd = e.read_psd()
    S = psd.shape[0]
    sym0 = sum(len(e.read_symbols(0, h)[1]) for h in hs)
    per_stream = psd[0].nbytes + sym0 * 12                       # soft as 2 x float32, hard as float32
    k = min(S, max(1, DUMP_STREAMS_BUDGET // max(1, per_stream)))
    idx = np.arange(S) if k == S else np.sort(np.random.default_rng(0).choice(S, k, replace=False))
    soft, hard, counts = [], [], np.zeros((k, len(hs)), np.float64)
    for i, s in enumerate(idx):
        for j, h in enumerate(hs):
            sf, hd = e.read_symbols(int(s), h)
            soft.append(sf)
            hard.append(hd)
            counts[i, j] = len(hd)
    soft = np.concatenate(soft) if soft else np.zeros(0, np.complex64)
    hard = np.concatenate(hard) if hard else np.zeros(0, np.uint8)
    write_dump(out_dir, {"psd": psd[idx], "soft_symbols": soft.view(np.float32).reshape(-1, 2),
                         "hard_symbols": hard.astype(np.float32), "symbol_counts": counts,
                         "streams": idx.astype(np.float64)})


# --------------------------------------------------------------------------------------------------
# CUDA arm
# --------------------------------------------------------------------------------------------------
def build_engine(sdb, name, streams, n, device):
    e = sdb.Engine(n_streams=streams, psd_size=N_FFT, psd_window="blackmann_harris", max_feed=n,
                   samp_rate=FS, device=device)
    hs = []
    for kind, f, baud, bw in workload_channels(name):
        f0, bwa = chan_angular(f, bw)
        h = e.open_channel(f0, bwa, 1.0)
        cls, kw = insp_kwargs(kind, baud, e.channel_rate(h))
        e.set_inspector(h, cls, **kw)
        hs.append(h)
    e.commit()
    return e, hs


def run_cuda(args):
    import torch
    import sigdigger_b200 as sdb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if sdb.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    affinity0 = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local)                      # undone before the CPU baseline leg below
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    name = args.workload
    S, H = args.streams, args.hops
    n = H * N_FFT // 2
    e, hs = build_engine(sdb, name, S, n, local)
    K = len(hs)

    # synthetic IQ, device resident: one modulated base signal per rank + independent noise per stream
    base = torch.from_numpy(make_base_signal(name, n, seed=1 + rank)).cuda()
    x = base.unsqueeze(0).repeat(S, 1).contiguous()
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    x += torch.view_as_complex(1e-3 * torch.randn((S, n, 2), generator=g, device="cuda"))
    xh = torch.empty((S, n), dtype=torch.complex64, pin_memory=True)
    xh.copy_(x)
    torch.cuda.synchronize()

    es = torch.cuda.ExternalStream(e.stream_ptr)
    samples_step = S * n

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(es)
        for _ in range(steps):
            fn()
        e.join()                 # the end event must also cover the inspector stream
        b.record(es)
        e.sync()
        ms = a.elapsed_time(b)
        barrier()
        if dist is not None:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- device-resident arm
    step_dev = lambda: e.feed_device_ptr(x.data_ptr(), x.stride(0), n)
    for _ in range(max(3, args.warmup)):
        step_dev()
    e.sync()
    l0 = e.launches
    with Clocks(local) as clk:
        ms = timed(step_dev, args.steps)
    launches = e.launches - l0
    if args.dump_outputs and rank == 0:
        dump_engine_outputs(args.dump_outputs, e, hs)
    value = samples_step * world * args.steps / (ms * 1e-3) / 1e6

    # ---- per-kernel device times: a separate pass in the engine's timing mode, which queues every kernel on ONE
    # stream (no two kernels overlap), so the CUDA-event spans recorded on that stream are the kernels' own warm
    # durations; the ncu launch list of the same command is committed under profiles/ (shares must agree)
    e.timing(True)
    timed_steps = 2
    for _ in range(timed_steps):
        step_dev()
    e.sync()
    fam = {f: e.kernel_time(f) for f in ("fft_cols", "fft_rows_psd", "fft_rows_chan", "chan_ifft", "inspector")}
    e.timing(False)
    # SURVEY 8(d): the algorithmic bytes of the path are B_alg per INPUT sample (8 B read once, shared by the PSD and
    # the channeliser, + 4 B of PSD + 9 B per symbol); intermediate streams are not algorithmic.  The dominant
    # kernel (largest total device time per step, the inspector kernel included) is charged with the B_alg of every
    # input sample its launches cover: achieved = B_alg x samples per launch / average launch duration.
    tot = {f: fam[f][0] * fam[f][1] / timed_steps for f in fam}            # ms of device time per step
    dom = max(tot, key=tot.get)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    launches_dom = max(1.0, fam[dom][1] / timed_steps)                     # launches per step
    alg_launch = B_ALG[name] * samples_step / launches_dom
    ach = alg_launch / (fam[dom][0] * 1e-3) / 1e9 if fam[dom][0] > 0 else 0.0
    traffic = None
    try:   # DRAM bytes per launch of that kernel from the committed single-pass ncu capture of this workload
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        if tr.get("workload") == name and dom in tr.get("kernels", {}):
            traffic = tr["kernels"][dom]["dram_bytes_per_launch"]
            # the capture was taken at tr["streams_per_gpu"] streams; the inspector / inverse-transform kernels
            # cover every stream in one launch, so their per-launch traffic scales with the stream count
            if dom in ("inspector", "chan_ifft") and tr.get("streams_per_gpu"):
                traffic = int(traffic * S / tr["streams_per_gpu"])
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": ach / peak, "traffic": traffic,
                "algorithmic_bytes_per_launch": alg_launch, "launch_ms": fam[dom][0],
                "note": "B_alg (SURVEY 8d) x input samples covered by one launch / its duration; durations are "
                        "CUDA-event spans of a serialised pass (one stream, no overlap). The kernel is bound by "
                        "instruction issue / recurrence latency, not by DRAM (profiles/r02_*.md)",
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                "kernel_share_of_device_time": tot[dom] / max(1e-9, sum(tot.values())),
                "device_ms_per_step": {f: round(tot[f], 4) for f in tot},
                "launch_ms_avg": {f: round(fam[f][0], 4) for f in fam},
                "path": {"b_alg_bytes_per_sample": B_ALG[name],
                         "achieved": B_ALG[name] * value * 1e6 / world / 1e9,
                         "frac": B_ALG[name] * value * 1e6 / world / 1e9 / peak}}
    # The path's other roofline: instruction issue.  Every input sample costs a fixed number of warp instructions
    # (64 inspectors' recurrences, filters and transforms; counted by ncu, profiles/r02_traffic.json), and an SM issues
    # at most 4 warp instructions per clock: the ceiling that count sets, whatever the memory system does.
    try:
        wi = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        if wi.get("workload") == name and "warp_instructions" in wi:
            w = wi["warp_instructions"]
            per_sample = sum(w["per_step_148_streams"].values()) / float(w["input_samples_per_step"])
            sm_clock = (clk.summary().get("sm_mhz") or 1965.0) * 1e6
            ceiling = 148 * 4 * sm_clock / per_sample / 1e6          # MS/s per GPU
            roofline["issue"] = {"warp_instructions_per_input_sample": round(per_sample, 2),
                                 "ceiling_msps_per_gpu": round(ceiling, 1),
                                 "frac": round(value / world / ceiling, 4),
                                 "ceiling_as_hbm_frac": round(B_ALG[name] * ceiling * 1e6 / 1e9 / peak, 4),
                                 "note": "148 SMs x 4 warp instructions per clock / instructions per sample: even a "
                                         "perfectly issue-bound run of this instruction stream stays below this "
                                         "fraction of the HBM roofline"}
    except Exception:
        pass
    if os.environ.get("SDB_LIB"):      # instrumented twin: busy cycles per role warp per chunk sample
        sdb.stage_cycles(reset=True)
        step_dev(); e.sync()
        roofline["inspector_role_cycles_per_sample"] = {k_: round(v_, 1) for k_, v_ in sdb.stage_cycles(reset=True).items()}
        sdb.cta_cycles(reset=True)
        step_dev(); e.sync()
        roofline["inspector_cta_by_class"] = sdb.cta_cycles(reset=True)
    wps, frames = H, H // 2

    # ---- end to end: pinned host IQ -> H2D -> path -> D2H of PSD frames and symbols, every step
    # Every step: H2D of that step's IQ from pinned memory, the whole path, D2H of its PSD frames and symbols
    # into pinned memory.  The engine pipelines the three (copy streams + double-buffered results), so the host
    # keeps two result sets in flight and only blocks at the end.
    cap = e.symbol_capacity
    pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()
    psd_h = [pin((S, frames, N_FFT), torch.float32) for _ in range(2)]
    cnt_h = [pin((S * K,), torch.int32).view(np.uint32) for _ in range(2)]
    # symbols come back packed (sdb_engine_read_symbols_packed_async: chain after chain, written by the GPU straight
    # into these pinned buffers), so PCIe carries the symbols that exist, not the [chains][cap] array they sit in
    cap_total = S * K * ((cap + 15) // 16 * 16)
    off_h = [pin((S * K + 1,), torch.int64).view(np.uint64) for _ in range(2)]
    soft_h = [pin((cap_total,), torch.complex64) for _ in range(2)]
    hard_h = [pin((cap_total,), torch.uint8) for _ in range(2)]
    e.sync()

    def run_e2e(eng, host_ptr, stride):
        step_no = [0]

        def step_e2e():
            b = step_no[0] & 1
            step_no[0] += 1
            eng.feed_host_ptr(host_ptr, stride, n)
            eng.read_psd_async(psd_h[b])
            eng.read_symbols_packed_async(cnt_h[b], off_h[b], soft_h[b], hard_h[b], cap_total)

        for _ in range(3):
            step_e2e()
        eng.sync()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        eng.sync()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return samples_step * world * args.steps / dt / 1e6

    e2e_v = run_e2e(e, xh.data_ptr(), xh.stride(0))
    h2d = samples_step * 8
    sym_extent = int(off_h[(args.steps + 3 - 1) & 1][-1])            # symbols (with alignment gaps) of the last step
    d2h = psd_h[0].nbytes + cnt_h[0].nbytes + off_h[0].nbytes + sym_extent * 9

    # ---- the same end-to-end loop with the IQ in native SDR sample formats (converted inside the first load):
    # 4 and 2 bytes per complex sample over PCIe instead of 8.  Extra information; `e2e` above is float32.
    e2e_fmt = {}
    if not args.no_formats:
        xr = torch.view_as_real(x)
        for fmt, tdt, scale, off in (("s16", torch.int16, 32768.0, 0.0), ("u8", torch.uint8, 128.0, 128.0)):
            lo, hi = (-32768, 32767) if fmt == "s16" else (0, 255)
            q = torch.clamp(torch.round(xr * scale + off), lo, hi).to(tdt)
            qh = torch.empty(q.shape, dtype=tdt, pin_memory=True)
            qh.copy_(q)
            del q
            ef = sdb.Engine(n_streams=S, psd_size=N_FFT, psd_window="blackmann_harris", max_feed=n, samp_rate=FS,
                            device=local, input_format=fmt)
            for kind, f, baud, bw in workload_channels(name):
                f0, bwa = chan_angular(f, bw)
                hh = ef.open_channel(f0, bwa, 1.0)
                cls, kw = insp_kwargs(kind, baud, ef.channel_rate(hh))
                ef.set_inspector(hh, cls, **kw)
            ef.commit()
            e2e_fmt[fmt] = {"value": run_e2e(ef, qh.data_ptr(), n), "unit": "MS/s",
                            "h2d_bytes_per_step": int(samples_step * (4 if fmt == "s16" else 2))}
            ef.close()
            del qh

    # ---- single-stream number (what one continuous source gets)
    single = None
    if rank == 0 and not args.no_single:
        e1, _ = build_engine(sdb, name, 1, n, local)
        x1 = x[:1].contiguous()
        for _ in range(3):
            e1.feed_device_ptr(x1.data_ptr(), x1.stride(0), n)
        e1.sync()
        es1 = torch.cuda.ExternalStream(e1.stream_ptr)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(es1)
        for _ in range(5):
            e1.feed_device_ptr(x1.data_ptr(), x1.stride(0), n)
        e1.join()
        b.record(es1)
        e1.sync()
        single = n * 5 / (a.elapsed_time(b) * 1e-3) / 1e6
        e1.close()

    # ---- bounded CPU baseline on rank 0, N=1 only
    try:
        os.sched_setaffinity(0, affinity0)                   # the CPU arm gets every core the process was given
    except OSError:
        pass
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores, kind, how = pick_threads(name)
        times, samples = cpu_run(name, cores, N_FFT // 2 * 16, cores, reps=2, warm=0, kind=kind)
        v = samples * len(times) / sum(times) / 1e6
        cpu = {"value": v, "unit": "MS/s", "cores": cores, "kind": "port", "build": CPU_FLAGS[kind],
               "per_thread_msps": v / cores,
               "sample": "%d streams x %d samples x %d reps of the same workload (oracle sources, speed build, OpenMP, "
                         "one stream per thread; %s)" % (cores, N_FFT // 2 * 16, len(times), how)}

    if rank == 0:
        out = {"metric": "complex MSamples/s ingested (%d-pt PSD + N inspectors)" % N_FFT, "value": value,
               "unit": "MS/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
               "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "f32", "data": "synthetic", "config": workload_config(args, S, H), "host_binding": numa,
               "clocks": clk.summary(), "gpu_launches": int(launches),
               "e2e": {"value": e2e_v, "unit": "MS/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
               "roofline": roofline, "cpu_baseline": cpu, "single_stream_msps": single,
               "e2e_native_formats": e2e_fmt}
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--streams", type=int, default=0)
    ap.add_argument("--hops", type=int, default=8)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-single", action="store_true")
    ap.add_argument("--no-formats", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="CUDA arm: write the outputs of the last timed step as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    global FS, N_FFT
    FS = FS_BY[args.workload]
    N_FFT = NFFT_BY[args.workload]
    if args.streams == 0:
        # cfg2: the (latency-bound) inspector kernel of 1024 single-channel streams takes about as long as their
        # transforms; 2048 streams put the transforms on the critical path (33.9 / 53.3 / 64.5 GS/s at 512 / 1024 /
        # 2048 streams on one B200, profiles/r01_batch.md)
        # cfg3: 148 streams are one wave of inspector CTAs (2 per SM); with 296 the CTAs of the faster inspector
        # classes are back-filled as they retire (15.2 / 15.8 / 16.1 / 16.1 GS/s at 148 / 222 / 296 / 444 streams,
        # profiles/r02_summary.md)
        args.streams = {"cfg2": 2048, "cfg3": 296, "cfg4": 1024, "cfg5": 0}[args.workload]
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "cfg5":
        run_cuda_cfg5(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
