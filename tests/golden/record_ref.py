#!/usr/bin/env python
"""Records the outputs of the reference's own code (oracle/_ref/libsdref.so and libsdref_suscan.so, built by
`make -C oracle ref` from the reference sources where they lie) on the inputs of tests/test_ref.py, so that the oracle is
held to the reference without the reference at test time.

    python tests/golden/record_ref.py          # CPU cases
    python tests/golden/record_ref.py --gpu    # LPFTask over the GPU tuner (the "lpf" entry)

The input builders below are the ones the tests use.  Outputs the tests compare bit for bit are stored as SHA-256 digests
of their bytes (with shape and dtype) in ref_compiled.json; outputs compared to a tolerance keep their values: short ones
in the JSON, longer ones in ref_compiled.npz (the histogram feeder's as a fixed strided sample).
"""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, HERE)

import make_golden as G                     # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "libsdref.so")
REF2 = os.path.join(ROOT, "oracle", "_ref", "libsdref_suscan.so")
SPACE = {"amplitude": 0, "phase": 1, "frequency": 2}


# ---- inputs (shared with tests/test_ref.py)
def sview_hist_case():
    """histogram mode: hops narrower than two destination bins"""
    rng = np.random.default_rng(3)
    fmin, fmax = 1.0e9, 1.0e9 + 65536 * 1000.0 * 40
    feeds = [((rng.random(512).astype(np.float32) * 10 - 80), fmin + (5 + 37.3 * h) * 40e3, 30e3) for h in range(200)]
    return fmin, fmax, feeds


WIDE = (-10e6, 25e6)        # zoom-out of the first case's range (Scanner::setViewRange)
DELAYS = (7, 500)
MANUAL = (("amplitude", "ask"), ("phase", "psk"), ("frequency", "psk"))
ZC_CASES = [("ask", "amplitude", True, 0.6 + 0.1j, 1 + 0j, 1.0 / 12),
            ("ask", "amplitude", False, 0.55 + 0.2j, np.exp(-0.3j), 1.0 / 12),
            ("psk", "phase", False, 0j, np.exp(0.1j), 1.0 / 12),
            ("ask", "amplitude", True, 0.6 + 0.1j, 1 + 0j, 1.0)]
ALPHAS = (0.25, 1.0)
TV_CASES = [(False, 40), (True, 61)]
TASK_N = 2 * 4096 + 777
HIST_N = 3 * 4096 + 55
LPF_N = 5 * 4096 + 300


def averager_frames():
    rng = np.random.default_rng(9)
    return rng.random((7, 4096)).astype(np.float32) * 40 - 100


def tv_case(interlace, lines):
    import test_oracle_tv as T
    x, _, _ = T.toy_signal(lines, interlace, frames=10)
    sp = T.toy_params(lines, interlace, 4, cls=T.ShimTvParams)
    W, H, cap, block = int(np.floor(T.LINE)), lines, 16, 7000
    return x, sp, W, H, cap, block


def psd_message_input():
    rng = np.random.default_rng(21)
    n = 8192
    lin = (rng.standard_normal(n) ** 2 * 10.0 ** rng.uniform(-9, 1, n)).astype(np.float32)
    lin[:4] = [0.0, 1e-12, 1.0, 123.5]
    return lin


def mq_input():
    rng = np.random.default_rng(22)
    return (rng.standard_normal(1000) + 1j * rng.standard_normal(1000)).astype(np.complex64)


def qpsk(n, seed=5):
    from sigdigger_b200 import synth
    x, _ = synth.multi_carrier(n, 1.0, [("qpsk", 0.01, 0.1, -6.0, {})], noise_db=-40.0, seed=seed)
    return np.ascontiguousarray(x, np.complex64)


def snr_cases():
    rng = np.random.default_rng(4)
    for bps, length in ((1, 256), (2, 256), (3, 400)):
        k = 1 << bps
        centres = (rng.integers(0, k, 200000) + 0.5) / k
        v = (centres + 0.03 * rng.standard_normal(200000)) % 1.0
        h = np.bincount((v * length).astype(int) % length, minlength=length).astype(np.uint32)
        yield bps, length, h


SNR_FEEDS = 6


def carrier_cases():
    rng = np.random.default_rng(12)
    for n, f0, notch in ((5000, 0.0371, 0.0), (16384, -0.212, 0.0), (3000, 0.11, 0.05), (9000, -0.4, 0.02)):
        t = np.arange(n)
        x = (np.exp(2j * np.pi * f0 * t) * (1 + 0.3 * np.cos(2 * np.pi * 0.001 * t))
             + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) + 0.5).astype(np.complex64)
        yield n, f0, notch, x


def lpf_input():
    return qpsk(LPF_N, seed=9)


JSON = os.path.join(HERE, "ref_compiled.json")
NPZ = os.path.join(HERE, "ref_compiled.npz")
SAMPLED = ("histogram_0", "histogram_1", "histogram_2")
STORED = ("quad_demod", "delayed_conj_7", "delayed_conj_500", "psd_message") + SAMPLED
VALUES = ("carrier_detect", "psd_message_fc_rate", "mq_inspector_id", "status_codes", "status_texts")
SAMPLE = 4096


def digest(a):
    a = np.ascontiguousarray(a)
    return {"sha256": hashlib.sha256(a.tobytes()).hexdigest(), "shape": list(a.shape), "dtype": a.dtype.str}


def same(entry, a):
    """a is, byte for byte, the recorded output (same shape and dtype)"""
    return digest(a) == entry


def sample(a):
    """the fixed strided sample kept of a long output"""
    return np.ascontiguousarray(a[::-(-len(a) // SAMPLE)])


def load():
    """the recorded reference outputs: JSON entries, with the stored arrays under "values" """
    with open(JSON) as f:
        rec = json.load(f)
    with np.load(NPZ, allow_pickle=False) as z:
        for k in z.files:
            rec[k]["values"] = z[k]
    return rec


# ---- the reference libraries
def _ref():
    L = C.CDLL(REF)
    L.ref_sview_new.restype = C.c_void_p
    L.ref_sview_read.restype = C.c_uint
    L.ref_wave_sampler.restype = C.c_long
    L.ref_wave_sampler.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int,
                                   C.c_float, C.c_float, C.c_float, C.c_float, C.c_size_t, C.c_double, C.c_void_p,
                                   C.c_void_p, C.c_size_t]
    L.ref_sview_set_range.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_float]
    L.ref_sview_feed.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ulong, C.c_double, C.c_int]
    L.ref_sview_feed_view.argtypes = [C.c_void_p, C.c_void_p]
    L.ref_sview_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ref_quad_demod.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.ref_delayed_conj.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_ulong]
    L.ref_averager.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_float, C.c_void_p]
    L.ref_tv_worker.restype = C.c_long
    L.ref_tv_worker.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                C.c_void_p]
    for fn, extra in (("ref_task_costas", [C.c_float, C.c_float, C.c_int]), ("ref_task_pll", [C.c_float]),
                      ("ref_task_agc", [C.c_float]), ("ref_task_xlate", [C.c_float, C.c_float]),
                      ("ref_task_lpf", [C.c_float])):
        getattr(L, fn).argtypes = [C.c_void_p, C.c_void_p, C.c_size_t] + extra
    L.ref_task_histogram.restype = C.c_long
    L.ref_task_histogram.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t]
    L.ref_snr_estimator.argtypes = [C.c_uint, C.c_float, C.c_float, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    L.ref_carrier_detect.restype = C.c_float
    L.ref_carrier_detect.argtypes = [C.c_void_p, C.c_size_t, C.c_double, C.c_double]
    return L


def _ref_suscan():
    L = C.CDLL(REF2)
    L.ref_suscan_psd_message.restype = C.c_long
    L.ref_suscan_psd_message.argtypes = [C.c_void_p, C.c_ulong, C.c_double, C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ref_suscan_mq_samples.restype = C.c_long
    L.ref_suscan_mq_samples.argtypes = [C.c_void_p, C.c_ulong, C.c_uint, C.c_void_p, C.c_void_p]
    L.ref_suscan_status_message.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_size_t]
    return L


def _sview(L, fmin, fmax, feeds, rel_bw=0.5):
    v = C.c_void_p(L.ref_sview_new())
    L.ref_sview_set_range(v, C.c_double(fmin), C.c_double(fmax), C.c_double(feeds[0][2]), C.c_float(rel_bw))
    for psd, fc, bw in feeds:
        p = np.ascontiguousarray(psd, np.float32)
        L.ref_sview_feed(v, p.ctypes.data, None, C.c_ulong(len(p)), C.c_double(fc), 1)
    return v


def _sview_read(L, v):
    out = [np.zeros(65536, np.float32) for _ in range(3)]
    n = L.ref_sview_read(v, out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data)
    return [o[:n].copy() for o in out]


def record_sview(L):
    out = {}
    fmin, fmax, fftbw, psize, feeds = G.sview_case()
    v = _sview(L, fmin, fmax, feeds)
    out["sview_linear"] = np.stack(_sview_read(L, v))
    fmin2, fmax2, feeds2 = sview_hist_case()
    out["sview_histogram"] = np.stack(_sview_read(L, _sview(L, fmin2, fmax2, feeds2)))
    wide = C.c_void_p(L.ref_sview_new())
    L.ref_sview_set_range(wide, C.c_double(fmin + WIDE[0]), C.c_double(fmax + WIDE[1]), C.c_double(fftbw), C.c_float(0.5))
    L.ref_sview_feed_view(wide, v)
    out["sview_wide"] = np.stack(_sview_read(L, wide))
    return out


def record_timewindow(L):
    out = {}
    c = G.timewindow_case()
    x = c["tone"][:5000]
    y = np.zeros_like(x)
    L.ref_quad_demod(x.ctypes.data, y.ctypes.data, C.c_size_t(len(x)))
    out["quad_demod"] = y
    for delay in DELAYS:
        x = c["tone"][:3000]
        y = np.zeros_like(x)
        L.ref_delayed_conj(x.ctypes.data, y.ctypes.data, C.c_size_t(len(x)), C.c_ulong(delay))
        out["delayed_conj_%d" % delay] = y
    for space, sig in MANUAL:
        x = np.ascontiguousarray(c[sig][:6000])
        y = np.zeros(1024, np.complex64)
        n = L.ref_wave_sampler(x.ctypes.data, C.c_size_t(len(x)), 0, SPACE[space], C.c_double(1.0), C.c_double(0.1),
                               C.c_double(0.1), 0, C.c_float(0), C.c_float(0), C.c_float(1), C.c_float(0), C.c_size_t(5),
                               C.c_double(487.3), y.ctypes.data, None, C.c_size_t(1024))
        out["manual_" + space] = y[:n].copy()
    for i, (sig, space, amp, thr, zc, bnor) in enumerate(ZC_CASES):
        x = np.ascontiguousarray(c[sig])
        sym = np.zeros(len(x), np.uint8)
        n = L.ref_wave_sampler(x.ctypes.data, C.c_size_t(len(x)), 2, SPACE[space], C.c_double(1.0), C.c_double(bnor),
                               C.c_double(0.1), int(amp), C.c_float(thr.real), C.c_float(thr.imag), C.c_float(np.real(zc)),
                               C.c_float(np.imag(zc)), C.c_size_t(0), C.c_double(100.0), None, sym.ctypes.data,
                               C.c_size_t(len(x)))
        out["zero_crossing_%d" % i] = sym[:n].copy()
    x = np.ascontiguousarray(c["psk"])
    y = np.zeros(len(x), np.complex64)
    n = L.ref_wave_sampler(x.ctypes.data, C.c_size_t(len(x)), 1, SPACE["frequency"], C.c_double(1.0), C.c_double(1.0 / 12),
                           C.c_double(0.2), 0, C.c_float(0), C.c_float(0), C.c_float(1), C.c_float(0), C.c_size_t(0),
                           C.c_double(100.0), y.ctypes.data, None, C.c_size_t(len(x)))
    out["gardner_frequency"] = y[:n].copy()
    frames = averager_frames()
    for i, alpha in enumerate(ALPHAS):
        y = np.zeros(4096, np.float32)
        L.ref_averager(frames.ctypes.data, 7, 4096, C.c_float(alpha), y.ctypes.data)
        out["averager_%d" % i] = y
    return out


def record_tv(L, interlace, lines):
    x, sp, W, H, cap, block = tv_case(interlace, lines)
    y = np.zeros((cap, H, W), np.float32)
    w, h = C.c_int(), C.c_int()
    got = L.ref_tv_worker(C.byref(sp), x.ctypes.data, x.size, block, y.ctypes.data, cap, C.byref(w), C.byref(h))
    assert got > 0 and (w.value, h.value) == (W, H)
    return y[:got].copy()


def record_tasks(L, S):
    out = {}
    x = qpsk(TASK_N)
    y = np.zeros(TASK_N, np.complex64)
    for kind in (1, 2, 3):
        assert L.ref_task_costas(x.ctypes.data, y.ctypes.data, TASK_N, 10.0, 2e-3, kind) == 0
        out["costas_%d" % kind] = y.copy()
    for name, fn, args in (("pll", L.ref_task_pll, (5e-3,)), ("agc", L.ref_task_agc, (20.0,)),
                           ("xlate", L.ref_task_xlate, (0.0123, 0.5))):
        assert fn(x.ctypes.data, y.ctypes.data, TASK_N, *args) == 0
        out[name] = y.copy()
    x = qpsk(HIST_N, seed=8)
    for space in (0, 1, 2):
        got = np.zeros(HIST_N, np.float32)
        k = L.ref_task_histogram(x.ctypes.data, HIST_N, space, got.ctypes.data, HIST_N)
        out["histogram_%d" % space] = got[:k].copy()
    for bps, length, h in snr_cases():
        hs = np.ascontiguousarray(np.tile(h, (SNR_FEEDS, 1)))
        sig, snr, model = np.zeros(SNR_FEEDS, np.float32), np.zeros(SNR_FEEDS, np.float32), np.zeros(length, np.float32)
        assert L.ref_snr_estimator(bps, C.c_float(0.5), C.c_float(0.0), hs.ctypes.data, length, SNR_FEEDS,
                                   sig.ctypes.data, snr.ctypes.data, model.ctypes.data) == length
        out["snr_%d_sigma" % bps], out["snr_%d_snr" % bps], out["snr_%d_model" % bps] = sig, snr, model
    out["carrier_detect"] = np.array([L.ref_carrier_detect(x.ctypes.data, n, 0.01, notch)
                                      for n, f0, notch, x in carrier_cases()], np.float32)
    # the reference's C++ facade over libsuscan
    lin = psd_message_input()
    y = np.zeros(lin.size, np.float32)
    fc, rate = C.c_double(), C.c_uint()
    assert S.ref_suscan_psd_message(lin.ctypes.data, lin.size, 433.92e6, 2000000, y.ctypes.data, C.byref(fc),
                                    C.byref(rate)) == lin.size
    out["psd_message"], out["psd_message_fc_rate"] = y, np.array([fc.value, rate.value])
    x = mq_input()
    y = np.zeros_like(x)
    iid = C.c_uint()
    assert S.ref_suscan_mq_samples(x.ctypes.data, x.size, 0xBEEF, y.ctypes.data, C.byref(iid)) == x.size
    out["mq_samples"], out["mq_inspector_id"] = y, np.array(iid.value, np.uint32)
    buf = C.create_string_buffer(64)
    codes = [S.ref_suscan_status_message(-1, b"source failed to start", buf, 64)]
    texts = [buf.value.decode()]
    codes.append(S.ref_suscan_status_message(0, None, buf, 64))
    texts.append(buf.value.decode())
    out["status_codes"], out["status_texts"] = np.array(codes, np.int32), np.array(texts)
    return out


def main():
    import sigdigger_b200
    sigdigger_b200.load_library()
    L = _ref()
    rec = {}
    if os.path.exists(JSON):
        with open(JSON) as f:
            rec = json.load(f)
    if "--gpu" in sys.argv:
        x = lpf_input()
        y = np.zeros(LPF_N, np.complex64)
        assert L.ref_task_lpf(x.ctypes.data, y.ctypes.data, LPF_N, 0.2) == 0
        rec["lpf"] = digest(y)
    else:
        out = dict(record_sview(L), **record_timewindow(L), **record_tasks(L, _ref_suscan()))
        stored = {}
        for k, a in out.items():
            if k in STORED:
                stored[k] = sample(a) if k in SAMPLED else a
                rec[k] = {"len": len(a)}
            elif k in VALUES or k.startswith("snr_"):
                rec[k] = {"values": a.tolist()}
            else:
                rec[k] = digest(a)
        for interlace, lines in TV_CASES:
            rec["tv_%d" % lines] = [digest(f) for f in record_tv(L, interlace, lines)]
        np.savez_compressed(NPZ, **stored)
    with open(JSON, "w") as f:          # one entry per line
        f.write("{\n%s\n}\n" % ",\n".join("%s: %s" % (json.dumps(k), json.dumps(rec[k])) for k in sorted(rec)))
    for p in (JSON, NPZ):
        print(p, os.path.getsize(p))


if __name__ == "__main__":
    main()
