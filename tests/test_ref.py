"""CPU: the oracle pinned to the REFERENCE ITSELF where the reference contains the arithmetic.  The reference's own code
(Panoramic/Scanner.cpp:1-293, Tasks/QuadDemodTask.cpp, Tasks/DelayedConjTask.cpp, Tasks/WaveSampler.cpp,
Misc/Averager.cpp, Default/GenericInspector/TVProcessorWorker.cpp, the Tasks/ and Misc/ classes named below and the
Suscan/ C++ facade), compiled where it lies behind no-behaviour Qt stubs (oracle/ref_shim/, oracle/ref_glue*.cpp,
`make -C oracle ref`) and run on the inputs below, produced the fixtures tests/golden/ref_compiled.{json,npz}
(tests/golden/record_ref.py: digests of the outputs compared bit for bit, values of those compared to a tolerance);
nothing of the reference is copied.  The restatements of oracle/*.c are compared with those
outputs here; the Python transcriptions of tests/golden/make_golden.py stay as a second opinion."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

import record_ref as R      # noqa: E402


@pytest.fixture(scope="module")
def ref():
    return R.load()


def _sview_oracle(oracle, fmin, fmax, feeds, rel_bw=0.5):
    L = oracle.lib()
    v = oracle.SpectrumView()
    assert L.sdo_sview_init(C.byref(v)) == 0
    L.sdo_sview_set_range(C.byref(v), fmin, fmax)
    v.fft_bandwidth = feeds[0][2]
    v.fft_rel_bw = rel_bw
    for psd, fc, bw in feeds:
        p = np.ascontiguousarray(psd, np.float32)
        L.sdo_sview_feed(C.byref(v), oracle.ptr(p), None, len(p), float(fc), 1)
    n = v.spectrum_size
    return [np.ctypeslib.as_array(q, shape=(65536,))[:n].copy() for q in (v.psd, v.psd_accum, v.psd_count)], v


def test_spectrumview_restatement_equals_the_compiled_reference(ref, oracle):
    """linear mode with revisits (forgetting rule, gap filling), histogram mode, and view-to-view feed"""
    import make_golden as G
    fmin, fmax, fftbw, psize, feeds = G.sview_case()
    got, ov = _sview_oracle(oracle, fmin, fmax, feeds)
    assert R.same(ref["sview_linear"], np.stack(got))
    fmin2, fmax2, feeds2 = R.sview_hist_case()
    got, ov2 = _sview_oracle(oracle, fmin2, fmax2, feeds2)
    assert R.same(ref["sview_histogram"], np.stack(got))
    # SpectrumView::feed(SpectrumView const &): zoom path of Scanner::setViewRange
    L = oracle.lib()
    wide_o = oracle.SpectrumView(); assert L.sdo_sview_init(C.byref(wide_o)) == 0
    L.sdo_sview_set_range(C.byref(wide_o), fmin + R.WIDE[0], fmax + R.WIDE[1])
    wide_o.fft_bandwidth = fftbw; wide_o.fft_rel_bw = 0.5
    L.sdo_sview_feed_view(C.byref(wide_o), C.byref(ov))
    L.sdo_sview_interpolate(C.byref(wide_o))
    n = wide_o.spectrum_size
    assert R.same(ref["sview_wide"], np.stack([np.ctypeslib.as_array(q, shape=(65536,))[:n]
                                               for q in (wide_o.psd, wide_o.psd_accum, wide_o.psd_count)]))


def test_timewindow_tasks_equal_the_compiled_reference(ref, oracle):
    import make_golden as G
    c = G.timewindow_case()
    # QuadDemodTask: the reference calls std::arg (libm), the oracle its SPEC M atan2: equal to rounding
    x = c["tone"][:5000]
    y = ref["quad_demod"]["values"]
    o = np.empty_like(x)
    prev = oracle.Cpx(0, 0); primed = C.c_int(0)
    oracle.lib().sdo_quad_demod(oracle.ptr(x), oracle.ptr(o), len(x), C.byref(prev), C.byref(primed))
    assert y.shape == x.shape and y[0] == 0 and np.all(y.real == 0) and np.max(np.abs(y.imag - o.imag)) < 2e-7
    # DelayedConjTask: to one ulp of cabsf (libm's hypot vs sqrtf of the sum of squares)
    for delay in R.DELAYS:
        x = c["tone"][:3000]
        y = ref["delayed_conj_%d" % delay]["values"]
        o = oracle.delayed_conj(x, delay)
        assert y.shape == o.shape and np.max(np.abs(y - o)) <= 4e-7 * np.max(np.abs(y))
    # WaveSampler MANUAL in the three decision spaces: soft symbols bit for bit
    for space, sig in R.MANUAL:
        x = np.ascontiguousarray(c[sig][:6000])
        o = oracle.sample_manual(x, space, 487.3, 5)
        assert len(o) == 487 and R.same(ref["manual_" + space], o), space
    # WaveSampler ZERO_CROSSING: recovered bit streams bit for bit
    for i, (sig, space, amp, thr, zc, bnor) in enumerate(R.ZC_CASES):
        x = np.ascontiguousarray(c[sig])
        o, k = oracle.sample_zero_crossing(x, space, bnor, amp, thr, zc)
        assert len(o) == k and R.same(ref["zero_crossing_%d" % i], np.asarray(o, np.uint8)), (sig, space, amp)


def test_gardner_sampler_of_the_reference_over_the_clock_detector_shim(ref, oracle):
    """Tasks/WaveSampler.cpp sampleGardner() compiled from the reference, running on THIS repo's su_clock_detector
    (libsigutils.so): equal to the oracle's Gardner detector fed the same way."""
    import make_golden as G
    import shim_build as SB
    x = np.ascontiguousarray(G.timewindow_case()["psk"])
    want = SB.oracle_gardner_frequency(oracle, x, 0.2, 1.0 / 12)
    assert R.same(ref["gardner_frequency"], want)


def test_averager_restatement_equals_the_compiled_reference(ref, oracle):
    frames = R.averager_frames()
    for i, alpha in enumerate(R.ALPHAS):
        last = frames[0].copy()
        L = oracle.lib()
        for f in range(1, 7):
            if alpha < 1.0:
                L.sdo_averager_feed(oracle.ptr(last), oracle.ptr(np.ascontiguousarray(frames[f])), 4096, C.c_float(alpha))
            else:
                last = frames[f].copy()
        assert R.same(ref["averager_%d" % i], last), alpha


@pytest.mark.parametrize("interlace,lines", R.TV_CASES)
def test_tv_worker_of_the_reference_over_the_tvproc_shim(ref, oracle, interlace, lines):
    """Default/GenericInspector/TVProcessorWorker.cpp COMPILED FROM THE REFERENCE (setParams / start / pushData /
    process / work with its acknowledgement window / returnFrame) drove this repo's <sigutils/tvproc.h> unmodified:
    the frames it emitted are, bit for bit, the oracle's (SPEC TV) and those of the reference-shaped TU."""
    import shim_build as SB
    import test_oracle_tv as T
    frames = ref["tv_%d" % lines]
    got = len(frames)
    x, sp, W, H, cap, block = R.tv_case(interlace, lines)
    assert got >= 5
    out_tu = np.zeros((cap, H, W), np.float32)
    w, h = C.c_int(), C.c_int()
    assert SB.reference_tu().tu_tv_worker(C.byref(sp), x.ctypes.data, x.size, block, out_tu.ctypes.data, cap,
                                          C.byref(w), C.byref(h)) == got
    assert (w.value, h.value) == (W, H)
    assert all(R.same(f, o) for f, o in zip(frames, out_tu)) and not out_tu[got:].any()
    t = T.OracleTv(T.toy_params(lines, interlace, 4))
    k = 0
    for p0 in range(0, x.size, block):
        blk, sent = x[p0:p0 + block], False
        for pos in range(0, blk.size, 64):
            f0 = t.frames
            t.feed(blk[pos:pos + 64])
            if t.frames > f0 and not sent:
                assert R.same(frames[k], t.frame(f0))
                k, sent = k + 1, True
    assert k == got
    t.close()


def test_psd_message_of_the_reference_over_the_shim_headers(ref, oracle):
    """Suscan/Messages/PSDMessage.cpp + Suscan/Message.cpp COMPILED FROM THE REFERENCE against include/analyzer/msg.h:
    the constructor's fft-shift + SU_POWER_DB pass (:26-39) is the reference's own; the oracle's sdo_psd_shift_db
    (= the PSD kernels' SDB_FLAG_PSD_SHIFT_DB epilogue, bit for bit) is held to it -- the layout exactly, the values to
    the difference between libm's log10f and the SPEC M polynomial."""
    lin = R.psd_message_input()
    n = lin.size
    out = ref["psd_message"]["values"]
    fc, rate = ref["psd_message_fc_rate"]["values"]
    assert out.shape == (n,) and fc == 433920000.0 and rate == 2000000
    mine = lin.copy()
    oracle.lib().sdo_psd_shift_db(oracle.ptr(mine), n)
    assert np.all(np.isfinite(out)) and out.min() >= -80.0 - 1e-3          # the 1e-8 floor of SU_POWER_DB
    assert np.max(np.abs(out - mine)) < 2e-5                                # dB; same bins in the same places
    want = 10.0 * np.log10(np.concatenate([lin[n // 2:], lin[:n // 2]]).astype(np.float64) + 1e-8)
    assert np.max(np.abs(out - want)) < 2e-5


class _SampleBatch(C.Structure):      # struct suscan_analyzer_sample_batch_msg (include/analyzer/msg.h)
    _fields_ = [("inspector_id", C.c_uint32), ("samples", C.c_void_p), ("sample_count", C.c_uint64),
                ("symbols", C.c_void_p)]


def test_mq_and_message_wrappers_of_the_reference_over_libsuscan(ref):
    """Suscan/MQ.cpp (caller-owned suscan_mq: init / read / finalize), SamplesMessage and StatusMessage over the shim
    library: a SAMPLES payload posted with suscan_mq_write came back through the reference's wrapper classes as posted.
    libsuscan's queue hands the same payload back here, and the recorded status messages carry the posted code / text."""
    import sigdigger_b200
    sigdigger_b200.load_library()
    S = C.CDLL(os.path.join(ROOT, "sigdigger_b200", "libsuscan.so"))
    S.suscan_mq_init.argtypes = S.suscan_mq_finalize.argtypes = [C.c_void_p]
    S.suscan_mq_write.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    S.suscan_mq_read.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    S.suscan_mq_read.restype = C.c_void_p
    x = R.mq_input()
    assert R.same(ref["mq_samples"], x) and ref["mq_inspector_id"]["values"] == 0xBEEF
    mq = C.c_void_p()                                          # struct suscan_mq { void *impl; }
    assert S.suscan_mq_init(C.byref(mq))
    m = _SampleBatch(0xBEEF, x.ctypes.data, x.size, None)
    assert S.suscan_mq_write(C.byref(mq), 6, C.byref(m))        # SUSCAN_ANALYZER_MESSAGE_TYPE_SAMPLES
    t = C.c_uint32()
    p = S.suscan_mq_read(C.byref(mq), C.byref(t))
    S.suscan_mq_finalize(C.byref(mq))
    assert t.value == 6 and p == C.addressof(m)
    back = _SampleBatch.from_address(p)
    assert back.inspector_id == 0xBEEF and back.sample_count == x.size
    assert R.same(ref["mq_samples"], np.ctypeslib.as_array((C.c_float * (2 * x.size)).from_address(back.samples))
                  .view(np.complex64))
    assert ref["status_codes"]["values"] == [-1, 0]
    assert ref["status_texts"]["values"] == ["source failed to start", ""]


def test_tasks_of_the_reference_over_the_sigutils_shim(ref, oracle):
    """Tasks/CostasRecoveryTask.cpp, PLLSyncTask.cpp, AGCTask.cpp, CarrierXlator.cpp COMPILED FROM THE REFERENCE
    (constructor + work() loops, `destination[p] = su_costas_feed(&costas, origin[p])`) over this repo's
    <sigutils/{pll,agc,ncqo}.h> and libsigutils.so: the north-star's "Tasks/ are drop-in".  Outputs equal the oracle's
    bit for bit (the shim's per-sample entry points run the kernels' step functions on the host)."""
    import shim_build as SB
    x = R.qpsk(R.TASK_N)
    for kind in (1, 2, 3):
        assert R.same(ref["costas_%d" % kind], SB.oracle_costas(oracle, x, kind, 0.1, 2e-3))
    assert R.same(ref["pll"], SB.oracle_pll(oracle, x, 5e-3))
    assert R.same(ref["agc"], SB.oracle_agc(oracle, x, 20.0))
    assert R.same(ref["xlate"], SB.oracle_xlate(oracle, x, 0.0123, 0.5))


def test_histogram_feeder_of_the_reference(ref, oracle):
    """Tasks/HistogramFeeder.cpp compiled from the reference against the oracle's restatement (SPEC Y.2): amplitude
    exactly; phase / frequency to one ulp of libm's cargf against the SPEC M atan2 (on the recorded strided sample)."""
    L = oracle.lib()
    L.sdo_histogram_feed.restype = C.c_size_t
    L.sdo_histogram_feed.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    n = R.HIST_N
    x = R.qpsk(n, seed=8)
    for space, tol in ((0, 0.0), (1, 4e-7), (2, 4e-7)):
        k = ref["histogram_%d" % space]["len"]
        mine = np.zeros(n, np.float32)
        m = L.sdo_histogram_feed(x.ctypes.data, mine.ctypes.data, n, space)
        assert k == m == (n - 1 if space == 2 else n)
        got, mine = ref["histogram_%d" % space]["values"], R.sample(mine[:k])
        k = len(got)
        assert k == len(mine)
        if tol == 0.0:
            assert np.max(np.abs(got[:k] - mine[:k]) / np.maximum(np.abs(mine[:k]), 1e-30)) < 2e-7   # cabsf vs SPEC M
        else:
            d = np.abs(got[:k] - mine[:k])
            d = np.minimum(d, np.abs(d - 2 * np.pi))                  # +-pi branch
            assert d.max() < tol


def test_snr_estimator_restatement_tracks_the_compiled_reference(ref, oracle):
    """Misc/SNREstimator.cpp compiled from the reference against the oracle's restatement (SPEC Y.7): same trajectory
    of sigma over successive feeds and the same model histogram, to the difference between libm's exp and SPEC M's."""
    for bps, length, h in R.snr_cases():
        sig, snr, model = (np.array(ref["snr_%d_%s" % (bps, k)]["values"], np.float32) for k in ("sigma", "snr", "model"))
        assert len(sig) == len(snr) == R.SNR_FEEDS and len(model) == length
        e = oracle.SnrEstimator(bps, length, alpha=0.5)
        for f in range(R.SNR_FEEDS):
            e.feed(h)
            assert abs(e.sigma - sig[f]) <= 5e-5 * abs(sig[f]), (bps, f, e.sigma, sig[f])
            assert abs(e.snr - snr[f]) <= 1e-4 * abs(snr[f])
        assert np.abs(e.model() - model).max() < 5e-5
        e.close()


def test_carrier_detector_restatement_tracks_the_compiled_reference(ref, oracle):
    """Tasks/CarrierDetector.cpp compiled from the reference (Blackman-Harris taps from this repo's <sigutils/taps.h>,
    its FFT through a binary64 stand-in for FFTW) against sdo_carrier_detect (SPEC Y.5, binary32 SPEC transform): the
    same peak to the transforms' rounding."""
    want = ref["carrier_detect"]["values"]
    cases = list(R.carrier_cases())
    assert len(want) == len(cases)
    for got, (n, f0, notch, x) in zip(want, cases):
        got = float(got)
        mine = float(oracle.carrier_detect(x, 0.01, notch))
        assert abs(got - mine) < 2e-5, (n, f0, got, mine)
        assert abs(got - 2 * np.pi * f0) < 2e-3 or notch > 0
