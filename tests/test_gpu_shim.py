"""-m gpu: the drop-in boundary (SURVEY.md 8(b)).  tests/shim/reference_tu.cpp -- the calling code of the reference's
Tasks/ objects and of Suscan::Analyzer, Qt removed -- is compiled with g++ against include/sigutils/*.h and
include/analyzer/*.h, linked with libsigutils.so / libsuscan.so, and its results are compared with the oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import parity
from sigdigger_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


import shim_build as SB


@pytest.fixture(scope="module")
def tu(sdb):
    return SB.reference_tu()


def _sig(n, seed=5):
    x, _ = synth.multi_carrier(n, 1.0, [("qpsk", 0.01, 0.1, -6.0, {})], noise_db=-40.0, seed=seed)
    return np.ascontiguousarray(x, np.complex64)


def test_costas_task_through_the_sigutils_names(tu, oracle):
    """su_costas_init(&costas, kind, 0, bw, 3, loopbw) + the per-sample su_costas_feed loop of
    Tasks/CostasRecoveryTask.cpp:36-61, and the same blocks through su_costas_feed_bulk (device, state in / out):
    both bit-identical to the oracle's Costas loop."""
    n = 3 * 4096 + 777
    x = _sig(n)
    for kind in (1, 2, 3):
        ref = SB.oracle_costas(oracle, x, kind, 0.1, 2e-3)
        for bulk in (0, 1):
            y = np.zeros(n, np.complex64)
            assert tu.tu_costas_task(x.ctypes.data, y.ctypes.data, C.c_size_t(n), C.c_float(10.0), C.c_float(2e-3), kind, bulk) == 0
            assert np.array_equal(y.view(np.uint32), ref.view(np.uint32)), (kind, bulk)


def test_pll_agc_xlate_tasks_through_the_sigutils_names(tu, oracle, sdb):
    n = 2 * 4096 + 100
    x = _sig(n, seed=6)
    ref = SB.oracle_pll(oracle, x, 5e-3)
    for bulk in (0, 1):
        y = np.zeros(n, np.complex64)
        assert tu.tu_pll_task(x.ctypes.data, y.ctypes.data, C.c_size_t(n), C.c_float(5e-3), bulk) == 0
        assert np.array_equal(y.view(np.uint32), ref.view(np.uint32)), bulk
    y = np.zeros(n, np.complex64)
    assert tu.tu_agc_task(x.ctypes.data, y.ctypes.data, C.c_size_t(n), C.c_float(20.0)) == 0
    ref = SB.oracle_agc(oracle, x, 20.0)
    assert np.array_equal(y.view(np.uint32), ref.view(np.uint32))
    for bulk in (0, 1):
        y = np.zeros(n, np.complex64)
        assert tu.tu_xlate_task(x.ctypes.data, y.ctypes.data, C.c_size_t(n), C.c_float(0.0123), C.c_float(0.5), bulk) == 0
        ref = sdb.carrier_xlate(x, 0.0123, 0.5)       # the engine's CarrierXlator task (itself oracle-checked)
        assert np.array_equal(y.view(np.uint32), ref.view(np.uint32)), bulk


def test_gardner_and_lpf_tasks_through_the_sigutils_names(tu, oracle, sdb):
    n = 5 * 4096
    x = _sig(n, seed=7)
    out = np.zeros(n, np.complex64)
    got = tu.tu_gardner_task(x.ctypes.data, C.c_size_t(n), C.c_float(0.1), C.c_float(0.1), out.ctypes.data, C.c_size_t(n))
    ref = SB.oracle_gardner_frequency(oracle, x, 0.1, 0.1)
    assert got == len(ref) and np.array_equal(out[:got].view(np.uint32), ref.view(np.uint32))
    # LPFTask: the specttuner shim against the engine's own LPF task (same kernels, block-wise feed vs one call)
    y = np.zeros(n, np.complex64)
    assert tu.tu_lpf_task(x.ctypes.data, y.ctypes.data, C.c_size_t(n), C.c_float(0.2)) == 0
    ref = sdb.lpf(x, 0.2)
    assert np.array_equal(y.view(np.uint32), ref.view(np.uint32))


def test_analyzer_session_through_the_suscan_names(tu, oracle):
    """Suscan::Analyzer's constructor / reader thread / openEx / setInspectorConfig / destructor against libsuscan.so:
    caller-owned suscan_mq, OPEN -> SET_ID -> SET_CONFIG handshake with a suscan_config_t bag, SAMPLES keyed by the
    caller's inspector id, every PSD frame, EOS.  Symbols bit-identical to the oracle from the block the
    configuration went live."""
    N, fs = 8192, 1000000
    baud = fs / 100.0
    blocks, per_block = 8, N * 4
    n = blocks * per_block
    x, _ = synth.multi_carrier(n, float(fs), [("qpsk", 0.125 * fs + 3.0, baud, -10.0, {})], noise_db=-50.0, seed=33)
    x = np.ascontiguousarray(x, np.complex64)
    fs_ch = fs * 256 / N
    cap = n
    soft = np.zeros(cap, np.complex64); hard = np.zeros(cap, np.uint8); psd = np.zeros(N, np.float32)
    cnt = C.c_ulong(0)
    got = tu.tu_analyzer_session(x.ctypes.data, n, fs, N, per_block, 0.125 * fs, 3 * baud, baud, fs_ch * 2e-3,
                                 soft.ctypes.data, hard.ctypes.data, cap, psd.ctypes.data, C.addressof(cnt))
    assert got > 0, got
    assert cnt.value == n // N
    ref_psd = oracle.psd_frames(x, N, "blackmann_harris")
    assert np.array_equal(psd.view(np.uint32), ref_psd[-1].view(np.uint32))
    # channel from block 2 on; blocks 2 and 3 ran the default configuration (matched filter bypassed, clock not
    # running: no samples), the new one (structural change -> fresh loops) is live from block 4
    kw = dict(baud=baud, costas_order=2, bits_per_symbol=2, loop_bw=fs_ch * 2e-3, mf_type=1, mf_rolloff=0.35,
              clock_type=1, clock_gain=0.1, clock_running=1)
    ic = oracle.insp_config("psk", fs_ch, **kw)
    f0, bw = float(np.float32(2.0 * np.pi * 0.125)), float(np.float32(2.0 * np.pi * (3 * baud) / fs))
    ref = oracle.analyzer_run(oracle.make_an_params(N, "blackmann_harris", [(f0, bw, 1.0, 0, ic)]), x[per_block:])
    chan = ref["chan"][0]
    hops = per_block // (N // 2)
    skip = (hops - 1) * 128 + hops * 128           # channel samples of blocks 2 and 3 (halfsz = 128)
    rs, rh = oracle.inspector_run(ic, chan[skip:])
    parity.assert_symbols_match(soft[:got], hard[:got], rs, rh, exact_soft=True)


def test_lpf_task_of_the_reference_over_the_specttuner_shim(oracle, sdb):
    """Tasks/LPFTask.cpp COMPILED FROM THE REFERENCE (su_specttuner_new / open_channel with guard = 2 pi / bw /
    feed_bulk / the zero flush of :104-107) over <sigutils/specttuner.h>, whose tuner is an engine on the GPU: its
    output, recorded in tests/golden/ref_compiled.json (tests/golden/record_ref.py --gpu), is the engine's own LPF
    task's, bit for bit."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import record_ref as R
    assert R.same(R.load()["lpf"], sdb.lpf(R.lpf_input(), 0.2))
