"""CPU tests (-m "not gpu"): the oracle against the float64 restatements of tests/f64_ref.py at every PSD size and
every channeliser window and inverse size the CUDA path dispatches differently (tests/size_cases.py).  The GPU tests
(tests/test_gpu_sizes.py) hold the kernels to the same references, so a mistake the oracle and the kernels share
cannot hide behind their bit-identity."""
import ctypes as C

import numpy as np
import pytest

import f64_ref
import parity
import size_cases as sc


def test_size_cases_cover_every_path():
    sizes, odd, precise, plain, below_dc, above_dc, wraps = set(), False, False, False, False, False, False
    for W in sc.TUNER_WINDOWS:
        for c in sc.channel_set(W):
            center, size, width = f64_ref.channel_geometry(W, c["f0"], c["bw"], c["guard"])
            sizes.add(size)
            odd |= width % 2 == 1
            precise |= c["precise"]
            plain |= not c["precise"]
            below_dc |= 0 < center < width // 2
            above_dc |= center + width // 2 > W
            wraps |= center == 0 and c["f0"] > np.pi
    assert sizes == set(sc.CHAN_SIZES)
    assert odd and precise and plain and below_dc and above_dc and wraps


@pytest.mark.parametrize("W", sc.TUNER_WINDOWS)
def test_geometry_and_weights_match_oracle(oracle, W):
    chans = sc.channel_set(W) + [sc.fullband_channel(W)] if W <= 16384 else sc.channel_set(W)
    for c in chans:
        cen, size, width = f64_ref.channel_geometry(W, c["f0"], c["bw"], c["guard"])
        assert (cen, size, width) == oracle.channel_geometry(W, c["f0"], c["bw"], c["guard"]), c
        h = np.empty(W, np.float32)
        oracle.lib().sdo_st_filter_response(W, width // 2, h.ctypes.data_as(C.POINTER(C.c_float)))
        assert np.abs(h / W - f64_ref.channel_weights(W, width // 2)).max() <= 6e-8 / W


def test_ncqo_phases_match_oracle(oracle):
    for fnor in (3e-4, -2.5e-3, 0.4, -0.9):
        o = oracle.Ncqo()
        oracle.lib().sdo_ncqo_init(C.byref(o), C.c_float(fnor))
        n = 3000
        ref = np.empty(n, np.float32)
        for i in range(n):
            ref[i] = o.phi
            oracle.lib().sdo_ncqo_read(C.byref(o))
        assert np.array_equal(f64_ref.ncqo_phases(fnor, n).view(np.uint32), ref.view(np.uint32)), fnor


@pytest.mark.parametrize("N", sc.PSD_SIZES)
def test_oracle_psd_vs_f64(oracle, N):
    kind = sc.psd_window(N)
    x = sc.psd_input(N, 2, seed=N % 101)
    assert np.abs(oracle.window(N, kind) - f64_ref.window(N, kind)).max() <= 6e-8
    parity.assert_psd_close(oracle.psd_frames(x, N, kind), f64_ref.psd_f64(x, N, kind))


@pytest.mark.parametrize("W", sc.TUNER_WINDOWS)
def test_oracle_specttuner_vs_f64(oracle, W):
    x = sc.tuner_input(W)
    chans = sc.channel_set(W)
    got = oracle.specttuner_run(x, W, chans)
    x_rms = float(np.sqrt(np.mean(np.abs(x) ** 2)))
    for c, g in zip(chans, got):
        _, size, _ = f64_ref.channel_geometry(W, c["f0"], c["bw"], c["guard"])
        ref = f64_ref.specttuner_f64(x, W, c["f0"], c["bw"], c["guard"], c["precise"])
        assert len(g) == len(ref) == (sc.tuner_halves(W) - 1) * size // 2
        parity.assert_channel_close(g, ref, x_rms, W // size)


@pytest.mark.parametrize("W", [64, 256, 4096, 16384])
@pytest.mark.parametrize("precise", [False, True])
def test_oracle_fullband_is_a_frequency_shift(oracle, W, precise):
    n = W // 2 * 12
    x = sc.noise(n, seed=W + precise)
    c = sc.fullband_channel(W, precise)
    center, size, width = f64_ref.channel_geometry(W, c["f0"], c["bw"], c["guard"])
    assert size == width == W and center % 2 == 0
    y = oracle.specttuner_run(x, W, [c])[0]
    phi = f64_ref.ncqo_phases(f64_ref.lo_fnor(W, c["f0"], center, size), len(y)) if precise else None
    ref = sc.fullband_expected(x[:len(y)], W, center, phi)
    assert np.abs(y - ref).max() < 3e-6


def test_oracle_precise_tone(oracle):
    W = 8192
    c, delta = sc.precise_tone_case(W)
    x = sc.precise_tone_input(W, 24, c, delta)
    _, size, _ = f64_ref.channel_geometry(W, c["f0"], c["bw"], c["guard"])
    sc.assert_precise_tone(oracle.specttuner_run(x, W, [c])[0], size, delta * (W // size))
