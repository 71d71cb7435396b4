"""-m gpu: every main-PSD size and every channeliser window / inverse size the CUDA path dispatches differently
(k_small_psd at N <= 4096, the F.4 / F.5 register passes, the generic four-step passes over several scratch chunks,
k_chan_ifft16 and k_chan_ifft<1, 2, 4>), each held to two references: the oracle bit for bit, and the float64
restatement of tests/f64_ref.py within the tolerances of tests/parity.py.  The second catches what the first cannot:
a mistake that the oracle and the kernels share."""
import numpy as np
import pytest

import f64_ref
import parity
import size_cases as sc

pytestmark = pytest.mark.gpu


def _same_bits(a, b):
    return np.asarray(a).shape == np.asarray(b).shape and np.array_equal(np.asarray(a).view(np.uint32),
                                                                         np.asarray(b).view(np.uint32))


def _psd_frames(N):
    """Frames per stream (2 streams): at least two, and past 2^17 enough to span several scratch chunks of the
    generic four-step path (64 MB / (8 N) windows: 32 at 2^18, 16 at 2^19, 8 at 2^20)."""
    return {1 << 18: 17, 1 << 19: 9, 1 << 20: 5}.get(N, 2)


# ------------------------------------------------------------------------------------------------
# main PSD
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", sc.PSD_SIZES)
def test_psd_size_paths(sdb, oracle, N):
    S, frames, kind = 2, _psd_frames(N), sc.psd_window(N)
    x = np.stack([sc.psd_input(N, frames, seed=N % 101 + s) for s in range(S)])
    # the channeliser window defaults to psd_size and has a floor of 64, so the two smallest PSDs name one
    e = sdb.Engine(n_streams=S, psd_size=N, psd_window=kind, max_feed=N * frames, st_window_size=max(N, 64))
    e.commit()
    e.feed(x)
    got = e.read_psd()
    for s in range(S):
        assert _same_bits(got[s], oracle.psd_frames(x[s], N, kind)), "stream %d not bit-identical" % s
        parity.assert_psd_close(got[s], f64_ref.psd_f64(x[s], N, kind))


@pytest.mark.parametrize("N", [256, 4096, 1 << 17, 1 << 20])
def test_psd_shift_db_size_paths(sdb, oracle, N):
    import torch
    S, frames, kind = 2, _psd_frames(N), "hann"
    x = np.stack([sc.psd_input(N, frames, seed=7 + s) for s in range(S)])
    e = sdb.Engine(n_streams=S, psd_size=N, psd_window=kind, max_feed=N * frames, flags=sdb.FLAG_PSD_SHIFT_DB)
    e.commit()
    e.feed(x)
    got = e.read_psd()
    lin = sdb.Engine(n_streams=S, psd_size=N, psd_window=kind, max_feed=N * frames)
    lin.commit()
    lin.feed(x)
    dl = torch.from_numpy(lin.read_psd()).cuda()
    db = torch.empty_like(dl)
    sdb.psd_shift_db(dl.data_ptr(), db.data_ptr(), S * frames, N)
    torch.cuda.synchronize()
    assert _same_bits(got, db.cpu().numpy()), "fused epilogue differs from the linear PSD + sdb.psd_shift_db"
    for s in range(S):
        ref = oracle.psd_frames(x[s], N, kind)
        for f in range(frames):
            oracle.lib().sdo_psd_shift_db(oracle.ptr(ref[f]), N)
        assert _same_bits(got[s], ref), "stream %d not bit-identical" % s
        # float64: the PSD tolerance carried through 10 log10, plus the float32 rounding of the dB value
        p = f64_ref.psd_f64(x[s], N, kind)
        M, Pmax = p.mean(axis=-1, keepdims=True), p.max(axis=-1, keepdims=True)
        tol = (parity.PSD_RTOL * p + parity.PSD_FLOOR * np.sqrt(p * M) + parity.PSD_LINE * np.sqrt(p * Pmax)
               + 1e-11 * M)
        tol_db = 10 / np.log(10) * np.fft.fftshift(tol / (p + 1e-8), axes=-1)
        ref_db = f64_ref.shift_db_f64(p)
        tol_db += 1e-6 * (np.abs(ref_db) + 1)
        worst = float(np.max(np.abs(got[s] - ref_db) / tol_db))
        assert worst <= 1.0, "dB PSD mismatch: worst bin at %.2f x tolerance" % worst


# ------------------------------------------------------------------------------------------------
# channeliser
# ------------------------------------------------------------------------------------------------
def _run_channels(sdb, W, chans, x, split, psd_size=0, psd_window="hann"):
    """One engine over x fed in pieces of `split` samples -> (per-channel outputs, channel infos, PSD or None)."""
    e = sdb.Engine(n_streams=1, psd_size=psd_size, psd_window=psd_window, st_window_size=W, max_feed=max(split))
    hs = [e.open_channel(c["f0"], c["bw"], c["guard"], c["precise"]) for c in chans]
    e.commit()
    outs, psd, off = [[] for _ in hs], [], 0
    for m in split:
        e.feed(x[None, off:off + m])
        off += m
        for i, h in enumerate(hs):
            outs[i].append(e.read_channel(0, h))
        if psd_size:
            psd.append(e.read_psd()[0].copy())
    infos = [e.channel_info(h) for h in hs]
    e.close()
    return [np.concatenate(o) for o in outs], infos, (np.concatenate(psd) if psd_size else None)


@pytest.mark.parametrize("W", sc.TUNER_WINDOWS)
def test_channeliser_size_paths(sdb, oracle, W):
    x = sc.tuner_input(W)
    chans = sc.channel_set(W)
    got, infos, _ = _run_channels(sdb, W, chans, x, [len(x)])
    ragged, _, _ = _run_channels(sdb, W, chans, x, sc.ragged_split(W, len(x)))
    ref = oracle.specttuner_run(x, W, chans)
    x_rms = float(np.sqrt(np.mean(np.abs(x) ** 2)))
    for i, (c, g, r, info) in enumerate(zip(chans, got, ref, infos)):
        assert info.size == f64_ref.channel_geometry(W, c["f0"], c["bw"], c["guard"])[1]
        assert len(g) == (sc.tuner_halves(W) - 1) * info.size // 2
        assert _same_bits(g, r), "channel %d (size %d) not bit-identical to the oracle" % (i, info.size)
        assert _same_bits(ragged[i], g), "channel %d (size %d): ragged feeds differ from one feed" % (i, info.size)
        parity.assert_channel_close(g, f64_ref.specttuner_f64(x, W, c["f0"], c["bw"], c["guard"], c["precise"]),
                                    x_rms, info.decimation)


@pytest.mark.parametrize("W", [64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384])
def test_fullband_channel_is_a_frequency_shift(sdb, oracle, W):
    """bw = 2 pi, guard = 1: the inverse size equals the window (k_chan_ifft<4> at 16384), and the output is the
    input moved down by the even centre bin -- and with `precise` also by the float32 LO phase."""
    n = W // 2 * 12
    x = sc.noise(n, seed=W)
    chans = [sc.fullband_channel(W, False), sc.fullband_channel(W, True)]
    got, infos, _ = _run_channels(sdb, W, chans, x, [n])
    ref = oracle.specttuner_run(x, W, chans)
    for c, g, r, info in zip(chans, got, ref, infos):
        assert info.size == info.width == W
        assert _same_bits(g, r), "precise=%s not bit-identical to the oracle" % c["precise"]
        phi = (f64_ref.ncqo_phases(f64_ref.lo_fnor(W, c["f0"], info.center, W), len(g)) if c["precise"] else None)
        assert np.abs(g - sc.fullband_expected(x[:len(g)], W, info.center, phi)).max() < 3e-6


@pytest.mark.parametrize("W", [8192, 65536])
def test_precise_tone_known_answer(sdb, W):
    c, delta = sc.precise_tone_case(W)
    x = sc.precise_tone_input(W, 16, c, delta)
    (y,), (info,), _ = _run_channels(sdb, W, [c], x, [len(x)])
    sc.assert_precise_tone(y, info.size, delta * info.decimation)


@pytest.mark.parametrize("psd_size,W", [(65536, 4096), (4096, 65536), (1 << 17, 8192)])
def test_mixed_psd_and_tuner_plans(sdb, oracle, psd_size, W):
    """psd_size != st_window_size in one engine: the scratch is sized for the larger plan and shared by both
    chains; both must equal single-purpose engines and the oracle."""
    step = max(psd_size, W // 2)
    n = step * max(3, 6 * (W // 2) // step)
    x = sc.noise(n, 5, 0.3)
    chans = sc.channel_set(W)[:2] + sc.channel_set(W)[-2:]
    split = [step, n - step]
    got, _, psd = _run_channels(sdb, W, chans, x, split, psd_size=psd_size, psd_window="hann")
    alone, _, _ = _run_channels(sdb, W, chans, x, split)
    p = sdb.Engine(n_streams=1, psd_size=psd_size, psd_window="hann", max_feed=n)
    p.commit()
    p.feed(x[None, :])
    assert _same_bits(psd, p.read_psd()[0])
    assert _same_bits(psd, oracle.psd_frames(x, psd_size, "hann"))
    for g, a, r in zip(got, alone, oracle.specttuner_run(x, W, chans)):
        assert _same_bits(g, a) and _same_bits(g, r)


def test_channel_size_limit(sdb):
    e = sdb.Engine(n_streams=1, psd_size=0, st_window_size=65536, max_feed=65536)
    h = e.open_channel(1.0, 2 * np.pi * 0.2)                   # 13108 bins -> 16384: the largest inverse size
    assert e.channel_info(h).size == 16384
    with pytest.raises(sdb.SdbError):
        e.open_channel(1.0, 2 * np.pi * 0.3)                   # 19661 bins -> 32768
