"""Inputs and channel sets for the size-path tests: every main-PSD size and every channeliser window the engine
dispatches differently, shared by the CPU tests (oracle vs float64) and the GPU tests (kernels vs oracle and float64).
"""
import numpy as np

PSD_SIZES = [1 << k for k in range(4, 21)]
TUNER_WINDOWS = [64, 128, 256, 1024, 2048, 4096, 8192, 16384, 32768, 65536, 1 << 17, 1 << 20]
CHAN_SIZES = [1 << k for k in range(2, 15)]            # inverse transforms 4 ... 16384

# inverse sizes per window: a child engine's window is its parent's channel size, so the small windows matter
_SIZES = {64: (4, 8, 16, 32, 64), 128: (8, 32, 128), 256: (16, 64, 256), 1024: (4, 128, 512, 1024),
          2048: (32, 256, 2048), 4096: (8, 512, 4096), 8192: (64, 1024, 8192), 16384: (16, 2048, 16384),
          32768: (4, 4096, 16384), 65536: (32, 8192, 16384), 1 << 17: (8, 1024, 16384), 1 << 20: (4, 2048, 16384)}


def psd_window(N):
    return ("hann", "flat_top", "blackmann_harris", "hamming", "none")[N.bit_length() % 5]


def noise(n, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    return ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * scale).astype(np.complex64)


def psd_input(N, frames, seed):
    t = np.arange(N * frames)
    x = noise(N * frames, seed, 0.3) + (0.5 * np.exp(2j * np.pi * 0.1234 * t)).astype(np.complex64)
    return x.astype(np.complex64)


def _bw_for(W, bins, guard):
    """bw such that S.2 keeps `bins` bins: guard * bw / 2 pi * W = bins - 0.5, which ceil() takes to `bins`."""
    return float(np.float32(2 * np.pi * (bins - 0.5) / W / guard))


def channel_set(W):
    """Channels for a window of W: one per inverse size of _SIZES[W] (guards 1, 1.5, 2 in turn, every other one
    precise, odd widths at guard 1), plus a precise channel straddling DC from below (small f0), a precise channel
    from just under 2 pi whose centre bin wraps to 0, and a channel centred on bin W - 2 whose upper bins wrap past
    W."""
    chans = []
    for i, s in enumerate(_SIZES[W]):
        bins = max(4, 3 * s // 4 + 1)                   # in (s/2, s]: the inverse size is s
        guard = (1.0, 1.5, 2.0)[i % 3]
        f0 = 2 * np.pi * ((0.137 + 0.29 * i) % 1.0)
        chans.append(dict(f0=float(np.float32(f0)), bw=_bw_for(W, bins, guard), guard=guard, precise=i % 2 == 1))
    wide = min(max(8, W // 16), 4096)
    chans.append(dict(f0=float(np.float32(2 * np.pi * 1.8 / W)), bw=_bw_for(W, wide, 1.0), guard=1.0, precise=True))
    chans.append(dict(f0=float(np.float32(2 * np.pi * (1 - 0.7 / W))), bw=_bw_for(W, max(6, W // 64), 1.0),
                      guard=1.0, precise=True))
    chans.append(dict(f0=float(np.float32(2 * np.pi * (1 - 2.6 / W))), bw=_bw_for(W, min(max(8, W // 32), 4096), 1.0),
                      guard=1.0, precise=False))
    return chans


def tuner_halves(W):
    """Input length in half windows: enough hops for the small windows, a few for the big ones (CPU oracle cost)."""
    return 40 if W <= 4096 else (12 if W <= 65536 else 5)


def tuner_input(W, seed=None):
    """Noise plus a tone inside every channel of channel_set(W), slightly off its centre."""
    n = W // 2 * tuner_halves(W)
    x = noise(n, W % 1009 if seed is None else seed, 0.05)
    t = np.arange(n)
    for i, c in enumerate(channel_set(W)):
        f = c["f0"] / (2 * np.pi) + 0.2 * c["bw"] / (2 * np.pi) / c["guard"]
        x += (0.3 * np.exp(2j * np.pi * f * t + 1j * i)).astype(np.complex64)
    return x


def ragged_split(W, n):
    """Feed lengths (multiples of W/2) of uneven size that add up to n."""
    h, left, out, k = W // 2, n // (W // 2), [], 1
    while left > 0:
        take = min(k, left)
        out.append(take * h)
        left -= take
        k = k * 2 + 1
    return out


# ---- known answers that do not depend on SPEC S numerics
def fullband_channel(W, precise=False):
    """bw = 2 pi, guard = 1: size = width = W, h = 1; the channel is the input shifted by the even centre bin."""
    return dict(f0=float(np.float32(2 * np.pi * 0.3)), bw=float(np.float32(2 * np.pi)), guard=1.0, precise=precise)


def fullband_expected(x, W, center, lo_phase=None):
    """y[n] = x[n] exp(-2 pi i c n / W) (times exp(-i phi_n) with the LO), the first half window faded in by
    sin^2(pi n / W)."""
    n = np.arange(len(x))
    y = x.astype(np.complex128) * np.exp(-2j * np.pi * ((center * n) % W) / W)
    if lo_phase is not None:
        y *= np.exp(-1j * lo_phase.astype(np.float64))
    y[:W // 2] *= np.sin(np.pi * n[:W // 2] / W) ** 2
    return y


def precise_tone_case(W):
    """A 40-bin precise channel whose f0 sits on an odd bin (one bin off its even centre bin, so the LO has work to
    do) and an offset delta of six bins: the tone f0 + delta is periodic in every window."""
    c = dict(f0=float(np.float32(2 * np.pi * 1731 / W)), bw=float(np.float32(2 * np.pi * 40 / W)), guard=1.0,
             precise=True)
    return c, float(np.float32(2 * np.pi * 6 / W))


def precise_tone_input(W, halves, c, delta, amp=0.7):
    return (amp * np.exp(1j * (np.float64(c["f0"]) + delta) * np.arange(W // 2 * halves))).astype(np.complex64)


def assert_precise_tone(y, size, omega, amp=0.7):
    """Past the fade-in the channel holds the tone at omega = delta * D rad/sample with the input amplitude."""
    y = np.asarray(y, np.complex128)[size:]
    assert np.abs(np.abs(y) - amp).max() < 1e-4 * amp
    step = np.angle(y[1:] * np.conj(y[:-1]))
    assert np.abs(step - omega).max() < 1e-5
