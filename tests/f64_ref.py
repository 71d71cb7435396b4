"""Float64 restatements of the main PSD (SPEC P) and the spectral tuner (SPEC S.1-S.4), written from SPEC.md alone.

The oracle and the CUDA kernels share their dataflows and twiddle tables, so a mistake common to both (a wrong bin
placement, cross-fade index or LO sign) would pass every bit-identity test.  These functions share nothing with
either: numpy's complex128 FFT, the geometry and weights recomputed here from the SPEC text.  Both sides are then
held to them with the tolerances of tests/parity.py (SPEC T).

The one float32 quantity kept on purpose is the LO phase of precise channels: SPEC N specifies a float32 phase
accumulator, whose rounding drifts from the exact phase by up to ~3e-3 rad over 57k samples.  That drift is part of
the specified output, so the phase sequence is reproduced in float32 and only its cos / sin are taken in float64.
"""
import numpy as np

PI_F = np.float32(np.pi)
TWO_PI_F = np.float32(2 * np.pi)
WINDOWS = ("none", "hamming", "hann", "flat_top", "blackmann_harris")


def window(n, kind):
    """SPEC W: symmetric taps, evaluated in binary64 and rounded once to binary32; returned as float64."""
    if kind == "none":
        return np.ones(n)
    x = 2 * np.pi * np.arange(n) / (n - 1)
    if kind == "hamming":
        v = 0.54 - 0.46 * np.cos(x)
    elif kind == "hann":
        v = 0.5 - 0.5 * np.cos(x)
    elif kind == "flat_top":
        v = 1 - 1.93 * np.cos(x) + 1.29 * np.cos(2 * x) - 0.388 * np.cos(3 * x) + 0.028 * np.cos(4 * x)
    elif kind == "blackmann_harris":
        v = 0.35875 - 0.48829 * np.cos(x) + 0.14128 * np.cos(2 * x) - 0.01168 * np.cos(3 * x)
    else:
        raise ValueError(kind)
    return v.astype(np.float32).astype(np.float64)


def psd_f64(x, N, kind):
    """SPEC P: |FFT(w x)|^2 / N of consecutive N-sample frames, DC first -> [frames, N] float64."""
    x = np.asarray(x)
    frames = len(x) // N
    u = x[:frames * N].astype(np.complex128).reshape(frames, N) * window(N, kind)
    return np.abs(np.fft.fft(u, axis=1)) ** 2 / N


def shift_db_f64(p):
    """The GUI layout (Suscan/Messages/PSDMessage.cpp:32-38): halves swapped, 10 log10(P + 1e-8)."""
    return 10 * np.log10(np.fft.fftshift(np.asarray(p, np.float64), axes=-1) + 1e-8)


def channel_geometry(W, f0, bw, guard):
    """SPEC S.2 in binary64 from the binary32 parameters -> (center, size, width)."""
    f0, bw, guard = (float(np.float32(v)) for v in (f0, bw, guard))
    c = 2 * np.floor(f0 / (4 * np.pi) * W + 0.5)
    m = int(min(max(np.ceil(guard * bw / (2 * np.pi) * W - 1e-3), 4), W))
    size = 1 << (m - 1).bit_length()
    width = int(min(max(np.ceil(m / guard - 1e-3), 2), size))
    return int(c) % W, size, width


def channel_weights(W, halfw):
    """SPEC S.3: h over the W bins of the window in FFT order (bin +i at i, bin -j at W - j), times k = 1/W.
    h is the brick wall over [-halfw, halfw) convolved with the periodic Blackman-Harris spectrum, or 1 when the
    channel spans the whole band (2 halfw >= W)."""
    if 2 * halfw >= W:
        return np.ones(W) / W
    c = (0.35875, 0.48829 / 2, 0.14128 / 2, 0.01168 / 2)
    k = np.arange(W)
    k = np.where(k < W // 2, k, k - W)
    h = np.zeros(W)
    for m in range(-3, 4):
        q = k - m
        h += c[abs(m)] * ((q >= -halfw) & (q < halfw))
    return h / W


def ncqo_phases(fnor, n):
    """SPEC N: the phases phi_0 .. phi_{n-1} that n reads of an NCQO at `fnor` return, accumulated in binary32
    (phi_0 = 0; phi <- wrap(phi + omega), omega = pi_f * fnor, wrap adds or subtracts 2 pi_f once)."""
    omega = np.float32(PI_F * np.float32(fnor))
    out = np.empty(n, np.float32)
    phi, i = np.float32(0.0), 0
    seg = 16 + (int(4 * np.pi / abs(float(omega))) if omega != 0 else n)
    while i < n:
        # ufunc.accumulate adds left to right, rounding every partial sum to binary32: phi, phi + w, (phi + w) + w ...
        run = np.full(min(n - i, seg), omega, np.float32)
        run[0] = phi
        acc = np.add.accumulate(run, dtype=np.float32)
        bad = np.flatnonzero((acc >= TWO_PI_F) | (acc < 0))
        k = int(bad[0]) if len(bad) else len(acc)
        out[i:i + k] = acc[:k]
        i += k
        if len(bad):
            v = acc[k]
            phi = np.float32(v - TWO_PI_F) if v >= TWO_PI_F else np.float32(v + TWO_PI_F)
        else:
            phi = np.float32(acc[-1] + omega)
            if phi >= TWO_PI_F:
                phi = np.float32(phi - TWO_PI_F)
            elif phi < 0:
                phi = np.float32(phi + TWO_PI_F)
    return out


def lo_fnor(W, f0, center, size):
    """S.4 precise channels: the LO runs at the residual offset from the even centre bin, scaled to the channel
    rate, wrapped into (-pi, pi]; fnor = omega / pi rounded to binary32."""
    resid = float(np.float32(f0)) - 2 * np.pi * center / W
    if resid > np.pi:
        resid -= 2 * np.pi
    return np.float32(resid * (W / size) / np.pi)


def specttuner_f64(x, W, f0, bw, guard=1.0, precise=False):
    """SPEC S.1-S.4 for one channel: windows of W samples with hop W/2 (the first once W samples are in), the
    channel's bins gathered circularly into slots +i and size - j, weighted, size * ifft, sin^2 cross-fade with the
    second half of the previous hop's transform.  Returns complex128, size/2 samples per hop."""
    x = np.asarray(x).astype(np.complex128)
    center, size, width = channel_geometry(W, f0, bw, guard)
    halfw, hs = width // 2, size // 2
    h = channel_weights(W, halfw)
    up = (center + np.arange(halfw)) % W                    # bins center + i -> slot i
    j = np.arange(1, halfw + 1)
    dn = (center - j) % W                                   # bins center - j -> slot size - j
    xf = np.sin(np.pi * np.arange(size) / size) ** 2
    hops = (len(x) - W) // (W // 2) + 1 if len(x) >= W else 0
    out = np.empty(hops * hs, np.complex128)
    prev = np.zeros(size, np.complex128)
    for m in range(hops):
        X = np.fft.fft(x[m * W // 2:m * W // 2 + W])
        B = np.zeros(size, np.complex128)
        B[:halfw] = X[up] * h[:halfw]
        B[size - j] = X[dn] * h[W - j]
        cur = np.fft.ifft(B) * size
        out[m * hs:(m + 1) * hs] = xf[:hs] * cur[:hs] + xf[hs:] * prev[hs:]
        prev = cur
    if precise:
        phi = ncqo_phases(lo_fnor(W, f0, center, size), len(out)).astype(np.float64)
        out *= np.exp(-1j * phi)
    return out
