"""Restatement of the wideband channelizer's contract (include/btle_b200.h, DESIGN.md §6.5) in numpy int64, and the float
form it is derived from.  Test infrastructure: product code never imports this.  The taps come from the library
(btle_b200.rx.wideband_taps), so nothing here depends on the last bit of libm."""
from __future__ import annotations

import numpy as np


def channelize(wide: np.ndarray, decim: int, taps: np.ndarray, q: int, shift: int) -> np.ndarray:
    """wide: int8 interleaved I,Q (N samples); taps: int16 [T, 2] (H_q re, im); q = (f_ch - fc) / 1 MHz.
    Returns int8 interleaved I,Q, ceil(N / decim) samples."""
    x = np.asarray(wide, dtype=np.int8).reshape(-1, 2).astype(np.int64)
    n, t_len = len(x), len(taps)
    c, m = (t_len - 1) // 2, -(-n // decim)
    xp = np.zeros((n + 2 * t_len + decim, 2), dtype=np.int64)           # x[k] = xp[k + t_len]; zero outside [0, N)
    xp[t_len:t_len + n] = x
    hr, hi = taps[:, 0].astype(np.int64), taps[:, 1].astype(np.int64)
    base = np.arange(m, dtype=np.int64) * decim + c + t_len
    ar = np.zeros(m, dtype=np.int64)
    ai = np.zeros(m, dtype=np.int64)
    for t in range(t_len):                                               # acc[m] = sum_t x[m*D + c - t] * H_q[t]
        v = xp[base - t]
        ar += v[:, 0] * hr[t] - v[:, 1] * hi[t]
        ai += v[:, 0] * hi[t] + v[:, 1] * hr[t]
    assert np.abs(ar).max(initial=0) < 2 ** 31 and np.abs(ai).max(initial=0) < 2 ** 31
    r = (q * np.arange(m, dtype=np.int64)) % 4                           # rot = acc * (-j)^r
    re = np.choose(r, [ar, ai, -ar, -ai])
    im = np.choose(r, [ai, -ar, -ai, ar])
    add = (1 << (shift - 1)) if shift else 0
    y = np.stack([re, im], axis=1)
    return np.clip((y + add) >> shift, -128, 127).astype(np.int8).reshape(-1)


def channelize_float(wide: np.ndarray, decim: int, proto: np.ndarray, q: int, shift: int) -> np.ndarray:
    """What the contract approximates: mix by exp(-j 2 pi q n / (4 decim)), filter with the real prototype `proto`
    (the q = 0 taps, int16 [T] or [T, 2]) centred on the output sample, decimate by `decim`, divide by 2^shift, round
    and saturate.  float64; equal to channelize() within 1 LSB."""
    x = np.asarray(wide, dtype=np.int8).reshape(-1, 2).astype(np.float64)
    x = x[:, 0] + 1j * x[:, 1]
    n = len(x)
    h = np.asarray(proto, dtype=np.float64)
    h = h[:, 0] if h.ndim == 2 else h
    t_len, c, m = len(h), (len(h) - 1) // 2, -(-n // decim)
    k = np.arange(n, dtype=np.int64)
    mixed = x * np.exp(-2j * np.pi * ((q * k) % (4 * decim)) / (4 * decim))
    full = np.convolve(mixed, h)                                         # full[k] = sum_t mixed[k - t] h[t]
    idx = np.arange(m, dtype=np.int64) * decim + c
    acc = np.where(idx < len(full), full[np.minimum(idx, len(full) - 1)], 0)
    y = np.stack([acc.real, acc.imag], axis=1) / 2.0 ** shift
    return np.clip(np.floor(y + 0.5), -128, 127).astype(np.int8).reshape(-1)
