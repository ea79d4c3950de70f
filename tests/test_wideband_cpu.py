"""Wideband channelizer on the CPU: the designed taps (btle_b200.rx.wideband_taps, host only), the int64 restatement of the
contract (oracle/wideband_port.py) against its float form, and the receiver behind the restatement on a synthesised
wideband capture."""
import os
import sys

import numpy as np
import pytest

import orc
from btle_b200 import BtleError, make_cfgs, synth
from btle_b200.hop import channel_freq_mhz
from btle_b200.rx import band_channels, wideband_taps

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import wideband_port as wp  # noqa: E402

DECIMS = (2, 5, 14, 20, 25, 64)


def _q(ch, fc):
    return channel_freq_mhz(ch) - fc


def _edge_centres(d):
    """Centres that put a channel exactly at the lower and at the upper band edge (|q| + 1 = fs/2 in MHz)."""
    return [2402 + 2 * d - 1, 2480 - 2 * d + 1]


def _proto(d):
    taps, shift = wideband_taps(d, 2440, 17)                       # channel 17 sits at 2440 MHz: q = 0
    return taps, shift


@pytest.mark.parametrize("d", DECIMS)
def test_prototype_design(d):
    taps, shift = _proto(d)
    t_len = len(taps)
    assert t_len % 2 == 1
    assert not taps[:, 1].any() and np.array_equal(taps[:, 0], taps[::-1, 0])     # real, symmetric
    h = taps[:, 0].astype(np.float64)
    fs = 4.0 * d
    nfft = 1 << 20
    resp = np.abs(np.fft.fft(h, nfft))
    f = np.abs(np.fft.fftfreq(nfft, 1.0 / fs))
    db = 20 * np.log10(np.maximum(resp, 1e-300) / resp[0])
    assert db[f >= 1.25].max() <= -50.0, db[f >= 1.25].max()
    assert db[f <= 0.6].min() >= -1.0, db[f <= 0.6].min()
    assert abs(h.sum() / 2.0 ** shift - 1.0) <= 0.10                                # default passband gain 1 +- 10 %
    assert np.abs(taps).max() <= 32767


@pytest.mark.parametrize("d", DECIMS)
def test_channel_taps(d):
    proto, shift0 = _proto(d)
    t_len = len(proto)
    c = (t_len - 1) // 2
    for fc in _edge_centres(d):
        chans = band_channels(d, fc)
        assert any(abs(_q(ch, fc)) + 1 == 2 * d for ch in chans)                      # a channel on the band edge
        for ch in chans:
            taps, shift = wideband_taps(d, fc, ch)
            assert len(taps) == t_len and shift == shift0
            t64 = taps.astype(np.int64)
            assert 128 * np.abs(t64).sum() < 2 ** 31                                     # no int32 overflow possible
            rot = proto[:, 0] * np.exp(2j * np.pi * _q(ch, fc) * (np.arange(t_len) - c) / (4 * d))
            assert np.abs(t64[:, 0] - rot.real).max() <= 1.0 and np.abs(t64[:, 1] - rot.imag).max() <= 1.0


def test_taps_reject_bad_arguments():
    for d in (1, 65):
        with pytest.raises(BtleError):
            wideband_taps(d, 2441, 37)
    with pytest.raises(BtleError):
        wideband_taps(5, 2426, 0)                                   # 2404 MHz: outside 2406..2446
    with pytest.raises(BtleError):
        wideband_taps(20, 2441, 40)
    with pytest.raises(BtleError):
        wideband_taps(5, 2426, 38, out_shift=32)
    assert band_channels(5, 2426) == [ch for ch in range(40) if 2418 <= channel_freq_mhz(ch) <= 2434]


@pytest.mark.parametrize("d,fc,ch", [(2, 2403, 37), (5, 2426, 13), (20, 2441, 17), (20, 2441, 39), (25, 2441, 37), (64, 2441, 0)])
def test_port_matches_float_form(d, fc, ch):
    rng = np.random.default_rng(d * 1000 + ch)
    taps, shift = wideband_taps(d, fc, ch)
    proto, _ = wideband_taps(d, channel_freq_mhz(ch), ch)          # q = 0 at the channel's own frequency
    for n in (1, len(taps) // 3, 20 * d + 3):
        wide = rng.integers(-128, 128, 2 * n, dtype=np.int8)
        a = wp.channelize(wide, d, taps, _q(ch, fc), shift)
        b = wp.channelize_float(wide, d, proto, _q(ch, fc), shift)
        assert a.size == 2 * (-(-n // d))
        assert np.abs(a.astype(np.int32) - b).max(initial=0) <= 1
    # a loud tone exactly on the channel comes out as a constant at unit gain: pins the mixer's sign and the centring
    n = 200 * d
    k = np.arange(n)
    tone = 60 * np.exp(2j * np.pi * _q(ch, fc) * k / (4 * d))
    wide = np.stack([np.round(tone.real), np.round(tone.imag)], axis=1).astype(np.int8).reshape(-1)
    y = wp.channelize(wide, d, taps, _q(ch, fc), shift).reshape(-1, 2)
    mid = y[len(y) // 4: 3 * len(y) // 4].astype(np.int32)
    assert np.abs(mid[:, 0] - 60).max() <= 2 and np.abs(mid[:, 1]).max() <= 2


# ---- end to end: synthesised wideband capture -> restatement -> receiver --------------------------------------------
AA_DATA, CRC_DATA = 0x60850A1B, 0x227BA7


def wideband_scenario(channels, decim, center_mhz, n_chunks=3, seed=5):
    """Per-channel 4 Msps captures with one packet each (the second channel's packet has a flipped bit, the third's
    straddles the first chunk boundary), their wideband capture and the receiver configs.  Packets on different
    channels are spread in time and quieter when there are many, so that their sum stays clear of int8 clipping."""
    amp = 40 if len(channels) <= 10 else 24
    m = n_chunks * 8192
    caps = np.zeros((len(channels), 2 * m), dtype=np.int8)
    cfgs = make_cfgs(len(channels))
    rng = np.random.default_rng(seed)
    slot = (m - 2000) // max(1, len(channels))
    for i, ch in enumerate(channels):
        adv = ch >= 37
        aa, crc = (synth.ADV_ACCESS_ADDR, synth.ADV_CRC_INIT) if adv else (AA_DATA, CRC_DATA)
        cfgs[i]["channel"], cfgs[i]["access_addr"], cfgs[i]["crc_init"] = ch, aa, crc
        body = rng.integers(0, 256, 6 + i % 20, dtype=np.uint8).tobytes()
        pdu = synth.adv_pdu(0, 1, 0, body) if adv else synth.ll_data_pdu(2, 0, 1, 0, body[:27])
        air = synth.air_bytes(pdu, ch, aa, crc, corrupt_bit=20 if i == 1 else None)
        wav = synth.modulate(air).astype(np.int32) * amp // 127
        start = 8192 - 300 if i == 2 else 600 + (i * slot) % (m - 2600)
        caps[i, 2 * start:2 * start + wav.size] = wav
    wide = synth.wideband_from_channels(caps, channels, decim, center_mhz, noise=1.0, seed=seed).numpy()
    return caps, cfgs, wide


def check_found(got, truth, n_expected=1):
    """`got` (records from the channelized capture) holds the packets of `truth` (records of the clean per-channel capture)
    exactly once, with the same bytes and CRC verdict, within +-2 samples."""
    assert len(truth) == n_expected and len(got) == len(truth), (len(got), len(truth))
    for a, b in zip(got, truth):
        assert a["n_bytes"] == b["n_bytes"] and bytes(a["bytes"]) == bytes(b["bytes"]) and a["crc_bad"] == b["crc_bad"]
        ta, tb = int(a["chunk"]) * 8192 + int(a["n0"]), int(b["chunk"]) * 8192 + int(b["n0"])
        assert abs(ta - tb) <= 2, (ta, tb)


def port_channels(wide, decim, center_mhz, channels):
    out = []
    for ch in channels:
        taps, shift = wideband_taps(decim, center_mhz, ch)
        out.append(wp.channelize(wide, decim, taps, channel_freq_mhz(ch) - center_mhz, shift))
    return np.stack(out)


def test_end_to_end_port_80msps():
    channels = [37, 0, 5, 10, 17, 25, 36, 39]
    caps, cfgs, wide = wideband_scenario(channels, 20, 2441)
    assert wide.size == 2 * 20 * caps.shape[1] // 2
    ys = port_channels(wide, 20, 2441, channels)
    for i, ch in enumerate(channels):
        c = cfgs[i]
        kw = dict(channel=ch, access_addr=int(c["access_addr"]), crc_init=int(c["crc_init"]))
        truth = orc.rx_stream(caps[i], **kw)
        check_found(orc.rx_stream(ys[i], **kw), truth)
        assert bool(truth["crc_bad"][0]) == (i == 1)
        if i == 2:
            assert truth["chunk"][0] == 0 and truth["n0"][0] > 8192 - 400
