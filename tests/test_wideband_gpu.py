"""Wideband channelizer on the B200: the kernel byte for byte against the int64 restatement (oracle/wideband_port.py), the
receiver behind it (rx_wideband == rx_batch(channelize)), connection following and the CLI on one wideband capture."""
import os
import subprocess

import numpy as np
import pytest
import torch

import orc
from btle_b200 import BtleError, BtleRx, synth
from btle_b200._native import BTLE_EINVAL, BTLE_EOVERFLOW
from btle_b200.hop import channel_freq_mhz, follow_connections_windowed, record_time
from btle_b200.rx import band_channels, wideband_taps
from test_wideband_cpu import check_found, port_channels, wideband_scenario, wp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "btle_b200", "btle_rx_b200")


@pytest.fixture(scope="module")
def rx():
    r = BtleRx(0)
    yield r
    r.close()


def _device_channelize(rx, wide, d, fc, chans, out_shift=-1):
    n = wide.size // 2
    width = 2 * (-(-n // d))
    stride = (width + 15) // 16 * 16 + 16
    d_wide = torch.from_numpy(wide).cuda()
    d_out = torch.full((len(chans), stride), 0x55, dtype=torch.int8, device="cuda")
    rx.channelize_device(d_wide, d, fc, chans, d_out, out_shift=out_shift)
    torch.cuda.synchronize()
    out = d_out.cpu().numpy()
    assert (out[:, width:] == 0x55).all()                            # the padding of each row is not written
    return out[:, :width]


def _port(wide, d, fc, chans, out_shift=-1):
    out = []
    for ch in chans:
        taps, shift = wideband_taps(d, fc, ch)
        out.append(wp.channelize(wide, d, taps, channel_freq_mhz(ch) - fc, shift if out_shift < 0 else out_shift))
    return np.stack(out)


@pytest.mark.parametrize("d,fc", [(2, 2403), (5, 2426), (20, 2441), (25, 2441), (64, 2441)])
def test_channelize_device_equals_port(rx, d, fc):
    rng = np.random.default_rng(d)
    band = band_channels(d, fc)
    t_len = len(wideband_taps(d, fc, band[0])[0])
    sets = [band, [band[-1], band[0], band[0], band[len(band) // 2]]]
    for n in (1, t_len // 2, 1100 * d + 7, 3 * 512 * d):
        wide = rng.integers(-128, 128, 2 * n, dtype=np.int8)                   # full-scale random
        for chans in sets:
            assert np.array_equal(_device_channelize(rx, wide, d, fc, chans), _port(wide, d, fc, chans)), (d, n, chans)
    wide = rng.integers(-128, 128, 2 * (700 * d + 3), dtype=np.int8)
    shift = wideband_taps(d, fc, band[0])[1]
    for s in (0, shift - 6):                                                     # outputs saturate at both rails
        got = _device_channelize(rx, wide, d, fc, sets[1], out_shift=s)
        assert (got == 127).any() and (got == -128).any()
        assert np.array_equal(got, _port(wide, d, fc, sets[1], out_shift=s))


def _check_e2e(rx, channels, d, fc):
    caps, cfgs, wide = wideband_scenario(channels, d, fc)
    cfgs["rssi"] = 1                                                  # the oracle always fills mag_sum
    ys = port_channels(wide, d, fc, channels)
    assert np.array_equal(rx.channelize(wide, d, fc, channels), ys)
    got = rx.rx_wideband(wide, d, fc, cfgs)
    assert got.tobytes() == rx.rx_batch(ys, cfgs).tobytes()
    for i, c in enumerate(cfgs):
        kw = dict(channel=int(c["channel"]), access_addr=int(c["access_addr"]), crc_init=int(c["crc_init"]))
        exp = orc.rx_stream(ys[i], stream=i, **kw)
        assert got[got["stream"] == i].tobytes() == exp.tobytes()
        check_found(exp, orc.rx_stream(caps[i], stream=i, **kw))
    return got


def test_end_to_end_80msps_40_channels(rx):
    got = _check_e2e(rx, list(range(40)), 20, 2441)
    assert len(got) == 40 and int(got["crc_bad"].sum()) == 1


def test_end_to_end_20msps_9_channels(rx):
    chans = band_channels(5, 2426)
    assert len(chans) == 9
    got = _check_e2e(rx, chans, 5, 2426)
    assert len(got) == 9


# ---- connection following on one 80 Msps capture (the scenario of test_hop, built here per channel, then wideband) ---
def _place(cap, ch, t_s, air, amp=64):
    wav = synth.modulate(air).astype(np.int32) * amp // 127
    p = 2 * int(round(t_s * 4e6))
    cap[ch, p:p + wav.size] = np.clip(cap[ch, p:p + wav.size].astype(np.int32) + wav, -128, 127)


def _connection_capture():
    n = 100 * 16384
    cap = np.zeros((40, n), dtype=np.int8)
    aa, crci, hop, interval = 0x60850A1B, 0x227BA7, 9, 16
    A, B = bytes.fromhex("5f96ea301800"), bytes.fromhex("9992b1ebd790")
    creq = synth.adv_pdu(5, 0, 0, A + B + aa.to_bytes(4, "little") + crci.to_bytes(3, "big") + bytes([2]) +
                         (15).to_bytes(2, "little") + interval.to_bytes(2, "little") + bytes(2) + (2000).to_bytes(2, "little") +
                         bytes.fromhex("ffffffff1f") + bytes([hop | (5 << 5)]))
    _place(cap, 37, 0.0030, synth.air_bytes(synth.adv_pdu(0, 0, 0, B + b"\x02\x01\x05"), 37))
    _place(cap, 37, 0.0050, synth.air_bytes(creq, 37))
    creq2 = bytearray(creq); creq2[2 + 28] = 0x0F
    _place(cap, 38, 0.0070, synth.air_bytes(bytes(creq2), 38))
    ch, t = 0, 0.012
    for k in range(9):
        ch = (ch + hop) % 37
        if k != 5:
            _place(cap, ch, t, synth.air_bytes(synth.ll_data_pdu(1, k & 1, k & 1, 0, bytes([k] * (k % 5))), ch, aa, crci))
            _place(cap, ch, t + 0.00035, synth.air_bytes(synth.ll_data_pdu(1, (k + 1) & 1, k & 1, 0, b""), ch, aa, crci))
        t += interval * 1.25e-3
    wide = synth.wideband_from_channels(torch.from_numpy(cap), list(range(40)), 20, 2441, noise=1.0, seed=9, device="cuda")
    return cap, wide.cpu().numpy()


@pytest.fixture(scope="module")
def connection_capture():
    return _connection_capture()


def _same(a, b, path="conns"):
    if isinstance(a, dict):
        assert set(a) == set(b), path
        for k in a:
            _same(a[k], b[k], f"{path}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), (path, len(a), len(b))
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, f"{path}[{i}]")
    elif isinstance(a, np.void):
        assert bytes(a["bytes"]) == bytes(b["bytes"]) and a["crc_bad"] == b["crc_bad"] and a["channel"] == b["channel"], path
        assert abs(record_time(a) - record_time(b)) <= 1e-6, path
    elif isinstance(a, float):
        assert abs(a - b) <= 1e-6 or a == b, (path, a, b)
    else:
        assert a == b, (path, a, b)


def test_follow_connections_from_wideband(rx, connection_capture):
    cap, wide = connection_capture
    adv_w, conns_w = follow_connections_windowed(rx, rx.channelize(wide, 20, 2441))
    adv_c, conns_c = follow_connections_windowed(rx, cap)
    assert len(conns_c) == 2 and sum(c["tracked"] for c in conns_c) == 1
    conns_w = [{k: v for k, v in c.items() if k != "chunks_decoded"} for c in conns_w]
    conns_c = [{k: v for k, v in c.items() if k != "chunks_decoded"} for c in conns_c]
    _same(list(adv_w), list(adv_c), "adv")
    _same(conns_w, conns_c)


@pytest.mark.parametrize("extra", [[], ["-j"], ["-j", "-Q", "-R"], ["-c", "37", "-o", "-v", "-j"], ["-c", "37", "-o", "-j", "-Q"]])
def test_cli_wideband_equals_iq_dir(rx, connection_capture, tmp_path, extra):
    _, wide = connection_capture
    wfile = tmp_path / "wide.bin"
    wide.tofile(wfile)
    ys = rx.channelize(wide, 20, 2441)
    for ch in range(40):
        ys[ch].tofile(tmp_path / f"ch{ch:02d}.bin")
    pcap = tmp_path / "out.pcap"
    outs = []
    for src in (["--iq-dir", str(tmp_path)], ["--wideband", f"{wfile}:80:2441"]):
        p = subprocess.run([CLI, *src, *extra, "-s", str(pcap)], capture_output=True, text=True)
        assert p.returncode == 0, p.stdout + p.stderr
        outs.append((p.stdout, pcap.read_bytes()))
        pcap.unlink()
    assert outs[0] == outs[1]
    assert len(outs[0][1]) > 24                                                  # pcap holds packets, not just its header


def test_cli_wideband_rejects_bad_rate(tmp_path):
    f = tmp_path / "w.bin"
    np.zeros(64, dtype=np.int8).tofile(f)
    p = subprocess.run([CLI, "--wideband", f"{f}:82:2441"], capture_output=True, text=True)
    assert p.returncode != 0 and "multiple of 4" in p.stdout


def test_error_paths(rx):
    wide = np.random.default_rng(0).integers(-128, 128, 2 * 4000, dtype=np.int8)
    for kwargs, word in ((dict(decim=1, center_mhz=2441, channels=[37]), "decim"),
                         (dict(decim=65, center_mhz=2441, channels=[37]), "decim"),
                         (dict(decim=20, center_mhz=2441, channels=[40]), "0~39"),
                         (dict(decim=5, center_mhz=2426, channels=[0]), "outside the band"),
                         (dict(decim=5, center_mhz=2426, channels=None), "all 40")):
        with pytest.raises(BtleError) as e:
            rx.channelize(wide, **kwargs)
        assert e.value.code == BTLE_EINVAL and word in str(e.value), str(e.value)
    d_wide = torch.from_numpy(wide).cuda()
    width = 2 * (4000 // 20)
    bad = ((d_wide, torch.zeros((2, width - 16), dtype=torch.int8, device="cuda"), "smaller"),
           (d_wide, torch.zeros((2, width + 8), dtype=torch.int8, device="cuda"), "multiple of 16"),
           (torch.zeros(2 * 4000 + 16, dtype=torch.int8, device="cuda")[2:2 + 2 * 4000], torch.zeros((2, width), dtype=torch.int8, device="cuda"), "aligned"),
           (d_wide, torch.zeros(2 * width + 16, dtype=torch.int8, device="cuda")[8:8 + 2 * width].view(2, width), "aligned"))
    for dw, do, word in bad:
        with pytest.raises(BtleError) as e:
            rx.channelize_device(dw, 20, 2441, [37, 38], do)
        assert e.value.code == BTLE_EINVAL and word in str(e.value), str(e.value)
    _, cfgs, wide = wideband_scenario(list(range(40)), 20, 2441)
    n_all = len(rx.rx_wideband(wide, 20, 2441, cfgs))
    with pytest.raises(BtleError) as e:
        rx.rx_wideband(wide, 20, 2441, cfgs, cap=3)
    assert e.value.code == BTLE_EOVERFLOW and f"{n_all} packets found" in str(e.value)
