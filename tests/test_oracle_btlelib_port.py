"""oracle/btlelib_port.py (numpy restatement of the reference's bit-true Python receiver) pinned to the reference through
golden vectors the imported reference btlelib produced (oracle/gen_golden_btlelib.py)."""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import btlelib_port as P  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden", "btlelib_rx.npz")
GOLD_RANDOM = os.path.join(ROOT, "tests", "golden", "btlelib_random.npz")


def _hex_le(h):            # 'A77B22' as btlelib passes it -> the -k style integer
    return int(h, 16)


def test_port_equals_reference_golden_vectors():
    z = np.load(GOLD)
    for n in range(int(z["n_cases"])):
        ch, crc_hex, aa_hex = int(z[f"c{n}_ch"]), str(z[f"c{n}_crc_hex"]), str(z[f"c{n}_aa_hex"])
        crc = int(crc_hex, 16) if crc_hex else 0x555555
        aa = int.from_bytes(bytes.fromhex(aa_hex), "little") if aa_hex else 0x8E89BED6
        r = P.rx_window(z[f"c{n}_i"], z[f"c{n}_q"], ch, crc, aa)
        assert r["crc_ok"] == bool(z[f"c{n}_crc_ok"]) and r["plen"] == int(z[f"c{n}_plen"]) and r["phase"] == int(z[f"c{n}_phase"]), n
        assert np.array_equal(r["pdu_bit"], z[f"c{n}_pdu_bit"]), n


def _noisy_window(z, k):
    """Case k's window as the reference's btle_rx saw it: its transmitter's waveform (= our 8-sps modulator over the PHY
    bits it sent) plus white Gaussian noise, seeded, at the case's SNR over a peak of 127 (sigma 127 / 10^(SNR/20) split
    evenly over I and Q), behind `pad` and ahead of 64 samples of noise alone, cut to whole symbols."""
    import torch
    from btle_b200 import synth
    lo = z["phy_bit_end"][k - 1] if k else 0
    ti, tq = synth.modulate_batch_8sps(torch.from_numpy(z["phy_bit"][lo:z["phy_bit_end"][k]][None, :]))
    np.random.seed(100 + k)
    sigma = 127 / np.power(10, z["snr"][k] / 20) / np.sqrt(2)
    ri = np.double(ti[0].numpy()) + np.random.normal(0, sigma, ti.shape[1])
    rq = np.double(tq[0].numpy()) + np.random.normal(0, sigma, tq.shape[1])
    pad = int(z["pad"][k])
    ri = np.concatenate((np.random.normal(0, 3, pad), ri, np.random.normal(0, 3, 64)))
    rq = np.concatenate((np.random.normal(0, 3, pad), rq, np.random.normal(0, 3, 64)))
    return ri[: len(ri) // 8 * 8], rq[: len(rq) // 8 * 8]


def test_port_equals_imported_reference_on_random_packets():
    """60 random packets at SNR 4..20 dB and arbitrary alignment, against what the reference's btle_rx returned for each
    (tests/golden/btlelib_random.npz, written by oracle/gen_golden_btlelib.py from the imported reference btlelib)."""
    z = np.load(GOLD_RANDOM)
    n_ok = n_bad = 0
    for k in range(len(z["ch"])):
        ri, rq = _noisy_window(z, k)
        ri, rq = np.int16(ri), np.int16(rq)
        assert hashlib.sha256(ri.tobytes() + rq.tobytes()).hexdigest() == z["sha256"][k], k       # the window the reference saw
        crc_hex, aa_hex = str(z["crc_hex"][k]), str(z["aa_hex"][k])
        got = P.rx_window(ri, rq, int(z["ch"][k]), int(crc_hex, 16) if crc_hex else 0x555555,
                          int.from_bytes(bytes.fromhex(aa_hex), "little") if aa_hex else 0x8E89BED6)
        lo = z["pdu_bit_end"][k - 1] if k else 0
        ref_ok = bool(z["crc_ok"][k])
        assert got["crc_ok"] == ref_ok and got["plen"] == int(z["plen"][k]) and got["phase"] == int(z["phase"][k]), (k, z["snr"][k])
        assert np.array_equal(got["pdu_bit"], z["pdu_bit"][lo:z["pdu_bit_end"][k]]), (k, z["snr"][k])
        n_ok += ref_ok; n_bad += not ref_ok
    assert n_ok > 20 and n_bad > 5


def test_port_stream_finds_what_it_sent():
    """The streaming rules on a synthetic 8-Msps capture built with the port's own transmitter bits and the 8-sps modulator:
    every packet comes back once, with its bytes, in order."""
    import torch
    from btle_b200 import synth
    rng = np.random.default_rng(9)
    pdus = [bytes([0x40, 6 + k % 20]) + rng.integers(0, 256, 6 + k % 20, dtype=np.uint8).tobytes() for k in range(12)]
    n = 12 * 6000 + 4096
    cap = rng.normal(0, 2.0, (n, 2))
    pos = []
    for k, pdu in enumerate(pdus):
        bits = P.tx_bits(pdu, 37)
        ti, tq = synth.modulate_batch_8sps(torch.from_numpy(bits[None, :]))
        p0 = 6000 * k + 500 + int(rng.integers(0, 1000))
        cap[p0:p0 + ti.shape[1], 0] += ti[0].numpy()
        cap[p0:p0 + ti.shape[1], 1] += tq[0].numpy()
        pos.append(p0)
    iq16 = cap.astype(np.int16)
    got = P.rx_stream(iq16, 37)
    assert len(got) == len(pdus)
    for g, pdu, p0 in zip(got, pdus, pos):
        assert g["crc_ok"] and bytes(np.packbits(g["pdu_bit"], bitorder="little")) == pdu
        assert 0 <= g["sample"] - p0 - 8 * 8 < 24                 # preamble (8 symbols) + modulator delay
