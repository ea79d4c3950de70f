#!/usr/bin/env python
"""Golden vectors for the btlelib-compatible shim, produced by importing the REFERENCE's own
python/btlelib.py here (from a writable copy: it writes table files next to itself on first TX
call, btlelib.py:90-91,155).  Writes tests/golden/btlelib_rx.npz and tests/golden/btlelib_random.npz (committed)."""
import hashlib
import os
import shutil
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("BTLE_REFERENCE", "/root/reference")


def main():
    td = tempfile.mkdtemp()
    shutil.copytree(os.path.join(REF, "python"), os.path.join(td, "python"))
    os.makedirs(os.path.join(td, "verilog"))
    os.chdir(os.path.join(td, "python"))
    sys.path.insert(0, os.getcwd())
    import btlelib as bl
    out = {}
    cases = [
        (37, "", "", "4225" + "0289674523" + "01" * 32, 20.0, 1),
        (37, "", "", "4225" + "0289674523" + "01" * 32, 7.0, 2),          # noisy: CRC may fail on early phases
        (9, "A77B22", "1B0A8560", "030c00020f0e50040706d007ffee", 15.0, 3),
        (10, "123456", "1B0A8511", "0100", 12.0, 4),
        (38, "", "", "40" + "10" + "a1b2c3d4e5f6" + "00112233445566778899", -3.0, 5),   # hopeless SNR
    ]
    for n, (ch, crc_hex, aa_hex, pdu_hex, snr, seed) in enumerate(cases):
        pdu_bit = bl.hex_string_to_bit(pdu_hex)
        crc_bits = bl.hex_string_to_bit(crc_hex) if crc_hex else []
        args_tx = [ch] + ([crc_bits, aa_hex] if crc_hex else [])
        tx_i, tx_q, _, _ = bl.btle_tx(pdu_bit, *args_tx)
        np.random.seed(seed)
        rx_i, rx_q = bl.add_noise(tx_i, tx_q, snr)
        args_rx = [ch] + ([crc_bits, aa_hex] if crc_hex else [])
        r = bl.btle_rx(rx_i, rx_q, *args_rx)
        out[f"c{n}_i"] = np.int16(rx_i); out[f"c{n}_q"] = np.int16(rx_q)
        out[f"c{n}_ch"] = ch; out[f"c{n}_crc_hex"] = crc_hex; out[f"c{n}_aa_hex"] = aa_hex
        out[f"c{n}_pdu_bit"] = np.asarray(r[0], dtype=np.int8); out[f"c{n}_crc_ok"] = bool(r[1])
        out[f"c{n}_plen"] = int(r[2]); out[f"c{n}_phy_bit"] = np.asarray(r[3], dtype=np.int8)
        out[f"c{n}_bit_all"] = r[4]; out[f"c{n}_sig_all"] = r[5]; out[f"c{n}_phase"] = int(r[6])
        print(n, "ch", ch, "snr", snr, "crc_ok", r[1], "plen", r[2], "phase", r[6])
    out["n_cases"] = len(cases)
    # TX waveforms (for the batched 8-sps synthesiser used by the BER harness)
    for n, (ch, crc_hex, aa_hex, pdu_hex) in enumerate([(37, "", "", "422506050403020119095344522f426c7565746f6f74682f4c6f772f456e657267791234567890"),
                                                       (11, "A77B22", "1B0A8560", "0103112233")]):
        pdu_bit = bl.hex_string_to_bit(pdu_hex)
        args_tx = [ch] + ([bl.hex_string_to_bit(crc_hex), aa_hex] if crc_hex else [])
        ti, tq, phy_bit, _ = bl.btle_tx(pdu_bit, *args_tx)
        out[f"tx{n}_i"], out[f"tx{n}_q"], out[f"tx{n}_phy_bit"], out[f"tx{n}_pdu_bit"] = np.int8(ti), np.int8(tq), np.int8(phy_bit), pdu_bit
        out[f"tx{n}_ch"], out[f"tx{n}_crc_hex"], out[f"tx{n}_aa_hex"] = ch, crc_hex, aa_hex
    out["gauss_fir_int8"] = np.int8(bl.gfsk_modulation_fixed_point.gauss_fir)
    out["cos_table"] = np.int8(bl.vco_fixed_point.cos_table)
    # leaf vectors
    rng = np.random.default_rng(3)
    bits = rng.integers(0, 2, 400).astype(np.int8)
    init = bl.hex_string_to_bit("A77B22")
    out["leaf_bits"] = bits
    out["leaf_crc_init"] = init
    out["leaf_crc24_core"] = bl.crc24_core(bits, init)
    for ch in (0, 17, 37):
        out[f"leaf_scramble_{ch}"] = bl.scramble_core(bits, ch)
    seq = bits[123:155].copy()
    out["leaf_seq"] = seq
    out["leaf_seq_idx"] = bl.search_unique_bit_sequence(bits, seq)
    out["leaf_seq_miss"] = bl.search_unique_bit_sequence(bits, 1 - np.zeros(64, dtype=np.int8))
    i16 = rng.integers(-300, 300, 777).astype(np.int16); q16 = rng.integers(-300, 300, 777).astype(np.int16)
    b, s = bl.gfsk_demodulation_fixed_point(i16, q16)
    out["leaf_i16"], out["leaf_q16"], out["leaf_gfsk_bit"], out["leaf_gfsk_sig"] = i16, q16, b, s
    out["hex_bits"] = bl.hex_string_to_bit("D6BE898E")
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "btlelib_rx.npz"), **out)
    random_packets(bl)


def random_packets(bl):
    """60 random packets through the reference's btle_tx + add_noise at SNR 4..20 dB, cut at an arbitrary alignment, and
    what its btle_rx made of each.  Stored: the transmitter's PHY bits and the noise parameters (the window is rebuilt by
    tests/test_oracle_btlelib_port.py: our 8-sps modulator, which equals btle_tx's waveform, plus the seeded noise), a
    digest of the int16 window, btle_rx's results."""
    import torch
    sys.path.insert(0, ROOT)
    from btle_b200 import synth
    cols = {f: [] for f in ("ch", "crc_hex", "aa_hex", "snr", "pad", "phy_bit", "sha256", "pdu_bit", "crc_ok", "plen", "phase")}
    rng = np.random.default_rng(5)
    for k in range(60):
        ch = int(rng.choice([37, 38, 39, 3, 20]))
        adv = ch >= 37
        plen = int(rng.integers(6, 38)) if adv else int(rng.integers(0, 28))
        pdu = bytes([int(rng.integers(0, 16)), plen]) + rng.integers(0, 256, plen, dtype=np.uint8).tobytes()
        crc_hex, aa_hex = ("", "") if adv else ("A77B22", "1B0A8560")
        pdu_bit = bl.hex_string_to_bit(pdu.hex())
        args = [ch] + ([bl.hex_string_to_bit(crc_hex), aa_hex] if crc_hex else [])
        ti, tq, phy_bit, _ = bl.btle_tx(pdu_bit, *args)
        phy_bit = np.asarray(phy_bit, dtype=np.uint8)
        mi, mq = synth.modulate_batch_8sps(torch.from_numpy(phy_bit[None, :]))
        assert np.array_equal(mi[0].numpy(), ti) and np.array_equal(mq[0].numpy(), tq)
        np.random.seed(100 + k)
        snr = float(rng.choice([4.0, 7.0, 9.0, 12.0, 20.0]))
        ri, rq = bl.add_noise(ti, tq, snr)
        pad = int(rng.integers(0, 5)) * 8 + int(rng.integers(0, 8))          # arbitrary alignment, like a window cut from a stream
        ri = np.concatenate((np.random.normal(0, 3, pad), ri, np.random.normal(0, 3, 64)))
        rq = np.concatenate((np.random.normal(0, 3, pad), rq, np.random.normal(0, 3, 64)))
        ri, rq = ri[: len(ri) // 8 * 8], rq[: len(rq) // 8 * 8]
        r = bl.btle_rx(ri, rq, *args)
        for f, v in (("ch", ch), ("crc_hex", crc_hex), ("aa_hex", aa_hex), ("snr", snr), ("pad", pad), ("phy_bit", phy_bit),
                     ("sha256", hashlib.sha256(np.int16(ri).tobytes() + np.int16(rq).tobytes()).hexdigest()),
                     ("pdu_bit", np.asarray(r[0], dtype=np.int8)), ("crc_ok", bool(r[1])), ("plen", int(r[2])), ("phase", int(r[6]))):
            cols[f].append(v)
    out = {f: np.array(v) for f, v in cols.items() if f not in ("phy_bit", "pdu_bit")}
    for f in ("phy_bit", "pdu_bit"):                    # ragged: concatenated, with the end offset of each case
        out[f], out[f + "_end"] = np.concatenate(cols[f]), np.cumsum([len(v) for v in cols[f]])
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "btlelib_random.npz"), **out)


if __name__ == "__main__":
    main()
