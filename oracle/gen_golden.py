#!/usr/bin/env python
"""Generates tests/golden/* by RUNNING THE REFERENCE ITSELF (oracle/_ref: btle_rx.c and
btle_tx.c from /root/reference compiled unmodified).  Run in the build container
(needs /root/reference); the fixtures it writes are committed and travel to the GPU box.

    python oracle/gen_golden.py
"""
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import orc  # noqa: E402
from btle_b200 import synth  # noqa: E402

REF = os.environ.get("BTLE_REFERENCE", "/root/reference")
GOLD = os.path.join(ROOT, "tests", "golden")
REF_TX = os.path.join(ROOT, "oracle", "_ref", "btle_ref_tx")


def ref_records(iq, **cfg):
    r = orc.ref_rx_stream(iq, live=True, **cfg)
    return dict(exp_chunk=r["chunk"], exp_n0=r["n0"], exp_nbytes=r["nbytes"], exp_crc_bad=r["crc_bad"],
                exp_bytes=r["bytes"])


def save(name, iq, cfg, extra=None):
    d = dict(iq=np.ascontiguousarray(iq, dtype=np.int8), cfg=json.dumps(cfg))
    d.update(ref_records(iq, **cfg))
    if extra:
        d.update(extra)
    np.savez_compressed(os.path.join(GOLD, name), **d)
    print(name, "packets:", len(d["exp_n0"]), "crc_bad:", int(np.sum(d["exp_crc_bad"])))


def ref_tx(descriptor):
    with tempfile.TemporaryDirectory() as td:
        p = subprocess.run([REF_TX, descriptor], cwd=td, capture_output=True)
        txt = open(os.path.join(td, "phy_sample.txt")).read()
        out = p.stdout.decode(errors="replace")
    return np.array([int(x) for x in re.findall(r"-?\d+", txt)], dtype=np.int8), out


def main():
    os.makedirs(GOLD, exist_ok=True)
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "ref", "oracle"], check=True, capture_output=True)
    # 1. tables / leaf known answers straight from the reference's own data
    kat = subprocess.run([orc.REF_DRIVER, "kat"], check=True, capture_output=True).stdout.decode()
    json.loads(kat)
    open(os.path.join(GOLD, "tables.json"), "w").write(kat)

    # 2. the reference's own capture (SURVEY.md App. B.1): keep the chunks around the 3 packets
    txt = open(os.path.join(REF, "matlab", "sample_iq_4msps.txt")).read()
    full = np.array([int(x) for x in re.findall(r"-?\d+", txt)], dtype=np.int8)
    assert full.size == 2097152
    rfull = orc.ref_rx_stream(full, live=True)
    assert list(rfull["chunk"].astype(np.int64) * 8192 + rfull["n0"]) == [97892, 501906, 905891]
    parts = [full[16384 * (k - 1):16384 * (k + 2)] for k in (11, 61, 110)]
    save("fixture_ch37.npz", np.concatenate(parts), dict(channel=37),
         dict(full_positions=np.array([97892, 501906, 905891])))

    # 3. reference TX -> reference RX loopbacks (SURVEY.md App. B.2 known answers)
    kats = [
        ("37-ADV_IND-TxAdd-1-RxAdd-0-AdvA-010203040506-AdvData-00112233445566778899AABBCCDDEEFF",
         dict(channel=37), "401606050403020100112233445566778899aabbccddeeff"),
        ("37-DISCOVERY-TxAdd-1-RxAdd-0-AdvA-010203040506-LOCAL_NAME09-SDR/Bluetooth/Low/Energy",
         dict(channel=37), "422006050403020119095344522f426c7565746f6f74682f4c6f772f456e65726779"),
        ("9-LL_CONNECTION_UPDATE_REQ-AA-60850A1B-LLID-3-NESN-0-SN-0-MD-0-WinSize-02-WinOffset-0e0F-Interval-0450-"
         "Latency-0607-Timeout-07D0-Instant-eeff-CRCInit-A77B22",
         dict(channel=9, access_addr=0x60850A1B, crc_init=0xA77B22), "030c00020f0e50040706d007ffee"),
        ("10-LL_DATA-AA-11850A1B-LLID-1-NESN-0-SN-0-MD-0-DATA-XX-CRCInit-123456",
         dict(channel=10, access_addr=0x11850A1B, crc_init=0x123456), "0100"),
    ]
    for i, (desc, cfg, pdu_hex) in enumerate(kats):
        wav, _ = ref_tx(desc)
        iq = np.zeros(3 * 16384, dtype=np.int8)
        rng = np.random.default_rng(i)
        iq[:] = rng.integers(-2, 3, iq.size)
        offs = [2 * 1000, 16384 + 2 * 3001, 2 * 16384 - 2 * 700]      # mid-chunk, odd phase, straddling a boundary
        for o in offs:
            iq[o:o + wav.size] = wav
        save(f"tx_loopback_{i}.npz", iq, cfg, dict(pdu_hex=pdu_hex, descriptor=desc, tx_wave=wav))

    # 4. synthetic ADV stream (noise floor + bursts, 1 in 5 corrupted)
    iq, truth = synth.make_adv_stream(24 * 16384, seed=4242, channel=38, corrupt_every=5, slot_samples=3000)
    save("synth_ch38.npz", iq.numpy(), dict(channel=38), dict(truth_start=truth["start_sample"], truth_corrupt=truth["corrupt"]))

    # 5. adversarial fuzz: full-scale random IQ, sparse masks (negative n0, tail hits, guards)
    rng = np.random.default_rng(20260922)
    cases = [dict(channel=37, access_addr=0x8E89BED6, access_mask=0x0000003F, crc_init=0x555555, raw=0),
             dict(channel=12, access_addr=0x80000000, access_mask=0xC0000001, crc_init=0xABCDEF, raw=0),
             dict(channel=39, access_addr=0x00000000, access_mask=0x00000000, crc_init=0x555555, raw=1)]
    for i, cfg in enumerate(cases):
        iq = rng.integers(-128, 128, 4 * 16384 + 1234, dtype=np.int8)
        save(f"fuzz_{i}.npz", iq, cfg)


if __name__ == "__main__":
    main()
