"""Pins our C restatement (oracle/btle_oracle.c) to the reference itself (oracle/_ref = the reference's btle_rx.c
compiled unmodified), through what its receiver() returned for these very inputs, recorded in tests/golden/ref_driver.npz
(tests/orc.py: ref_driver)."""
import numpy as np
import pytest
import torch

import orc
from btle_b200 import synth


def _cmp(iq, **cfg):
    rec = orc.rx_stream(iq, **cfg)
    ref = orc.ref_rx_stream(iq, **cfg)
    orc.assert_same_as_ref(rec, ref)
    return rec


def test_synth_adv_stream_all_adv_channels():
    for ch in (37, 38, 39):
        iq, truth = synth.make_adv_stream(512 * 1024, seed=100 + ch, channel=ch, corrupt_every=7)
        rec = _cmp(iq.numpy(), channel=ch)
        assert len(rec) >= 60
        assert rec["crc_bad"].sum() >= 1


def test_data_channels_custom_aa_crcinit():
    for ch in (0, 9, 10, 36):
        aa, ci = 0x60850A1B + ch, 0xA77B22 ^ ch
        iq, _ = synth.make_adv_stream(256 * 1024, seed=200 + ch, channel=ch, access_addr=aa, crc_init=ci,
                                      data_channel_pdu=True, corrupt_every=5, slot_samples=2048)
        rec = _cmp(iq.numpy(), channel=ch, access_addr=aa, crc_init=ci)
        assert len(rec) >= 50


def test_raw_mode():
    iq, _ = synth.make_adv_stream(256 * 1024, seed=5, channel=37)
    rec = _cmp(iq.numpy(), channel=37, raw=1)
    assert len(rec) >= 30 and (rec["n_bytes"] == 42).all()


@pytest.mark.parametrize("seed", range(6))
def test_fuzz_random_iq_loose_masks(seed):
    """Adversarial: full-scale random IQ with sparse masks -> very many hits, negative
    n0 through the zeroed history (App. A.2), hits in the look-ahead tail, length-guard
    breaks, bad ADV lengths."""
    rng = np.random.default_rng(seed)
    iq = rng.integers(-128, 128, 8 * 16384 + 5000, dtype=np.int8)
    masks = [0x0000000F, 0x000000FF, 0x80000001, 0x00000000, 0xF0000000, 0x00010100]
    aas = [0x8E89BED6, 0x00000000, 0xFFFFFFFF, 0x55555555, 0x80000000, 0x12345678]
    for ch in (37, 3):
        for raw in (0, 1):
            rec = _cmp(iq, channel=ch, access_addr=aas[seed], access_mask=masks[seed], raw=raw,
                       crc_init=0x123456)
            assert len(rec) > 8


def test_fuzz_small_amplitude_zero_products():
    """d uses a strict > 0 (btle_rx.c:1533): zeros and tiny amplitudes must give bit 0."""
    rng = np.random.default_rng(99)
    iq = rng.integers(-1, 2, 6 * 16384, dtype=np.int8)
    _cmp(iq, channel=38, access_mask=0x000003FF, access_addr=0x2AA)
    _cmp(np.zeros(3 * 16384, dtype=np.int8), channel=37, access_addr=0, access_mask=0xFFFFFFFF)


def test_short_and_ragged_lengths():
    rng = np.random.default_rng(3)
    for n in (0, 100, 16383, 16384, 16385, 16384 + 3007, 2 * 16384 + 1):
        iq = rng.integers(-128, 128, n, dtype=np.int8)
        _cmp(iq, channel=37, access_mask=0xFF)


def test_worst_case_packets_per_chunk():
    """BTLE_MAX_PKTS_PER_CHUNK (include/btle_b200.h): with mask 0 every window matches, through the zeroed
    history up to 31 symbols before the restart point, so a zero-length data PDU advances the cursor by only
    328 int8 -> 51 packets in one chunk; with bit 0 of the mask set it is 576 int8 -> at most 34."""
    z = np.zeros(2 * 16384 + 3008, dtype=np.int8)
    best = 0
    for ch in range(37):
        rec = _cmp(z, channel=ch, access_addr=0, access_mask=0)
        best = max(best, int(np.bincount(rec["chunk"]).max()))
    assert best == 51
    # a 1 in bit 0 of the masked access address cannot be matched by the zeroed history
    rng = np.random.default_rng(0)
    for iq in (rng.integers(-128, 128, z.size, dtype=np.int8), rng.integers(-1, 2, z.size, dtype=np.int8)):
        for ch in (1, 9, 20):
            rec = _cmp(iq, channel=ch, access_addr=1, access_mask=1)
            assert len(rec) > 10 and int(np.bincount(rec["chunk"]).max()) <= 34
