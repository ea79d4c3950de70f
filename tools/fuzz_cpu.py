#!/usr/bin/env python
"""Long-running CPU fuzz (no GPU): unmodified reference (oracle/_ref) vs the C restatement (oracle/) vs the
CPU emulation of the kernel logic (tests/emul), on random access addresses / masks / channels / CRC inits and a
mix of input kinds.  FUZZ_SECONDS (default 300), argv[1] = seed."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import emul, orc
from btle_b200 import synth

rng = np.random.default_rng(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
t0, n_case, n_pkt = time.time(), 0, 0
kinds = {}
while time.time() - t0 < float(os.environ.get("FUZZ_SECONDS", "300")):
    kind = int(rng.integers(0, 5))
    nchunks = int(rng.integers(1, 7))
    n = nchunks * 16384 + int(rng.choice([0, 0, 1, 2, 3007, 3008, 3009, int(rng.integers(0, 16384))]))
    ch = int(rng.integers(0, 40))
    aa = int(rng.integers(0, 1 << 32))
    crc_init = int(rng.integers(0, 1 << 24))
    raw = int(rng.integers(0, 4) == 0)
    pop = int(rng.choice([0, 1, 2, 4, 8, 12, 16, 24, 32]))
    mask = 0
    for p in rng.permutation(32)[:pop]:
        mask |= 1 << int(p)
    if kind == 0:      # full-scale random IQ
        iq = rng.integers(-128, 128, n, dtype=np.int8)
    elif kind == 1:    # tiny amplitudes: products are 0 / +-1
        iq = rng.integers(-1, 2, n, dtype=np.int8)
    elif kind == 2:    # real bursts with the full mask on a random channel, dense slots
        adv = ch >= 37
        iq_t, _ = synth.make_adv_stream(n, seed=int(rng.integers(0, 1 << 30)), channel=ch, access_addr=aa, crc_init=crc_init,
                                        corrupt_every=int(rng.choice([0, 3, 50])), slot_samples=int(rng.choice([1500, 2048, 3000, 4096])),
                                        data_channel_pdu=not adv)
        iq = iq_t.numpy()
        mask = 0xFFFFFFFF if rng.integers(0, 2) else (mask | 0xFF)
    elif kind == 3:    # bursts + strong random interference in stretches
        iq_t, _ = synth.make_adv_stream(n, seed=int(rng.integers(0, 1 << 30)), channel=37 + ch % 3, access_addr=aa, crc_init=crc_init,
                                        slot_samples=2048)
        iq = iq_t.numpy().copy()
        ch = 37 + ch % 3
        for _ in range(8):
            a = int(rng.integers(0, max(1, n - 4000)))
            iq[a:a + 4000] = rng.integers(-128, 128, min(4000, n - a), dtype=np.int8)
        mask = 0xFFFFFFFF
    else:              # constant / periodic patterns (long runs of identical d-bits)
        period = int(rng.choice([2, 4, 6, 8, 16, 64]))
        base = rng.integers(-100, 101, period, dtype=np.int8)
        iq = np.resize(base, n).astype(np.int8)
    cfg = dict(channel=ch, access_addr=aa, access_mask=mask, crc_init=crc_init, raw=raw)
    o = orc.rx_stream(iq, **cfg)
    e = emul.rx_stream(iq, span_chunks=int(rng.choice([1, 2, 5, 16])), **cfg)
    assert o.tobytes() == e.tobytes(), ("emul != oracle", kind, n, cfg)
    # the kernel's unit plan + list-driven chain + decode pass + unit directory
    from btle_b200._native import CFG_DTYPE
    c1 = np.zeros(1, dtype=CFG_DTYPE)
    c1[0] = (ch, aa, mask, crc_init, raw, 1)
    ur, ud = emul.rx_batch_units(iq[None, :], c1, grid=int(rng.choice([1, 3, 148])), reverse_units=bool(rng.integers(0, 2)))
    uw = np.concatenate([ur[int(b):int(b) + int(c)] for b, c in ud]) if len(ud) else ur[:0]
    assert uw.tobytes() == o.tobytes(), ("emul units != oracle", kind, n, cfg)
    if orc.ref_available():
        orc.assert_same_as_ref(o, orc.ref_rx_stream(iq, live=True, **cfg))
    n_case += 1; n_pkt += len(o); kinds[kind] = kinds.get(kind, 0) + len(o)
print(f"fuzz ok: {n_case} cases, {n_pkt} packets compared, packets per input kind {kinds}, ref={'yes' if orc.ref_available() else 'no'}")
