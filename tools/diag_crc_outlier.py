#!/usr/bin/env python
"""The bench stream has one CRC failure more than the bursts that were corrupted on purpose.  Find it and run
the whole 1 GiB capture through the CPU oracle around it: the verdict must be the reference's, not ours."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import orc
import bench
from btle_b200 import BtleRx, make_cfgs, synth, REC_DTYPE

n_int8 = bench.STREAM_INT8
iq, truth = synth.make_adv_stream(n_int8, seed=bench.SEED, channel=37, slot_samples=bench.SLOT_SAMPLES, corrupt_every=100, device="cuda")
rx = BtleRx(0)
cfgs = make_cfgs(1, rssi=1)     # the oracle always fills mag_sum
cap = n_int8 // 16384 * 3
d_out = torch.empty(cap * 64, dtype=torch.uint8, device="cuda")
d_cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
rx.rx_device(iq.view(1, -1), cfgs, d_out, d_cnt, torch.cuda.current_stream().cuda_stream)
torch.cuda.synchronize()
n = int(d_cnt.item())
rec = rx.sort_records(d_out[: n * 64].cpu().numpy().view(REC_DTYPE))
pos = rec["chunk"].astype(np.int64) * 8192 + rec["n0"]
starts = truth["start_sample"]
# burst s starts (preamble) at starts[s]; its access address 8 symbols = 32 samples later
idx = np.searchsorted(starts, pos, side="right") - 1
bad = rec["crc_bad"] != 0
extra = np.nonzero(bad & ~truth["corrupt"][idx])[0]
print("records", n, "crc bad", int(bad.sum()), "corrupted on purpose", int(truth["corrupt"].sum()), "extra", extra.tolist())
host = iq.cpu().numpy()
for e in extra:
    c = int(rec["chunk"][e])
    base = max(0, c - 1)
    lo, hi = base * 16384, min(n_int8, (c + 3) * 16384)
    nch = (hi - lo) // 16384
    exp = orc.rx_stream(host[lo:hi])
    mine = rec[(rec["chunk"] >= base) & (rec["chunk"] < base + nch)].copy()
    mine["chunk"] -= base
    print("chunk", c, "n0", int(rec["n0"][e]), "offset from burst start", int(pos[e] - starts[idx[e]]), "n_bytes", int(rec["n_bytes"][e]),
          "| oracle on chunks", base, "..", base + nch - 1, "equal:", mine.tobytes() == exp.tobytes(), "records", len(mine), len(exp))
    pdu = truth["pdus"][idx[e]]
    got = bytes(rec["bytes"][e][: int(rec["n_bytes"][e])])
    sent = bytes(pdu) if not isinstance(pdu, bytes) else pdu
    diff = [(i, got[i] ^ sent[i]) for i in range(min(len(got), len(sent))) if got[i] != sent[i]]
    print("   decoded vs transmitted PDU (byte index, xor):", diff, "lengths", len(got), len(sent))
    if orc.ref_available():
        try:
            orc.assert_same_as_ref(mine, orc.ref_rx_stream(host[lo:hi], live=True))
            print("   unmodified reference: equal")
        except AssertionError as ex:
            print("   unmodified reference: DIFFERENT", ex)
