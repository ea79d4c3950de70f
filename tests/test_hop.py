"""Offline connection following (btle_b200/hop.py).  The logic is host-side; on the CPU it is driven
by an oracle-backed stand-in for BtleRx (tests only), on the GPU by the real thing."""
import os

import numpy as np
import pytest
import torch

import orc
from btle_b200 import REC_DTYPE, synth
from btle_b200.hop import channel_freq_mhz, follow_connections, hop_events_ndjson, parse_connect_req


class OracleRx:
    """rx_batch() with the oracle — test infrastructure, lets the hop logic run without a GPU."""

    def rx_batch(self, iq, cfgs):
        out = [orc.rx_stream(iq[s], channel=int(c["channel"]), access_addr=int(c["access_addr"]),
                             access_mask=int(c["access_mask"]), crc_init=int(c["crc_init"]), stream=s)
               for s, c in enumerate(cfgs)]
        return np.concatenate(out) if out else np.zeros(0, dtype=REC_DTYPE)


def _place(cap, ch, t_s, air, amp=64):
    wav = synth.modulate(air).astype(np.int32) * amp // 127
    p = 2 * int(round(t_s * 4e6))
    seg = cap[ch, p:p + wav.size].astype(np.int32) + wav
    cap[ch, p:p + wav.size] = np.clip(seg, -128, 127).astype(np.int8)


def _capture_with_connection():
    n = 100 * 16384                                       # 205 ms on every channel
    gen = torch.Generator(); gen.manual_seed(3)
    cap = synth.noise_floor(40 * n, gen).numpy().reshape(40, n).copy()
    aa, crci, hop, interval = 0x60850A1B, 0x227BA7, 9, 16  # 16 x 1.25 ms = 20 ms (the reference's guards need > 11 ms)
    A = bytes.fromhex("5f96ea301800"); B = bytes.fromhex("9992b1ebd790")
    creq = synth.adv_pdu(5, 0, 0, A + B + aa.to_bytes(4, "little") + crci.to_bytes(3, "big") + bytes([2]) +
                         (15).to_bytes(2, "little") + interval.to_bytes(2, "little") + bytes(2) + (2000).to_bytes(2, "little") +
                         bytes.fromhex("ffffffff1f") + bytes([hop | (5 << 5)]))
    _place(cap, 37, 0.0030, synth.air_bytes(synth.adv_pdu(0, 0, 0, B + b"\x02\x01\x05"), 37))
    _place(cap, 37, 0.0050, synth.air_bytes(creq, 37))
    # a second initiator with a partial channel map: must be reported, not tracked
    creq2 = bytearray(creq); creq2[2 + 28] = 0x0F
    _place(cap, 38, 0.0070, synth.air_bytes(bytes(creq2), 38))
    sent, ch, t = [], 0, 0.012
    for k in range(9):
        ch = (ch + hop) % 37
        if k != 5:                                        # event 5 is missed entirely -> "skip"
            m = synth.ll_data_pdu(1, k & 1, k & 1, 0, bytes([k] * (k % 5)))
            s_ = synth.ll_data_pdu(1, (k + 1) & 1, k & 1, 0, b"")
            _place(cap, ch, t, synth.air_bytes(m, ch, aa, crci))
            _place(cap, ch, t + 0.00035, synth.air_bytes(s_, ch, aa, crci))
            sent.append((k, ch, m, s_))
        t += interval * 1.25e-3
    return cap, dict(aa=aa, crci=crci, hop=hop, interval=interval), sent


def _check(rx):
    cap, p, sent = _capture_with_connection()
    adv, conns = follow_connections(rx, cap)
    assert len(adv) == 3 and len(conns) == 2
    c = next(c for c in conns if c["tracked"])
    d = next(c for c in conns if not c["tracked"])
    assert d["chm"] == "1fffffff0f" and d["adv_channel"] == 38
    assert c["access_addr"] == p["aa"] and c["crc_init"] == p["crci"] and c["hop"] == 9 and c["interval"] == 16
    assert c["init_a"] == "001830ea965f" and c["adv_a"] == "90d7ebb19299" and c["win_offset"] == 15 and c["sca"] == 5
    ev = {e["k"]: e for e in c["events"]}
    for k, ch, m, s_ in sent:
        e = ev[k]
        assert e["channel"] == ch and len(e["packets"]) == 2, (k, e["channel"], len(e["packets"]))
        assert bytes(e["packets"][0]["bytes"][:len(m)]) == m and bytes(e["packets"][1]["bytes"][:2]) == s_
        assert not e["packets"][0]["crc_bad"] and not e["packets"][1]["crc_bad"]
    assert ev[5]["packets"] == [] and ev[5]["channel"] == (6 * 9) % 37
    chans = [e["channel"] for e in c["events"][:9]]
    assert chans == [((k + 1) * 9) % 37 for k in range(9)]
    _check_hop_events(conns, c, d)


def _check_hop_events(conns, c, d):
    """NDJSON `hop` lines (btle_json.h:21-24) for the two CONNECT_REQs of the test capture."""
    import json
    text = hop_events_ndjson(conns)
    lines = text.splitlines()
    ev = [json.loads(l) for l in lines]
    assert all(l.startswith('{"v":1,"t":"hop","ts":') for l in lines)          # btj_emit_hop's field order
    assert [list(e) for e in ev] == [["v", "t", "ts", "event", "state_from", "state_to", "ch", "freq_mhz", "aa", "crc_init",
                                      "interval_us", "hop", "chm"]] * len(ev)
    assert [e["ts"] for e in ev] == sorted(e["ts"] for e in ev)
    drop = [e for e in ev if e["event"] == "track_drop"]
    assert len(drop) == 1 and drop[0]["ch"] == 38 and drop[0]["chm"] == "1fffffff0f" and drop[0]["freq_mhz"] == 0 \
        and (drop[0]["state_from"], drop[0]["state_to"], drop[0]["interval_us"]) == (0, 0, 0)      # btle_rx.c:2420-2422
    start = [e for e in ev if e["event"] == "track_start"]
    assert len(start) == 1 and start[0]["ch"] == 9 and start[0]["freq_mhz"] == 2422 and start[0]["interval_us"] == 20000 \
        and start[0]["aa"] == "60850a1b" and start[0]["crc_init"] == "227ba7" and start[0]["hop"] == 9 \
        and (start[0]["state_from"], start[0]["state_to"]) == (0, 1) and abs(start[0]["ts"] - 0.005) < 1e-3
    chg = [e for e in ev if e["event"] == "chan_change"]
    assert len(chg) == len(c["events"]) - 1 and len(chg) >= 8
    assert [e["ch"] for e in chg[:8]] == [((k + 2) * 9) % 37 for k in range(8)]
    # event 5 had no packet: the hop out of it is a "skip" (3 -> 3), all others follow a CRC-ok packet (2 -> 3)
    assert [(e["state_from"], e["state_to"]) for e in chg[:8]] == [(2, 3)] * 5 + [(3, 3)] + [(2, 3)] * 2
    # a hop happens one interval minus the 7 ms guard after the previous anchor (btle_rx.c:2404, :2431, :2472)
    e1 = c["events"][0]
    assert abs(chg[0]["ts"] - (e1["t"] + 0.020 - 0.007)) < 1e-6
    # the reference's own NDJSON consumer (btle_cli.events.parse_line) took every one of these lines for a HopEvent
    accepted = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cli_consumers.json")))["hop_lines"]
    assert all(accepted.get(l) == "HopEvent" for l in lines), [l for l in lines if l not in accepted]


def test_parse_connect_req_rejects_other_pdus():
    r = np.zeros(1, dtype=REC_DTYPE)[0]
    r["bytes"][0], r["bytes"][1] = 0x05, 33
    assert parse_connect_req(r) is None
    r["bytes"][1] = 34; r["crc_bad"] = 1
    assert parse_connect_req(r) is None


def test_follow_connections_logic_with_oracle_backend():
    _check(OracleRx())


@pytest.mark.gpu
def test_follow_connections_on_gpu():
    import __graft_entry__ as ge
    ge.build()
    from btle_b200 import BtleRx
    _check(BtleRx(0))


def test_channel_freq_mhz_is_the_reference_mapping():
    # get_freq_by_channel_number, btle_rx.c:1006-1022
    assert [channel_freq_mhz(c) for c in (37, 38, 39, 0, 10, 11, 36)] == [2402, 2426, 2480, 2404, 2424, 2428, 2478]
    with pytest.raises(ValueError):
        channel_freq_mhz(40)


# ---- the C connection follower (btle_b200_receiver_controller) against the reference's own receiver_controller --------
def _write_dir(tmp, cap):
    for c in range(40):
        cap[c].tofile(os.path.join(tmp, f"ch{c:02d}.bin"))


def _ref_hop_lines(tmp, verbose=1):
    return orc.ref_driver(["hop", tmp, "37", "8e89bed6", "555555", "ffffffff", "0", "1", str(verbose)], inputs=[tmp]).splitlines()


def test_c_controller_replays_the_reference_state_machine(tmp_path):
    """Feeds btle_b200_receiver_controller() / btle_b200_note_packet() / the payload parsers (host C, no GPU) with the
    packet trace the UNMODIFIED reference produced while following the connection on a virtual radio (oracle/_ref `hop`
    mode: the reference's receiver() + receiver_controller() over 40 per-channel captures), chunk by chunk, and expects
    the same hop events, byte for byte as NDJSON."""
    import ctypes
    import json
    from btle_b200 import _native
    cap, p, sent = _capture_with_connection()
    _write_dir(str(tmp_path), cap)
    lines = _ref_hop_lines(str(tmp_path))
    ref_events = [ln for ln in lines if ln.startswith('{"v":1,"t":"hop"')]
    pkts = [json.loads(ln) for ln in lines if ln.startswith('{"v":1,"t":"pkt"')]
    assert len(ref_events) >= 8 and any('"state_from":3,"state_to":3' in e for e in ref_events)       # a "skip" is in there

    L = _native.load()
    i64, vp = ctypes.c_int64, ctypes.c_void_p

    class Ev(ctypes.Structure):
        _fields_ = [("ts_us", i64), ("event", ctypes.c_char * 16), ("state_from", ctypes.c_int), ("state_to", ctypes.c_int), ("ch", ctypes.c_int),
                    ("freq_mhz", ctypes.c_int), ("access_addr", ctypes.c_uint32), ("crc_init", ctypes.c_uint32), ("interval_us", ctypes.c_int),
                    ("hop", ctypes.c_int), ("chm", ctypes.c_uint8 * 5)]
    NOW = ctypes.CFUNCTYPE(i64, vp)
    SETF = ctypes.CFUNCTYPE(ctypes.c_int, vp, ctypes.c_uint64)
    EVT = ctypes.CFUNCTYPE(None, vp, ctypes.POINTER(Ev))

    class Hooks(ctypes.Structure):
        _fields_ = [("now_us", NOW), ("set_freq", SETF), ("event", EVT), ("user", vp), ("quiet_text", ctypes.c_int)]
    state = {"now": 0}
    got = []

    def on_event(_u, e):
        e = e.contents
        got.append('{"v":1,"t":"hop","ts":%.6f,"event":"%s","state_from":%d,"state_to":%d,"ch":%d,"freq_mhz":%d,"aa":"%08x","crc_init":"%06x",'
                   '"interval_us":%d,"hop":%d,"chm":"%s"}' % (e.ts_us / 1e6, e.event.decode(), e.state_from, e.state_to, e.ch, e.freq_mhz, e.access_addr,
                                                               e.crc_init & 0xFFFFFF, e.interval_us, e.hop, bytes(e.chm).hex()))
    hooks = Hooks(NOW(lambda u: state["now"]), SETF(lambda u, f: 0), EVT(on_event), None, int(os.environ.get("HOP_QUIET", "1")))
    L.btle_b200_set_hop_hooks.argtypes = [ctypes.POINTER(Hooks)]
    L.btle_b200_receiver_controller.argtypes = [vp, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint32)]
    L.btle_b200_parse_adv_pdu_payload_byte.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp]
    L.btle_b200_parse_ll_pdu_payload_byte.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp]
    L.btle_b200_note_packet.argtypes = [vp]
    L.btle_b200_hop_reset()
    L.btle_b200_set_hop_hooks(ctypes.byref(hooks))
    try:
        nchunks = cap.shape[1] // 16384
        by_chunk = {}
        for pk in pkts:                                 # the reference stamps packets with the virtual time of their chunk
            k = round((pk["ts"] * 1e6 * 4 - 1504) / 8192) - 1
            by_chunk.setdefault(k, []).append(pk)
        chan, aa, crc = ctypes.c_int(37), ctypes.c_uint32(0x8E89BED6), ctypes.c_uint32(0)
        scratch = ctypes.create_string_buffer(64)
        for k in range(nchunks):
            for pk in by_chunk.get(k, []):
                assert pk["ch"] == chan.value and int(pk["aa"], 16) == aa.value      # our machine is on the channel / AA the reference was on
                rec = np.zeros(1, dtype=REC_DTYPE)
                rec["crc_bad"] = 0 if pk["crc_ok"] else 1
                L.btle_b200_note_packet(rec.ctypes.data)
                payload = bytes.fromhex(pk["payload_hex"])
                if pk["kind"] == "adv":
                    assert L.btle_b200_parse_adv_pdu_payload_byte(payload, len(payload), pk["pdu_type"], scratch) == 0
                else:
                    assert L.btle_b200_parse_ll_pdu_payload_byte(payload, len(payload), pk["ll_pdu_type"], scratch) >= 0
            state["now"] = ((k + 1) * 8192 + 1504) // 4
            assert L.btle_b200_receiver_controller(None, 1, ctypes.byref(chan), ctypes.byref(aa), ctypes.byref(crc)) == 0
    finally:
        L.btle_b200_set_hop_hooks(None)
    assert got == ref_events


def test_payload_parsers_keep_the_reference_contract(capfd):
    """parse_adv_pdu_payload_byte / parse_ll_pdu_payload_byte: 0 / -1 / opcode, the reference's messages, its struct layouts."""
    import ctypes
    from btle_b200 import _native
    L = _native.load()
    L.btle_b200_parse_adv_pdu_payload_byte.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    L.btle_b200_parse_ll_pdu_payload_byte.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    out = ctypes.create_string_buffer(64)
    adva = bytes.fromhex("060504030201")
    assert L.btle_b200_parse_adv_pdu_payload_byte(adva + b"\x02\x01\x06", 9, 0, out) == 0
    assert out.raw[:6] == adva[::-1] and out.raw[6:9] == b"\x02\x01\x06"                     # AdvA MSB first, Data as sent
    assert L.btle_b200_parse_adv_pdu_payload_byte(adva, 5, 0, out) == -1                      # too short
    assert L.btle_b200_parse_adv_pdu_payload_byte(adva + adva[:5], 11, 3, out) == -1          # SCAN_REQ must be 12
    creq = bytes(range(34))
    assert L.btle_b200_parse_adv_pdu_payload_byte(creq, 33, 5, out) == -1
    assert L.btle_b200_parse_adv_pdu_payload_byte(creq, 34, 5, out) == 0
    import struct as st_
    # ADV_PDU_PAYLOAD_TYPE_5: InitA[6] AdvA[6] AA[4] CRCInit(u32) WinSize(u8) pad WinOffset Interval Latency Timeout (u16) ChM[5] Hop SCA
    assert out.raw[:6] == creq[0:6][::-1] and out.raw[6:12] == creq[6:12][::-1] and out.raw[12:16] == creq[12:16][::-1]
    assert st_.unpack_from("<I", out.raw, 16)[0] == (creq[16] << 16 | creq[17] << 8 | creq[18])
    assert out.raw[20] == creq[19] and st_.unpack_from("<HHHH", out.raw, 22) == tuple(creq[20 + 2 * i] | creq[21 + 2 * i] << 8 for i in range(4))
    assert out.raw[30:35] == creq[28:33][::-1] and out.raw[35] == creq[33] & 0x1F and out.raw[36] == creq[33] >> 5
    status = ctypes.cast(L.btle_b200_receiver_status, ctypes.c_void_p)
    assert L.btle_b200_parse_ll_pdu_payload_byte(b"", 0, 1, out) == 0
    assert L.btle_b200_parse_ll_pdu_payload_byte(b"", 0, 3, out) == -1
    assert L.btle_b200_parse_ll_pdu_payload_byte(bytes([12, 9, 0x0f, 0, 1, 2]), 6, 3, out) == 12        # LL_VERSION_IND
    assert out.raw[0] == 12 and out.raw[1] == 9 and st_.unpack_from("<HH", out.raw, 2) == (0x000f, 0x0201)
    assert L.btle_b200_parse_ll_pdu_payload_byte(bytes([12, 9, 0x0f, 0, 1]), 5, 3, out) == -1
    assert L.btle_b200_parse_ll_pdu_payload_byte(bytes([0x33, 1, 2]), 3, 3, out) == 0x33                 # unknown opcode: kept
    text = capfd.readouterr().out
    for msg in ("Error: Payload Too Short (only 5 bytes)!", "Error: Payload length 11 bytes. Need to be 12 for PDU Type SCAN_REQ!",
                "Error: Payload length 33 bytes. Need to be 34 for PDU Type CONNECT_REQ!", "Error: LL PDU TYPE3(LL_CTRL) should not have payload length 0!",
                "Error: LL CTRL PDU TYPE12(LL_VERSION_IND) should have payload length 6!"):
        assert msg in text


# ---- many connections at once: windowed follower == full follower, in three launches ---------------------------------
def _capture_with_many_connections(n_conn=6, intervals=(16, 20, 24, 16, 20, 18, 22, 16)):
    n = 100 * 16384
    gen = torch.Generator(); gen.manual_seed(11)
    cap = synth.noise_floor(40 * n, gen).numpy().reshape(40, n).copy()
    rng = np.random.default_rng(4)
    A = lambda: rng.integers(0, 256, 6, dtype=np.uint8).tobytes()
    conns = []
    for i in range(n_conn):
        aa, crci = 0x50850A1B + 0x01010101 * i, 0x227BA7 ^ (i * 0x010203)
        hop, interval = [9, 5, 11, 16, 7, 13, 6, 10][i % 8], intervals[i % 8]
        creq = synth.adv_pdu(5, 0, 0, A() + A() + aa.to_bytes(4, "little") + crci.to_bytes(3, "big") + bytes([2]) + (15).to_bytes(2, "little") +
                             interval.to_bytes(2, "little") + bytes(2) + (2000).to_bytes(2, "little") + bytes.fromhex("ffffffff1f") + bytes([hop | (5 << 5)]))
        adv_ch = 37 + i % 3
        t_creq = 0.002 + 0.0031 * i
        _place(cap, adv_ch, t_creq, synth.air_bytes(creq, adv_ch))
        ch, t = 0, t_creq + 0.006
        missing = {int(x) for x in rng.choice(np.arange(1, 9), size=2, replace=False)} if i % 2 else set()
        k = 0
        while t < 0.195:
            ch = (ch + hop) % 37
            if k not in missing:
                m = synth.ll_data_pdu(1, k & 1, k & 1, 0, bytes([i, k] * (k % 4)))
                _place(cap, ch, t, synth.air_bytes(m, ch, aa, crci), amp=60 + i)
                _place(cap, ch, t + 0.0004, synth.air_bytes(synth.ll_data_pdu(1, (k + 1) & 1, k & 1, 0, b""), ch, aa, crci))
            t += interval * 1.25e-3
            k += 1
        conns.append(dict(aa=aa, crci=crci, hop=hop, interval=interval))
    return cap, conns


class CountingRx:
    def __init__(self, inner):
        self.inner, self.calls, self.chunks = inner, 0, 0

    def rx_batch(self, iq, cfgs):
        self.calls += 1
        self.chunks += iq.shape[0] * (iq.shape[1] // 16384)
        return self.inner.rx_batch(iq, cfgs)


def _check_windowed(rx, intervals=(16, 20, 24, 16, 20, 18, 22, 16), expect_calls=3):
    from btle_b200.hop import follow_connections_windowed
    cap, truth = _capture_with_many_connections(6, intervals)
    full_rx, win_rx = CountingRx(rx), CountingRx(rx)
    _, full = follow_connections(full_rx, cap)
    _, win = follow_connections_windowed(win_rx, cap)
    assert len(full) == len(win) == 6 and all(c["tracked"] for c in win)
    assert win_rx.calls == expect_calls and full_rx.calls == 1 + 6           # three launches whatever the number of connections
    if expect_calls == 3:
        assert win_rx.chunks * 6 < full_rx.chunks                            # and several times less decoding
    by_aa = lambda xs, key: sorted(xs, key=lambda c: c[key])
    for a, b, t in zip(by_aa(full, "access_addr"), by_aa(win, "access_addr"), by_aa(truth, "aa")):
        assert a["access_addr"] == b["access_addr"] == t["aa"] and a["hop"] == b["hop"] == t["hop"]
        assert len(a["events"]) == len(b["events"]) >= 5
        for x, y in zip(a["events"], b["events"]):
            assert (x["channel"], x["anchored"], len(x["packets"])) == (y["channel"], y["anchored"], len(y["packets"]))
            assert abs(x["t"] - y["t"]) < 1e-12 and abs(x["t_hop"] - y["t_hop"]) < 1e-12
            for p, q in zip(x["packets"], y["packets"]):
                assert p.tobytes()[4:] == q.tobytes()[4:]                    # everything but the batch-local stream index
        assert any(not e["anchored"] for e in a["events"]) == any(not e["anchored"] for e in b["events"])
    assert hop_events_ndjson(full) == hop_events_ndjson(win)


def test_windowed_follower_equals_full_follower_with_oracle_backend():
    _check_windowed(OracleRx())


def test_windowed_follower_falls_back_when_the_reference_machine_loses_the_connection():
    """15 ms interval and two missed events in a row: the reference's state machine arrives earlier and earlier and never
    re-anchors (its dwell ends before the packet comes).  The windowed follower notices that the walk left its predicted
    windows and redoes that one connection with full passes — same result as the full follower."""
    _check_windowed(OracleRx(), intervals=(16, 12, 24, 16, 20, 18, 22, 16), expect_calls=4)


@pytest.mark.gpu
def test_windowed_follower_on_gpu():
    import __graft_entry__ as ge
    ge.build()
    from btle_b200 import BtleRx
    _check_windowed(BtleRx(0))
