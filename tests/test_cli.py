"""The btle_rx-compatible host program (btle_b200/btle_rx_b200): option surface and exit codes on
the CPU; on the GPU its text / NDJSON / pcap output against the reference's own sinks
(oracle/_ref/btle_ref_driver sinks, as recorded in tests/golden/ref_driver.npz) for the same capture, modulo time stamps."""
import os
import re
import subprocess
import zlib

import numpy as np
import pytest

import orc
from btle_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "btle_b200", "btle_rx_b200")


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__ as ge
    ge.build()
    assert os.path.exists(CLI)


def run(args, **kw):
    return subprocess.run([CLI] + args, capture_output=True, text=True, **kw)


def test_bad_arguments_print_usage_and_exit_minus_one():
    for args in (["-c", "40"], ["-g", "63"], ["-l", "41"], ["--nope"], ["-c", "37", "extra"], ["-h"],
                 ["-F", "zz"], ["-T", "16"]):
        p = run(args)
        assert p.returncode == 255, args          # exit(-1), btle_rx.c:1457
        assert "Usage" in p.stdout


def test_no_capture_is_a_board_failure():
    p = run(["-c", "38", "-j", "-Q"])
    assert p.returncode == 1                      # btle_rx.c:2586
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    import json
    ev = [json.loads(l) for l in lines]
    assert [e["event"] for e in ev] == ["start", "stop"] and ev[0]["ch"] == 38 and ev[0]["freq_hz"] == 2426000000


def _adv_pdus(rng):
    A = lambda: rng.integers(0, 256, 6, dtype=np.uint8).tobytes()
    out = []
    for t in (0, 2, 4, 6):
        out.append(synth.adv_pdu(t, 1, 0, A() + rng.integers(0, 256, int(rng.integers(0, 32)), dtype=np.uint8).tobytes()))
    out.append(synth.adv_pdu(1, 0, 1, A() + A()))
    out.append(synth.adv_pdu(3, 1, 1, A() + A()))
    out.append(synth.adv_pdu(3, 1, 1, A() + A() + b"\x01"))              # SCAN_REQ with a wrong length -> dropped
    out.append(synth.adv_pdu(5, 0, 0, A() + A() + bytes.fromhex("1b0a8560") + bytes.fromhex("227ba7") +
                             bytes([2]) + bytes.fromhex("0f00500000000d07") + bytes.fromhex("ffffffff1f") + bytes([0xA9])))
    out.append(synth.adv_pdu(5, 0, 0, A() * 3))                           # CONNECT_REQ with a wrong length -> dropped
    out.append(synth.adv_pdu(9, 0, 0, rng.integers(0, 256, 20, dtype=np.uint8).tobytes()))   # reserved type
    out.append(synth.adv_pdu(0, 0, 0, bytes.fromhex("a1b2c3d4e5f6") + b"hello"))
    return out


def _ll_pdus(rng):
    R = lambda n: rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    out = [synth.ll_data_pdu(1, 0, 1, 0, b""), synth.ll_data_pdu(2, 1, 0, 1, R(9)), synth.ll_data_pdu(2, 1, 0, 1, b""),
           synth.ll_data_pdu(0, 0, 0, 0, R(3)), synth.ll_data_pdu(3, 0, 0, 0, b"")]
    for op, n in ((0, 12), (1, 8), (2, 2), (7, 2), (13, 2), (3, 23), (4, 13), (5, 1), (6, 1), (10, 1), (11, 1), (8, 9),
                  (9, 9), (12, 6), (14, 5), (200, 4), (0, 11), (12, 7)):
        out.append(synth.ll_data_pdu(3, 0, 1, 0, bytes([op]) + R(n - 1)))
    return out


def _undefined_in_reference(line):
    """Data-channel PDUs that are not LL control PDUs and carry a payload: the reference decides whether to drop them
    from an UNINITIALISED int (parse_ll_pdu_payload_byte, btle_rx.c:1742 / :1936, checked at :2350-2353).  oracle/_ref is
    built with -ftrivial-auto-var-init=zero, which pins that int to 0 = "kept" — the behaviour this repo defines
    (DESIGN.md §2) — so nothing has to be left out of the comparison any more."""
    return False


def _normalise_text(s):
    keep = []
    for l in s.splitlines():
        if _undefined_in_reference(l):
            continue
        if re.match(r"^\d+us Pkt", l):
            keep.append(re.sub(r"^\d+us ", "T ", l))
        elif re.match(r"^\d+\.\d+ Pkt", l):
            keep.append(re.sub(r"^\d+\.\d+ ", "T ", l))
        elif l.startswith("Error:") or l.startswith("XXXus PktBAD") or l.startswith("Hop:"):
            keep.append(l)
        elif l.startswith("{") and '"t":"hop"' in l:
            keep.append(l)
        elif l.startswith("{") and '"t":"pkt"' in l:
            keep.append(re.sub(r'"ts":[0-9.]+', '"ts":0', l))
    return keep


def _pcap_records(path):
    b = open(path, "rb").read()
    assert b[:24] == bytes.fromhex("a1b2c3d4000200040000000000000000000005dc00000100")      # btle_rx.c:110
    recs, off = [], 24
    while off < len(b):
        caplen = int.from_bytes(b[off + 8:off + 12], "big")
        assert caplen == int.from_bytes(b[off + 12:off + 16], "big")
        rec = b[off + 16:off + 16 + caplen]
        off += 16 + caplen
        ch, hdr0, plen = rec[0], rec[14], rec[15] & 0x1F
        recs.append(rec)
    return recs


CASES = [
    ("adv", 37, 0x8E89BED6, 0x555555, [], _adv_pdus),
    ("adv_filter_type", 38, 0x8E89BED6, 0x555555, ["-T", "0,3,5"], _adv_pdus),
    ("adv_filter_adva", 39, 0x8E89BED6, 0x555555, ["-F", "f6:e5:d4:c3:b2:a1"], _adv_pdus),
    ("adv_raw", 37, 0x8E89BED6, 0x555555, ["-r"], _adv_pdus),
    ("data", 9, 0x60850A1B, 0xA77B22, [], _ll_pdus),
    ("data_filter_adva", 20, 0x11850A1B, 0x123456, ["-F", "010203040506"], _ll_pdus),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,ch,aa,crc,extra,mk", CASES)
def test_cli_output_equals_reference_sinks(tmp_path, name, ch, aa, crc, extra, mk):
    rng = np.random.default_rng(zlib.crc32(name.encode()) & 0xFFFF)      # a seed that is the same in every process
    pdus = mk(rng)
    iq = synth.make_pdu_stream(pdus, ch, aa, crc, seed=5, corrupt={1, 7})
    f = tmp_path / "iq.bin"
    iq.tofile(f)
    mine_pcap, ref_pcap = tmp_path / "mine.pcap", tmp_path / "ref.pcap"
    p = run(["-i", str(f), "-c", str(ch), "-a", f"{aa:x}", "-k", f"{crc:x}", "-j", "-R", "-s", str(mine_pcap)] + extra)
    assert p.returncode == 0, p.stdout + p.stderr
    fa = extra[extra.index("-F") + 1] if "-F" in extra else "-"
    ft = extra[extra.index("-T") + 1] if "-T" in extra else "-"
    q = orc.ref_driver(["sinks", f, ch, f"{aa:x}", f"{crc:x}", "ffffffff", "1" if "-r" in extra else "0", "0", "1", "1", ref_pcap, fa, ft],
                       inputs=[f], outputs=[ref_pcap])
    mine, ref = _normalise_text(p.stdout), _normalise_text(q)
    assert len(ref) >= 4
    assert mine == ref
    assert _pcap_records(mine_pcap) == _pcap_records(ref_pcap)


@pytest.mark.gpu
def test_cli_sc16_input_equals_int8_input(tmp_path):
    iq8, _ = synth.make_adv_stream(6 * 16384, seed=4, channel=37, slot_samples=2500)
    iq8 = iq8.numpy()
    (tmp_path / "a.int8").write_bytes(iq8.tobytes())
    (tmp_path / "a.sc16").write_bytes((iq8.astype(np.int16) << 4).tobytes())
    a = run(["-i", str(tmp_path / "a.int8"), "-Q", "-j"])
    b = run(["--iq-sc16", str(tmp_path / "a.sc16"), "-Q", "-j"])
    assert a.returncode == 0 and b.returncode == 0
    pk = lambda s_: [l for l in s_.splitlines() if '"t":"pkt"' in l]
    assert len(pk(a.stdout)) > 10 and pk(a.stdout) == pk(b.stdout)


@pytest.mark.gpu
def test_cli_verbose_prints_the_reference_pktbad_lines(tmp_path):
    """-v: access-address hits whose ADV header length is outside 6..37 are printed as "PktBAD" and not counted
    (btle_rx.c:2291-2298).  They come back from the GPU as BTLE_REC_REJECTED records."""
    rng = np.random.default_rng(11)
    pdus = _adv_pdus(rng)
    pdus.insert(2, synth.adv_pdu(0, 1, 0, b"\x01\x02\x03"))                   # PloadL3
    pdus.insert(5, bytes([0x02, 45]) + bytes(range(20)))                      # header says PloadL45
    pdus.append(synth.adv_pdu(6, 0, 1, bytes(5)))                             # PloadL5
    iq = synth.make_pdu_stream(pdus, 37, seed=9, corrupt={1})
    f = tmp_path / "iq.bin"
    iq.tofile(f)
    p = run(["-i", str(f), "-c", "37", "-v", "-j"])
    assert p.returncode == 0, p.stdout + p.stderr
    q = orc.ref_driver(["sinks", f, "37", "8e89bed6", "555555", "ffffffff", "0", "0", "1", "0", "-", "-", "-", "1"], inputs=[f])
    mine, ref = _normalise_text(p.stdout), _normalise_text(q)
    assert sum(l.startswith("XXXus PktBAD") for l in ref) == 3
    assert mine == ref
    quiet = run(["-i", str(f), "-c", "37", "-j"])                             # without -v: same packets, no PktBAD lines
    assert [l for l in mine if not l.startswith("XXXus")] == _normalise_text(quiet.stdout)


@pytest.mark.gpu
def test_cli_hop_follows_the_connection_like_the_reference(tmp_path):
    """-o over per-channel captures (--iq-dir): text lines, packet events and hop events equal what the UNMODIFIED reference
    prints when its receiver() + receiver_controller() drive a virtual radio over the same 40 captures (oracle/_ref hop)."""
    import test_hop as T
    cap, prm, sent = T._capture_with_connection()
    T._write_dir(str(tmp_path), cap)
    p = run(["--iq-dir", str(tmp_path), "-c", "37", "-o", "-v", "-j"])
    assert p.returncode == 0, p.stdout + p.stderr
    ref = T._ref_hop_lines(str(tmp_path), verbose=1)
    mine_n, ref_n = _normalise_text(p.stdout), _normalise_text("\n".join(ref))
    assert sum('"t":"hop"' in l for l in ref_n) >= 8 and sum("Ch8 " in l or '"ch":8,' in l for l in ref_n) >= 2
    assert mine_n == ref_n
    # the consumer side: -Q -j only, every line is NDJSON the reference front-end accepts
    q = run(["--iq-dir", str(tmp_path), "-c", "37", "-o", "-j", "-Q"])
    import json
    ev = [json.loads(l) for l in q.stdout.splitlines() if l.startswith("{")]
    assert [e["t"] for e in ev].count("hop") == sum('"t":"hop"' in l for l in ref_n) and ev[0]["event"] == "start" and ev[-1]["event"] == "stop"


@pytest.mark.gpu
def test_cli_multi_capture_batch_equals_single_runs(tmp_path):
    """-i FILE:CH[:AA[:CRCINIT]] given several times: one batched launch, packets merged in time order."""
    a, _ = synth.make_adv_stream(12 * 16384, seed=21, channel=37, slot_samples=2600, straddle_every=4)
    b, _ = synth.make_adv_stream(12 * 16384, seed=22, channel=9, slot_samples=3100, access_addr=0x60850A24, crc_init=0xA77B2B, data_channel_pdu=True)
    c, _ = synth.make_adv_stream(12 * 16384, seed=23, channel=39, slot_samples=2900)
    for name, t in (("a.bin", a), ("b.bin", b), ("c.bin", c)):
        t.numpy().tofile(tmp_path / name)
    multi = run(["-i", f"{tmp_path}/a.bin:37", "-i", f"{tmp_path}/b.bin:9:60850a24:a77b2b", "-i", f"{tmp_path}/c.bin:39", "-j", "-Q"])
    assert multi.returncode == 0, multi.stdout + multi.stderr
    import json
    pk = lambda s_: [json.loads(l) for l in s_.splitlines() if '"t":"pkt"' in l]
    singles = []
    for args in (["-i", f"{tmp_path}/a.bin", "-c", "37"], ["-i", f"{tmp_path}/b.bin", "-c", "9", "-a", "60850a24", "-k", "a77b2b"],
                 ["-i", f"{tmp_path}/c.bin", "-c", "39"]):
        r = run(args + ["-j", "-Q"])
        assert r.returncode == 0
        singles += pk(r.stdout)
    got = pk(multi.stdout)
    assert len(got) == len(singles) > 30
    assert [e["ts"] for e in got] == sorted(e["ts"] for e in got)
    strip = lambda e: {k: v for k, v in e.items() if k != "pkt"}
    assert sorted(map(json.dumps, map(strip, got))) == sorted(map(json.dumps, map(strip, singles)))


@pytest.mark.gpu
def test_cli_streams_a_capture_in_segments_and_from_a_pipe(tmp_path):
    """A single capture is read in segments straight into page-locked buffers and decoded while the next segment is read
    (btle_b200_stream_*): any segment size, a file or a pipe, gives the records of the whole-capture call."""
    iq, _ = synth.make_adv_stream(45 * 16384 + 5000, seed=31, channel=38, slot_samples=2300, straddle_every=3, corrupt_every=5)
    f = tmp_path / "iq.bin"
    iq.numpy().tofile(f)
    pk = lambda s_: [l for l in s_.splitlines() if '"t":"pkt"' in l]
    whole = run(["-i", str(f), "-c", "38", "-j", "-Q", "-R"])
    assert whole.returncode == 0 and len(pk(whole.stdout)) > 60
    for seg in ("1", "3", "16", "44", "45", "46"):
        r = run(["-i", str(f), "-c", "38", "-j", "-Q", "-R", "--segment-chunks", seg])
        assert r.returncode == 0, r.stdout + r.stderr
        assert pk(r.stdout) == pk(whole.stdout), seg
    with open(f, "rb") as fh:
        piped = subprocess.run([CLI, "-i", "-", "-c", "38", "-j", "-Q", "-R", "--segment-chunks", "7"], stdin=fh, capture_output=True, text=True)
    assert piped.returncode == 0 and pk(piped.stdout) == pk(whole.stdout)
    # and it equals the oracle
    exp = orc.rx_stream(iq.numpy(), channel=38)
    assert len(pk(whole.stdout)) == len(exp)


@pytest.mark.gpu
def test_cli_live_pipe_sigint_like_the_front_end(tmp_path):
    """What the reference's btle_cli does to its sniffer (rx_proc.py:64-81 argv, :101-117 SIGINT stop, :119-137 line
    stream): long options --json --quiet-text --rssi-est, NDJSON lines as packets arrive on a live stream, SIGINT ends the
    run with a 'stop' status and exit code 0."""
    import json
    import signal
    import time
    iq, _ = synth.make_adv_stream(64 * 16384, seed=41, channel=37, slot_samples=3000)
    raw = iq.numpy().tobytes()
    p = subprocess.Popen([CLI, "-c", "37", "-g", "24", "-l", "32", "--rssi-est", "--json", "--quiet-text", "-i", "-", "--segment-chunks", "8"],
                         stdin=subprocess.PIPE, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    half = 40 * 16384
    p.stdin.write(raw[:half])
    p.stdin.flush()
    lines = []
    t0 = time.time()
    while time.time() - t0 < 60:                         # packets of the completed segments arrive while the pipe is still open
        line = p.stdout.readline().decode()
        if line.startswith("{"):
            lines.append(json.loads(line))
        if sum(e["t"] == "pkt" for e in lines) >= 20:
            break
    assert sum(e["t"] == "pkt" for e in lines) >= 20 and lines[0]["t"] == "status" and lines[0]["event"] == "start"
    p.send_signal(signal.SIGINT)                         # rx_proc.py:107-117
    try:
        p.stdin.close()
    except BrokenPipeError:
        pass
    out = p.stdout.read().decode()
    assert p.wait(timeout=30) == 0
    rest = [json.loads(l) for l in out.splitlines() if l.startswith("{")]
    assert rest and rest[-1]["t"] == "status" and rest[-1]["event"] == "stop"
