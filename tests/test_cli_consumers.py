"""What `btle_rx_b200 -j -R -s file.pcap` printed and wrote on a B200 for two small captures (committed under
tests/golden/ by tools/make_cli_fixture.py), fed to the consumers on the other side of the process boundary:
structural checks, and what the reference's OWN front-end code (host/python/btle_cli: events.parse_line,
pcap_loader.load, aggregate.ScanAggregator, rx_proc.RxOptions — SURVEY.md §8b seam 2) made of them, as recorded in
tests/golden/cli_consumers.json by oracle/gen_golden_cli_consumers.py."""
import hashlib
import json
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
CASES = [("adv", 37, 0x8E89BED6), ("data", 9, 0x60850A1B)]


def _lines(name):
    return open(os.path.join(GOLD, f"cli_fixture_{name}.out")).read().splitlines()


def _pcap_bodies(name):
    b = open(os.path.join(GOLD, f"cli_fixture_{name}.pcap"), "rb").read()
    assert b[:24] == bytes.fromhex("a1b2c3d4000200040000000000000000000005dc00000100")      # btle_rx.c:110
    out, off = [], 24
    while off < len(b):
        caplen = int.from_bytes(b[off + 8:off + 12], "big")
        out.append(b[off + 16:off + 16 + caplen])
        off += 16 + caplen
    return out


@pytest.mark.parametrize("name,ch,aa", CASES)
def test_fixture_is_self_consistent(name, ch, aa):
    ev = [json.loads(l) for l in _lines(name) if l.startswith("{")]
    assert ev[0]["t"] == "status" and ev[0]["event"] == "start" and ev[-1]["event"] == "stop"      # btle_rx.c:2588, :2669
    pk = [e for e in ev if e["t"] == "pkt"]
    assert len(pk) >= 8 and [e["pkt"] for e in pk] == sorted(e["pkt"] for e in pk)
    assert all(e["ch"] == ch and e["aa"] == f"{aa:08x}" and e["v"] == 1 for e in pk)
    assert any(not e["crc_ok"] for e in pk) and any(e["crc_ok"] for e in pk)
    bodies = _pcap_bodies(name)
    assert len(bodies) == len(pk)                                     # every printed packet is stored, :2361-2362
    for e, body in zip(pk, bodies):
        assert body[0] == ch and int.from_bytes(body[10:14], "little") == aa                   # phdr + AA, :184-207
        pdu = body[14:]
        assert pdu[2:2 + e["plen"]].hex() == e["payload_hex"] if "payload_hex" in e else True


def _front_end():
    return json.load(open(os.path.join(GOLD, "cli_consumers.json")))


@pytest.mark.parametrize("name,ch,aa", CASES)
def test_reference_front_end_consumes_our_output(name, ch, aa):
    g = _front_end()["fixtures"][name]
    for f, digest in g["sha256"].items():          # the fixture the front-end was run on
        assert hashlib.sha256(open(os.path.join(GOLD, f), "rb").read()).hexdigest() == digest, \
            f"{f} changed: re-run oracle/gen_golden_cli_consumers.py"
    lines = _lines(name)
    kinds = g["line_kinds"]
    # text lines are tolerated (rx_proc.py:125-137), every JSON line is a valid v1 event
    assert len(kinds) == len(lines) and all((k is None) == (not l.startswith("{")) for k, l in zip(kinds, lines))
    ev = [k for k in kinds if k is not None]
    assert ev[0] == "StatusEvent" and ev[-1] == "StatusEvent"
    pk = g["pkt"]
    assert len(pk) == ev.count("PktEvent") == sum('"t":"pkt"' in l for l in lines)
    ours = [json.loads(l) for l in lines if '"t":"pkt"' in l]
    assert g["pcap_linktype"] == g["dlt_bluetooth_le_ll_with_phdr"] and len(g["pcap"]) == len(pk)
    for e, p, o in zip(pk, g["pcap"], ours):
        assert p["channel"] == ch == e["ch"] == o["ch"] and p["access_addr"] == aa
        assert p["pdu_header"][3] == e["plen"] == o["plen"]
        if name == "adv" and e["adv_a"] is not None:
            assert p["adv_a"] == e["adv_a"]                                # same AdvA from the pcap bytes and from the NDJSON
        if e["rssi_est"] is not None:
            assert p["rssi_dbm"] == e["rssi_est"]
    if name == "adv":
        snap = g["scan_pkt_counts"]
        assert len(snap) >= 4 and sum(snap) <= len(pk)


def test_reference_rxprocess_spawns_our_binary():
    """The reference's own process wrapper (btle_cli.rx_proc.RxProcess: $BTLE_RX lookup rx_proc.py:31-33, argv :64-81,
    line stream :119-137, stop :101-117) drives btle_rx_b200 with the argv its RxOptions built (recorded).  In a GPU-less
    container the program reports the reference's "board failure" (exit code 1, btle_rx.c:2586) after the start / stop
    status events; on a B200 the same argv streams packets (tests/test_cli.py::test_cli_live_pipe_sigint_like_the_front_end)."""
    root = os.path.dirname(HERE)
    exe = os.path.join(root, "btle_b200", "btle_rx_b200")
    if not os.path.exists(exe):
        import __graft_entry__ as ge
        ge.build()
    argv = _front_end()["rx_argv"]
    assert argv[:7] == ["<exe>", "-c", "38", "-g", "24", "-l", "32"] and "--json" in argv and "-o" in argv
    repl = {"<exe>": exe, "<input>": os.path.join(GOLD, "cli_fixture_adv.out")}     # any readable file: there is no GPU to decode it
    p = subprocess.run([repl.get(a, a) for a in argv], capture_output=True, text=True, timeout=120)
    lines = p.stdout.splitlines()
    ev = [json.loads(l) for l in lines if l.startswith("{")]
    banner = [l for l in lines if l and not l.startswith("{")]
    import torch
    if not torch.cuda.is_available():
        assert p.returncode == 1 and any("btle_b200_create" in b for b in banner)
    assert ev and ev[0]["t"] == "status" and ev[0].get("event") == "start"
