#!/usr/bin/env python
"""Runs the reference's OWN front-end code (host/python/btle_cli: events.parse_line, pcap_loader.load,
aggregate.ScanAggregator, rx_proc.RxOptions) over what btle_rx_b200 prints and writes — the committed CLI fixtures
(tests/golden/cli_fixture_*) and the NDJSON hop lines of tests/test_hop.py's capture — and writes what it made of them
to tests/golden/cli_consumers.json (committed; read by tests/test_cli_consumers.py and tests/test_hop.py).

    BTLE_REFERENCE=<reference checkout> python oracle/gen_golden_cli_consumers.py
"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REF = os.environ["BTLE_REFERENCE"]          # a checkout of the reference project


def main():
    sys.dont_write_bytecode = True
    sys.path.insert(0, os.path.join(REF, "host", "python", "btle_cli", "src"))
    from btle_cli.aggregate import ScanAggregator
    from btle_cli.events import PktEvent, parse_line
    from btle_cli.pcap_loader import DLT_BLUETOOTH_LE_LL_WITH_PHDR, load
    from btle_cli.rx_proc import RxOptions
    out = {"fixtures": {}}
    for name in ("adv", "data"):
        out_path, pcap_path = (os.path.join(GOLD, f"cli_fixture_{name}.{ext}") for ext in ("out", "pcap"))
        parsed = [parse_line(l) for l in open(out_path).read().splitlines()]
        pk = [e for e in parsed if isinstance(e, PktEvent)]
        cap = load(pcap_path)
        d = {"sha256": {os.path.basename(p): hashlib.sha256(open(p, "rb").read()).hexdigest() for p in (out_path, pcap_path)},
             "line_kinds": [type(e).__name__ if e is not None else None for e in parsed],
             "pkt": [{"ch": e.ch, "plen": e.plen, "adv_a": e.adv_a, "rssi_est": e.rssi_est} for e in pk],
             "pcap_linktype": cap.linktype, "dlt_bluetooth_le_ll_with_phdr": DLT_BLUETOOTH_LE_LL_WITH_PHDR,
             "pcap": [{"channel": p.channel, "access_addr": p.access_addr, "pdu_header": list(p.pdu_header), "adv_a": p.adv_a,
                       "rssi_dbm": p.rssi_dbm} for p in cap.packets]}
        if name == "adv":
            agg = ScanAggregator()
            for e in pk:
                agg.update(e)
            d["scan_pkt_counts"] = [r.pkt_count for r in agg.snapshot()]
        out["fixtures"][name] = d
    out["rx_argv"] = RxOptions(channel=38, hop=True, filter_pdu_type="0,5", filter_adva="AA:BB:CC:DD:EE:FF",
                               extra_args=["-i", "<input>"]).to_argv("<exe>")
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_hop as T
    from btle_b200.hop import follow_connections, hop_events_ndjson
    cap, _, _ = T._capture_with_connection()
    _, conns = follow_connections(T.OracleRx(), cap)
    out["hop_lines"] = {l: type(parse_line(l)).__name__ for l in hop_events_ndjson(conns).splitlines()}
    with open(os.path.join(GOLD, "cli_consumers.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
