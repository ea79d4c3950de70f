"""Wideband channelizer measurement (DESIGN.md §6.5): 1 s of one int8 capture of the band -> 4 Msps captures of every
channel -> the receiver, on one GPU.  Prints a markdown report (profiles/wideband_r01.md holds one).

The input is a synth.wideband_from_channels segment with packets on every channel, tiled to 1 s (larger than L2, so the
timed passes read HBM).  Timed with CUDA events after warm-up:
  channelize   btle_b200_channelize_device alone;
  receiver     btle_b200_rx_device on its output;
  end to end   btle_b200_rx_wideband from page-locked host memory (copy, channelize, receive, records back).
The IDP-pipe bound is 2*T*n_ch*M lane-ops at 148 SMs x 64 lanes/clk (2 IDP warp-instructions/clk/SM, DESIGN.md §4.1) at
the SM clock nvidia-smi reports while the timed channelizer loop runs."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from btle_b200 import BtleRx, make_cfgs, synth  # noqa: E402
from btle_b200.rx import band_channels, wideband_taps  # noqa: E402

SHAPES = [(20, 2441), (5, 2426), (25, 2441)]     # 80 Msps / 40 channels (the target), 20 Msps / 9, 100 Msps / 40


def smi(fields):
    p = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), f"--query-gpu={fields}", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    return [x.strip() for x in p.stdout.strip().split(",")] if p.returncode == 0 else ["?"] * len(fields.split(","))


def segment(channels, decim, center_mhz, m_seg, seed):
    """Per-channel captures with packets (advertising PDUs on 37..39, LL data PDUs elsewhere) -> one wideband segment."""
    caps = torch.empty((len(channels), 2 * m_seg), dtype=torch.int8, device="cuda")
    for i, ch in enumerate(channels):
        iq, _ = synth.make_adv_stream(2 * m_seg, seed=seed + ch, channel=ch, slot_samples=4096, amplitude=20, corrupt_every=7,
                                      device="cuda", data_channel_pdu=ch < 37)
        caps[i] = iq
    return synth.wideband_from_channels(caps, channels, decim, center_mhz, noise=1.0, seed=seed, device="cuda")


def events_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def run_shape(rx, decim, center_mhz, seconds, reps):
    channels = band_channels(decim, center_mhz)
    n_ch, fs = len(channels), 4e6 * decim
    n = int(seconds * fs)
    seg = segment(channels, decim, center_mhz, 8 * 8192, seed=1)
    d_wide = seg.repeat((2 * n + seg.numel() - 1) // seg.numel())[:2 * n].contiguous()
    m = (n + decim - 1) // decim
    stride = (2 * m + 15) // 16 * 16
    d_out = torch.empty((n_ch, stride), dtype=torch.int8, device="cuda")
    cfgs = make_cfgs(n_ch, channel=channels)
    cap = n_ch * (2 * m // 16384) * 34 + 16
    d_recs = torch.empty(cap * 64, dtype=torch.uint8, device="cuda")
    d_count = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def chan():
        rx.channelize_device(d_wide, decim, center_mhz, channels, d_out, stream_ptr=stream)

    def recv():
        rx.rx_device(d_out[:, :2 * m], cfgs, d_recs, d_count, stream_ptr=stream)

    for _ in range(3):
        chan(); recv()
    torch.cuda.synchronize()
    # channelizer: the clock is read while the timed loop is on the GPU
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        chan()
    b.record()
    sm_mhz = smi("clocks.sm")[0]
    b.synchronize()
    t_chan = a.elapsed_time(b) / reps
    t_recv = events_ms(recv, reps)
    n_pkts = int(d_count.item())
    # end to end from page-locked host memory
    h_wide = torch.empty(2 * n, dtype=torch.int8, pin_memory=True)
    h_wide.copy_(d_wide)
    rx.rx_wideband(h_wide, decim, center_mhz, cfgs)
    t0 = time.perf_counter()
    for _ in range(max(1, reps // 4)):
        recs = rx.rx_wideband(h_wide, decim, center_mhz, cfgs)
    t_e2e = (time.perf_counter() - t0) * 1e3 / max(1, reps // 4)
    d_tmp = torch.empty_like(d_wide)
    t_h2d = events_ms(lambda: d_tmp.copy_(h_wide, non_blocking=True), max(1, reps // 4))
    t_taps = len(wideband_taps(decim, center_mhz, channels[0])[0])
    ops = 2.0 * t_taps * n_ch * m
    try:
        clk = float(sm_mhz) * 1e6
        bound_ms = ops / (148 * 64 * clk) * 1e3
        share = f"{bound_ms / t_chan:.3f} (bound {bound_ms:.2f} ms at {sm_mhz} MHz)"
    except ValueError:
        share = "not measured (no SM clock reading)"
    return {
        "shape": f"{fs / 1e6:.0f} Msps, D = {decim}, fc = {center_mhz} MHz, {n_ch} channels, T = {t_taps}, {seconds:g} s = {2 * n / 1e6:.0f} MB",
        "rows": [
            ("channelize_device", f"{t_chan:.3f} ms", f"{n / t_chan / 1e6:.2f} G wideband samples/s, real-time x{seconds * 1e3 / t_chan:.1f}"),
            ("IDP-pipe share", share, f"{ops / 1e9:.1f} G lane-ops"),
            ("receiver on its output", f"{t_recv:.3f} ms", f"{n_ch} x {2 * m / 1e6:.1f} MB, {n_pkts} packets"),
            ("rx_wideband end to end (page-locked)", f"{t_e2e:.3f} ms", f"real-time x{seconds * 1e3 / t_e2e:.1f}, {len(recs)} packets"),
            ("  of which H2D copy", f"{t_h2d:.3f} ms", f"PCIe share {t_h2d / t_e2e:.2f}, {2 * n / t_h2d / 1e6:.1f} GB/s"),
        ],
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the wideband measurement needs a CUDA device"
    name, plimit, maxclk = smi("name,power.limit,clocks.max.sm")
    rx = BtleRx(0)
    print(f"# Wideband channelizer (tools/wideband_bench.py)\n\nCard: {name}, power limit {plimit} W, max SM clock {maxclk} MHz.  "
          f"CUDA events, mean of {args.reps} after 3 warm-up passes; input tiled from a packet segment, larger than L2.\n")
    for decim, fc in SHAPES:
        r = run_shape(rx, decim, fc, args.seconds, args.reps)
        print(f"## {r['shape']}\n\n| step | time | |\n|---|---|---|")
        for row in r["rows"]:
            print("| " + " | ".join(row) + " |")
        print()
        torch.cuda.empty_cache()
    rx.close()


if __name__ == "__main__":
    main()
