"""Synthetic BLE 1M-PHY packet / IQ-stream generator (input data for tests and bench).

This is plumbing around the receive hot path: it produces int8 IQ at 4 samples per
symbol that the receiver must decode.  The integer GFSK modulator follows the
behaviour of the reference transmitter's `gen_sample_from_phy_bit`
(/root/reference/host/btle-tools/src/btle_tx.c:1022-1063): +-1 impulses every 4th
sample, 9 integer Gaussian taps {2,11,32,53,60,53,32,11,2} (sum 256 = a quarter turn of
the 1024-step phase wheel per symbol, i.e. modulation index 0.5), phase accumulated
modulo 1024 and mapped through round(127*cos/sin(2*pi*k/1024))
(gauss_cos_sin_table.h; the waveform is checked sample for sample against the reference
transmitter's own output in tests/test_tx_modulator_gpu.py and tests/test_oracle_golden.py).  CRC-24 and whitening follow
btle_tx.c:1441-1530 / the BLE Core spec.  Written from the behaviour, vectorised over
whole batches of packets with torch integer ops so the same code runs on CPU and CUDA.
"""
from __future__ import annotations

import numpy as np
import torch

GAUSS_TAPS = (2, 11, 32, 53, 60, 53, 32, 11, 2)
SPS = 4
ADV_ACCESS_ADDR = 0x8E89BED6
ADV_CRC_INIT = 0x555555


def _phase_tables(device=None):
    k = np.arange(1024)
    c = np.round(127.0 * np.cos(2 * np.pi * k / 1024)).astype(np.int8)
    s = np.round(127.0 * np.sin(2 * np.pi * k / 1024)).astype(np.int8)
    return torch.from_numpy(c).to(device), torch.from_numpy(s).to(device)


def whitening_table() -> np.ndarray:
    """uint8 [40, 42]: per-channel whitening bytes (LFSR x^7+x^4+1, seed 1|channel)."""
    tab = np.zeros((40, 42), dtype=np.uint8)
    for ch in range(40):
        reg = [1] + [(ch >> (5 - i)) & 1 for i in range(6)]
        for byte in range(42):
            v = 0
            for bit in range(8):
                o = reg[6]
                v |= o << bit
                n4 = reg[3] ^ reg[6]
                reg = [o, reg[0], reg[1], reg[2], n4, reg[4], reg[5]]
            tab[ch, byte] = v
    return tab


_WHITEN = whitening_table()


def crc_init_reorder(crc_init: int) -> int:
    """Bit-reverse each of the three bytes (btle_rx.c:1969-1993)."""
    out = 0
    for b in range(3):
        v = (crc_init >> (8 * b)) & 0xFF
        out |= int(f"{v:08b}"[::-1], 2) << (8 * b)
    return out


def crc24(data: bytes, crc_init: int = ADV_CRC_INIT) -> int:
    """Reflected CRC-24 (poly 0xDA6000) over `data`, register seeded with reorder(crc_init)."""
    crc = crc_init_reorder(crc_init)
    for b in data:
        for j in range(8):
            fb = (crc ^ (b >> j)) & 1
            crc >>= 1
            if fb:
                crc ^= 0xDA6000
    return crc


def adv_pdu(pdu_type: int, tx_add: int, rx_add: int, payload: bytes) -> bytes:
    assert 0 <= len(payload) <= 63
    return bytes([(pdu_type & 0xF) | ((tx_add & 1) << 6) | ((rx_add & 1) << 7), len(payload)]) + bytes(payload)


def ll_data_pdu(llid: int, nesn: int, sn: int, md: int, payload: bytes) -> bytes:
    assert 0 <= len(payload) <= 31
    return bytes([(llid & 3) | ((nesn & 1) << 2) | ((sn & 1) << 3) | ((md & 1) << 4), len(payload)]) + bytes(payload)


def air_bytes(pdu: bytes, channel: int, access_addr: int = ADV_ACCESS_ADDR, crc_init: int = ADV_CRC_INIT,
              corrupt_bit: int | None = None) -> bytes:
    """preamble + access address + whitened(PDU + CRC), in transmission order."""
    crc = crc24(pdu, crc_init)
    body = bytearray(pdu + bytes([crc & 0xFF, (crc >> 8) & 0xFF, (crc >> 16) & 0xFF]))
    if corrupt_bit is not None:
        body[corrupt_bit // 8] ^= 1 << (corrupt_bit % 8)
    w = _WHITEN[channel]
    body = bytes(b ^ int(w[i]) for i, b in enumerate(body))
    preamble = 0x55 if (access_addr & 1) else 0xAA
    return bytes([preamble]) + int(access_addr).to_bytes(4, "little") + body


def modulate_batch(air: torch.Tensor, n_bytes: torch.Tensor) -> torch.Tensor:
    """Integer GFSK modulation of a batch of packets.

    air: uint8 [B, Lmax] air bytes (zero padded); n_bytes: int [B] valid lengths.
    Returns int8 [B, 2*(8*Lmax*4+16)] interleaved IQ; samples after each packet's own
    8*n*4+16 samples are zero."""
    dev = air.device
    B, L = air.shape
    nbit = 8 * L
    shifts = torch.arange(8, device=dev, dtype=torch.int32)
    bits = ((air.to(torch.int32).unsqueeze(-1) >> shifts) & 1).reshape(B, nbit)       # LSB first
    valid_bits = (torch.arange(nbit, device=dev).unsqueeze(0) < (8 * n_bytes.to(dev)).unsqueeze(1))
    imp = torch.where(valid_bits, 2 * bits - 1, torch.zeros_like(bits))               # +-1 / 0
    nsamp = nbit * SPS + 16
    # impulse train: symbol k sits at over-sampled index 15 + 4k (btle_tx.c:1030-1041)
    os_len = nsamp + 32
    os_ = torch.zeros((B, os_len), dtype=torch.int32, device=dev)
    os_[:, 15:15 + nbit * SPS:SPS] = imp
    # acc_i = sum_{j=3..11} g[15-j] * os[i+j]  (btle_tx.c:1052-1056); taps are symmetric
    acc = torch.zeros((B, nsamp - 1), dtype=torch.int32, device=dev)
    for t, g in enumerate(GAUSS_TAPS):
        j = 3 + t
        acc += g * os_[:, j:j + nsamp - 1]
    phase = torch.cumsum(acc, dim=1) & 1023
    phase = torch.cat([torch.zeros((B, 1), dtype=phase.dtype, device=dev), phase], dim=1)
    cos_t, sin_t = _phase_tables(dev)
    i = cos_t[phase.long()]
    q = sin_t[phase.long()]
    valid_s = (torch.arange(nsamp, device=dev).unsqueeze(0) < (8 * n_bytes.to(dev) * SPS + 16).unsqueeze(1))
    i = torch.where(valid_s, i, torch.zeros_like(i))
    q = torch.where(valid_s, q, torch.zeros_like(q))
    return torch.stack([i, q], dim=-1).reshape(B, 2 * nsamp)


def modulate(air: bytes) -> np.ndarray:
    """int8 interleaved IQ for one packet (8*len*4+16 samples)."""
    t = torch.tensor(list(air), dtype=torch.uint8).unsqueeze(0)
    return modulate_batch(t, torch.tensor([len(air)])).squeeze(0).numpy().copy()


def noise_floor(n_int8: int, gen: torch.Generator, device=None) -> torch.Tensor:
    """Integer background noise like the off-packet floor of the reference capture
    (matlab/sample_iq_4msps.txt: std ~0.8 LSB, mean ~-0.3, range -7..6; SURVEY.md §8d C2)."""
    x = torch.randn(n_int8, generator=gen, device=device, dtype=torch.float32) * 0.8 - 0.3
    return torch.clamp(torch.round(x), -7, 6).to(torch.int8)


def make_adv_stream(n_int8: int, seed: int, channel: int = 37, slot_samples: int = 4096, amplitude: int = 64,
                    corrupt_every: int = 100, device=None, access_addr: int = ADV_ACCESS_ADDR,
                    crc_init: int = ADV_CRC_INIT, data_channel_pdu: bool = False, batch: int = 8192,
                    use_cuda_modulator: bool = True, straddle_every: int = 0):
    """Noise floor + one burst per `slot_samples` slot at a random sample offset
    (SURVEY.md §8d C2/C3).  ADV_IND (TxAdd=1, AdvA = counter, AdvData random 0..31 B) on
    advertising channels, LL data PDUs (len 0..27) when data_channel_pdu.  Every
    `corrupt_every`-th burst gets one flipped payload bit (CRC must fail).  Every
    `straddle_every`-th burst (when its slot allows it) is placed ACROSS the next 8192-sample chunk
    boundary of the reference's ring (btle_rx.c:2619-2651) at a random cut point, so that its decode
    needs the look-ahead behind the chunk (SURVEY.md §8d C2: "1 % straddle a chunk boundary by
    construction"); truth["straddle"] marks them.
    Returns (iq int8 tensor [n_int8] on `device`, truth dict of numpy arrays)."""
    dev = torch.device(device) if device is not None else torch.device("cpu")
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    iq = noise_floor(n_int8, gen, dev)
    n_samples = n_int8 // 2
    n_slots = n_samples // slot_samples
    rng = np.random.default_rng(seed + 1)
    Lmax = 1 + 4 + 2 + 37 + 3
    burst_samples = 8 * Lmax * SPS + 16
    starts = np.zeros(n_slots, dtype=np.int64)
    pdus, corrupt = [], np.zeros(n_slots, dtype=bool)
    straddle = np.zeros(n_slots, dtype=bool)
    prev_end = 0                                            # first sample behind the previous burst
    air = np.zeros((n_slots, Lmax), dtype=np.uint8)
    nby = np.zeros(n_slots, dtype=np.int64)
    for s in range(n_slots):
        if data_channel_pdu:
            plen = int(rng.integers(0, 28))
            pdu = ll_data_pdu(int(rng.integers(1, 3)), s & 1, (s >> 1) & 1, 0, rng.integers(0, 256, plen, dtype=np.uint8).tobytes())
        else:
            dlen = int(rng.integers(0, 32))
            adva = int(s).to_bytes(6, "little")
            pdu = adv_pdu(0, 1, 0, adva + rng.integers(0, 256, dlen, dtype=np.uint8).tobytes())
        cb = None
        if corrupt_every and s % corrupt_every == corrupt_every - 1:
            cb = int(rng.integers(16, 8 * len(pdu))) if len(pdu) > 2 else 8 * len(pdu) + 3
            corrupt[s] = True
        a = air_bytes(pdu, channel, access_addr, crc_init, cb)
        air[s, :len(a)] = np.frombuffer(a, dtype=np.uint8)
        nby[s] = len(a)
        n_s = 8 * len(a) * SPS + 16
        lo = max(s * slot_samples, prev_end + 32)           # keep clear of a burst that spilled over from the slot before
        hi = max(lo + 1, (s + 1) * slot_samples - n_s)
        starts[s] = int(rng.integers(lo, hi))
        if straddle_every and s % straddle_every == straddle_every - 1:
            edge = (lo // 8192 + 1) * 8192                  # next chunk boundary behind the earliest start
            first = max(lo, edge - n_s + 1)
            if first < edge and edge + n_s < n_samples and edge <= (s + 1) * slot_samples:
                starts[s] = int(rng.integers(first, edge))  # edge falls strictly inside the burst
                straddle[s] = True
        prev_end = int(starts[s]) + n_s
        pdus.append(pdu)
    for b0 in range(0, n_slots, batch):
        b1 = min(n_slots, b0 + batch)
        if dev.type == "cuda" and use_cuda_modulator:
            wav = modulate_batch_cuda(torch.from_numpy(air[b0:b1]).to(dev).contiguous(), torch.from_numpy(nby[b0:b1]).to(dev))
        else:
            wav = modulate_batch(torch.from_numpy(air[b0:b1]).to(dev), torch.from_numpy(nby[b0:b1]).to(dev))
        wav = (wav.to(torch.int32) * amplitude) // 127
        idx = (2 * torch.from_numpy(starts[b0:b1]).to(dev)).unsqueeze(1) + torch.arange(2 * burst_samples, device=dev).unsqueeze(0)
        # only the burst's own samples are written: the zero padding of a short burst may overlap
        # the next burst's slot, and duplicate indices in one scatter would race on CUDA
        own = torch.arange(2 * burst_samples, device=dev).unsqueeze(0) < (2 * (8 * torch.from_numpy(nby[b0:b1]).to(dev) * SPS + 16)).unsqueeze(1)
        ok = (idx < n_int8) & own
        idx = torch.where(ok, idx, torch.zeros_like(idx))
        cur = iq[idx.reshape(-1)].to(torch.int32).reshape(idx.shape)
        new = torch.clamp(cur + wav, -128, 127).to(torch.int8)
        iq[idx[ok]] = new[ok]
    truth = {"start_sample": starts, "n_air_bytes": nby, "corrupt": corrupt, "pdus": pdus, "straddle": straddle}
    return iq, truth


def make_pdu_stream(pdus, channel: int, access_addr: int = ADV_ACCESS_ADDR, crc_init: int = ADV_CRC_INIT, seed: int = 0,
                    slot_samples: int = 2048, amplitude: int = 64, corrupt=()):
    """Noise floor + the given PDUs (bytes), one per slot, at pseudo-random offsets.  PDUs whose
    index is in `corrupt` get one flipped payload/CRC bit.  Returns int8 numpy array."""
    n_slots = len(pdus) + 1
    n_int8 = ((2 * n_slots * slot_samples + 16383) // 16384 + 1) * 16384
    gen = torch.Generator()
    gen.manual_seed(seed)
    iq = noise_floor(n_int8, gen).numpy().copy()
    rng = np.random.default_rng(seed + 1)
    for s, pdu in enumerate(pdus):
        cb = (8 * len(pdu) + 5) if s in corrupt else None
        wav = modulate(air_bytes(bytes(pdu), channel, access_addr, crc_init, cb)).astype(np.int32) * amplitude // 127
        start = s * slot_samples + int(rng.integers(0, max(1, slot_samples - wav.size // 2 - 8)))
        seg = iq[2 * start:2 * start + wav.size].astype(np.int32) + wav
        iq[2 * start:2 * start + wav.size] = np.clip(seg, -128, 127).astype(np.int8)
    return iq


# ---- 8 samples/symbol modulator of the reference's Python model (input generator of the BER sweep) ----
GAUSS_TAPS_8SPS = (0, 0, 0, 1, 4, 9, 15, 22, 24, 22, 15, 9, 4, 1, 0, 0, 0)   # btlelib.py:146-160 (int8, x128)


def modulate_batch_8sps(phy_bits: torch.Tensor):
    """phy_bits: int8/uint8 [B, n] of 0/1 (preamble + AA + whitened PDU+CRC).  Returns (i, q) int8
    [B, 8n+16], the behaviour of btlelib.gfsk_modulation_fixed_point (btlelib.py:146-189): NRZ at
    8 samples/symbol preceded by 17 samples of -1, 17-tap integer Gaussian FIR, >>1, phase
    accumulated modulo 2048, round(127 cos/sin) lookup.  Equality with the reference's waveform
    is asserted against golden vectors in tests."""
    dev = phy_bits.device
    B, n = phy_bits.shape
    L = len(GAUSS_TAPS_8SPS)
    nrz = (phy_bits.to(torch.int32) * 2 - 1).repeat_interleave(8, dim=1)
    x = torch.cat([-torch.ones((B, L), dtype=torch.int32, device=dev), nrz,
                   torch.zeros((B, L - 1), dtype=torch.int32, device=dev)], dim=1)     # zero tail of the full convolution
    m = 8 * n + L - 1                                       # outputs kept: full-conv indices L .. L+m-1
    y = torch.zeros((B, m), dtype=torch.int32, device=dev)
    for j, g in enumerate(GAUSS_TAPS_8SPS):
        if g:
            y += g * x[:, L - j:L - j + m]
    v = y >> 1
    phase = torch.cumsum(v, dim=1) & 2047
    k = torch.arange(2048, device=dev, dtype=torch.float64)
    cos_t = torch.round(127 * torch.cos(2 * torch.pi * k / 2048)).to(torch.int8)
    sin_t = torch.round(127 * torch.sin(2 * torch.pi * k / 2048)).to(torch.int8)
    return cos_t[phase.long()], sin_t[phase.long()]


# ---- the same two modulators as hand-written CUDA kernels (btle_b200_tx_modulate_device) ----------
_tx_ctx = None


def modulate_batch_cuda(air: torch.Tensor, n_bytes: torch.Tensor, sps: int = 4):
    """air uint8 [B, Lmax] on a CUDA device, n_bytes int [B].  sps=4 -> int8 [B, 2*(32*Lmax+16)]
    interleaved IQ (== modulate_batch); sps=8 -> (i, q) int8 [B, 64*Lmax+16] (== modulate_batch_8sps
    of the unpacked bits).  Runs tx_modulate_kernel through the C-ABI on the current stream."""
    import ctypes
    from .rx import BtleRx
    global _tx_ctx
    assert air.is_cuda and air.dtype == torch.uint8 and air.is_contiguous()
    if _tx_ctx is None or _tx_ctx.device != air.device.index:
        _tx_ctx = BtleRx(air.device.index)
    B, L = air.shape
    nb = n_bytes.to(device=air.device, dtype=torch.int32).contiguous()
    nsamp = 8 * L * sps + 16
    st = ctypes.c_void_p(torch.cuda.current_stream(air.device).cuda_stream)
    if sps == 4:
        out = torch.empty((B, 2 * nsamp), dtype=torch.int8, device=air.device)
        _tx_ctx._check(_tx_ctx._L.btle_b200_tx_modulate_device(_tx_ctx._h, air.data_ptr(), nb.data_ptr(), B, L, 4, out.data_ptr(), None, st))
        return out
    oi = torch.empty((B, nsamp), dtype=torch.int8, device=air.device)
    oq = torch.empty((B, nsamp), dtype=torch.int8, device=air.device)
    _tx_ctx._check(_tx_ctx._L.btle_b200_tx_modulate_device(_tx_ctx._h, air.data_ptr(), nb.data_ptr(), B, L, 8, oi.data_ptr(), oq.data_ptr(), st))
    return oi, oq


# ---- whole captures generated on the device (btle_b200_synth_streams_device) --------------------------
def synth_streams_device(cfgs: np.ndarray, n_int8: int, seed: int, device=None, slot_samples: int = 4096, amplitude: int = 64,
                         corrupt_every: int = 100, straddle_every: int = 100, noise: int = 0, want_truth: bool = True,
                         out: torch.Tensor | None = None):
    """len(cfgs) captures of n_int8 bytes each: noise floor + one burst per slot with the stream's channel / access
    address / CRC init (ADV_IND on 37..39, LL data PDUs elsewhere), generated by synth_noise_kernel +
    synth_bursts_kernel on the current CUDA stream.  Returns (iq int8 CUDA tensor [n_streams, n_int8] — a view of
    a 16-byte-pitched buffer —, truth: SYNTH_TRUTH_DTYPE array [n_streams * n_slots] or None)."""
    import ctypes
    from ._native import CFG_DTYPE, SYNTH_CFG_DTYPE, SYNTH_TRUTH_DTYPE
    from .rx import BtleRx
    global _tx_ctx
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if _tx_ctx is None or _tx_ctx.device != dev.index:
        _tx_ctx = BtleRx(dev.index)
    cfgs = np.ascontiguousarray(cfgs, dtype=CFG_DTYPE)
    ns = len(cfgs)
    pitch = (n_int8 + 15) // 16 * 16
    if out is None:
        out = torch.empty((ns, pitch), dtype=torch.int8, device=dev)
    assert out.shape[0] == ns and out.stride(1) == 1 and out.shape[1] >= n_int8
    sc = np.zeros(1, dtype=SYNTH_CFG_DTYPE)
    sc["seed"], sc["slot_samples"], sc["amplitude"] = seed, slot_samples, amplitude
    sc["corrupt_every"], sc["straddle_every"], sc["noise"] = corrupt_every, straddle_every, noise
    n_slots = (n_int8 // 2) // slot_samples
    d_truth = torch.empty((max(1, ns * n_slots), 64), dtype=torch.uint8, device=dev) if want_truth else None
    got = ctypes.c_size_t(0)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _tx_ctx._check(_tx_ctx._L.btle_b200_synth_streams_device(
        _tx_ctx._h, out.data_ptr(), ns, out.stride(0), n_int8, cfgs.ctypes.data, sc.ctypes.data,
        d_truth.data_ptr() if want_truth else None, ns * n_slots if want_truth else 0, ctypes.byref(got), st))
    truth = None
    if want_truth:
        truth = d_truth[: ns * n_slots].cpu().numpy().view(SYNTH_TRUTH_DTYPE).reshape(-1)
    return out[:, :n_int8], truth


def channel_plan(n_streams: int, rssi: int = 0) -> np.ndarray:
    """btle_stream_cfg array of SURVEY.md §8d C3/C5: stream k on BLE channel k mod 40; advertising parameters on
    37..39, data channels with access address 0x60850A1B + ch and CRC init 0xA77B22 ^ ch."""
    from .rx import make_cfgs
    c = make_cfgs(n_streams, rssi=rssi)
    ch = np.arange(n_streams) % 40
    adv = ch >= 37
    c["channel"] = ch
    c["access_addr"] = np.where(adv, ADV_ACCESS_ADDR, 0x60850A1B + ch).astype(np.uint32)
    c["crc_init"] = np.where(adv, ADV_CRC_INIT, 0xA77B22 ^ ch).astype(np.uint32)
    return c


def wideband_from_channels(caps, channels, decim: int, center_mhz: int, noise: float = 0.0, seed: int = 0, device=None):
    """One int8 interleaved I,Q capture at 4 MHz * decim centred on center_mhz that carries per-channel 4 Msps captures
    caps [n_ch, 2M] (int8, M a multiple of 4) on `channels`: each is band-limited to +-1 MHz in the FFT domain, placed at
    bin offset q*M/4 (q = f_ch - fc in MHz) of an N = M*decim point spectrum, so that wideband sample m*decim carries
    sample m of the channel; then the inverse FFT, seeded Gaussian noise of `noise` LSB per component, rounding and
    clipping.  Deliberately independent of the library's channelizer taps.  torch only; runs on `device` (CPU default).
    Returns an int8 tensor of 2N values."""
    from .hop import channel_freq_mhz
    dev = torch.device(device) if device is not None else torch.device("cpu")
    caps = torch.as_tensor(np.ascontiguousarray(caps, dtype=np.int8) if not torch.is_tensor(caps) else caps).to(dev)
    caps = caps.reshape(len(channels), -1)
    m = caps.shape[1] // 2
    assert m % 4 == 0, "channel captures must hold a multiple of 4 samples"
    n = m * decim
    spec = torch.zeros(n, dtype=torch.complex128, device=dev)
    k = torch.fft.fftfreq(m, d=1.0 / m, device=dev).round().to(torch.int64)          # signed bin index
    keep = k.abs() <= m // 4                                                          # |f| <= 1 MHz
    for i, ch in enumerate(channels):
        q = channel_freq_mhz(int(ch)) - int(center_mhz)
        assert abs(q) + 1 <= 2 * decim, f"channel {ch} is outside the band"
        x = caps[i].to(torch.float64).reshape(m, 2)
        xs = torch.fft.fft(torch.complex(x[:, 0], x[:, 1]))
        spec.index_add_(0, (k[keep] + q * m // 4) % n, xs[keep] * decim)
    w = torch.fft.ifft(spec)
    out = torch.stack([w.real, w.imag], dim=1)
    if noise:
        gen = torch.Generator(device=dev)
        gen.manual_seed(seed)
        out = out + noise * torch.randn(out.shape, generator=gen, device=dev, dtype=torch.float64)
    return torch.clamp(torch.round(out), -128, 127).to(torch.int8).reshape(-1)
