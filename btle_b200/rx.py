"""Python face of the receive path: thin object over the C-ABI context.

`BtleRx.rx()` / `rx_batch()` take host int8 IQ (numpy) and return packet records
(numpy structured array, `REC_DTYPE`) in the order the reference's receiver() emits them.
`rx_device()` works on CUDA tensors already resident in HBM (torch is only used for the
device memory and the stream)."""
from __future__ import annotations

import ctypes

import numpy as np

from . import _native
from ._native import BTLE_EINVAL, BTLE_EOVERFLOW, BtleError, CFG_DTYPE, DIR_DTYPE, REC_DTYPE, WIDEBAND_CFG_DTYPE

DEFAULT_ACCESS_ADDR = 0x8E89BED6     # btle_rx.c:231
DEFAULT_CRC_INIT = 0x555555          # btle_rx.c:232
DEFAULT_CHANNEL = 37                 # btle_rx.c:230


def make_cfgs(n_streams=1, channel=DEFAULT_CHANNEL, access_addr=DEFAULT_ACCESS_ADDR, access_mask=0xFFFFFFFF,
              crc_init=DEFAULT_CRC_INIT, raw=0, rssi=0) -> np.ndarray:
    """btle_stream_cfg array; every argument may be a scalar or a per-stream sequence."""
    c = np.zeros(n_streams, dtype=CFG_DTYPE)
    c["channel"], c["access_addr"], c["access_mask"] = channel, access_addr, access_mask
    c["crc_init"], c["raw"], c["rssi"] = crc_init, raw, rssi
    return c


def _wideband_cfg(decim: int, center_mhz: int, out_shift: int = -1) -> np.ndarray:
    c = np.zeros(1, dtype=WIDEBAND_CFG_DTYPE)
    c["decim"], c["center_mhz"], c["out_shift"] = decim, center_mhz, out_shift
    return c


def band_channels(decim: int, center_mhz: int) -> list:
    """The BLE channels inside a capture at 4 MHz * decim centred on center_mhz (|f_ch - fc| + 1 MHz <= fs / 2)."""
    from .hop import channel_freq_mhz
    return [ch for ch in range(40) if abs(channel_freq_mhz(ch) - int(center_mhz)) + 1 <= 2 * int(decim)]


def wideband_taps(decim: int, center_mhz: int, channel: int, out_shift: int = -1):
    """The channelizer's complex int16 taps of `channel` (btle_b200_wideband_taps): (int16 [T, 2] = Re, Im; output
    shift).  Host only: needs no GPU."""
    L = _native.load()
    cfg = _wideband_cfg(decim, center_mhz, out_shift)
    n, shift = ctypes.c_size_t(0), ctypes.c_int(0)
    rc = L.btle_b200_wideband_taps(cfg.ctypes.data, int(channel), None, 0, ctypes.byref(n), ctypes.byref(shift))
    if rc not in (0, BTLE_EOVERFLOW):
        raise BtleError(rc, f"no wideband taps for decim={decim}, center={center_mhz} MHz, channel={channel} "
                            "(decim must be 2..64, the channel 0..39 and inside the band)")
    taps = np.zeros((n.value, 2), dtype=np.int16)
    rc = L.btle_b200_wideband_taps(cfg.ctypes.data, int(channel), taps.ctypes.data, n.value, ctypes.byref(n), ctypes.byref(shift))
    if rc != 0:
        raise BtleError(rc, L.btle_b200_strerror(rc).decode())
    return taps, shift.value


class BtleRx:
    def __init__(self, device: int = 0):
        self._L = _native.load()
        h = ctypes.c_void_p()
        rc = self._L.btle_b200_create(ctypes.byref(h), int(device))
        if rc != 0:
            raise BtleError(rc, self._L.btle_b200_strerror(rc).decode())
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._L.btle_b200_destroy(self._h)
            self._h = None

    __del__ = close

    def _check(self, rc):
        if rc != 0:
            raise BtleError(rc, self._L.btle_b200_last_error(self._h).decode() or self._L.btle_b200_strerror(rc).decode())

    @property
    def last_launches(self) -> int:
        return self._L.btle_b200_last_launches(self._h)

    # ---- host buffers -------------------------------------------------------------------
    def rx_batch(self, iq: np.ndarray, cfgs: np.ndarray, cap: int | None = None) -> np.ndarray:
        """iq: int8 [n_streams, n_int8] (C-contiguous) or [n_int8]; cfgs: CFG_DTYPE [n_streams]."""
        iq = np.ascontiguousarray(iq, dtype=np.int8)
        if iq.ndim == 1:
            iq = iq[None, :]
        ns, n = iq.shape
        cfgs = np.ascontiguousarray(cfgs, dtype=CFG_DTYPE)
        assert cfgs.shape == (ns,)
        grow = cap is None                  # default capacity: typical worst case; grown once on BTLE_EOVERFLOW
        if cap is None:
            cap = ns * (n // 16384) * 34 + 16
        while True:
            out = np.empty(cap, dtype=REC_DTYPE)
            n_out = ctypes.c_size_t(0)
            rc = self._L.btle_b200_rx_batch(self._h, iq.ctypes.data, ns, n, n, cfgs.ctypes.data, out.ctypes.data, cap,
                                            ctypes.byref(n_out))
            if rc == BTLE_EOVERFLOW and grow:
                cap, grow = n_out.value, False
                continue
            self._check(rc)
            return out[:n_out.value]

    def rx(self, iq: np.ndarray, **cfg) -> np.ndarray:
        return self.rx_batch(np.asarray(iq).reshape(1, -1), make_cfgs(1, **cfg))

    def rx_iq16(self, iq16: np.ndarray, shift: int = 4, **cfg) -> np.ndarray:
        """int16 interleaved IQ (bladeRF SC16Q11: shift 4, btle_rx.c:307-308) -> records."""
        iq16 = np.ascontiguousarray(iq16, dtype=np.int16)
        cfgs = make_cfgs(1, **cfg)
        cap = (iq16.size // 16384) * 34 + 16
        for attempt in range(2):
            out = np.empty(cap, dtype=REC_DTYPE)
            n_out = ctypes.c_size_t(0)
            rc = self._L.btle_b200_rx_iq16(self._h, iq16.ctypes.data, iq16.size, shift, cfgs.ctypes.data, out.ctypes.data, cap,
                                           ctypes.byref(n_out))
            if rc == BTLE_EOVERFLOW and attempt == 0:
                cap = n_out.value
                continue
            self._check(rc)
            return out[:n_out.value]

    def rx_sps8(self, iq16: np.ndarray, channel=DEFAULT_CHANNEL, crc_init=DEFAULT_CRC_INIT, access_addr=DEFAULT_ACCESS_ADDR) -> np.ndarray:
        """Interleaved int16 I,Q at 8 samples per symbol (a `btle_ll -q` .bin capture) -> SPS8_REC_DTYPE array: the Python
        model's receiver (8 phases, first CRC-ok phase wins) on every packet the GPU finds in the capture."""
        from ._native import SPS8_REC_DTYPE
        iq16 = np.ascontiguousarray(iq16, dtype=np.int16).reshape(-1)
        n = iq16.size // 2
        cap = n // 576 + 16
        out = np.zeros(cap, dtype=SPS8_REC_DTYPE)
        n_out = ctypes.c_size_t(0)
        self._check(self._L.btle_b200_rx_sps8(self._h, iq16.ctypes.data, n, int(channel), int(crc_init), int(access_addr), out.ctypes.data, cap,
                                              ctypes.byref(n_out)))
        return out[:n_out.value]

    # ---- wideband captures (one capture of the band -> per-channel 4 Msps captures) --------------------------------
    def _wide_channels(self, decim, center_mhz, channels):
        if channels is None:
            channels = band_channels(decim, center_mhz)
            if len(channels) != 40:
                raise BtleError(BTLE_EINVAL, f"a capture at {4 * decim} Msps around {center_mhz} MHz does not hold all 40 channels; "
                                             "pass `channels`")
        return np.ascontiguousarray(channels, dtype=np.int32).reshape(-1)

    def channelize(self, wide: np.ndarray, decim: int, center_mhz: int, channels=None, out_shift: int = -1) -> np.ndarray:
        """wide: int8 interleaved I,Q at 4 MHz * decim -> int8 [n_ch, 2 * ceil(N / decim)]: the 4 Msps captures of
        `channels` (None = all 40, which the band must hold), e.g. for hop.follow_connections_windowed."""
        wide = np.ascontiguousarray(wide, dtype=np.int8).reshape(-1)
        ch = self._wide_channels(decim, center_mhz, channels)
        n = wide.size // 2
        width = 2 * ((n + decim - 1) // decim) if decim > 0 else 0
        stride = (width + 15) & ~15
        out = np.zeros((ch.size, max(stride, 16)), dtype=np.int8)
        cfg = _wideband_cfg(decim, center_mhz, out_shift)
        self._check(self._L.btle_b200_channelize(self._h, wide.ctypes.data, n, cfg.ctypes.data, ch.ctypes.data, ch.size,
                                                 out.ctypes.data, out.shape[1]))
        return np.ascontiguousarray(out[:, :width])

    def channelize_device(self, d_wide, decim: int, center_mhz: int, channels, d_out, out_shift: int = -1, stream_ptr: int = 0):
        """d_wide: torch int8 CUDA tensor (2N, interleaved I,Q); d_out: torch int8 CUDA tensor [n_ch, stride] (stride a
        multiple of 16, >= 2 * ceil(N / decim)).  Enqueued on `stream_ptr`, not synchronised."""
        ch = self._wide_channels(decim, center_mhz, channels)
        assert d_out.dim() == 2 and d_out.shape[0] == ch.size and d_out.stride(1) == 1
        cfg = _wideband_cfg(decim, center_mhz, out_shift)
        self._check(self._L.btle_b200_channelize_device(self._h, d_wide.data_ptr(), d_wide.numel() // 2, cfg.ctypes.data, ch.ctypes.data,
                                                        ch.size, d_out.data_ptr(), d_out.stride(0), ctypes.c_void_p(stream_ptr)))

    def rx_wideband(self, wide, decim: int, center_mhz: int, cfgs: np.ndarray, cap: int | None = None) -> np.ndarray:
        """Channelize `wide` (numpy int8, or a page-locked torch CPU tensor) and decode channel cfgs[i]["channel"] as
        stream i, in one receiver launch (btle_b200_rx_wideband)."""
        if hasattr(wide, "data_ptr"):
            assert wide.dtype.itemsize == 1 and wide.is_contiguous() and not wide.is_cuda
            ptr, n = wide.data_ptr(), wide.numel() // 2
        else:
            wide = np.ascontiguousarray(wide, dtype=np.int8).reshape(-1)
            ptr, n = wide.ctypes.data, wide.size // 2
        cfgs = np.ascontiguousarray(cfgs, dtype=CFG_DTYPE).reshape(-1)
        cfg = _wideband_cfg(decim, center_mhz)
        m = (n + decim - 1) // decim if decim > 0 else 0
        grow = cap is None
        if cap is None:
            cap = cfgs.size * (2 * m // 16384) * 34 + 16
        while True:
            out = np.empty(cap, dtype=REC_DTYPE)
            n_out = ctypes.c_size_t(0)
            rc = self._L.btle_b200_rx_wideband(self._h, ptr, n, cfg.ctypes.data, cfgs.ctypes.data, cfgs.size, out.ctypes.data, cap,
                                               ctypes.byref(n_out))
            if rc == BTLE_EOVERFLOW and grow:
                cap, grow = n_out.value, False
                continue
            if rc == BTLE_EOVERFLOW:
                raise BtleError(rc, f"{n_out.value} packets found, capacity {cap}")
            self._check(rc)
            return out[:n_out.value]

    # ---- unbounded capture, pushed in pieces (btle_b200_stream_*) -----------------------------
    def stream(self, segment_chunks: int = 0, **cfg) -> "RxStream":
        """Streaming session over one capture of any length: `with rx.stream(channel=37) as s: recs = s.push(iq_piece) ...;
        recs = s.finish()`.  Segments are double-buffered in page-locked memory; records come back in reference order,
        `chunk` counted from the start of the stream, as segments complete."""
        return RxStream(self, make_cfgs(1, **cfg), segment_chunks)

    # ---- device-resident ------------------------------------------------------------------
    def rx_device(self, d_iq, cfgs: np.ndarray, d_out, d_count, stream_ptr: int = 0):
        """d_iq: torch int8 CUDA tensor [n_streams, n_int8]; d_out: torch uint8 CUDA tensor
        [cap*64]; d_count: torch int32 CUDA tensor [1].  Enqueues on `stream_ptr` (no sync).  Records land in
        one block per unit of work (see include/btle_b200.h); sort_records() gives reference order."""
        ns, n = d_iq.shape
        cfgs = np.ascontiguousarray(cfgs, dtype=CFG_DTYPE)
        assert d_iq.stride(1) == 1 and cfgs.shape == (ns,)
        cap = d_out.numel() // 64
        rc = self._L.btle_b200_rx_device(self._h, d_iq.data_ptr(), ns, d_iq.stride(0), n, cfgs.ctypes.data,
                                         d_out.data_ptr(), cap, d_count.data_ptr(), ctypes.c_void_p(stream_ptr))
        self._check(rc)

    def units(self, n_streams: int, n_int8: int) -> int:
        """Number of unit-directory entries a launch over this shape writes (btle_b200_rx_units)."""
        return int(self._L.btle_b200_rx_units(self._h, n_streams, n_int8))

    def rx_device_dir(self, d_iq, cfgs: np.ndarray, d_out, d_count, d_dir, stream_ptr: int = 0):
        """Like rx_device, with the unit directory in the caller's buffer: d_dir is a torch CUDA tensor of at least
        units(...) * 8 bytes.  d_out / d_dir may be views of PEER memory (another GPU's buffer mapped here): the kernel
        then stores records and directory straight over NVLink.  Walking the directory (gather_ordered) yields the
        records in the reference's order.  d_count may be None (the packet count is the sum of the directory's counts):
        no memset is then enqueued in front of the kernel."""
        ns, n = d_iq.shape
        cfgs = np.ascontiguousarray(cfgs, dtype=CFG_DTYPE)
        assert d_iq.stride(1) == 1 and cfgs.shape == (ns,)
        cap = d_out.numel() * d_out.element_size() // 64
        dir_cap = d_dir.numel() * d_dir.element_size() // 8
        rc = self._L.btle_b200_rx_device_dir(self._h, d_iq.data_ptr(), ns, d_iq.stride(0), n, cfgs.ctypes.data, d_out.data_ptr(),
                                             cap, d_count.data_ptr() if d_count is not None else None, d_dir.data_ptr(), dir_cap,
                                             ctypes.c_void_p(stream_ptr))
        self._check(rc)

    def gather_ordered(self, recs: np.ndarray, unit_dir: np.ndarray) -> np.ndarray:
        """Host copies of a launch's record buffer and unit directory -> records in reference order."""
        recs = np.ascontiguousarray(recs, dtype=REC_DTYPE)
        unit_dir = np.ascontiguousarray(unit_dir, dtype=DIR_DTYPE)
        total = int(unit_dir["count"].sum())
        out = np.empty(total, dtype=REC_DTYPE)
        n_out = ctypes.c_size_t(0)
        rc = self._L.btle_b200_gather_ordered(recs.ctypes.data, recs.size, unit_dir.ctypes.data, unit_dir.size, out.ctypes.data,
                                              total, ctypes.byref(n_out))
        if rc != 0:
            raise BtleError(rc, "record buffer holds fewer records than the directory describes (capacity overflow)")
        return out

    def sort_records(self, recs: np.ndarray) -> np.ndarray:
        recs = np.ascontiguousarray(recs, dtype=REC_DTYPE)
        self._L.btle_b200_sort_records(recs.ctypes.data, recs.size)
        return recs

    # ---- leaf functions with the reference's signatures ----------------------------------
    def search_unique_bits(self, rxp: np.ndarray, search_len: int, unique_bits, unique_bits_mask, num_bits=32) -> int:
        rxp = np.ascontiguousarray(rxp, dtype=np.int8)
        assert rxp.size >= 8 * search_len + 2
        ub = np.ascontiguousarray(unique_bits, dtype=np.uint8)
        um = np.ascontiguousarray(unique_bits_mask, dtype=np.uint8)
        r = self._L.btle_b200_search_unique_bits(self._h, rxp.ctypes.data, search_len, ub.ctypes.data, um.ctypes.data, num_bits)
        if r <= -1000:                     # BTLE_SEARCH_ERR(code): errors live below every possible hit index
            self._check(r + 1000)
        return r

    def demod_byte(self, rxp: np.ndarray, num_byte: int) -> np.ndarray:
        rxp = np.ascontiguousarray(rxp, dtype=np.int8)
        out = np.zeros(num_byte, dtype=np.uint8)
        self._check(self._L.btle_b200_demod_byte(self._h, rxp.ctypes.data, num_byte, out.ctypes.data))
        return out

    def scramble_byte(self, byte_in, channel: int, table_offset: int = 0) -> np.ndarray:
        b = np.ascontiguousarray(byte_in, dtype=np.uint8)
        out = np.zeros_like(b)
        self._check(self._L.btle_b200_scramble_byte(self._h, b.ctypes.data, b.size, channel, table_offset, out.ctypes.data))
        return out

    def crc24_byte(self, byte_in, init_hex: int) -> int:
        b = np.ascontiguousarray(byte_in, dtype=np.uint8)
        out = ctypes.c_uint32(0)
        self._check(self._L.btle_b200_crc24_byte(self._h, b.ctypes.data, b.size, init_hex, ctypes.byref(out)))
        return out.value

    def crc_init_reorder(self, crc_init: int) -> int:
        return self._L.btle_b200_crc_init_reorder(crc_init)

    def dbits(self, iq: np.ndarray) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.int8)
        n = iq.size // 2 - 1
        out = np.zeros(max(n, 0), dtype=np.uint8)
        if n > 0:
            self._check(self._L.btle_b200_dbits(self._h, iq.ctypes.data, n, out.ctypes.data))
        return out


class RxStream:
    """Python face of btle_b200_stream_open / push / finish / close."""

    def __init__(self, rx: BtleRx, cfgs: np.ndarray, segment_chunks: int):
        self._rx, self._L = rx, rx._L
        self._L.btle_b200_stream_open.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p)]
        self._L.btle_b200_stream_push.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t,
                                                  ctypes.POINTER(ctypes.c_size_t)]
        self._L.btle_b200_stream_finish.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]
        self._L.btle_b200_stream_close.argtypes = [ctypes.c_void_p]
        self._L.btle_b200_stream_close.restype = None
        self._cfg = np.ascontiguousarray(cfgs, dtype=CFG_DTYPE)
        h = ctypes.c_void_p()
        rx._check(self._L.btle_b200_stream_open(rx._h, self._cfg.ctypes.data, int(segment_chunks), ctypes.byref(h)))
        self._h = h
        self._buf = np.empty(65536, dtype=REC_DTYPE)

    def push(self, iq) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.int8).reshape(-1)
        out, done, step = [], 0, 64 << 20
        while done < iq.size:                   # a push never returns more records than the buffer holds: feed it in bounded pieces
            piece = iq[done:done + step]
            n = ctypes.c_size_t(0)
            self._rx._check(self._L.btle_b200_stream_push(self._h, piece.ctypes.data, piece.size, self._buf.ctypes.data, self._buf.size, ctypes.byref(n)))
            out.append(self._buf[:n.value].copy())
            done += piece.size
        return np.concatenate(out) if out else self._buf[:0].copy()

    def finish(self) -> np.ndarray:
        out = []
        while True:
            n = ctypes.c_size_t(0)
            rc = self._L.btle_b200_stream_finish(self._h, self._buf.ctypes.data, self._buf.size, ctypes.byref(n))
            out.append(self._buf[:n.value].copy())
            if rc != BTLE_EOVERFLOW:
                self._rx._check(rc)
                break
        return np.concatenate(out)

    def close(self):
        if getattr(self, "_h", None):
            self._L.btle_b200_stream_close(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    __del__ = close
