"""ctypes binding of the C-ABI (include/btle_b200.h -> btle_b200/libbtle_b200.so).

There is no CPU fallback: if the CUDA library is missing or no CUDA device is usable this module
raises.  Nothing here imports the test oracle."""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BTLE_B200_LIB") or os.path.join(_HERE, "libbtle_b200.so")   # env override: A/B builds

BTLE_OK, BTLE_EINVAL, BTLE_ENODEV, BTLE_ENOMEM, BTLE_ECUDA, BTLE_EOVERFLOW = 0, -1, -2, -3, -4, -5

# btle_pkt_rec, 64 bytes
REC_DTYPE = np.dtype([
    ("stream", "<i4"), ("chunk", "<i4"), ("n0", "<i4"),
    ("channel", "u1"), ("n_bytes", "u1"), ("crc_bad", "u1"), ("flags", "u1"),
    ("access_addr", "<u4"), ("mag_sum", "<u2"), ("bytes", "u1", 42),
])
# btle_stream_cfg, 24 bytes
CFG_DTYPE = np.dtype([("channel", "<i4"), ("access_addr", "<u4"), ("access_mask", "<u4"), ("crc_init", "<u4"),
                      ("raw", "<i4"), ("rssi", "<i4")])
# btle_model_rx_rec, 80 bytes
MODEL_REC_DTYPE = np.dtype([("start", "<i4"), ("n_pdu_bits", "<u2"), ("crc_ok", "u1"), ("phase", "u1"), ("payload_len", "u1"),
                            ("found", "u1"), ("pdu", "u1", 70)])
# btle_synth_cfg (32 bytes) / btle_synth_truth (64 bytes)
SYNTH_CFG_DTYPE = np.dtype([("seed", "<u8"), ("slot_samples", "<i4"), ("amplitude", "<i4"), ("corrupt_every", "<i4"),
                            ("straddle_every", "<i4"), ("noise", "<i4"), ("reserved", "<i4")])
SYNTH_TRUTH_DTYPE = np.dtype([("start_sample", "<i8"), ("stream", "<i4"), ("slot", "<i4"), ("n_air_bytes", "u1"), ("corrupt", "u1"),
                              ("straddle", "u1"), ("pdu_len", "u1"), ("pdu", "u1", 44)])
assert SYNTH_CFG_DTYPE.itemsize == 32 and SYNTH_TRUTH_DTYPE.itemsize == 64
DIR_DTYPE = np.dtype([("base", "<u4"), ("count", "<u4")])      # btle_unit_dir
BER_CFG_DTYPE = np.dtype([("seed", "<u8"), ("snr_db", "<f4"), ("ppm", "<f4"), ("channel", "<i4"), ("crc_init", "<u4"), ("access_addr", "<u4"),
                          ("reserved", "<u4")])
BER_RESULT_DTYPE = np.dtype([("packets", "<u8"), ("pkt_err", "<u8"), ("bit_err", "<u8"), ("bit_total", "<u8"), ("aa_miss", "<u8"), ("seconds", "<f8")])
assert BER_CFG_DTYPE.itemsize == 32 and BER_RESULT_DTYPE.itemsize == 48
SPS8_REC_DTYPE = np.dtype([("sample", "<i8"), ("window", "<i8"), ("rx", MODEL_REC_DTYPE)])     # btle_sps8_rec
# btle_wideband_cfg, 16 bytes
WIDEBAND_CFG_DTYPE = np.dtype([("decim", "<i4"), ("center_mhz", "<i4"), ("out_shift", "<i4"), ("reserved", "<i4")])
assert WIDEBAND_CFG_DTYPE.itemsize == 16
assert REC_DTYPE.itemsize == 64 and CFG_DTYPE.itemsize == 24 and MODEL_REC_DTYPE.itemsize == 80 and SPS8_REC_DTYPE.itemsize == 96

EXPORTS = [
    "btle_b200_create", "btle_b200_destroy", "btle_b200_bind_host_numa", "btle_b200_last_error", "btle_b200_strerror", "btle_b200_version",
    "btle_b200_rx_batch", "btle_b200_rx", "btle_b200_rx_device", "btle_b200_rx_device_dir", "btle_b200_rx_units",
    "btle_b200_gather_ordered", "btle_b200_sort_records", "btle_b200_last_launches",
    "btle_b200_search_unique_bits", "btle_b200_demod_byte", "btle_b200_scramble_byte", "btle_b200_crc24_byte",
    "btle_b200_crc_init_reorder", "btle_b200_parse_adv_pdu_header_byte", "btle_b200_parse_ll_pdu_header_byte",
    "btle_b200_dbits", "btle_b200_gfsk_demod_i16", "btle_b200_search_bit_sequence", "btle_b200_crc24_bits",
    "btle_b200_scramble_bits", "btle_b200_model_rx_batch_device", "btle_b200_model_rx_batch",
    "btle_b200_tx_modulate_device", "btle_b200_rx_iq16", "btle_b200_synth_streams_device", "btle_b200_rx_sps8", "btle_b200_sps8_hits_device", "btle_b200_ber_run",
    "btle_b200_stream_open", "btle_b200_stream_push", "btle_b200_stream_acquire", "btle_b200_stream_commit", "btle_b200_stream_finish",
    "btle_b200_stream_close", "btle_b200_stream_set_cfg", "btle_b200_parse_adv_pdu_payload_byte", "btle_b200_parse_ll_pdu_payload_byte",
    "btle_b200_receiver_controller", "btle_b200_receiver_status", "btle_b200_note_packet", "btle_b200_set_hop_hooks", "btle_b200_hop_reset",
    "btle_b200_get_freq_by_channel_number", "btle_b200_chm_is_full_map",
    "btle_b200_wideband_taps", "btle_b200_channelize_device", "btle_b200_channelize", "btle_b200_rx_wideband",
]


class BtleError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"btle_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load():
    """Load libbtle_b200.so (built in-tree by __graft_entry__.build()).  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BtleError(BTLE_ENODEV, f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = ctypes.CDLL(LIB_PATH)
    vp, sz, i32, u32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_uint32
    L.btle_b200_create.argtypes = [ctypes.POINTER(vp), i32]
    L.btle_b200_bind_host_numa.argtypes = [i32, ctypes.POINTER(ctypes.c_int)]
    L.btle_b200_destroy.argtypes = [vp]
    L.btle_b200_destroy.restype = None
    L.btle_b200_last_error.argtypes = [vp]
    L.btle_b200_last_error.restype = ctypes.c_char_p
    L.btle_b200_strerror.argtypes = [i32]
    L.btle_b200_strerror.restype = ctypes.c_char_p
    L.btle_b200_version.restype = u32
    L.btle_b200_rx_batch.argtypes = [vp, vp, sz, sz, sz, vp, vp, sz, ctypes.POINTER(sz)]
    L.btle_b200_rx.argtypes = [vp, vp, sz, vp, vp, sz, ctypes.POINTER(sz)]
    L.btle_b200_rx_device.argtypes = [vp, vp, sz, sz, sz, vp, vp, sz, vp, vp]
    L.btle_b200_rx_device_dir.argtypes = [vp, vp, sz, sz, sz, vp, vp, sz, vp, vp, sz, vp]
    L.btle_b200_rx_units.argtypes = [vp, sz, sz]
    L.btle_b200_rx_units.restype = sz
    L.btle_b200_gather_ordered.argtypes = [vp, sz, vp, sz, vp, sz, ctypes.POINTER(sz)]
    L.btle_b200_sort_records.argtypes = [vp, sz]
    L.btle_b200_sort_records.restype = None
    L.btle_b200_last_launches.argtypes = [vp]
    L.btle_b200_search_unique_bits.argtypes = [vp, vp, i32, vp, vp, i32]
    L.btle_b200_demod_byte.argtypes = [vp, vp, i32, vp]
    L.btle_b200_scramble_byte.argtypes = [vp, vp, i32, i32, i32, vp]
    L.btle_b200_crc24_byte.argtypes = [vp, vp, i32, u32, ctypes.POINTER(u32)]
    L.btle_b200_crc_init_reorder.argtypes = [u32]
    L.btle_b200_crc_init_reorder.restype = u32
    ip = ctypes.POINTER(ctypes.c_int)
    L.btle_b200_parse_adv_pdu_header_byte.argtypes = [vp, ip, ip, ip, ip]
    L.btle_b200_parse_adv_pdu_header_byte.restype = None
    L.btle_b200_parse_ll_pdu_header_byte.argtypes = [vp, ip, ip, ip, ip, ip]
    L.btle_b200_parse_ll_pdu_header_byte.restype = None
    L.btle_b200_dbits.argtypes = [vp, vp, sz, vp]
    L.btle_b200_gfsk_demod_i16.argtypes = [vp, vp, vp, sz, vp, vp]
    L.btle_b200_search_bit_sequence.argtypes = [vp, vp, sz, vp, sz]
    L.btle_b200_search_bit_sequence.restype = ctypes.c_long
    L.btle_b200_crc24_bits.argtypes = [vp, vp, sz, vp, vp]
    L.btle_b200_scramble_bits.argtypes = [vp, vp, sz, i32, vp]
    L.btle_b200_model_rx_batch_device.argtypes = [vp, vp, vp, sz, sz, i32, i32, u32, u32, vp, vp]
    L.btle_b200_model_rx_batch.argtypes = [vp, vp, vp, sz, sz, i32, i32, u32, u32, vp]
    L.btle_b200_tx_modulate_device.argtypes = [vp, vp, vp, sz, sz, i32, vp, vp, vp]
    L.btle_b200_rx_iq16.argtypes = [vp, vp, sz, i32, vp, vp, sz, ctypes.POINTER(sz)]
    L.btle_b200_ber_run.argtypes = [vp, vp, sz, vp]
    L.btle_b200_sps8_hits_device.argtypes = [vp, vp, sz, u32, vp, sz, vp, vp]
    L.btle_b200_rx_sps8.argtypes = [vp, vp, sz, i32, u32, u32, vp, sz, ctypes.POINTER(sz)]
    L.btle_b200_synth_streams_device.argtypes = [vp, vp, sz, sz, sz, vp, vp, vp, sz, ctypes.POINTER(sz), vp]
    L.btle_b200_wideband_taps.argtypes = [vp, i32, vp, sz, ctypes.POINTER(sz), ctypes.POINTER(ctypes.c_int)]
    L.btle_b200_channelize_device.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz, vp]
    L.btle_b200_channelize.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz]
    L.btle_b200_rx_wideband.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz, ctypes.POINTER(sz)]
    _lib = L
    return L


def bind_host_numa(device: int) -> int:
    """Bind the calling thread (CPU affinity + preferred memory node) to the NUMA node of CUDA device `device`
    (btle_b200_bind_host_numa).  Returns the node or -1."""
    node = ctypes.c_int(-1)
    load().btle_b200_bind_host_numa(int(device), ctypes.byref(node))
    return node.value
