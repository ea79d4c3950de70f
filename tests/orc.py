"""Test-side access to the oracle (oracle/libbtle_oracle.so = our C restatement,
oracle/_ref/btle_ref_driver = the unmodified reference receiver).  Only tests,
__graft_entry__.smoke() and bench.py's CPU-baseline legs may import this."""
from __future__ import annotations

import atexit
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "libbtle_oracle.so")
REF_DRIVER = os.path.join(ORACLE_DIR, "_ref", "btle_ref_driver")

# layout shared by orc_rec (oracle/btle_oracle.h) and btle_pkt_rec (include/btle_b200.h)
REC_DTYPE = np.dtype([
    ("stream", "<i4"), ("chunk", "<i4"), ("n0", "<i4"),
    ("channel", "u1"), ("n_bytes", "u1"), ("crc_bad", "u1"), ("flags", "u1"),
    ("access_addr", "<u4"), ("mag_sum", "<u2"), ("bytes", "u1", 42),
])
assert REC_DTYPE.itemsize == 64
REF_DTYPE = np.dtype([("chunk", "<i4"), ("n0", "<i4"), ("nbytes", "<i4"), ("crc_bad", "<i4"), ("bytes", "u1", 48)])


class OrcCfg(ctypes.Structure):
    _fields_ = [("channel", ctypes.c_int32), ("access_addr", ctypes.c_uint32), ("access_mask", ctypes.c_uint32),
                ("crc_init", ctypes.c_uint32), ("raw", ctypes.c_int32)]


def build_oracle():
    src = os.path.join(ORACLE_DIR, "btle_oracle.c")
    if (not os.path.exists(ORACLE_SO)) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(src):
        subprocess.run(["make", "-C", ORACLE_DIR, "oracle"], check=True, capture_output=True)
    return ORACLE_SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build_oracle())
        _lib.orc_crc_init_reorder.restype = ctypes.c_uint32
        _lib.orc_crc_init_reorder.argtypes = [ctypes.c_uint32]
        _lib.orc_crc24.restype = ctypes.c_uint32
        _lib.orc_crc24.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32]
        _lib.orc_whiten_byte.restype = ctypes.c_uint8
        _lib.orc_whiten_byte.argtypes = [ctypes.c_int, ctypes.c_int]
        _lib.orc_dbits.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_void_p]
        _lib.orc_search.restype = ctypes.c_int
        _lib.orc_search.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32,
                                    ctypes.POINTER(ctypes.c_int)]
        _lib.orc_demod_bytes.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        _lib.orc_rx_stream.restype = ctypes.c_long
        _lib.orc_rx_stream.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.POINTER(OrcCfg), ctypes.c_int32,
                                       ctypes.c_void_p, ctypes.c_long]
    return _lib


def rx_stream(iq: np.ndarray, channel=37, access_addr=0x8E89BED6, access_mask=0xFFFFFFFF, crc_init=0x555555,
              raw=0, stream=0) -> np.ndarray:
    """Our C restatement over one capture -> REC_DTYPE array in reference order."""
    iq = np.ascontiguousarray(iq, dtype=np.int8)
    cfg = OrcCfg(channel, access_addr, access_mask, crc_init, raw)
    cap = (iq.size // 16384) * 51 + 8      # BTLE_MAX_PKTS_PER_CHUNK
    out = np.zeros(cap, dtype=REC_DTYPE)
    n = lib().orc_rx_stream(iq.ctypes.data, iq.size, ctypes.byref(cfg), stream, out.ctypes.data, cap)
    assert n <= cap
    return out[:n]


def dbits(iq: np.ndarray) -> np.ndarray:
    """d[n] for n in [0, len/2 - 1)."""
    iq = np.ascontiguousarray(iq, dtype=np.int8)
    n = iq.size // 2 - 1
    d = np.zeros(n, dtype=np.uint8)
    lib().orc_dbits(iq.ctypes.data, n, d.ctypes.data)
    return d


def ref_available() -> bool:
    return os.path.exists(REF_DRIVER)


# What btle_ref_driver printed and wrote, recorded once per (arguments, input contents) so that the comparisons with the
# reference run wherever the tests run, without the reference sources.  Re-record (where oracle/_ref is built, on a
# machine with a GPU so that the CLI cases run) with
#     BTLE_REF_RECORD=/tmp/ref_driver.npz python -m pytest tests   and copy the file over REF_GOLDEN.
REF_GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_driver.npz")
_RECORD_TO = os.environ.get("BTLE_REF_RECORD")
_recorded = {}
_golden = None


def _case_key(args, inputs, outputs):
    """Digest of the driver's arguments (paths replaced by their role) and of the contents of its inputs."""
    h = hashlib.sha256()
    names = {p: f"<in{i}>" for i, p in enumerate(inputs)}
    names.update({p: f"<out{i}>" for i, p in enumerate(outputs)})
    for a in args:
        h.update(names.get(a, a).encode() + b"\0")
    for p in inputs:
        files = [os.path.join(p, f) for f in sorted(os.listdir(p))] if os.path.isdir(p) else [p]
        for f in files:
            h.update(os.path.basename(f).encode() + b"\0")
            with open(f, "rb") as fh:
                h.update(hashlib.sha256(fh.read()).digest())
    return h.hexdigest()[:32]


def _save_recorded():
    old = dict(np.load(_RECORD_TO)) if os.path.exists(_RECORD_TO) else {}
    old.update(_recorded)
    np.savez_compressed(_RECORD_TO, **old)


def ref_driver(args, inputs=(), outputs=(), live=False, stdout=True) -> str:
    """btle_ref_driver (the unmodified reference) with `args` -> its stdout (if `stdout`); the files it writes land at
    `outputs`.  `inputs` are the files / directories among `args` it reads.  Served from REF_GOLDEN unless `live` or recording."""
    args, inputs, outputs = [str(a) for a in args], [str(p) for p in inputs], [str(p) for p in outputs]
    key = _case_key(args, inputs, outputs)
    if live or _RECORD_TO:
        p = subprocess.run([REF_DRIVER] + args, check=True, capture_output=True)
        if _RECORD_TO and not live:
            if not _recorded:
                atexit.register(_save_recorded)
            _recorded[key + ".stdout"] = np.frombuffer(p.stdout if stdout else b"", dtype=np.uint8)
            for i, o in enumerate(outputs):
                _recorded[f"{key}.out{i}"] = np.fromfile(o, dtype=np.uint8)
        return p.stdout.decode()
    global _golden
    if _golden is None:
        _golden = np.load(REF_GOLDEN)
    assert key + ".stdout" in _golden.files, (
        f"no recorded reference output for btle_ref_driver {' '.join(args[:1])} on this input (case {key}): the test's input "
        f"or arguments changed; re-record {os.path.relpath(REF_GOLDEN, ROOT)} (see tests/orc.py)")
    for i, o in enumerate(outputs):
        _golden[f"{key}.out{i}"].tofile(o)
    return _golden[key + ".stdout"].tobytes().decode()


def ref_rx_stream(iq: np.ndarray, channel=37, access_addr=0x8E89BED6, access_mask=0xFFFFFFFF, crc_init=0x555555,
                  raw=0, live=False) -> np.ndarray:
    """The unmodified reference receiver() over one capture -> REF_DTYPE array."""
    iq = np.ascontiguousarray(iq, dtype=np.int8)
    with tempfile.TemporaryDirectory() as td:
        fi, fo = os.path.join(td, "iq.bin"), os.path.join(td, "out.rec")
        iq.tofile(fi)
        ref_driver(["run", fi, str(channel), f"{access_addr:x}", f"{crc_init:x}", f"{access_mask:x}", str(int(raw)), fo],
                   inputs=[fi], outputs=[fo], live=live, stdout=False)
        return np.fromfile(fo, dtype=REF_DTYPE)


def ref_time(iq_path: str, channel=37, access_addr=0x8E89BED6, access_mask=0xFFFFFFFF, crc_init=0x555555, raw=0,
             procs=1, reps=1) -> dict:
    import json
    p = subprocess.run([REF_DRIVER, "time", iq_path, str(channel), f"{access_addr:x}", f"{crc_init:x}",
                        f"{access_mask:x}", str(int(raw)), str(procs), str(reps)], check=True, capture_output=True)
    return json.loads(p.stdout.decode().strip().splitlines()[-1])


def assert_same_as_ref(rec: np.ndarray, ref: np.ndarray):
    """REC_DTYPE records (oracle or GPU) vs REF_DTYPE records (reference)."""
    assert len(rec) == len(ref), f"packet count {len(rec)} != reference {len(ref)}"
    for a, b in zip(rec, ref):
        assert a["chunk"] == b["chunk"] and a["n0"] == b["n0"], (a["chunk"], a["n0"], b["chunk"], b["n0"])
        assert a["n_bytes"] == b["nbytes"] and a["crc_bad"] == b["crc_bad"]
        nb = int(b["nbytes"])
        assert bytes(a["bytes"][:nb]) == bytes(b["bytes"][:nb])
