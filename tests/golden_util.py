import glob
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def cases():
    return sorted(os.path.basename(p) for p in glob.glob(os.path.join(GOLD, "*.npz"))
                  if not os.path.basename(p).startswith(("btlelib", "ref_driver")))


def load(name):
    z = np.load(os.path.join(GOLD, name), allow_pickle=False)
    cfg = json.loads(str(z["cfg"]))
    return z, cfg


def assert_matches_golden(rec, z):
    """rec: REC_DTYPE records from the implementation under test; z: golden npz written by
    oracle/gen_golden.py from the reference's own receiver()."""
    assert len(rec) == len(z["exp_n0"]), f"{len(rec)} packets, reference found {len(z['exp_n0'])}"
    for i, a in enumerate(rec):
        assert a["chunk"] == z["exp_chunk"][i] and a["n0"] == z["exp_n0"][i], (i, a["chunk"], a["n0"])
        nb = int(z["exp_nbytes"][i])
        assert a["n_bytes"] == nb and a["crc_bad"] == z["exp_crc_bad"][i], i
        assert bytes(a["bytes"][:nb]) == bytes(z["exp_bytes"][i][:nb]), i


def tables():
    return json.load(open(os.path.join(GOLD, "tables.json")))
