#!/usr/bin/env python
"""Capture the reference's own compiled portable_hash (dpark/portable_hash.pyx, cythonized as-is) on seeded
random ints, floats and byte strings, so that the oracle's hash is checked against it without the reference.

    python tests/golden/make_refhash_golden.py      # writes tests/golden/ref_portable_hash.json

The inputs are regenerated from the seed by `inputs()` in the test.  Stored per kind: the SHA-256 of all the
reference's hashes as little-endian int64 (every value is compared through it) and every STRIDE-th hash in the
clear, so that a mismatch can be located.  Needs the reference sources (DPARK_REFERENCE, as make_golden.py);
only the hashes are stored."""
import hashlib
import importlib.util
import json
import os
import random
import shutil
import sys
import sysconfig
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "ref_portable_hash.json")
STRIDE = {"ints": 20, "floats": 10, "bytes": 5}


def inputs():
    rnd = random.Random(7)
    xs = [rnd.randint(-2 ** 63, 2 ** 63 - 1) for _ in range(20000)]
    fs = [rnd.uniform(-1e9, 1e9) for _ in range(5000)] + [rnd.random() * 2.0 ** rnd.randint(-1000, 1000) for _ in range(5000)]
    bs = [bytes(rnd.randrange(256) for _ in range(rnd.randrange(0, 64))) for _ in range(5000)]
    return {"ints": xs, "floats": fs, "bytes": bs}


def digest(hashes):
    return hashlib.sha256(np.asarray(hashes, dtype="<i8").tobytes()).hexdigest()


def main():
    sys.path.insert(0, HERE)
    from make_golden import build_reference
    scratch = tempfile.mkdtemp(prefix="dpark_ref_")
    try:
        build_reference(scratch)
        so = os.path.join(scratch, "dpark", "portable_hash" + sysconfig.get_config_var("EXT_SUFFIX"))
        spec = importlib.util.spec_from_file_location("portable_hash", so)
        ph = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ph)
        out = {}
        for kind, xs in inputs().items():
            h = [ph.portable_hash(x) for x in xs]
            out[kind] = {"n": len(h), "sha256": digest(h), "stride": STRIDE[kind], "sample": h[::STRIDE[kind]]}
    finally:
        shutil.rmtree(scratch, ignore_errors=True)
    with open(OUT, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print("wrote %s: %s" % (OUT, {k: v["n"] for k, v in out.items()}))


if __name__ == "__main__":
    main()
