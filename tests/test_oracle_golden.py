"""Pins the oracle (oracle/dpk_oracle.c + oracle/oracle.py) against the golden
vectors captured from the real reference (tests/golden/make_golden.py).  CPU only."""
import json

import numpy as np
import pytest

from oracle import oracle as orc
from tests.golden_util import dec, load, split_rows

HV = load("hash_vectors.json")
SC = load("shuffle_cases.json")


def test_portable_hash_all_golden_keys():
    bad = []
    for row in HV["rows"]:
        k = dec(row["key"])
        if orc.portable_hash(k) != row["hash"]:
            bad.append((k, orc.portable_hash(k), row["hash"]))
    assert not bad, bad[:5]


def test_get_partition_all_golden_keys():
    for row in HV["rows"]:
        k = dec(row["key"])
        got = [orc.get_partition(k, p) for p in HV["partitions"]]
        assert got == row["part"], (k, got, row["part"])


def test_unhashable_types_raise_like_reference():
    assert [u["raises"] for u in HV["unhashable"]] == ["TypeError"] * 4
    for k in (True, [1, 2], {1: 2}, 1 + 2j):
        with pytest.raises(TypeError):
            orc.portable_hash(k)


def test_thresholds_bisect():
    thr = HV["thresholds"]
    for row in HV["threshold_rows"]:
        assert orc.get_partition(row["key"], 8, thr) == row["part"]
    for row in HV["threshold_rows_small"]:
        assert orc.get_partition(row["key"], 3, HV["thresholds_small"]) == row["part"]


def test_vector_hash_matches_scalar_and_golden():
    ints = [dec(r["key"]) for r in HV["rows"] if isinstance(r["key"], int)
            and -2 ** 63 <= r["key"] < 2 ** 63]
    want = [r["hash"] for r in HV["rows"] if isinstance(r["key"], int)
            and -2 ** 63 <= r["key"] < 2 ** 63]
    assert orc.hash_vec(np.array(ints, dtype=np.int64)).tolist() == want
    fl = [(dec(r["key"]), r["hash"]) for r in HV["rows"]
          if isinstance(r["key"], dict) and "f" in r["key"]]
    got = orc.hash_vec(np.array([f for f, _ in fl], dtype=np.float64)).tolist()
    assert got == [h for _, h in fl]
    # bytes and str (as UTF-8) columns
    for tag, mode, encf in (("b", 0, lambda b: b), ("s", 1, lambda s: s.encode("utf-8", "surrogatepass"))):
        ks = [(dec(r["key"]), r["hash"]) for r in HV["rows"]
              if isinstance(r["key"], dict) and tag in r["key"]]
        blobs = [encf(k) for k, _ in ks]
        offs = np.zeros(len(blobs) + 1, dtype=np.int64)
        offs[1:] = np.cumsum([len(b) for b in blobs])
        data = np.frombuffer(b"".join(blobs), dtype=np.uint8)
        got = orc.hash_bytes_vec(data, offs, mode).tolist()
        assert got == [h for _, h in ks]


FUNCS = {"add": lambda x, y: x + y, "min": lambda x, y: min(x, y), "max": lambda x, y: max(x, y),
         "mul": lambda x, y: x * y, "or": lambda x, y: x | y, "and": lambda x, y: x & y,
         "xor": lambda x, y: x ^ y}
OPNAME = {"add": "sum", "min": "min", "max": "max", "mul": "prod", "or": "or", "and": "and",
          "xor": "xor"}


def _canon_py(parts):
    from tests.golden.make_golden import enc
    return [sorted(([enc(k), enc(v)] for k, v in p.items()), key=json.dumps) for p in parts]


@pytest.mark.parametrize("case", SC["cases"], ids=[c["name"] for c in SC["cases"]])
def test_python_restatement_matches_reference(case):
    rows = [(dec(k), dec(v)) for k, v in case["rows"]]
    splits = split_rows(rows, case["split_sizes"])
    if case["op"] == "reduceByKey":
        got = orc.py_reduce_by_key(splits, case["P"], FUNCS[case["func"]], case["thresholds"])
    else:
        got = orc.py_group_by_key(splits, case["P"])
    if case["name"].startswith("f32_vals_add") or case["name"] == "i32_keys_f_vals":
        # float sums: reference merge order is not deterministic -> tolerance
        want = [{json.dumps(k): dec(v) for k, v in part} for part in case["parts"]]
        from tests.golden.make_golden import enc
        for p, part in enumerate(got):
            assert len(part) == len(want[p])
            for k, v in part.items():
                assert abs(v - want[p][json.dumps(enc(k))]) <= 1e-9 * max(1.0, abs(v))
    else:
        assert _canon_py(got) == case["parts"]


def _numeric_case(case):
    if not case["rows"]:
        return True
    k, v = case["rows"][0]
    kk, vv = dec(k), dec(v)
    return type(kk) is int and type(vv) in (int, float)


NUM_CASES = [c for c in SC["cases"] if _numeric_case(c)]


@pytest.mark.parametrize("case", NUM_CASES, ids=[c["name"] for c in NUM_CASES])
def test_c_restatement_matches_reference(case):
    rows = [(dec(k), dec(v)) for k, v in case["rows"]]
    splits = split_rows(rows, case["split_sizes"])
    isf = bool(rows) and type(rows[0][1]) is float
    ks = [np.array([k for k, _ in s], dtype=np.int64) for s in splits]
    vs = [np.array([v for _, v in s], dtype=np.float64 if isf else np.int64) for s in splits]
    P = case["P"]
    if case["op"] == "reduceByKey":
        if case["func"] == "mul":
            pytest.skip("products overflow int64; covered by the Python restatement")
        got = orc.reduce_by_key(ks, vs, P, OPNAME[case["func"]], case["thresholds"])
        for p in range(P):
            want = {k: dec(v) for k, v in case["parts"][p]}
            gk, gv = got[p]
            assert sorted(gk.tolist()) == sorted(want)
            for k, v in zip(gk.tolist(), gv.tolist()):
                if isf and case["func"] == "add":
                    assert abs(v - want[k]) <= 1e-9 * max(1.0, abs(v))
                else:
                    assert v == want[k]
    else:
        got = orc.group_by_key(ks, vs, P)
        for p in range(P):
            want = {k: dec(v) for k, v in case["parts"][p]}
            gk, go, gv = got[p]
            assert sorted(gk.tolist()) == sorted(want)
            for i, k in enumerate(gk.tolist()):
                assert gv[go[i]:go[i + 1]].tolist() == want[k]


def test_split_like_parallelize_matches_reference_split_sizes():
    for case in SC["cases"]:
        rows = case["rows"]
        got = [len(s) for s in orc.split_like_parallelize(rows, case["M"])]
        assert got == case["split_sizes"], case["name"]


def test_oracle_hash_vs_compiled_reference_extension():
    """The reference's own Cython portable_hash, compiled as-is, on 35000 seeded ints, floats and byte strings
    (tests/golden/make_refhash_golden.py): every hash through the stored SHA-256, a stride sample value by value."""
    from tests.golden.make_refhash_golden import digest, inputs
    want = load("ref_portable_hash.json")
    xs = inputs()
    got = {"ints": orc.hash_vec(np.array(xs["ints"], dtype=np.int64)).tolist(),
           "floats": orc.hash_vec(np.array(xs["floats"], dtype=np.float64)).tolist(),
           "bytes": [orc.portable_hash(b) for b in xs["bytes"]]}
    for kind, w in want.items():
        assert len(got[kind]) == w["n"], kind
        assert got[kind][::w["stride"]] == w["sample"], kind
        assert digest(got[kind]) == w["sha256"], kind
