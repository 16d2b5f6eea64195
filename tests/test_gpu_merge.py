"""dpk_combine -- the reduce-side merge behind every reduceByKey / combineByKey (DESIGN.md a9) -- under every merge
variant dpk_set_option can select, against an exact reference computed with numpy / Python from the raw input
columns (not from the oracle's merge, which casts every key to int64).  -m gpu, apart from the CPU check that the
data shapes reach the kernel paths they are named after.

Reference rules:
  keys   grouped by their bits, float -0.0 spelled 0.0 (one key, DESIGN.md §7); every output key must sit in the
         reference's partition orc.partition_vec(orc.hash_vec(key), P) and be spelled canonically
  int    sum / min / max / and / or / xor exact (numpy reduceat); prod in Python ints (inputs keep it inside int64)
  float  sum: |got - fsum| <= (n_k - 1) * 2^-53 * sum|v| per key, and the sign of a zero result exact: -0.0 iff
         every value of the key is -0.0 (IEEE sums of anything else that cancel give +0.0);
         min / max: bit-exact up to the sign of a zero (DESIGN.md §7);
         prod: rtol 1e-12 and the sign exact (the sign of a product does not depend on the order)
No NaN keys or values: their behaviour is not defined.
"""
import ctypes as C
import functools
import math
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc

# kernel constants the shapes are built around (dpk_aggregate2.cuh, dpk_combine.cu)
AG2_CAP = 2048        # staged rows per window of k_smem_aggregate2: no pass holds more distinct keys
AG2_MINW = 256        # a pass whose free room falls below this splits: <= AG2_CAP - AG2_MINW distinct keys always fit
AG2_MAX_M = 1 << 16   # hash-disjoint passes filter on slot_hash32 bits 12..27
AG_MAX_SB2 = 10       # the second-level split is at most 1024-way

# built-in values of the dpk_set_option switches that select the merge (dpk_combine.cu)
DEFAULTS = {"reduce_impl": 2, "agg_impl": 1, "agg_wide": 1, "agg_ctas": 4, "agg_split": 1, "agg_cursor": 1,
            "agg_pipe": 0, "agg_batched": 0, "agg_target_rows": 2048}

# every variant, spelled as in DPK_OPTIONS
VARIANTS = ["default", "agg_split=0", "agg_cursor=0", "agg_batched=1", "agg_ctas=3", "agg_pipe=1", "agg_pipe=2",
            "agg_pipe=1,agg_batched=1", "agg_impl=0,agg_wide=1", "agg_impl=0,agg_wide=0", "reduce_impl=1",
            "reduce_impl=0"]

KEY_KINDS = ["int64", "int32", "float64", "float32", "uint64"]
VAL_KINDS = ["int64", "int32", "float64", "float32"]
INT_OPS = ["sum", "min", "max", "prod", "and", "or", "xor"]
FLOAT_OPS = ["sum", "min", "max", "prod"]
COMBOS = [(kk, vk, op) for kk in KEY_KINDS for vk in VAL_KINDS
          for op in (FLOAT_OPS if vk.startswith("float") else INT_OPS)]
LARGE_COMBOS = [("int64", "int64", "sum"), ("int64", "float64", "sum")]


def nv():
    from dpark_b200 import _native
    return _native


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _parse(spec):
    """"name=value,..." -> dict, the way _native parses DPK_OPTIONS."""
    out = {}
    for item in filter(None, spec.split(",")):
        name, _, value = item.partition("=")
        out[name.strip()] = int(value)
    return out


def _set(opts):
    for name, value in opts.items():
        nv().set_option(name, value)


def _restore():
    """The settings are global to the process and have no getter: back to the built-in values with the DPK_OPTIONS
    overrides on top, as the library stands after loading."""
    _set(dict(DEFAULTS, **_parse(os.environ.get("DPK_OPTIONS", ""))))


@pytest.fixture
def variant(request):
    spec = request.param
    opts = dict(DEFAULTS, **({} if spec == "default" else _parse(spec)))
    try:
        _set(opts)
        yield opts
    finally:
        _restore()


def _shared_memory_merge(opts):
    """The variant merges fine buckets in shared-memory tables with a bounded number of hash-disjoint passes."""
    return opts["reduce_impl"] == 2 and (opts["agg_impl"] == 1 or opts["agg_pipe"] != 0)


def _choose_sb2(n, F, target=DEFAULTS["agg_target_rows"]):
    """choose_sb2 (dpk_combine.cu): bits of the second-level split for n received rows in F first-level buckets."""
    sb2 = 0
    while sb2 < AG_MAX_SB2 and n // (F << sb2) > target:
        sb2 += 1
    return sb2


# ---------------------------------------------------------------- keys and values
KEY_DTYPES = {"int64": np.int64, "int32": np.int32, "float64": np.float64, "float32": np.float32,
              "uint64": np.uint64}
F61 = 2.0 ** 61
EDGE_KEYS = {
    "int64": [-2 ** 63, 2 ** 63 - 1, -1, -2, 0, 1, 2 ** 61 - 2, 2 ** 61 - 1, 2 ** 61, 2 ** 61 + 1, -(2 ** 61 - 1),
              -2 ** 61, 2 ** 62],
    "int32": [-2 ** 31, 2 ** 31 - 1, -1, -2, 0, 1],
    "uint64": [2 ** 63, 2 ** 64 - 1, 2 ** 63 - 1, 2 ** 63 + 1, 0, 1, 2 ** 61 - 1, 2 ** 61, 2 ** 61 + 1],
    "float64": [-0.0, 0.0, np.inf, -np.inf, 5e-324, -5e-324, 2.225073858507201e-308, 1e-310, np.nextafter(F61, 0),
                F61, np.nextafter(F61, np.inf), 1.0, -1.0, -2.0, 1.7976931348623157e308, -1.7976931348623157e308],
    "float32": [-0.0, 0.0, np.inf, -np.inf, 1e-45, -1e-45, 1.1754942e-38, np.nextafter(np.float32(F61), np.float32(0)),
                F61, np.nextafter(np.float32(F61), np.float32(np.inf)), 1.0, -1.0, -2.0, 3.4028235e38],
}


def _random_keys(rng, kk, n):
    if kk == "int64":
        return rng.integers(-2 ** 63, 2 ** 63 - 1, n, dtype=np.int64, endpoint=True)
    if kk == "int32":
        return rng.integers(-2 ** 31, 2 ** 31 - 1, n, dtype=np.int32, endpoint=True)
    if kk == "uint64":
        return rng.integers(0, 2 ** 64 - 1, n, dtype=np.uint64, endpoint=True)
    if kk == "float64":
        return rng.standard_normal(n) * 10.0 ** rng.integers(-300, 300, n)
    return (rng.standard_normal(n) * 10.0 ** rng.integers(-35, 35, n)).astype(np.float32)


def _values(rng, vk, op, n):
    if vk.startswith("int"):
        if op == "prod":       # |product| <= 2^(rows of the key): < 2^63 for every shape prod runs on (checked)
            v = rng.choice(np.array([-2, -1, -1, 1, 1, 2]), n)
            v[rng.random(n) < 0.01] = 0
        elif vk == "int64":
            v = rng.integers(-2 ** 40, 2 ** 40, n)
        else:
            v = rng.integers(-2 ** 31, 2 ** 31 - 1, n, endpoint=True)
    elif op == "prod":
        v = rng.uniform(0.5, 2.0, n) * rng.choice(np.array([-1.0, 1.0]), n)
    else:
        v = rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4, n)
    return v.astype(KEY_DTYPES[vk])


def _seed(*parts):
    return int.from_bytes(repr(parts).encode(), "little") % (2 ** 63)


# Colliding keys.  For keys below 2^32, slot_hash32 (dpk_common.cuh) is lo * 0xCC9E2D51 + 0x7F4A7C15 followed by
# murmur3 fmix32; both steps invert, so keys can be computed from the slot hashes they are meant to have.
def _inv32(c):
    return np.uint32(pow(c, -1, 2 ** 32))


def keys_with_slot_hash(h):
    """int64 keys in [0, 2^32) whose slot_hash32 values are the uint32 array h."""
    x = np.asarray(h, dtype=np.uint32).copy()
    x ^= x >> np.uint32(16)
    x *= _inv32(0xC2B2AE35)
    x ^= (x >> np.uint32(13)) ^ (x >> np.uint32(26))
    x *= _inv32(0x85EBCA6B)
    x ^= x >> np.uint32(16)
    return ((x - np.uint32(0x7F4A7C15)) * _inv32(0xCC9E2D51)).astype(np.int64)


def colliding_keys(count, lo_bit, hi_bit, seed, even=False):
    """count distinct keys < 2^32 whose slot_hash32 values agree in bits lo_bit..hi_bit (even keys only: hash_i64(k)
    = k for small k, so they all land in partition 0 of P = 2)."""
    rng = np.random.default_rng(seed)
    width = hi_bit - lo_bit + 1
    fixed = np.uint32(int(rng.integers(0, 1 << width)) << lo_bit)
    nfree = 32 - width
    free = np.unique(rng.integers(0, 1 << nfree, min(1 << nfree, 8 * count), dtype=np.int64))
    rng.shuffle(free)
    low = (free & ((1 << lo_bit) - 1)).astype(np.uint32)
    high = ((free >> lo_bit) << (hi_bit + 1)).astype(np.uint32)
    k = keys_with_slot_hash(low | fixed | high)
    if even:
        k = k[k % 2 == 0]
    assert len(k) >= count, "only %d keys" % len(k)
    return k[:count]


# ---------------------------------------------------------------- data shapes
class Case(object):
    def __init__(self, keys, vals, P, sub_bits, opts=None):
        self.keys, self.vals, self.P, self.sub_bits, self.opts = keys, vals, P, sub_bits, opts or {}


def shape_keys(shape, kk):
    """(keys, P, sub_bits, options) of a shape; the values come from _values per (value kind, op)."""
    rng = np.random.default_rng(_seed(shape, kk))
    if shape == "fast":
        # 2·10^5 rows, P = 3, sub_bits = 2: F = 12 first-level buckets of ~16.7 k rows; choose_sb2 takes sb2 = 4
        # (16 667 / 8 = 2083 > 2048, / 16 = 1042), so the ~192 fine buckets hold ~1042 rows each, all well below
        # AG2_CAP = 2048: the one-window path.  Three quarters of the rows have random (distinct) keys, a quarter
        # repeat 5000 pooled keys (~10 rows each).
        n = 200_000
        k = _random_keys(rng, kk, n)
        pool = _random_keys(rng, kk, 5000)
        k[: n // 4] = pool[rng.integers(0, len(pool), n // 4)]
        rng.shuffle(k)
        return k, 3, 2, {}
    if shape == "edge":
        # the edge keys of the kind, 40 rows each, among 1.3·10^5 random and pooled rows; P = 5, sub_bits = 1
        n = 130_000
        k = _random_keys(rng, kk, n)
        pool = _random_keys(rng, kk, 3000)
        k[: n // 4] = pool[rng.integers(0, len(pool), n // 4)]
        edges = np.array(EDGE_KEYS[kk], dtype=object).astype(KEY_DTYPES[kk])
        k = np.concatenate([k, np.repeat(edges, 40)])
        rng.shuffle(k)
        return k, 5, 1, {}
    if shape == "hot":
        # The general path with m = 1 (and, under agg_pipe, the big-bucket list).  3 hot keys x 10^5 rows + 2·10^5
        # rows of distinct keys = 5·10^5 rows; P = 4, sub_bits = 1: F = 8, choose_sb2 takes sb2 = 5 (62 500 / 32 =
        # 1953), so 256 fine buckets of ~780 distinct keys.  A hot key's fine bucket holds > 10^5 rows (> AG2_CAP:
        # more than one window) but ~780 distinct keys (<= AG2_CAP - AG2_MINW = 1792: every window finds room), so it
        # is merged in one pass behind its resident distinct rows.
        d = rng.integers(-2 ** 62, 2 ** 62, 200_000)
        k = np.concatenate([d, np.repeat(np.array([7, -123456789, 2 ** 40 + 3], dtype=np.int64), 100_000)])
        rng.shuffle(k)
        return k, 4, 1, {}
    if shape == "passes":
        # Hash-disjoint passes.  P = 1, sub_bits = 0, 2.7·10^6 rows over 2.65·10^6 distinct keys: choose_sb2 stops at
        # its cap sb2 = 10 (2.7·10^6 / 1024 = 2636 > 2048), so every fine bucket holds ~2590 distinct keys
        # > AG2_CAP = 2048.  No single pass can hold them; each bucket is merged in passes m >= 2.
        d = rng.permutation(2_650_000).astype(np.int64) * 2_654_435_761 - 2 ** 45
        k = np.concatenate([d, d[rng.integers(0, len(d), 50_000)]])
        rng.shuffle(k)
        return k, 1, 0, {}
    if shape == "deep":
        # Deep passes.  agg_target_rows = 3584, P = 1, sub_bits = 0: 3000 distinct keys + 500 repeated rows = 3500
        # rows <= 3584, so sb2 = 0 and all rows form one fine bucket (> AG2_CAP rows: the general path).  The keys'
        # slot_hash32 values agree in bits 12..19, the bits passes m <= 256 filter on, so each of those passes holds
        # either none or all 3000 > AG2_CAP distinct keys and fails; bit 20 (m = 512) splits them ~1500 / 1500
        # <= 1792.  Nine levels of splitting, and the result must still be exact.
        d = colliding_keys(3000, 12, 19, _seed(shape))
        k = np.concatenate([d, d[rng.integers(0, len(d), 500)]])
        rng.shuffle(k)
        return k, 1, 0, {"agg_target_rows": 3584}
    if shape == "exhausted":
        # Passes that run out of hash bits.  P = 2, sub_bits = 0: 3500 rows in partition 0 and 500 in partition 1,
        # n = 4000, choose_sb2 = 0 (2000 <= 2048): one fine bucket per partition.  Partition 0 holds 3000 even keys
        # (hash_i64(k) = k, even -> partition 0) whose slot_hash32 values agree in bits 12..27, so every pass down to
        # m = AG2_MAX_M = 2^16 holds all 3000 > AG2_CAP distinct keys: the shared-memory merge cannot complete and
        # must say so (out_counts = -1 -> NativeError).  Partition 1 holds 400 ordinary odd keys.
        d = colliding_keys(3000, 12, 27, _seed(shape), even=True)
        odd = rng.integers(0, 2 ** 40, 400) * 2 + 1
        k = np.concatenate([d, d[rng.integers(0, len(d), 500)], odd, odd[rng.integers(0, len(odd), 100)]])
        rng.shuffle(k)
        return k, 2, 0, {}
    if shape == "signed_zero":
        # keys whose values are all -0.0 (1..4 rows), mixed -0.0 / +0.0 (2..5 rows), +0.0 only, {x, -x, -0.0}
        # (cancel exactly: +0.0), and ordinary keys (1..3 rows); P = 4, sub_bits = 0
        u = _random_keys(rng, kk, 60_000)
        u = u[np.unique(_canon_bits(u), return_index=True)[1]]
        rng.shuffle(u)
        groups = [(u[:2000], 1, 4), (u[2000:4000], 2, 5), (u[4000:5000], 1, 3), (u[5000:6000], 3, 3),
                  (u[6000:36000], 1, 3)]
        ks = [np.repeat(g, rng.integers(lo, hi + 1, len(g))) for g, lo, hi in groups]
        return ks, 4, 0, {}
    raise ValueError(shape)


def _signed_zero_values(rng, ks, vk, op):
    """Values of the signed_zero shape, group by group (keys stay grouped: the shape's caller shuffles)."""
    a, b, c, d, e = ks
    va = np.full(len(a), -0.0)
    vb = rng.choice(np.array([-0.0, 0.0]), len(b))
    starts = np.flatnonzero(np.r_[True, b[1:] != b[:-1]])
    vb[starts] = -0.0                      # every mixed key has both signs: first row -0.0, last row +0.0
    vb[np.r_[starts[1:], len(b)] - 1] = 0.0
    vc = np.zeros(len(c))
    x = rng.standard_normal(len(d) // 3) * 10.0 ** rng.integers(-3, 4, len(d) // 3)
    vd = np.stack([x, -x, np.full(len(x), -0.0)], axis=1).ravel()
    ve = _values(rng, "float64", op, len(e))
    return np.concatenate([va, vb, vc, vd, ve]).astype(KEY_DTYPES[vk])


@functools.lru_cache(maxsize=4)
def make_case(shape, kk, vk, op):
    k, P, sb, opts = shape_keys(shape, kk)
    rng = np.random.default_rng(_seed(shape, kk, vk, op))
    if shape == "signed_zero":
        v = _signed_zero_values(rng, k, vk, op)
        k = np.concatenate(k)
        perm = rng.permutation(len(k))
        k, v = k[perm], v[perm]
    else:
        v = _values(rng, vk, op, len(k))
    case = Case(k, v, P, sb, opts)
    case.expect = _reference(k, v, P, op)
    return case


# ---------------------------------------------------------------- exact reference
def _canon_bits(keys):
    """Identity of a key as int64 bits, float -0.0 spelled 0.0."""
    if keys.dtype.kind == "f":
        keys = keys.copy()
        keys[keys == 0] = 0
    return _raw_bits(keys)


def _raw_bits(keys):
    if keys.dtype == np.float64 or keys.dtype == np.uint64:
        return keys.view(np.int64)
    if keys.dtype == np.float32:
        return keys.view(np.int32).astype(np.int64)
    return keys.astype(np.int64)


class Expect(object):
    pass


def _reference(keys, vals, P, op):
    bits = _canon_bits(keys)
    order = np.argsort(bits, kind="stable")
    sb, sv = bits[order], vals[order]
    starts = np.flatnonzero(np.r_[True, sb[1:] != sb[:-1]])
    nk = np.diff(np.r_[starts, len(sb)])
    ukeys = keys[order][starts]
    if ukeys.dtype.kind == "f":
        ukeys[ukeys == 0] = 0
    e = Expect()
    e.bits, e.nk, e.tol = sb[starts], nk, None
    e.part = orc.partition_vec(orc.hash_vec(ukeys), P)
    multi = np.flatnonzero(nk > 1)
    if vals.dtype.kind == "i":
        v = sv.astype(np.int64)
        if op == "prod":
            out = v[starts].copy()
            for g in multi:
                p = math.prod(v[starts[g]:starts[g] + nk[g]].tolist())
                assert -2 ** 63 <= p < 2 ** 63, "the inputs must keep every product inside int64"
                out[g] = p
        else:
            if op == "sum":
                assert np.add.reduceat(np.abs(v.astype(np.float64)), starts).max() < 2.0 ** 62
            uf = {"sum": np.add, "min": np.minimum, "max": np.maximum, "and": np.bitwise_and, "or": np.bitwise_or,
                  "xor": np.bitwise_xor}[op]
            out = uf.reduceat(v, starts)
    else:
        v = sv.astype(np.float64)
        if op == "sum":
            out = v[starts].copy()
            for g in multi:
                out[g] = math.fsum(v[starts[g]:starts[g] + nk[g]].tolist())
            negzero = np.logical_and.reduceat((v == 0) & np.signbit(v), starts)
            out[negzero] = -0.0              # math.fsum drops the sign of an all -0.0 sum
            e.tol = (nk - 1) * 2.0 ** -53 * np.add.reduceat(np.abs(v), starts)
        else:
            uf = {"min": np.minimum, "max": np.maximum, "prod": np.multiply}[op]
            out = uf.reduceat(v, starts)
    e.vals = out
    return e


def _run(case, op):
    from dpark_b200 import shuffle
    ks, vs = np.array_split(case.keys, 2), np.array_split(case.vals, 2)
    _set(case.opts)
    try:
        return shuffle.reduce_by_key([dev(x) for x in ks], [dev(x) for x in vs], case.P, op, sub_bits=case.sub_bits)
    finally:
        _set({name: DEFAULTS[name] for name in case.opts})


def _check(res, case, op):
    e = case.expect
    assert sorted(p for p, _, _ in res) == list(range(case.P))
    isfloat = case.vals.dtype.kind == "f"
    kdt = torch.from_numpy(case.keys[:1]).dtype
    for p, gk, gv in res:
        assert gk.dtype == kdt
        assert gv.dtype == (torch.float64 if isfloat else torch.int64)
        gk, gv = gk.cpu().numpy(), gv.cpu().numpy()
        sel = e.part == p
        wb, wv = e.bits[sel], e.vals[sel]
        gb = _raw_bits(gk)                     # not canonicalised: a key must come out spelled canonically
        o = np.argsort(gb, kind="stable")
        gb, gv = gb[o], gv[o]
        if not np.array_equal(gb, wb):
            pytest.fail("partition %d: %d keys, want %d; missing %s, unexpected %s" % (
                p, len(gb), len(wb), np.setdiff1d(wb, gb)[:5].tolist(), np.setdiff1d(gb, wb)[:5].tolist()))
        if not isfloat or op in ("min", "max"):
            bad = gv != wv
        elif op == "sum":
            bad = ~(np.abs(gv - wv) <= e.tol[sel])
            bad |= (gv == 0) & (wv == 0) & (np.signbit(gv) != np.signbit(wv))
        else:
            bad = ~np.isclose(gv, wv, rtol=1e-12, atol=0) | (np.signbit(gv) != np.signbit(wv))
        if bad.any():
            i = np.flatnonzero(bad)[:5]
            pytest.fail("partition %d, %s: %d of %d values differ; key bits %s got %s want %s (rows %s)" % (
                p, op, int(bad.sum()), len(bad), wb[i].tolist(), gv[i].tolist(), wv[i].tolist(),
                e.nk[sel][i].tolist()))


def _need_key_kind(kk):
    if kk == "uint64" and getattr(torch, "uint64", None) not in nv()._KEY_KIND:
        pytest.skip("this torch has no uint64 tensors")


# ---------------------------------------------------------------- the matrix
# the variant varies fastest, so that the cached input and reference of a case serve all variants in a row
@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, indirect=True)
@pytest.mark.parametrize("kk,vk,op", COMBOS)
@pytest.mark.parametrize("shape", ["fast", "edge"])
def test_merge_matches_the_exact_reference(shape, kk, vk, op, variant):
    _need_key_kind(kk)
    case = make_case(shape, kk, vk, op)
    _check(_run(case, op), case, op)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, indirect=True)
@pytest.mark.parametrize("op", FLOAT_OPS)
@pytest.mark.parametrize("vk", ["float64", "float32"])
@pytest.mark.parametrize("kk", KEY_KINDS)
def test_signed_zero_values_keep_their_sign(kk, vk, op, variant):
    """A key whose values are all -0.0 sums to -0.0 (createCombiner is the identity, DESIGN.md §7) in every variant;
    mixed +-0.0 and exactly cancelling values sum to +0.0; products of zeros carry the sign of the product."""
    _need_key_kind(kk)
    case = make_case("signed_zero", kk, vk, op)
    _check(_run(case, op), case, op)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, indirect=True)
@pytest.mark.parametrize("kk,vk,op", LARGE_COMBOS)
@pytest.mark.parametrize("shape", ["hot", "passes", "deep"])
def test_slow_paths_match_the_exact_reference(shape, kk, vk, op, variant):
    case = make_case(shape, kk, vk, op)
    _check(_run(case, op), case, op)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS, indirect=True)
@pytest.mark.parametrize("kk,vk,op", LARGE_COMBOS)
def test_a_merge_that_runs_out_of_hash_bits_raises(kk, vk, op, variant):
    """The exhausted shape: every variant returns the exact result or raises NativeError, never a short partition;
    the shared-memory merges (agg_impl 1, any agg_pipe) cannot complete it and must raise."""
    case = make_case("exhausted", kk, vk, op)
    if _shared_memory_merge(variant):
        with pytest.raises(nv().NativeError):
            _run(case, op)
    else:
        _check(_run(case, op), case, op)


@pytest.mark.gpu
def test_str_key_reduce_by_key_raises_when_a_partition_merge_failed(monkeypatch):
    """reduceByKey over str keys (strings.reduce_by_key_bytes) must surface a partition whose merge failed
    (out_counts = -1) as NativeError instead of returning it empty.  The failure is injected: a real one cannot be
    built for row-id keys at a sane size."""
    import sys
    from dpark_b200 import _native
    sys.argv = [sys.argv[0]]
    from dpark_b200 import DparkContext
    dc = DparkContext("local")
    rows = [("w%d" % (i % 97), i) for i in range(5000)]
    want = {}
    for w, i in rows:
        want[w] = want.get(w, 0) + i
    assert dict(dc.parallelize(rows, 4).reduceByKey(lambda x, y: x + y, 3).collect()) == want
    real, calls = _native.combine, []

    def failing(*a, **kw):
        ok, ov, off, cnt = real(*a, **kw)
        calls.append(cnt.numel())
        cnt[cnt.numel() - 1] = -1
        return ok, ov, off, cnt
    monkeypatch.setattr(_native, "combine", failing)
    with pytest.raises(_native.NativeError):
        dc.parallelize(rows, 4).reduceByKey(lambda x, y: x + y, 3).collect()
    assert calls


# ---------------------------------------------------------------- CPU: the shapes reach their paths
def _fine_buckets(L, keys, P, sub_bits, target=DEFAULTS["agg_target_rows"]):
    """(rows, distinct keys) per fine bucket of the reduce side, by the product's own bucket arithmetic."""
    from tests.test_host_logic import _p
    h = orc.hash_vec(keys)
    n, F = len(keys), P << sub_bits
    sb2 = _choose_sb2(n, F, target)
    b1 = np.empty(n, dtype=np.int32)
    assert L.hc_bucket(_p(h), C.c_int64(n), C.c_int32(P), C.c_int32(sub_bits), _p(b1)) == 0
    b2 = np.empty(n, dtype=np.int32)
    L.hc_fine_bucket(_p(h), C.c_int64(n), C.c_int32(sub_bits), C.c_int32(sb2), _p(b2))
    assert b2.min() >= 0 and b2.max() < (1 << sb2)
    fb = (b1.astype(np.int64) << sb2) | b2
    first = np.unique(_canon_bits(keys), return_index=True)[1]
    return np.bincount(fb, minlength=F << sb2), np.bincount(fb[first], minlength=F << sb2), fb


def _slot_hash(L, keys):
    from tests.test_host_logic import _p
    keys = np.ascontiguousarray(keys, dtype=np.int64)
    o = np.empty(len(keys), dtype=np.uint32)
    L.hc_slot_hash32(_p(keys), C.c_int64(len(keys)), _p(o))
    return o


def test_shapes_reach_the_paths_they_are_named_after():
    """The arithmetic in the shapes' comments, checked with the product's own hash and bucket functions (hostcheck)."""
    from tests.test_host_logic import _hostcheck
    L = _hostcheck()
    # the colliding-key constructor inverts slot_hash32 exactly
    rng = np.random.default_rng(1)
    want = rng.integers(0, 2 ** 32, 10000, dtype=np.int64).astype(np.uint32)
    k = keys_with_slot_hash(want)
    assert (k >= 0).all() and (k < 2 ** 32).all() and np.array_equal(_slot_hash(L, k), want)
    for kk in KEY_KINDS:
        k, P, sb, _ = shape_keys("fast", kk)
        rows, _, _ = _fine_buckets(L, k, P, sb)
        assert rows.max() <= AG2_CAP, kk
    k, P, sb, _ = shape_keys("hot", "int64")
    rows, distinct, fb = _fine_buckets(L, k, P, sb)
    hot = np.unique(fb[np.isin(k, [7, -123456789, 2 ** 40 + 3])])
    assert (rows[hot] > AG2_CAP).all() and (distinct[hot] <= AG2_CAP - AG2_MINW).all()
    assert np.delete(rows, hot).max() <= AG2_CAP
    k, P, sb, _ = shape_keys("passes", "int64")
    rows, distinct, _ = _fine_buckets(L, k, P, sb)
    assert len(rows) == 1 << AG_MAX_SB2 and distinct.min() > AG2_CAP
    k, P, sb, opts = shape_keys("deep", "int64")
    rows, distinct, _ = _fine_buckets(L, k, P, sb, opts["agg_target_rows"])
    assert len(rows) == 1 and rows[0] > AG2_CAP and distinct[0] == 3000
    s = _slot_hash(L, np.unique(k))
    assert len(np.unique((s >> 12) & 0xFF)) == 1                  # passes m <= 256 keep all keys together
    halves = np.bincount((s >> 20) & 1, minlength=2)               # m = 512 separates them
    assert halves.max() <= AG2_CAP - AG2_MINW
    k, P, sb, _ = shape_keys("exhausted", "int64")
    rows, distinct, fb = _fine_buckets(L, k, P, sb)
    part = orc.partition_vec(orc.hash_vec(k), P)
    assert len(rows) == 2 and rows[0] > AG2_CAP and distinct[0] == 3000 and (fb == part).all()
    s = _slot_hash(L, np.unique(k[part == 0]))
    assert len(np.unique((s >> 12) & (AG2_MAX_M - 1))) == 1        # bits 12..27: every pass holds all 3000 keys
    assert (k[part == 1] % 2 == 1).all()
