"""Sub-bucketed layout (sub_bits > 0): an internal refinement of each reduce
partition.  What the reference defines must be unchanged: which keys a partition
owns, and the (map split, position) order of rows -- now per fine bucket.  -m gpu."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def nv():
    from dpark_b200 import _native
    return _native


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("P,sb", [(1, 4), (3, 2), (8, 5), (8, 7), (64, 4), (5, 9)])
def test_partition_with_sub_buckets_refines_reference_partitions(P, sb):
    rng = np.random.default_rng(P * 100 + sb)
    n = 400000
    k = rng.integers(-2 ** 63, 2 ** 63 - 1, n, dtype=np.int64)
    k[: n // 2] = rng.integers(0, 20000, n // 2)
    v = np.arange(n, dtype=np.int64)
    ok, ov, off = nv().partition(dev(k), dev(v), P, sub_bits=sb)
    ok, ov, off = ok.cpu().numpy(), ov.cpu().numpy(), off.cpu().numpy()
    S = 1 << sb
    assert len(off) == P * S + 1 and off[0] == 0 and off[-1] == n
    pid = orc.partition_vec(orc.hash_vec(k), P)
    want_off = np.zeros(P + 1, dtype=np.int64)
    want_off[1:] = np.cumsum(np.bincount(pid, minlength=P))
    assert np.array_equal(off[::S], want_off)                # partition boundaries == the reference's
    bucket_of_row = np.searchsorted(off, np.arange(n), side="right") - 1
    assert np.array_equal(bucket_of_row >> sb, orc.partition_vec(orc.hash_vec(ok), P))
    assert np.array_equal(k[ov], ok)                         # (key, value) pairs intact
    # stable inside every fine bucket: the row-index payload ascends
    brk = np.zeros(n, dtype=bool)
    brk[off[1:-1][off[1:-1] < n]] = True
    asc = (ov[1:] > ov[:-1]) | brk[1:]
    assert asc.all()
    # equal keys share one fine bucket
    order = np.argsort(ok, kind="stable")
    same = ok[order][1:] == ok[order][:-1]
    assert (bucket_of_row[order][1:][same] == bucket_of_row[order][:-1][same]).all()
    # sub-buckets of a big partition are all used and roughly balanced
    if n / (P * S) > 200:
        cnt = np.diff(off)
        assert cnt.min() > 0


@pytest.mark.parametrize("sb", [0, 3, 6])
@pytest.mark.parametrize("op", ["sum", "max"])
def test_reduce_by_key_same_result_for_any_sub_bits(sb, op):
    from dpark_b200 import shuffle
    rng = np.random.default_rng(31 + sb)
    n, P, M = 600000, 8, 3
    k = rng.integers(-40000, 40000, n, dtype=np.int64)
    k[:4] = [-1, -2, -2 ** 63, 2 ** 63 - 1]
    v = rng.integers(-2 ** 20, 2 ** 20, n, dtype=np.int64)
    ks, vs = np.array_split(k, M), np.array_split(v, M)
    res = shuffle.reduce_by_key([dev(x) for x in ks], [dev(x) for x in vs], P, op, sub_bits=sb)
    want = orc.reduce_by_key(ks, vs, P, op)
    for p, gk, gv in res:
        gk, gv = gk.cpu().numpy(), gv.cpu().numpy()
        o1, o2 = np.argsort(gk), np.argsort(want[p][0])
        assert np.array_equal(gk[o1], want[p][0][o2])
        assert np.array_equal(gv[o1], want[p][1][o2])


@pytest.mark.parametrize("impl", [0, 1, 2])
@pytest.mark.parametrize("shape", ["distinct_overflow", "hot_keys", "sentinel_key"])
def test_every_reduce_implementation_gives_the_oracle_result(impl, shape):
    """The three reduce-side implementations (dpk_set_option reduce_impl) must agree with
    the oracle, including the cases that stress implementation 2: fine buckets with more
    distinct keys than the shared-memory table holds (hash-disjoint passes), a few very hot
    keys, and the key whose bits equal the free-slot marker (INT64_MIN)."""
    from dpark_b200 import shuffle
    rng = np.random.default_rng(77)
    P, sb = 2, 0
    if shape == "distinct_overflow":
        # P = 1, one first-level bucket: the second-level split stops at its cap of 1024 fine buckets, so each holds
        # ~3e6 / 1024 = 2930 distinct keys > 2048 (AG2_CAP, the most one pass of the shared-memory merge can hold)
        P, n = 1, 3_000_000
        k = rng.permutation(n).astype(np.int64) * 7919 - 10 ** 9
    elif shape == "hot_keys":
        n = 1_000_000
        k = rng.integers(0, 5, n, dtype=np.int64)
        k[::7] = rng.integers(0, 10 ** 6, len(k[::7]))
    else:
        n = 200_000
        k = rng.integers(-100, 100, n, dtype=np.int64)
        k[::3] = -2 ** 63
    v = rng.integers(-1000, 1000, n, dtype=np.int64)
    nv().set_option("reduce_impl", impl)
    try:
        res = shuffle.reduce_by_key([dev(k)], [dev(v)], P, "sum", sub_bits=sb)
    finally:
        nv().set_option("reduce_impl", 2)
    want = orc.reduce_by_key([k], [v], P, "sum")
    for p, gk, gv in res:
        gk, gv = gk.cpu().numpy(), gv.cpu().numpy()
        o1, o2 = np.argsort(gk), np.argsort(want[p][0])
        assert np.array_equal(gk[o1], want[p][0][o2])
        assert np.array_equal(gv[o1], want[p][1][o2])


def test_reduce_with_thresholds_and_sub_buckets():
    from dpark_b200 import shuffle
    rng = np.random.default_rng(41)
    n, P = 300000, 4
    k = rng.integers(-1000, 1000, n, dtype=np.int64)
    v = np.ones(n, dtype=np.int64)
    thr = [-500, 0, 500]
    res = shuffle.reduce_by_key([dev(k)], [dev(v)], P, "sum", thresholds=thr, sub_bits=4)
    want = orc.reduce_by_key([k], [v], P, "sum", thr)
    for p, gk, gv in res:
        gk, gv = gk.cpu().numpy(), gv.cpu().numpy()
        o1, o2 = np.argsort(gk), np.argsort(want[p][0])
        assert np.array_equal(gk[o1], want[p][0][o2])
        assert np.array_equal(gv[o1], want[p][1][o2])


def test_pointer_mode_scatter_equals_plain_scatter():
    """dpk_partition_scatter_ptrs (the fused scatter + exchange entry point) with pointers that
    happen to be local: two chunks interleaved into one bucket-major buffer, bit-identical to
    the plain multi-chunk scatter."""
    from dpark_b200 import shuffle
    rng = np.random.default_rng(99)
    n, P, sb = 500000, 4, 3
    F = P << sb
    k = rng.integers(-2 ** 40, 2 ** 40, n, dtype=np.int64)
    v = np.arange(n, dtype=np.int64)
    cut = 123457
    kc = [dev(k[:cut]), dev(k[cut:])]
    vc = [dev(v[:cut]), dev(v[cut:])]
    mo = shuffle.map_side(kc, vc, P, sub_bits=sb)
    counts, wss = [], []
    for x in kc:
        c, ws = nv().partition_count(x, P, sub_bits=sb)
        counts.append(c)
        wss.append(ws)
    cm = torch.stack(counts)
    off = torch.zeros(F + 1, dtype=torch.int64, device="cuda")
    off[1:] = torch.cumsum(cm.sum(0), 0)
    base = off[:-1].unsqueeze(0) + (torch.cumsum(cm, 0) - cm)
    ok = torch.empty(n, dtype=torch.int64, device="cuda")
    ov = torch.empty(n, dtype=torch.int64, device="cuda")
    for m in range(2):
        kp = (ok.data_ptr() + base[m] * 8).contiguous()
        vp = (ov.data_ptr() + base[m] * 8).contiguous()
        nv().partition_scatter_ptrs(kc[m], vc[m], P, kp, vp, wss[m], sub_bits=sb)
    assert torch.equal(ok, mo.keys) and torch.equal(ov, mo.vals) and torch.equal(off, mo.offsets)


@pytest.mark.parametrize("threads", [512, 1024])
@pytest.mark.parametrize("kinds", [("int64", "int64"), ("int32", "float32"), ("int64", None)])
def test_pointer_mode_bulk_scatter_unordered(kinds, threads):
    """The fused scatter + exchange for unordered multisplits (reduceByKey map side): k_part_scatter_bulk in pointer
    mode -- bucket runs leave through the TMA to per-bucket absolute addresses.  With local addresses of buckets laid
    out in a PERMUTED order (as in a peer's receive buffer, where a bucket's slot has nothing to do with its number)
    every bucket must hold exactly the rows the plain multisplit puts there, as a multiset of (key, value) pairs."""
    rng = np.random.default_rng(7)
    n, P, sb = 700001, 8, 5
    F = P << sb
    kdt, vdt = kinds
    k = rng.integers(-2 ** 30, 2 ** 30, n).astype(kdt)
    v = None if vdt is None else (np.arange(n).astype(vdt))
    dk, dv = dev(k), (None if v is None else dev(v))
    nv().set_option("scatter_ptr_threads", threads)
    try:
        pk, pv, off = nv().partition(dk, dv, P, sub_bits=sb, unordered=True)
        counts, ws = nv().partition_count(dk, P, sub_bits=sb, unordered=True)
        assert torch.equal(counts, off[1:] - off[:-1])
        perm = torch.from_numpy(rng.permutation(F)).cuda()
        # bucket b's slot: buckets laid out in perm order, 3 pad rows between slots (odd alignment phases)
        c_perm = counts[perm]
        start_perm = torch.cumsum(c_perm + 3, 0) - (c_perm + 3)
        start = torch.empty(F, dtype=torch.int64, device="cuda")
        start[perm] = start_perm
        total = int((c_perm + 3).sum().item())
        ok = torch.zeros(total, dtype=dk.dtype, device="cuda")
        ov = None if dv is None else torch.zeros(total, dtype=dv.dtype, device="cuda")
        kp = (ok.data_ptr() + start * ok.element_size()).contiguous()
        vp = None if dv is None else (ov.data_ptr() + start * ov.element_size()).contiguous()
        nv().partition_scatter_ptrs(dk, dv, P, kp, vp, ws, sub_bits=sb, unordered=True)
        torch.cuda.synchronize()
    finally:
        nv().set_option("scatter_ptr_threads", 1024)
    okh, pkh = ok.cpu().numpy(), pk.cpu().numpy()
    ovh, pvh = (None, None) if dv is None else (ov.cpu().numpy(), pv.cpu().numpy())
    offh, sth, ch = off.cpu().numpy(), start.cpu().numpy(), counts.cpu().numpy()
    for b in range(F):
        got_k = okh[sth[b]:sth[b] + ch[b]]
        want_k = pkh[offh[b]:offh[b + 1]]
        if dv is None:
            assert np.array_equal(np.sort(got_k), np.sort(want_k)), b
        else:
            got = np.stack([got_k.astype(np.int64), ovh[sth[b]:sth[b] + ch[b]].astype(np.int64)])
            want = np.stack([want_k.astype(np.int64), pvh[offh[b]:offh[b + 1]].astype(np.int64)])
            assert np.array_equal(got[:, np.lexsort(got)], want[:, np.lexsort(want)]), b
        assert not okh[sth[b] + ch[b]:sth[b] + ch[b] + 3].any(), "pad rows behind bucket %d were written" % b


def test_fused_plan_matches_the_push_layout_and_diverts_overflow():
    """dpk_fused_plan: slot of (source rank, bucket) in the owner's receive buffer = source-rank-major, bucket-major
    (what exchange_push delivers); a bucket that would end past the capacity goes to the dump columns."""
    rng = np.random.default_rng(3)
    G, P, sb = 4, 6, 2           # 6 partitions on 4 ranks: blocks of 2, the last rank owns none
    F = P << sb
    per_block = ((P + G - 1) // G) << sb
    counts = rng.integers(0, 50, (G, F)).astype(np.int64)
    allc = dev(counts)
    base = np.arange(1, 2 * G + 1, dtype=np.int64) * (1 << 30)       # fake receive-buffer addresses [2][G]
    dump_k = torch.empty(int(counts.sum()), dtype=torch.int64, device="cuda")
    dump_v = torch.empty(int(counts.sum()), dtype=torch.float32, device="cuda")
    for cap in (1 << 20, 300):
        for rank in range(G):
            err = torch.zeros(1, dtype=torch.int64, device="cuda")
            kp, vp, seg = nv().fused_plan(allc, G, per_block, rank, dev(base), 8, 4, cap, dump_k, dump_v, err)
            kp, vp, seg = kp.cpu().numpy(), vp.cpu().numpy(), seg.cpu().numpy()
            b0, b1 = min(F, rank * per_block), min(F, (rank + 1) * per_block)
            assert np.array_equal(seg, counts[:, b0:b1])
            over = 0
            for d in range(G):
                lo, hi = min(F, d * per_block), min(F, (d + 1) * per_block)
                first = counts[:rank, lo:hi].sum()
                over = max(over, counts[:, lo:hi].sum() - cap)
                run = 0
                for b in range(lo, hi):
                    local = counts[rank, :b].sum()
                    if first + run + counts[rank, b] <= cap:
                        assert kp[b] == base[d] + (first + run) * 8 and vp[b] == base[G + d] + (first + run) * 4
                    else:
                        assert kp[b] == dump_k.data_ptr() + local * 8 and vp[b] == dump_v.data_ptr() + local * 4
                    run += counts[rank, b]
            assert int(err.item()) == max(0, over)


@pytest.mark.parametrize("H,Q", [(1, 1), (2, 2), (3, 4)])
def test_push_plan_parts_tile_the_blocks(H, Q):
    """dpk_push_plan_part: pushing every destination's block in Q parts into Q regions of the receive buffers, from H
    groups per rank, must (a) cover every row of the map output exactly once, (b) land each part's rows
    (rank, group)-major then bucket-major inside its region -- the layout dpk_combine reads with the part's seg matrix."""
    rng = np.random.default_rng(17)
    G, P, sb = 4, 16, 3
    F = P << sb
    per_parts = P // G
    per_block = per_parts << sb
    part_blk = (per_parts // Q) << sb
    S = G * H
    counts = rng.integers(0, 40, (S, F)).astype(np.int64)
    allc = dev(counts)
    region = 5000
    base = (np.arange(1, 2 * G + 1, dtype=np.int64) << 32)          # fake receive-buffer addresses [2][G]
    for rank in range(G):
        for h in range(H):
            my = rank * H + h
            n_mine = int(counts[my].sum())
            out_k = torch.empty(max(n_mine, 1), dtype=torch.int64, device="cuda")
            out_v = torch.empty(max(n_mine, 1), dtype=torch.float32, device="cuda")
            covered = 0
            for q in range(Q):
                err = torch.zeros(1, dtype=torch.int64, device="cuda")
                src, dst, nby, seg = nv().push_plan(allc, G, per_block, my, rank, out_k, out_v, dev(base), region, err,
                                                    part=(q * part_blk, (q + 1) * part_blk), dst_row0=q * region)
                src, dst, nby, seg = src.cpu().numpy(), dst.cpu().numpy(), nby.cpu().numpy(), seg.cpu().numpy()
                assert int(err.item()) == 0
                lo_r, hi_r = rank * per_block + q * part_blk, rank * per_block + (q + 1) * part_blk
                assert np.array_equal(seg, counts[:, lo_r:hi_r])
                for d in range(G):
                    lo, hi = d * per_block + q * part_blk, d * per_block + (q + 1) * part_blk
                    rows = counts[my, lo:hi].sum()
                    first_src = counts[my, :lo].sum()
                    first_dst = counts[:my, lo:hi].sum()
                    assert nby[d] == rows * 8 and nby[G + d] == rows * 4
                    assert src[d] == out_k.data_ptr() + first_src * 8 and src[G + d] == out_v.data_ptr() + first_src * 4
                    assert dst[d] == base[d] + (q * region + first_dst) * 8
                    assert dst[G + d] == base[G + d] + (q * region + first_dst) * 4
                    covered += rows
            assert covered == n_mine
    # a region that is too small: clamped, and reported
    err = torch.zeros(1, dtype=torch.int64, device="cuda")
    out_k = torch.empty(int(counts[0].sum()), dtype=torch.int64, device="cuda")
    src, dst, nby, _ = nv().push_plan(allc, G, per_block, S - 1, G - 1, out_k, None, dev(base[:G]), 100, err,
                                      part=(0, part_blk), dst_row0=0)
    need = max(counts[:, d * per_block:d * per_block + part_blk].sum() for d in range(G))
    assert int(err.item()) == need - 100
    for d in range(G):
        first_dst = counts[:S - 1, d * per_block:d * per_block + part_blk].sum()
        assert nby.cpu().numpy()[d] == 8 * max(0, min(counts[S - 1, d * per_block:d * per_block + part_blk].sum(), 100 - first_dst))


@pytest.mark.parametrize("H,Q,kdt,vdt", [(1, 1, torch.int64, torch.int64), (2, 2, torch.int64, torch.int64),
                                         (3, 4, torch.int32, torch.float32), (2, 2, torch.int64, None)])
def test_pipe_plan_layout(H, Q, kdt, vdt):
    """dpk_pipe_plan: the padded send layout (bucket_base) and the Q push tables of one group.  Blocks follow each other
    in (destination, part) order, buckets inside a block are dense, every push is congruent mod 16 bytes to its landing
    place, lands (rank, group)-major inside region q, and the pads fit the promised spare rows."""
    rng = np.random.default_rng(23)
    G, P, sb = 4, 16, 2
    F = P << sb
    per_block = (P // G) << sb
    part_blk = per_block // Q
    S = G * H
    counts = rng.integers(0, 60, (S, F)).astype(np.int64)
    allc = dev(counts)
    region = 4096
    ksz = torch.empty(0, dtype=kdt).element_size()
    vsz = None if vdt is None else torch.empty(0, dtype=vdt).element_size()
    A = 16 // min(ksz, vsz or ksz)
    pad = nv().pipe_pad_rows(G, Q, ksz, vsz)
    ncols = 1 if vdt is None else 2
    base_addr = (np.arange(1, ncols * G + 1, dtype=np.int64) << 32)
    for rank in (0, G - 1):
        for h in range(H):
            my = rank * H + h
            n_mine = int(counts[my].sum())
            out_k = torch.empty(n_mine + pad, dtype=kdt, device="cuda")
            out_v = None if vdt is None else torch.empty(n_mine + pad, dtype=vdt, device="cuda")
            err = torch.zeros(1, dtype=torch.int64, device="cuda")
            bb, src, dst, nby, seg = nv().pipe_plan(allc, G, per_block, Q, region, my, rank, out_k, out_v, dev(base_addr), err)
            bb, src, dst, nby, seg = (t.cpu().numpy() for t in (bb, src, dst, nby, seg))
            assert int(err.item()) == 0
            pos = 0
            for d in range(G):
                for q in range(Q):
                    lo, hi = d * per_block + q * part_blk, d * per_block + (q + 1) * part_blk
                    first_dst = counts[:my, lo:hi].sum()
                    landing = q * region + first_dst
                    start = bb[lo]
                    assert pos <= start < pos + A and (start - landing) % A == 0
                    assert np.array_equal(bb[lo:hi], start + np.cumsum(counts[my, lo:hi]) - counts[my, lo:hi])
                    rows = counts[my, lo:hi].sum()
                    assert nby[q, d] == rows * ksz and src[q, d] == out_k.data_ptr() + start * ksz
                    assert dst[q, d] == base_addr[d] + landing * ksz and (src[q, d] - dst[q, d]) % 16 == 0
                    if vdt is not None:
                        assert nby[q, G + d] == rows * vsz and src[q, G + d] == out_v.data_ptr() + start * vsz
                        assert dst[q, G + d] == base_addr[G + d] + landing * vsz and (src[q, G + d] - dst[q, G + d]) % 16 == 0
                    pos = start + rows
            assert pos <= n_mine + pad
            for q in range(Q):
                lo = rank * per_block + q * part_blk
                assert np.array_equal(seg[q], counts[:, lo:lo + part_blk])


@pytest.mark.parametrize("tma", [0, 1])
def test_copy_segments_on_a_few_sms(tma):
    """dpk_copy_segments restricted to whole SMs (the overlapped pushes): the TMA ring (congruent segments: head / aligned
    middle / tail; incongruent ones by loads and stores) and the load/store form must both copy exactly the bytes of
    every segment and nothing else."""
    rng = np.random.default_rng(31 + tma)
    sizes = [0, 1, 8, 15, 16, 17, 4096, 32768, 32769, 65536 + 24, 300000, 1 << 20]
    src = torch.from_numpy(rng.integers(0, 256, 8 << 20, dtype=np.uint8)).cuda()
    dst = torch.zeros(8 << 20, dtype=torch.uint8, device="cuda")
    want = np.zeros(8 << 20, dtype=np.uint8)
    srch = src.cpu().numpy()
    so, do, nb = [], [], []
    s_at, d_at = 5, 64
    for i, n in enumerate(sizes * 2):
        s_off = s_at + (i * 7) % 16              # every alignment of the source ...
        d_off = d_at + ((s_off - d_at) % 16 if i < len(sizes) else (i * 3) % 16)   # ... congruent first, arbitrary after
        so.append(src.data_ptr() + s_off)
        do.append(dst.data_ptr() + d_off)
        nb.append(n)
        want[d_off:d_off + n] = srch[s_off:s_off + n]
        s_at = s_off + n + 40
        d_at = d_off + n + 40
    nv().set_option("copy_tma", tma)
    try:
        nv().copy_segments(dev(np.array(so, dtype=np.int64)), dev(np.array(do, dtype=np.int64)), dev(np.array(nb, dtype=np.int64)), sms=3)
        torch.cuda.synchronize()
    finally:
        nv().set_option("copy_tma", 1)
    assert np.array_equal(dst.cpu().numpy(), want)


def test_choose_sub_bits_bounds():
    from dpark_b200 import shuffle
    assert shuffle.choose_sub_bits(1000, 8) == 0
    assert shuffle.choose_sub_bits(10 ** 8, 8) == 5
    for n in (10 ** 6, 10 ** 8, 10 ** 9, 4 * 10 ** 9):
        for P in (1, 4, 8, 64, 1000, 4096):
            sb = shuffle.choose_sub_bits(n, P)
            assert (P << sb) <= max(P, 1024)


@pytest.mark.parametrize("wide", [0, 1])
@pytest.mark.parametrize("op", ["sum", "min", "max"])
@pytest.mark.parametrize("vkind", ["i64", "f64"])
def test_slot_claim_variants_agree_with_the_oracle(wide, op, vkind):
    """dpk_set_option("agg_wide"): claiming a shared-memory slot and depositing the first value with one
    128-bit CAS (1) or with a 64-bit key CAS followed by an atomic on the accumulator (0) must both give
    the reference's createCombiner/mergeValue result (dpark/rdd.py:303-327) for every op and value kind,
    with negative values (high half of the 64-bit add) and mostly-distinct as well as repeated keys.
    The switch belongs to the round-1 kernel k_smem_aggregate, which runs only with agg_impl = 0."""
    from dpark_b200 import shuffle
    rng = np.random.default_rng(5 + wide)
    n, P = 700_000, 3
    k = rng.integers(-2 ** 40, 2 ** 40, n, dtype=np.int64)
    k[: n // 4] = rng.integers(0, 300, n // 4)
    if vkind == "i64":
        v = rng.integers(-2 ** 40, 2 ** 40, n, dtype=np.int64)
    else:
        v = rng.standard_normal(n) * 1e6
    nv().set_option("agg_impl", 0)
    nv().set_option("agg_wide", wide)
    try:
        res = shuffle.reduce_by_key([dev(k[: n // 2]), dev(k[n // 2:])], [dev(v[: n // 2]), dev(v[n // 2:])], P, op)
    finally:
        nv().set_option("agg_wide", 1)
        nv().set_option("agg_impl", 1)
    want = orc.reduce_by_key([k[: n // 2], k[n // 2:]], [v[: n // 2], v[n // 2:]], P, op)
    for p, gk, gv in res:
        gk, gv = gk.cpu().numpy(), gv.cpu().numpy()
        o1, o2 = np.argsort(gk), np.argsort(want[p][0])
        assert np.array_equal(gk[o1], want[p][0][o2])
        if vkind == "i64" or op != "sum":
            assert np.array_equal(gv[o1], want[p][1][o2])
        else:   # float sums: accumulation order differs; tolerance 1e-9 * sum|v| (DESIGN.md §7)
            assert np.allclose(gv[o1], want[p][1][o2], rtol=0, atol=1e-9 * np.abs(v).sum())


@pytest.mark.parametrize("unordered", [False, True])
def test_consecutive_slices_are_partitioned_in_one_launch_with_the_same_result(unordered):
    """Map splits that are consecutive slices of one buffer take ONE count + scatter launch pair (shuffle._as_one);
    the bucket-major output must equal the per-split path's: bit-identical when stable, the same rows per bucket when
    the order inside a bucket is free."""
    from dpark_b200 import shuffle
    rng = np.random.default_rng(3)
    n, P, sb, M = 300_001, 6, 3, 5
    k = torch.from_numpy(rng.integers(-10 ** 6, 10 ** 6, n, dtype=np.int64)).cuda()
    v = torch.arange(n, dtype=torch.int64, device="cuda")
    per = -(-n // M)
    kc = [k[i * per:min(n, (i + 1) * per)] for i in range(M)]
    vc = [v[i * per:min(n, (i + 1) * per)] for i in range(M)]
    assert shuffle._as_one(kc) is not None
    before = nv().launch_count()
    one = shuffle.map_side(kc, vc, P, None, False, sb, unordered=unordered)
    launches_one = nv().launch_count() - before
    sep = shuffle.map_side([c.clone() for c in kc], [c.clone() for c in vc], P, None, False, sb, unordered=unordered)
    assert launches_one <= 4 and torch.equal(one.offsets, sep.offsets)
    if not unordered:
        assert torch.equal(one.keys, sep.keys) and torch.equal(one.vals, sep.vals)
    else:
        off = one.offsets.cpu().tolist()
        for b in range(P << sb):
            a, e = off[b], off[b + 1]
            assert torch.equal(one.vals[a:e].sort().values, sep.vals[a:e].sort().values)
            assert torch.equal(one.keys[a:e], k[one.vals[a:e]])
