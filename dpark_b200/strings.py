"""reduceByKey over str / bytes keys (examples/wc.py's shape).

Columnar form of the keys: one uint8 buffer + int64 offsets.  On the device:

    hash_bytes     portable_hash per row (string_hash over signed chars for bytes,
                   unicode_hash over code points for str; dpark/portable_hash.pyx:17-48)
    dict_encode    representative row id per row (key identity by VALUE, like the
                   reference's dicts -- the 64-bit hash is never trusted as identity)
    partition_count + combine(DPK_K_ROWID)
                   rows are routed by their hash to the reference's partitions and
                   merged per representative id (map-side combine and reduce-side
                   merge collapse into one pass on a single GPU, because every row
                   of a key is local).

Only (representative id, combined value) pairs come back; the host decodes each
distinct key once from the byte buffer it already holds.

Under torch.distributed the rows are first routed to the rank owning their partition (dpark_b200.engine._routed_shuffle);
this module is the one-GPU stage that then runs on the owner.
"""
import numpy as np
import torch

from . import _native as nv
from . import columnar, shuffle


def _concat(splits):
    datas, offs, vals, base, rows = [], [np.zeros(1, np.int64)], [], 0, 0
    for c in splits:
        if c.n == 0:
            continue
        datas.append(c.keys)
        offs.append(c.key_offsets[1:] + base)
        base += int(c.key_offsets[-1])
        vals.append(c.vals)
        rows += c.n
    data = np.concatenate(datas) if datas else np.zeros(0, np.uint8)
    offsets = np.concatenate(offs)
    v = np.concatenate(vals) if vals else np.zeros(0, np.int64)
    return data, offsets, v, rows


def reduce_by_key_bytes(splits, key_kind, P, thresholds, op, dev, res):
    if shuffle._world() > 1:
        raise NotImplementedError("this is the one-GPU stage; under torch.distributed the rows are first routed to the "
                                  "rank owning their partition (dpark_b200.engine._routed_shuffle)")
    data, offsets, vals, n = _concat(splits)
    if n == 0:
        for p in range(P):
            res.parts[p] = ([], [])
        return res
    d_data = torch.from_numpy(data if data.size else np.zeros(1, np.uint8)).to(dev)
    d_off = torch.from_numpy(offsets).to(dev)
    d_vals = torch.from_numpy(vals).to(dev)
    key_objs = None
    if key_kind == columnar.KEY_TUPLE:       # identity = the canonical bytes; hash = tuple_hash of the leaves, on the device
        key_objs = [k for c in splits if c.n for k in c.key_objs]
        h = columnar.tuple_hashes_on_device(key_objs, dev)
    else:
        h = nv.hash_bytes(d_data, d_off, nv.STR_UTF8 if key_kind == columnar.KEY_STR else nv.BYTES_SIGNED)
    rep = nv.dict_encode(d_data, d_off, h)
    # map side: bucket-major by the hash of the string each id stands for; reduce side: merge per id
    sb = shuffle.choose_sub_bits(n, P)
    mo = shuffle.map_side([rep], [d_vals], P, thresholds, False, sb, row_hash=h, unordered=True)
    rx = shuffle.exchange(mo)
    ok, ov, off, cnt = nv.combine(rx.keys, rx.vals, op, P, rx.seg.contiguous(), rx.part_first, rx.nparts,
                                  thresholds, sb, row_hash=h)
    off_h, cnt_h = off.cpu().tolist(), cnt.cpu().tolist()
    shuffle.check_counts(cnt_h)
    ok_h, ov_h = ok.cpu().numpy(), ov.cpu().numpy()
    raw = data.tobytes()
    offs_l = offsets
    is_str = key_kind == columnar.KEY_STR
    for p in range(P):
        ids = ok_h[off_h[p]:off_h[p] + cnt_h[p]]
        keys = []
        for r in ids.tolist():
            if key_objs is not None:
                keys.append(key_objs[r])
                continue
            b = raw[offs_l[r]:offs_l[r + 1]]
            keys.append(b.decode("utf-8", "surrogatepass") if is_str else b)
        res.parts[p] = (keys, ov_h[off_h[p]:off_h[p] + cnt_h[p]].tolist())
    return res
