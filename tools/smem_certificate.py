"""Certificate of an SMEM result set without an oracle, from exact searches on the same index (fmb_search_exact).

For the SMEMs (qidx, begin, end, lb, len) of a batch, reported with min_len = 0, these checks together prove the set is complete and
exact:
  - Q[b:e] has the reported interval;
  - Q[b-1:e] (b > 0) and Q[b:e+1] (e < m) have none: every SMEM is maximal;
  - for consecutive SMEMs of a query with b2 <= e1, Q[b2-1:e1+1] has none: no occurring interval lies between two of them;
  - every query position outside all SMEMs holds a symbol that occurs nowhere (0, >= sigma, or absent from the text).
The last two imply that every occurring interval lies inside a reported one, so no SMEM is missing.  Used by tests/test_gpu_smem.py
and tools/smem_bench.py.
"""
import numpy as np


def _gather(symbols, offsets, qidx, begin, end):
    """flat symbols and offsets of the substrings Q[qidx][begin:end]"""
    lens = (end - begin).astype(np.int64)
    sub_off = np.zeros(lens.size + 1, dtype=np.uint64)
    np.cumsum(lens, out=sub_off[1:].view(np.int64))
    starts = offsets[qidx].astype(np.int64) + begin.astype(np.int64)
    idx = np.repeat(starts - sub_off[:-1].astype(np.int64), lens) + np.arange(int(sub_off[-1]), dtype=np.int64)
    return symbols[idx], sub_off


def _exact(index, symbols, offsets):
    """(lb, len) per query of fmb_search_exact (len 0: does not occur)"""
    nq = offsets.size - 1
    lb, ln = np.zeros(nq, dtype=np.uint64), np.zeros(nq, dtype=np.uint64)
    if nq == 0:
        return lb, ln
    q = index.upload(symbols, offsets)
    h = index.search_exact(q).hits()
    lb[h["qidx"].astype(np.int64)] = h["lb"]
    ln[h["qidx"].astype(np.int64)] = h["len"]
    return lb, ln


def certify(index, symbols, offsets, smems, absent_symbols=()):
    """True when `smems` (numpy SMEM records of every query, min_len = 0) passes every check; `absent_symbols`: symbols below sigma
    that do not occur in the text"""
    symbols = np.ascontiguousarray(symbols, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    sigma = index.info.sigma
    nq = offsets.size - 1
    m = (offsets[1:] - offsets[:-1]).astype(np.int64)
    q, b, e = (smems[f].astype(np.int64) for f in ("qidx", "begin", "end"))
    if q.size and (q.min() < 0 or q.max() >= nq or (b >= e).any() or (e > m[q]).any()):
        return False
    # order: by qidx, then begin; within a query starts and ends strictly increase
    same = q[1:] == q[:-1]
    if (q[1:] < q[:-1]).any() or (same & ((b[1:] <= b[:-1]) | (e[1:] <= e[:-1]))).any():
        return False
    # the reported intervals
    lb, ln = _exact(index, *_gather(symbols, offsets, q, b, e))
    if not (np.array_equal(lb, smems["lb"].astype(np.uint64)) and np.array_equal(ln, smems["len"].astype(np.uint64))):
        return False
    # maximality on both sides, and nothing occurring between consecutive SMEMs
    tests = []
    left = b > 0
    tests.append((q[left], b[left] - 1, e[left]))
    right = e < m[q]
    tests.append((q[right], b[right], e[right] + 1))
    k = np.flatnonzero(same & (b[1:] <= e[:-1]))
    tests.append((q[k], b[k + 1] - 1, e[k] + 1))
    tq, tb, te = (np.concatenate(x) for x in zip(*tests))
    _, ln = _exact(index, *_gather(symbols, offsets, tq, tb, te))
    if ln.any():
        return False
    # positions outside every SMEM hold symbols that occur nowhere
    cover = np.zeros(symbols.size + 1, dtype=np.int64)
    np.add.at(cover, offsets[q].astype(np.int64) + b, 1)
    np.add.at(cover, offsets[q].astype(np.int64) + e, -1)
    covered = np.cumsum(cover)[:-1] > 0
    lo, hi = int(offsets[0]), int(offsets[-1])
    out = symbols[lo:hi][~covered[lo:hi]]
    occurs = np.zeros(256, dtype=bool)
    occurs[1:sigma] = True
    occurs[list(absent_symbols)] = False
    return not occurs[out].any()
