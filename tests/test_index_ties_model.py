"""The parallel restatement behind adb_index_sort_ref_ties (csrc/index_ties.cu), checked on the
CPU against the reference's quicksort (oracle.port(): index.c:25-46,89-101).  No GPU needed:
this is the specification of the kernels, level by level.

A Lomuto partition of [lo, hi] with pivot x = v[hi] in closed form:
  * the m = hi - lo scanned rows j = lo .. hi-1; L rows (v[j] < x) keep their order at lo ..;
  * the pivot lands at lo + nL;
  * rows >= x act as a FIFO queue.  `lead` = number of L rows before the first push.  Every
    scanned row from the first push on is an event, event index k = (j - lo) - lead: a push
    holds its own row, an L row is a rotation holding S[Lb - lead] (Lb = L rows before it);
    if there was a push, one closing rotation, event m - lead, holds S[nL - lead];
  * with R rotations, S[R + s] lands at lo + nL + 1 + s (s < Q, Q = pushes).
Segments whose keys are pairwise distinct (no K[k] == K[k-1] inside, K = sorted keys) finish
in one scatter; non-decreasing segments finish with every run of equal keys rotated right by
one.  Both are exactly what the recursion would leave."""
import numpy as np
import pytest


def _partition(v, p, lo, hi):
    x = v[hi]
    m = hi - lo
    is_l = v[lo:hi] < x
    lb = np.concatenate([[0], np.cumsum(is_l)])[:-1]        # L rows before each scanned row
    n_l = int(is_l.sum())
    q = m - n_l
    pushes = np.flatnonzero(~is_l)
    lead = int(pushes[0]) if q else m
    ev = [None] * (m - lead + 1 if q else 0)               # ("push", row) or ("rot", index)
    for r in range(lead, m):
        k = r - lead
        ev[k] = ("rot", int(lb[r]) - lead) if is_l[r] else ("push", lo + r)
    rot = n_l - lead + 1 if q else 0
    if q:
        ev[m - lead] = ("rot", n_l - lead)

    def resolve(k):
        while ev[k][0] == "rot":
            k = ev[k][1]
        return ev[k][1]

    order = [lo + r for r in range(m) if is_l[r]] + [hi] + [resolve(rot + s) for s in range(q)]
    v[lo:hi + 1], p[lo:hi + 1] = v[order].copy(), p[order].copy()
    return lo + n_l


def model_index_sort(col, small=0):
    """Level-synchronous: every live segment of a level is finished or partitioned at once."""
    n = col.size
    v, p = col.astype(np.int64).copy(), np.arange(n, dtype=np.int64)
    key = np.sort(col.astype(np.int64), kind="stable")
    dup = np.concatenate([[0], np.cumsum(key[1:] == key[:-1])])   # dup[k] = #(K[i] == K[i-1], i <= k)
    out = np.full(n, -1, dtype=np.int64)
    live = [(0, n - 1)] if n > 1 else []
    if n == 1:
        out[0] = 0
    levels = 0
    while live:
        levels += 1
        nxt = []
        for lo, hi in live:
            if dup[hi] - dup[lo] == 0:                          # pairwise distinct
                dest = lo + np.searchsorted(key[lo:hi + 1], v[lo:hi + 1], side="left")
                out[dest] = p[lo:hi + 1]
                continue
            seg = v[lo:hi + 1]
            if np.all(seg[:-1] <= seg[1:]):                      # non-decreasing
                for i in range(lo, hi + 1):
                    last = i == hi or v[i + 1] != v[i]
                    dest = lo + int(np.searchsorted(key[lo:i + 1], v[i], side="left")) if last else i + 1
                    out[dest] = p[i]
                continue
            pv = _partition(v, p, lo, hi)
            out[pv] = p[pv]
            for a, b in ((lo, pv - 1), (pv + 1, hi)):
                if b == a:
                    out[a] = p[a]
                elif b > a:
                    nxt.append((a, b))
        live = nxt
    assert (out >= 0).all()
    return key.astype(np.int32), out.astype(np.uint64), levels


def _shapes(rng, n):
    yield rng.integers(0, 2, n)
    yield rng.integers(0, 4, n)
    yield rng.integers(-5, 300, n)
    yield np.minimum(rng.zipf(1.3, n), 1000)
    yield np.sort(rng.integers(0, 10, n))
    yield np.sort(rng.integers(0, 10, n))[::-1]
    yield np.full(n, 7)
    yield rng.permutation(n)
    yield np.where(np.arange(n) % 2 == 0, np.iinfo(np.int32).min, np.iinfo(np.int32).max)


@pytest.fixture(scope="module")
def port():
    from oracle import oracle
    return oracle.port()


@pytest.mark.parametrize("seed", range(12))
def test_level_model_equals_the_quicksort(port, seed):
    rng = np.random.default_rng(seed)
    for n in (1, 2, 3, 5, 17, 64, 257):
        for col in _shapes(rng, n):
            col = np.asarray(col, dtype=np.int32)
            ev, ep = port.index_sort(col)
            mv, mp, _ = model_index_sort(col)
            assert np.array_equal(mv, ev), (n, col)
            assert np.array_equal(mp, ep), (n, col)


def test_distinct_keys_take_one_level(port):
    col = np.random.default_rng(5).permutation(1000).astype(np.int32)
    _, mp, levels = model_index_sort(col)
    assert levels == 1 and np.array_equal(mp, port.index_sort(col)[1])
