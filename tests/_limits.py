"""Inputs and a reference for the tests at the int32 index limit: extents of exactly 2^31, so that index 2^31 - 1 is legal in
every dimension (the reference's IndexT is int32).

The oracle's row-wise multiply_mm allocates dense arrays of the inner and the column extent (about 36 GB at 2^31).
relabeled_mm instead maps each of the three dimensions of the product (rows of op(A), the inner index, columns of op(B))
monotonically onto 0..u-1, where u is the number of distinct indices any operand, scale vectors included, uses there; it runs
the oracle on that small problem and maps the result back.  A monotone map keeps every order and every equality the product
depends on -- which terms meet, in which order they are summed, which scale entries join -- so the values are bit-identical."""
from __future__ import annotations

import numpy as np

import _cases
from oracle.oracle import Coo

N = 1 << 31
TOP = N - 1
EDGE = np.array([0, 1, 2, N - 3, N - 2, N - 1], dtype=np.int64)


def _op_dims(M: Coo, t: str):
    """(leading, trailing) index arrays of op(M)."""
    return (M.idx[1], M.idx[0]) if t == "T" else (M.idx[0], M.idx[1])


def _relabel(M: Coo, t: str, lead_map, trail_map, lead_n, trail_n) -> Coo:
    lead, trail = _op_dims(M, t)
    a, b = np.searchsorted(lead_map, lead), np.searchsorted(trail_map, trail)
    if t == "T":
        return Coo((trail_n, lead_n), [b, a], M.val, M.sort_order)
    return Coo((lead_n, trail_n), [a, b], M.val, M.sort_order)


def _relabel_vec(v, umap, n):
    if v is None:
        return None
    return Coo((n,), [np.searchsorted(umap, v.idx[0])], v.val, v.sort_order)


def _union(*arrays):
    u = np.unique(np.concatenate([np.asarray(a, dtype=np.int64) for a in arrays if a is not None] + [np.zeros(0, np.int64)]))
    return u, max(len(u), 1)


def relabeled_mm(orc, Cst, si, A: Coo, tA, sj, B: Coo, tB, sk, policy=1, zero_nan=False, want_stats=False):
    """orc.multiply_mm on the problem with every dimension compressed to the indices in use, mapped back (see the module
    docstring).  Scale vectors must lie inside their dimension's extent, as they do here."""
    a_rows, a_in = _op_dims(A, tA)
    b_in, b_cols = _op_dims(B, tB)
    ur, nr = _union(a_rows, None if si is None else si.idx[0])
    uj, nj = _union(a_in, b_in, None if sj is None else sj.idx[0])
    uk, nk = _union(b_cols, None if sk is None else sk.idx[0])
    Ar = _relabel(A, tA, ur, uj, nr, nj)
    Br = _relabel(B, tB, uj, uk, nj, nk)
    out, st = orc.multiply_mm(Cst, _relabel_vec(si, ur, nr), Ar, tA, _relabel_vec(sj, uj, nj), Br, tB, _relabel_vec(sk, uk, nk),
                              policy, zero_nan, want_stats=True)
    shape = (A.shape[1] if tA == "T" else A.shape[0], B.shape[0] if tB == "T" else B.shape[1])
    res = Coo(shape, [ur[out.idx[0]] if out.n else out.idx[0], uk[out.idx[1]] if out.n else out.idx[1]], out.val, None)
    return (res, st) if want_stats else res


def crowded(rng, n, extreme=True, pool=None):
    """n indices in [0, 2^31): with `extreme`, half from both ends (EDGE) and half from random middles; otherwise middles only.
    `pool`: draw the middles from this many distinct values (so that rows, inner indices and columns meet)."""
    mids = rng.integers(3, N - 3, pool or n)
    x = mids[rng.integers(0, len(mids), n)]
    if extreme:
        e = rng.random(n) < 0.5
        x[e] = EDGE[rng.integers(0, len(EDGE), int(e.sum()))]
    return x.astype(np.int64)


def mm_inputs(seed, roles, row_len=None, flavour=None, b_len=8, inner_lo=None):
    """op(A) (rows x inner) and op(B) (inner x cols), extents 2^31.  `roles` names the dimensions that hold extreme indices
    ("i" rows, "j" inner, "k" columns); the others use middles only.  row_len: every row of op(A) has exactly that many
    distinct inner indices (1..8: the register merge's builds), else 1..6; rows of op(B) hold 0..b_len entries.  inner_lo: the
    inner indices lie in inner_lo .. inner_lo + 599 instead (a stretch of B short enough for a block to stage it).
    Outputs at column 2^31-1 (when "k" is a role): two rows whose terms there cancel to exactly 0 (dropped) and one whose
    terms are +inf and -inf (NaN, kept)."""
    rng = np.random.default_rng(seed)
    flavour = flavour or ["pos", "int", "mixed"][seed % 3]
    rows = np.unique(crowded(rng, 60, "i" in roles))
    if inner_lo is None:
        inner = np.unique(crowded(rng, 40, "j" in roles))
    else:   # the last index of the stretch always in use (2^31-1 for inner_lo = 2^31-600)
        inner = np.unique(np.append(inner_lo + rng.integers(0, 599, 40), inner_lo + 599))
    cols_pool = crowded(rng, 300, "k" in roles, pool=120)
    ai, aj = [], []
    for r in rows:
        ln = row_len if row_len else int(rng.integers(1, 7))
        js = rng.choice(inner, min(ln, len(inner)), replace=False)
        ai += [r] * len(js); aj += js.tolist()
    av = _cases._values(rng, len(ai), flavour)
    bj, bk = [], []
    for j in inner:
        ln = int(rng.integers(0, b_len + 1))
        ks = rng.choice(cols_pool, ln)          # repeats: duplicates that consolidate folds
        bj += [j] * ln; bk += ks.tolist()
    bv = _cases._values(rng, len(bj), flavour)
    ai, aj, av = list(ai), list(aj), list(av)
    bj, bk, bv = list(bj), list(bk), list(bv)
    if "k" in roles:
        # two fresh inner indices whose B rows are identical and hold column 2^31-1 (and a middle column)
        cand = crowded(rng, 30, "j" in roles) if inner_lo is None else inner_lo + rng.integers(0, 600, 30)
        free_j = rng.permutation(np.setdiff1d(cand, inner))[:2]
        mid_k = int(cols_pool[0])
        for j in free_j:
            bj += [int(j), int(j)]; bk += [TOP, mid_k]; bv += [3.0, 1.5]
        free_i = rng.permutation(np.setdiff1d(crowded(rng, 30, "i" in roles), rows))[:3]
        if len(free_j) == 2:
            for r, (x, y) in zip(free_i, ((2.0, -2.0), (0.25, -0.25), (np.inf, -np.inf))):
                ai += [int(r), int(r)]; aj += [int(free_j[0]), int(free_j[1])]; av += [x, y]
    A = Coo((N, N), [np.array(ai, np.int64), np.array(aj, np.int64)], np.array(av, np.float64))
    B = Coo((N, N), [np.array(bj, np.int64), np.array(bk, np.int64)], np.array(bv, np.float64))
    return A, B


def transposed(M: Coo, t: str) -> Coo:
    """The stored operand whose op(.) under transpose flag t is M."""
    return Coo((M.shape[1], M.shape[0]), [M.idx[1], M.idx[0]], M.val, None) if t == "T" else M


def scale_vector(rng, used, mode):
    """Ascending scale vector over the indices `used` (most of them present, some explicit zeros) with index 2^31-1
    handled by `mode`: "nonzero" present and non-zero, "zero" present and 0, "absent" left out."""
    u = np.unique(np.asarray(used, dtype=np.int64))
    u = u[u != TOP]
    keep = u[rng.random(len(u)) < 0.85]
    val = 0.5 + rng.random(len(keep))
    val[rng.random(len(keep)) < 0.1] = 0.0
    if mode == "nonzero":
        keep, val = np.append(keep, TOP), np.append(val, 1.75)
    elif mode == "zero":
        keep, val = np.append(keep, TOP), np.append(val, 0.0)
    return Coo((N,), [keep], val, (0,))
