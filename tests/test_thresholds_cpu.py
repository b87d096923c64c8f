"""The multiply threshold cases (tests/_thresholds.py) checked without a GPU: every row sits where its builder says it
does, and the values make the order of summation visible."""
import math

import numpy as np
import pytest

import _thresholds as T

CASES = T.all_cases()


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_rows_sit_on_their_thresholds(case):
    an = T.analyse(case)
    # the bins the code's rules give, recounted from the arrays, are the builder's
    assert an["bins"] == [tuple(r) for r in case["rows"]]
    for r, what, value, thr in case["claims"]:
        got = {"entries": an["entries"], "products": an["products"], "outputs": an["outputs"], "words": an["words"]}[what][r]
        assert got == value and abs(value - thr) <= 1, (r, what, got, value, thr)


def test_every_threshold_is_met_from_both_sides():
    seen = {}
    for c in CASES:
        for _, what, value, thr in c["claims"]:
            seen.setdefault((what, thr), set()).add(value - thr)
    for key in [("entries", T.MERGE_MAX_LISTS), ("products", T.MERGE_MAX_PRODUCTS), ("products", T.HASH_MIN_PRODUCTS),
                ("products", T.HSM_CAP), ("words", T.HS_LIST_CAP), ("outputs", 16)] + \
               [("outputs", cap) for cap in T.HASH_CAP.values()] + [("outputs", 2 * cap) for cap in T.HASH_CAP.values()]:
        # (the 8-entry limit and 2 CAP outputs: on it and above it)
        two_sided = key != ("entries", T.MERGE_MAX_LISTS) and key[1] not in [2 * c for c in T.HASH_CAP.values()]
        assert seen.get(key, set()) >= ({-1, 0, 1} if two_sided else {0, 1}), key
    widths = {c["B"].shape[1] for c in CASES}
    assert {T.HASH_MAX_COLS, T.HASH_MAX_COLS + 1, 2 * T.HASH_MAX_COLS + 1} <= widths


def test_hash_step_cases_take_both_step_kinds():
    for v in T.HASH_NT:
        traces = {s: T.hash_trace(next(c for c in CASES if c["name"] == f"hash_steps_v{v}_{s}"), v) for s in (31, 32, 33, 0)}
        assert traces[31]["piped"] == traces[32]["piped"] == 0 and traces[31]["barriers"] > 0 and traces[32]["barriers"] > 0
        assert traces[33]["piped"] == traces[33]["steps"] > 0 and traces[0]["piped"] > 0


def test_panel_cuts_around_a_row_start():
    """Two panels whose chunk is the first product of row PANEL_CUT_ROW minus 1, exactly, or plus 1: the cut lands on that
    row, on it, and on the next row."""
    for delta, cut in ((-2, T.PANEL_CUT_ROW), (0, T.PANEL_CUT_ROW), (1, T.PANEL_CUT_ROW + 1)):
        case = next(c for c in CASES if c["name"] == f"panels_{delta}")
        prod = T.analyse(case, columns=False)["products"]
        S, F = int(prod[:T.PANEL_CUT_ROW].sum()), int(prod.sum())
        assert F == 2 * S + delta and -(-F // 2) == S + {-2: -1, 0: 0, 1: 1}[delta]
        for mp in (-(-F // 2), F - 1):
            assert T.panel_rows(prod, mp) == [0, cut], (delta, mp)


@pytest.mark.parametrize("offset", [0, 1])
def test_esc_chunk_cases_reach_the_chunk_at_a_row_end(offset):
    case = T.esc_chunk(offset)
    an = T.analyse(case, columns=False)
    bins = [b for b, _ in an["bins"]]
    assert bins == [b for b, _ in case["rows"]]
    esc = np.where(np.array(bins) == "esc", an["products"], 0)
    prefix = np.cumsum(esc)
    r = T.ESC_BOUNDARY_ROW
    assert prefix[r] == T.ESC_CHUNK + offset and prefix[r - 1] < T.ESC_CHUNK and prefix[-1] < 2 * T.ESC_CHUNK
    assert an["products"][r] == 510 + offset and max(esc) < T.HASH_MIN_PRODUCTS


def _terms(case):
    """Every product of the case as (output number, term), in ascending j within each output, and the output keys."""
    A, B = case["A"], case["B"]
    m, nj = A.shape
    si_d, _ = T._dense(case["si"], m)
    sj_d, sj_on = T._dense(case["sj"], nj)
    sk_d, _ = T._dense(case["sk"], B.shape[1])
    if case["si"] is None:
        si_d[:] = 1.0
    if case["sj"] is None:
        sj_on[:] = True
        sj_d[:] = 1.0
    if case["sk"] is None:
        sk_d[:] = 1.0
    bo = np.lexsort((B.idx[1], B.idx[0]))
    bj, bk, bv = B.idx[0][bo].astype(np.int64), B.idx[1][bo].astype(np.int64), B.val[bo]
    bptr = np.searchsorted(bj, np.arange(nj + 1))
    keep = sj_on[A.idx[1]] & (si_d[A.idx[0]] != 0)
    ai, aj = A.idx[0][keep].astype(np.int64), A.idx[1][keep].astype(np.int64)
    asv = A.val[keep] * (sj_d[aj] if case["sj"] is not None else 1.0)   # (a*s) first
    cnt = bptr[aj + 1] - bptr[aj]
    e = np.repeat(np.arange(len(ai)), cnt)
    pos = np.arange(len(e)) - np.repeat(np.cumsum(cnt) - cnt, cnt) + bptr[aj][e]
    i, j, k, t = ai[e], aj[e], bk[pos], asv[e] * bv[pos]
    keep = sk_d[k] != 0
    i, j, k, t = i[keep], j[keep], k[keep], t[keep]
    o = np.lexsort((j, k, i))
    i, k, t = i[o], k[o], t[o]
    first = np.concatenate([[True], (i[1:] != i[:-1]) | (k[1:] != k[:-1])])
    grp = np.cumsum(first) - 1
    return grp, t, i[first], k[first], si_d, sk_d


def _ordered_sum(grp, t, n, reverse=False):
    """Sums from 0, one term after the other (ascending position in the group, or descending)."""
    start = np.flatnonzero(np.concatenate([[True], grp[1:] != grp[:-1]]))
    size = np.diff(np.concatenate([start, [len(grp)]]))
    acc = np.zeros(n)
    for p in range(int(size.max()) if len(size) else 0):
        live = size > p
        idx = start[live] + (size[live] - 1 - p if reverse else p)
        acc[live] = acc[live] + t[idx]
    return acc, size


# cases whose outputs cannot show a summation order, and why
NO_ORDER = {
    "nl1_shortB": "rows of one entry: one term per output",
    "nl1_longB": "rows of one entry: one term per output",
    "nl2_shortB": "rows of at most two entries: two terms commute",
    "nl2_longB": "rows of at most two entries: two terms commute",
    "onepass_pass": "rows of two entries, so that the one-pass merge takes them",
    "small_8191_distinct": "all-distinct columns by construction",
    "small_8192_distinct": "all-distinct columns by construction",
    "small_8193_distinct": "all-distinct columns by construction",
}


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_values_are_order_sensitive(orc, case):
    grp, t, oi, ok, si_d, sk_d = _terms(case)
    n = len(oi)
    fwd, size = _ordered_sum(grp, t, n)
    rev, _ = _ordered_sum(grp, t, n, reverse=True)
    # the oracle forms every sum in ascending j from 0: its product is exactly the forward sums that are not 0
    want = orc.multiply_mm(case["C"], case["si"], case["A"], ".", case["sj"], case["B"], ".", case["sk"])
    live = fwd != 0
    assert np.array_equal(want.idx[0], oi[live]) and np.array_equal(want.idx[1], ok[live])
    scaled = fwd[live] * case["C"] * si_d[oi[live]] * sk_d[ok[live]]
    assert np.array_equal(want.val.view(np.uint64), scaled.view(np.uint64))
    # and lies within n eps sum|t| of the exact sum
    start = np.flatnonzero(np.concatenate([[True], grp[1:] != grp[:-1]]))
    mag = np.add.reduceat(np.abs(t), start) if n else np.zeros(0)
    for g in range(0, n, max(1, n // 2000)):
        exact = math.fsum(t[start[g]:start[g] + size[g]])
        assert abs(fwd[g] - exact) <= size[g] * 2.0 ** -52 * mag[g], (case["name"], g)
    # reversed order changes the bits of many outputs: of those with four or more terms at least 30 %, of those with three
    # (where only the first two terms trade places with the last) at least 15 %; two terms commute exactly
    # -- every case but those listed in NO_ORDER has such outputs
    if case["name"] in NO_ORDER:
        return
    long_sums = size >= 32   # (a few outputs of hundreds of terms suffice: most of them must change)
    assert np.count_nonzero(size >= 3) >= 8 or np.count_nonzero(long_sums) >= 1, case["name"]
    if np.count_nonzero(long_sums):
        assert np.count_nonzero(fwd[long_sums] != rev[long_sums]) >= 0.5 * np.count_nonzero(long_sums), case["name"]
    for least, share in ((4, 0.3), (3, 0.15)):
        multi = size >= least
        if np.count_nonzero(multi) >= 8:
            differ = np.count_nonzero(fwd[multi] != rev[multi]) / np.count_nonzero(multi)
            assert differ >= share, (case["name"], least, differ)
