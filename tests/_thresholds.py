"""Multiply inputs whose rows sit exactly on, one below and one above the thresholds at which multiply changes bin,
kernel build or branch (spgemm.cuh, multiply_core in spb_api.cu).

Every builder returns a case dict: the operands (oracle Coo, A is m x nj, B is nj x n_cols, both untransposed), the
scale vectors, and what the code is expected to do with them:
  rows      per A row: the bin it must land in ('merge', 'esc', 'hash', 'skip') and, for hash rows, whether the
            shared-memory sort lists its columns ('small') -- written down by the builder from its construction;
  claims    (row, quantity, value, threshold): the row's entries / products / outputs / 32-column words, which must equal
            value, and value sits on the threshold or one away from it;
  expect    the bin totals the library reports in spb_mm_stats.
tests/test_thresholds_cpu.py recounts all of it from the arrays with numpy; tests/test_gpu_multiply_thresholds.py runs it.

Values are order-sensitive: N(0,1) * 2^U(-E, E), never small integers, so that adding an output's terms in another order
than ascending j changes the bits of most outputs with three or more terms.  The exception is a cancelling pair: two B
rows with the same columns and values under A values +a and -a, whose outputs sum to exactly 0 (the reference drops them).
"""
from __future__ import annotations

import numpy as np

from oracle.oracle import Coo

# thresholds, as the library has them
MERGE_MAX_LISTS = 8         # spgemm.cuh: longest row the register merge takes
MERGE_MAX_PRODUCTS = 1024   # SPB_MERGE_MAX_PRODUCTS default (count_row: f > max_products -> ESC)
HASH_MIN_PRODUCTS = 512     # SPB_HASH_MIN_PRODUCTS default (k_esc_row_products: f >= -> hash)
HASH_MAX_COLS = 1572864     # bitmap columns (one column window)
HSM_CAP = 8192              # products of a row the shared-memory sort takes (wide matrices only)
HS_LIST_CAP = 4608          # non-zero bitmap words of a unit the sparse walk takes
ESC_CHUNK = 1 << 27         # SPB_ESC_CHUNK default
HASH_CAP = {2: 2560, 1: 5120, 0: 10240}   # outputs per hash numeric work item, by SPB_HASH_VARIANT
HASH_NT = {2: 256, 1: 512, 0: 1024}       # threads of the hash numeric kernel (products per step)
EXP = 3


def values(rng, n):
    return rng.standard_normal(n) * np.exp2(rng.uniform(-EXP, EXP, n))


class Build:
    """Rows of A and B written one by one.  brow() adds a row j of B (its columns), arow() a row of A (its inner indices)."""

    def __init__(self, seed, n_cols):
        self.rng = np.random.default_rng(seed)
        self.n_cols = int(n_cols)
        self.bcols, self.bvals = [], []
        self.arows = []          # (js, a values or None)
        self.bins, self.small, self.claims = [], [], []

    def brow(self, cols, vals=None):
        cols = np.asarray(cols, np.int64)
        assert len(np.unique(cols)) == len(cols) and (len(cols) == 0 or (cols.min() >= 0 and cols.max() < self.n_cols))
        order = np.argsort(cols)
        v = values(self.rng, len(cols)) if vals is None else np.asarray(vals, np.float64)
        self.bcols.append(cols[order]); self.bvals.append(v[order])
        return len(self.bcols) - 1

    def pair(self, cols):
        """Two B rows with the same columns and values (a cancelling pair under A values +a, -a)."""
        v = values(self.rng, len(cols))
        return self.brow(cols, v), self.brow(cols, v.copy())

    def arow(self, js, bin, small=False, avals=None, claim=None):
        assert len(set(js)) == len(js)
        self.arows.append((list(js), avals))
        self.bins.append(bin); self.small.append(bool(small))
        if claim is not None:
            self.claims.append((len(self.arows) - 1,) + tuple(claim))
        return len(self.arows) - 1

    def plen(self, js, masked=()):
        return int(sum(len(self.bcols[j]) for j in js if j not in masked))

    def finish(self, name, C=1.0, si=None, sj=None, sk=None, **extra):
        m, nj = len(self.arows), len(self.bcols)
        ai = np.concatenate([np.full(len(js), i) for i, (js, _) in enumerate(self.arows)]).astype(np.int32)
        aj = np.concatenate([js for js, _ in self.arows]).astype(np.int32)
        av = np.concatenate([values(self.rng, len(js)) if a is None else np.asarray(a, np.float64) for js, a in self.arows])
        bj = np.concatenate([np.full(len(c), j) for j, c in enumerate(self.bcols)]).astype(np.int32)
        bk = np.concatenate(self.bcols).astype(np.int32)
        bv = np.concatenate(self.bvals)
        case = dict(name=name, C=C, si=si, sj=sj, sk=sk, A=Coo((m, nj), [ai, aj], av), B=Coo((nj, self.n_cols), [bj, bk], bv),
                    rows=list(zip(self.bins, self.small)), claims=list(self.claims), env={}, ctx_env={})
        case.update(extra)
        case["expect"] = _expect(case)
        return case


def _expect(case):
    """Bin totals from the builder's per-row bins; products from the construction (masked j and si-zero rows form none)."""
    an = analyse(case, columns=False)
    e = dict(merge=0, esc=0, hash=0, small=0, products_hash=0, products_esc=0)
    for r, (b, small) in enumerate(case["rows"]):
        if b in ("merge", "esc", "hash"):
            e[b] += 1
        if b == "hash":
            e["products_hash"] += int(an["products"][r]); e["small"] += small
        if b == "esc":
            e["products_esc"] += int(an["products"][r])
    return e


# ---- numpy recount: per-row entries, products, distinct output columns, what the rules of the code make of them -----
def _dense(vec, n, fill=0.0):
    d = np.full(n, fill)
    present = np.zeros(n, bool)
    if vec is not None:
        d[vec.idx[0]] = vec.val
        present[vec.idx[0]] = True
    return d, present


def analyse(case, columns=True):
    A, B = case["A"], case["B"]
    m, nj = A.shape
    n_cols = B.shape[1]
    bptr = np.zeros(nj + 1, np.int64)
    np.add.at(bptr, B.idx[0].astype(np.int64) + 1, 1)
    bptr = np.cumsum(bptr)
    border = np.lexsort((B.idx[1], B.idx[0]))
    bk = B.idx[1][border].astype(np.int64)
    aorder = np.lexsort((A.idx[1], A.idx[0]))
    ai, aj = A.idx[0][aorder].astype(np.int64), A.idx[1][aorder].astype(np.int64)
    si_d, _ = _dense(case["si"], m)
    si_on = si_d != 0 if case["si"] is not None else np.ones(m, bool)
    _, sj_on = _dense(case["sj"], nj)
    if case["sj"] is None:
        sj_on[:] = True
    sk_d, _ = _dense(case["sk"], n_cols)
    sk_on = sk_d != 0 if case["sk"] is not None else None
    blen = np.diff(bptr)
    eprod = np.where(sj_on[aj] & si_on[ai], blen[aj], 0)
    entries = np.bincount(ai, minlength=m)
    products = np.bincount(ai, weights=eprod, minlength=m).astype(np.int64)
    astart = np.concatenate([[0], np.cumsum(entries)])
    outputs, words, cols = np.zeros(m, np.int64), np.zeros(m, np.int64), []
    for r in range(m if columns else 0):
        js = aj[astart[r]:astart[r + 1]]
        js = js[sj_on[js]]
        c = np.unique(np.concatenate([bk[bptr[j]:bptr[j + 1]] for j in js])) if len(js) else np.zeros(0, np.int64)
        if sk_on is not None:
            c = c[sk_on[c]]
        cols.append(c)
        outputs[r] = len(c)
        words[r] = len(np.unique(c // 32))
    # the rules: k_merge_count / count_row, k_esc_row_products, the small-row sort's cap (only for wide matrices)
    wide = n_cols > HASH_MAX_COLS
    bins = []
    for r in range(m):
        if entries[r] == 0 or not si_on[r]:
            bins.append(("skip", False))
        elif entries[r] <= MERGE_MAX_LISTS and products[r] == 0:
            bins.append(("skip", False))
        elif entries[r] <= MERGE_MAX_LISTS and products[r] <= MERGE_MAX_PRODUCTS:
            bins.append(("merge", False))
        elif products[r] >= HASH_MIN_PRODUCTS:
            bins.append(("hash", bool(wide and products[r] <= HSM_CAP)))
        else:
            bins.append(("esc", False))
    return dict(entries=entries, products=products, outputs=outputs, words=words, cols=cols, bins=bins,
                astart=astart, aj=aj, bptr=bptr, bk=bk, sj_on=sj_on)


def hash_trace(case, variant):
    """What k_hash_numeric's trace counts for the case's hash rows: work items, staged chunks, steps, warp-pipelined steps
    and barriers between entries.  Replays the item cut of k_hash_items, the windows of k_hash_splits, the staging of
    NT entries at a time and the choice per step (fewer than 32 entry changes: barrier per entry; else warp-pipelined)."""
    an = analyse(case)
    cap, NT = HASH_CAP[variant], HASH_NT[variant]
    items = chunks = steps = piped = rounds = 0
    for r, (b, _) in enumerate(an["bins"]):
        if b != "hash" or an["outputs"][r] == 0:
            continue
        out = an["cols"][r]
        total = len(out)
        n_items = -(-total // cap)
        per = -(-total // n_items)
        js = an["aj"][an["astart"][r]:an["astart"][r + 1]]
        for p in range(n_items):
            items += 1
            lo = out[p * per] if p > 0 else -1
            hi = out[(p + 1) * per] if p + 1 < n_items else 1 << 40
            lens = []
            for j in js:
                if not an["sj_on"][j]:
                    lens.append(0)
                    continue
                c = an["bk"][an["bptr"][j]:an["bptr"][j + 1]]
                lens.append(int(np.count_nonzero((c >= lo) & (c < hi))))
            for c0 in range(0, len(lens), NT):
                chunks += 1
                ln = [x for x in lens[c0:c0 + NT] if x]
                pre = np.concatenate([[0], np.cumsum(ln)])
                T = int(pre[-1])
                last = None
                for b0 in range(0, T, NT):
                    steps += 1
                    xf = int(np.searchsorted(pre, b0, "right")) - 1
                    xl = int(np.searchsorted(pre, min(b0 + NT, T) - 1, "right")) - 1
                    if xl - xf < 32:
                        for xi in range(xf, xl + 1):
                            if last != xi:
                                rounds += 1
                            last = xi
                    else:
                        piped += 1
                        last = None
    return dict(items=items, chunks=chunks, steps=steps, piped=piped, barriers=rounds)


# ---- builders ---------------------------------------------------------------------------------------------------------
def _overlapping(b, cols, n_rows, cover=0.6):
    """n_rows B rows over the columns `cols`: every column in at least one row, most in several (multi-term outputs)."""
    cols = np.asarray(cols, np.int64)
    owner = b.rng.integers(0, n_rows, len(cols))
    js = []
    for t in range(n_rows):
        take = (owner == t) | (b.rng.random(len(cols)) < cover)
        js.append(b.brow(cols[take]))
    return js


def _sized(b, pool, sizes):
    """B rows of the given sizes, columns drawn from `pool` (shared between rows: multi-term outputs)."""
    return [b.brow(b.rng.choice(pool, s, replace=False)) for s in sizes]


def merge_bin():
    """<= 8 inner indices and <= 1024 products: register merge; 9 entries or 1025 products: long row."""
    b = Build(11, 400)
    pool = np.arange(0, 400, 3)
    short = _sized(b, pool, [12] * 9)
    for n in (7, 8):
        b.arow(short[:n], "merge", claim=("entries", n, MERGE_MAX_LISTS))
    b.arow(short[:9], "esc", claim=("entries", 9, MERGE_MAX_LISTS))
    for f in (1023, 1024, 1025):   # eight B rows of 128 columns, the last one trimmed or grown
        js = _sized(b, np.arange(400), [128] * 7 + [128 - 1024 + f])
        b.arow(js, "merge" if f <= 1024 else "hash", claim=("products", f, MERGE_MAX_PRODUCTS))
    empty = b.brow([])
    b.arow(short[:8] + [empty], "esc", claim=("entries", 9, MERGE_MAX_LISTS))   # 9 entries, 8 lists that form products
    masked = b.brow(b.rng.choice(pool, 12, replace=False))
    b.arow(short[:8] + [masked], "esc", claim=("entries", 9, MERGE_MAX_LISTS))  # the 9th j is absent from scalej
    zi = b.arow(short[:9], "skip")   # zeroed by si (entry 0.0)
    ai = b.arow(short[:5], "skip")   # absent from si
    m = len(b.arows)
    nj = len(b.bcols)
    sj_idx = np.array([j for j in range(nj) if j != masked], np.int32)
    sj = Coo((nj,), [sj_idx], 1.0 + b.rng.random(len(sj_idx)), (0,))
    si_idx = np.array([i for i in range(m) if i != ai], np.int32)
    si_val = 0.5 + b.rng.random(len(si_idx))
    si_val[si_idx == zi] = 0.0
    si = Coo((m,), [si_idx], si_val, (0,))
    return b.finish("merge_bin", C=-1.5, si=si, sj=sj)


def hash_vs_esc():
    """Long rows (9+ entries) of 511, 512 and 513 products next to merge rows."""
    b = Build(12, 3000)
    pool = np.arange(0, 3000, 25)   # 120 columns: outputs of several terms
    for f in (511, 512, 513):
        js = _sized(b, pool, [50] * 9 + [f - 450])
        b.arow(js, "esc" if f < HASH_MIN_PRODUCTS else "hash", claim=("products", f, HASH_MIN_PRODUCTS))
    for _ in range(40):
        b.arow(_sized(b, pool, [6, 9, 7]), "merge")
    return b.finish("hash_vs_esc", C=0.75)


def nl_build(longest, long_b):
    """Longest row of A exactly `longest` (1..8): the merge kernels are built for 2/4/6/8 lists after it.  Mean B row
    at most 16 (the count kernel reports the longest row) or above 16 (k_row_maxlen runs first)."""
    b = Build(100 + longest, 2000)
    size = 24 if long_b else 10
    js = _sized(b, np.arange(0, 2000, 7)[:2 * size], [size] * 16)
    for t in range(120):
        n = longest if t % 5 == 0 else 1 + t % longest
        sel = b.rng.choice(16, n, replace=False)
        b.arow([js[s] for s in sel], "merge", claim=("entries", n, n) if t == 0 else None)
    return b.finish(f"nl{longest}_{'long' if long_b else 'short'}B")


def merge_staging(cancel=True):
    """Rows of 15, 16, 17, 32 and 33 outputs (the numeric pass flushes every 16, 8 or 4 outputs of a lane), and rows whose
    first or last output of a flushed run cancels exactly (tombstone, then compaction).  cancel=False: the same matrix with
    +a / +a on the pairs instead, so that nothing cancels."""
    b = Build(13, 600)
    for n in (15, 16, 17, 32, 33):
        for rep in range(3):
            cols = b.rng.choice(600, n, replace=False)
            b.arow(_overlapping(b, cols, 5, cover=0.7), "merge", claim=("outputs", n, 16 if n < 24 else 32))
    for n, where in ((16, 0), (16, 15), (17, 15), (32, 16), (8, 7)):
        cols = np.sort(b.rng.choice(600, n, replace=False))
        p, q = b.pair(cols[[where]])
        rest = np.delete(cols, where)
        js = _overlapping(b, rest, 4, cover=0.7)
        b.arow(js[:1] + [p, q] + js[1:], "merge", avals=None)
        # +a / -a on the pair (values in the order of the list above: js[0], p, q, js[1:])
        a = values(b.rng, 6)
        a[2] = -a[1] if cancel else a[1]
        b.arows[-1] = (b.arows[-1][0], a)
    return b.finish("merge_staging" if cancel else "merge_staging_no_cancel", C=2.0)


def onepass(kind):
    """SPB_MERGE_ONEPASS=1: a matrix it takes ('pass'), one with a row of 17 outputs ('outputs') and one with a row of
    more than merge_max_products products ('products'); both of the latter must fall back to the two-pass answer."""
    b = Build(14, 5000)
    pool = np.arange(5000)
    small = _sized(b, pool, [3] * 600)
    for t in range(1500):
        b.arow([small[(t * 7 + u) % 600] for u in range(2)], "merge")
    if kind == "outputs":
        b.arow(_overlapping(b, b.rng.choice(5000, 17, replace=False), 5, cover=0.7), "merge", claim=("outputs", 17, 16))
    if kind == "products":
        js = _sized(b, pool[:300], [128] * 7 + [129])
        b.arow(js, "hash", claim=("products", 1025, MERGE_MAX_PRODUCTS))
    return b.finish(f"onepass_{kind}")


def _pattern_row(b, pool, lens, cancel_cols=None):
    """A hash row from B rows of the given lengths over `pool`; optionally a cancelling pair over cancel_cols (which no
    other B row of the row touches)."""
    js = _sized(b, pool, lens)
    avals = None
    if cancel_cols is not None:
        p, q = b.pair(cancel_cols)
        js = js + [p, q]
        avals = values(b.rng, len(js))
        avals[-1] = -avals[-2]
    return js, avals


def hash_items(variant, with_sk=False):
    """Hash rows of CAP-1, CAP, CAP+1, 2 CAP and 2 CAP+1 outputs (CAP = outputs per work item of the variant), and a row of
    2 CAP outputs whose first, last and middle outputs (an item's first and last) cancel exactly.  with_sk: a scale vector
    that excludes every fifth column, so the rows have fewer outputs than distinct columns."""
    cap = HASH_CAP[variant]
    n_cols = 3 * cap
    b = Build(20 + variant, n_cols)
    for n in (cap - 1, cap, cap + 1, 2 * cap, 2 * cap + 1):
        cols = b.rng.choice(n_cols, n, replace=False)
        b.arow(_overlapping(b, cols, 5, cover=0.7), "hash", claim=None if with_sk else ("outputs", n, cap if n < 2 * cap else 2 * cap))
    cols = np.sort(b.rng.choice(n_cols, 2 * cap, replace=False))
    edge = [0, cap - 1, cap, 2 * cap - 1]
    js = _overlapping(b, np.delete(cols, edge), 5, cover=0.7)
    p, q = b.pair(cols[edge])
    a = values(b.rng, 7)
    a[6] = -a[5]
    b.arow(js + [p, q], "hash", avals=a)
    sk = None
    if with_sk:
        k = np.arange(n_cols)
        sk = Coo((n_cols,), [k[k % 5 != 2].astype(np.int32)], 0.5 + b.rng.random(int(np.count_nonzero(k % 5 != 2))), (0,))
    return b.finish(f"hash_items_v{variant}{'_sk' if with_sk else ''}", C=1.25, sk=sk, ctx_env={"SPB_HASH_VARIANT": str(variant)})


def hash_steps(variant, span):
    """Hash rows whose every step of NT products spans exactly `span` entries (31 and 32: a barrier per entry change;
    33: warp-pipelined).  span 0: 2 NT one-product entries that all hit one column (32 lanes per output: the most rounds)."""
    NT = HASH_NT[variant]
    L = NT // 32
    b = Build(30 + variant * 10 + span, 4 * NT)
    pool = np.arange(0, 6 * L, 2)   # 3 L columns: ~20 terms per output
    if span == 0:
        for r in range(2):
            js = [b.brow([r]) for _ in range(2 * NT)]
            b.arow(js, "hash", claim=("products", 2 * NT, HASH_MIN_PRODUCTS) if NT == 256 else None)
    else:
        step = {31: [L] * 30 + [2 * L], 32: [L] * 32, 33: [L] * 31 + [L // 2] * 2}[span]
        lens = step * max(2, -(-HASH_MIN_PRODUCTS // NT))
        for r in range(3):
            js, _ = _pattern_row(b, pool, lens)
            b.arow(js, "hash")
    return b.finish(f"hash_steps_v{variant}_{span}", ctx_env={"SPB_HASH_VARIANT": str(variant)})


def bitmap_width(n_cols):
    """n_cols = W, W+1 (a one-column second window) or 2W+1; outputs at columns W-1, W and n_cols-1 (those that exist).
    Rows of more than HSM_CAP products, so that wide matrices list their columns with the bitmap in windows."""
    W = HASH_MAX_COLS
    b = Build(40 + n_cols % 7, n_cols)
    edge = np.unique([c for c in (0, W - 1, W, n_cols - 1) if c < n_cols])
    shared = np.setdiff1d(b.rng.choice(n_cols, 3600, replace=False), edge)   # the rows' B rows overlap: multi-term outputs
    for r in range(3):
        js = []
        for t in range(3):
            cols = np.union1d(b.rng.choice(shared, 3000, replace=False), edge)
            js.append(b.brow(cols))
        b.arow(js, "hash")
    for r in range(20):
        b.arow([b.brow(np.union1d(b.rng.choice(n_cols, 3, replace=False), edge[-1:]))], "merge")
    return b.finish(f"bitmap_{n_cols}", C=-0.5)


def small_sort(f, collapse):
    """A row of f products (8191, 8192, 8193) in a matrix wider than the bitmap: at most HSM_CAP products, its columns are
    listed by the shared-memory sort.  All-distinct columns, or collapsing onto 8 columns.  Next to it a row of 12000
    products (always the bitmap)."""
    n_cols = 2 * HASH_MAX_COLS
    b = Build(50 + f % 10 + 10 * collapse, n_cols)
    if collapse:
        lens = [8] * (f // 8) + ([f % 8] if f % 8 else [])
        js = [b.brow(np.arange(1000, 1000 + n) * 977) for n in lens]
    else:
        cols = b.rng.choice(n_cols, f, replace=False)
        js = [b.brow(cols[t::4]) for t in range(4)]
    b.arow(js, "hash", small=f <= HSM_CAP, claim=("products", f, HSM_CAP))
    b.arow([b.brow(b.rng.choice(n_cols, 4000, replace=False)) for _ in range(3)], "hash")
    return b.finish(f"small_{f}_{'collapse' if collapse else 'distinct'}")


def sparse_walk(words):
    """A hash row whose outputs occupy exactly `words` (4607, 4608, 4609) 32-column bitmap words, next to a dense row."""
    n_cols = 32 * 5000
    b = Build(60 + words % 10, n_cols)
    cols = 32 * np.arange(words) + b.rng.integers(0, 32, words)
    b.arow(_overlapping(b, cols, 5, cover=0.7), "hash", claim=("words", words, HS_LIST_CAP))
    b.arow(_overlapping(b, np.arange(20000, 40000), 5, cover=0.7), "hash")
    return b.finish(f"walk_{words}")


def esc_chunk(offset):
    """ESC rows (9 entries, < 512 products) whose products add up to ESC_CHUNK exactly at the end of row ESC_BOUNDARY_ROW
    (offset 0), or one product past it (offset 1), followed by more ESC rows: two chunks, cut at a row boundary either
    way (k_esc_chunks: the first row whose ESC product offset is >= ESC_CHUNK)."""
    b = Build(70 + offset, 200)
    # 262148 rows of 511 products and 510 of 510: 2^27 exactly (2^27 = 1 mod 511)
    j511 = _sized(b, np.arange(200), [56] * 8 + [63])
    j510 = j511[:8] + [b.brow(b.rng.choice(200, 62, replace=False))]
    j512 = j511[:8] + [b.brow(b.rng.choice(200, 64, replace=False))]
    b.arows = [(j511, None)] * 262148 + [(j510, None)] * 510
    if offset:   # one row of 512 would be hash: move the extra product to a row of 510 -> 511
        b.arows[-1] = (j511, None)
    b.arows += [(j511, None)] * 1000 + [(j512, None)] * 3
    b.bins = ["esc"] * (len(b.arows) - 3) + ["hash"] * 3
    b.small = [False] * len(b.arows)
    return b.finish(f"esc_chunk_{offset}")


ESC_BOUNDARY_ROW = 262148 + 510 - 1


def panel_rows(row_products, max_products):
    """First row of every panel spb_mm_plan_create makes: nch = ceil(F / max_products) even chunks of ceil(F / nch)
    products, cut c at the first row whose first product is >= c * chunk (k_panel_bounds), empty panels dropped."""
    prod = np.asarray(row_products, np.int64)
    F, nrows = int(prod.sum()), len(prod)
    nch = min(-(-max(F, 1) // max_products), nrows)
    chunk = -(-max(F, 1) // nch)
    starts = np.concatenate([[0], np.cumsum(prod)[:-1]])
    rb = [0] + [int(np.searchsorted(starts, c * chunk, "left")) for c in range(1, nch)] + [nrows]
    lo = []
    for c in range(nch + 1):
        if 0 < c < nch and rb[c] == lo[-1]:
            continue
        if c == nch and lo and rb[c] == lo[-1]:
            break
        lo.append(rb[c])
    return lo[:-1]   # (lo ends with nrows)


PANEL_CUT_ROW = 30


def panels(delta):
    """Two halves of 30 rows: the first has S products, the second S + delta.  With two panels (max_products from
    ceil(F / 2) to F - 1) the chunk is ceil((2 S + delta) / 2): S - 1 (delta -2), S (delta 0) or S + 1 (delta 1), so
    the cut falls one product before, on and one product after the first product of row PANEL_CUT_ROW."""
    b = Build(80, 5000)
    pool = np.arange(0, 5000, 50)   # 100 columns: outputs of several terms
    sizes = [list(b.rng.integers(5, 40, 1 + t % 11)) for t in range(PANEL_CUT_ROW)]
    sizes = sizes + [list(x) for x in sizes]
    sizes[-1][0] += delta
    for sz in sizes:
        js = _sized(b, pool, sz)
        n, f = len(js), b.plen(js)
        b.arow(js, ("merge" if f <= MERGE_MAX_PRODUCTS else "hash") if n <= MERGE_MAX_LISTS else ("hash" if f >= HASH_MIN_PRODUCTS else "esc"))
    return b.finish(f"panels_{delta}")


def all_cases():
    """Every builder's cases but the ESC chunk ones (large: tests/test_thresholds_cpu.py recounts them on their own)."""
    out = [merge_bin(), hash_vs_esc(), merge_staging(), merge_staging(cancel=False)] + [panels(d) for d in (-2, 0, 1)]
    out += [nl_build(n, lb) for n in range(1, 9) for lb in (False, True)]
    out += [onepass(k) for k in ("pass", "outputs", "products")]
    out += [hash_items(v, s) for v in (2, 1, 0) for s in (False, True)]
    out += [hash_steps(v, s) for v in (2, 1, 0) for s in (31, 32, 33, 0)]
    out += [bitmap_width(n) for n in (HASH_MAX_COLS, HASH_MAX_COLS + 1, 2 * HASH_MAX_COLS + 1)]
    out += [small_sort(f, c) for f in (8191, 8192, 8193) for c in (False, True)]
    out += [sparse_walk(w) for w in (4607, 4608, 4609)]
    return out
