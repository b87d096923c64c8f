"""The reference the index-limit GPU tests use (tests/_limits.py: the oracle on a monotonically relabelled problem), checked on
the CPU against the oracle's literal loop nest (pairs=True, O(nnz) memory) at extents of exactly 2^31, and against the
row-wise oracle itself where the extents are small enough for it."""
import numpy as np
import pytest

import _cases
import _limits as L
from oracle import oracle as O


@pytest.mark.parametrize("roles", ["i", "j", "k", "ijk"])
@pytest.mark.parametrize("tA,tB", [(".", "."), ("T", "."), (".", "T"), ("T", "T")])
def test_relabelled_reference_matches_the_loop_nest_at_2_31(orc, roles, tA, tB):
    for seed in range(3):
        A, B = L.mm_inputs(100 + seed, roles)
        rng = np.random.default_rng(seed)
        modes = ["nonzero", "zero", "absent"]
        si = L.scale_vector(rng, A.idx[0], modes[seed]) if seed != 1 else None
        sj = L.scale_vector(rng, np.concatenate([A.idx[1], B.idx[0]]), modes[(seed + 1) % 3]) if seed != 2 else None
        sk = L.scale_vector(rng, B.idx[1], modes[(seed + 2) % 3]) if seed != 0 else None
        for scales in ((None, None, None), (si, sj, sk)):
            args = (1.5, scales[0], L.transposed(A, tA), tA, scales[1], L.transposed(B, tB), tB, scales[2])
            want = orc.multiply_mm(*args, pairs=True)
            got = L.relabeled_mm(orc, *args)
            assert got.shape == (L.N, L.N)
            assert _cases.same_coo(got, want), (roles, tA, tB, seed, scales[0] is not None)
            if "k" in roles and scales[0] is None:   # the cancelling rows are dropped, the +inf - inf row is kept as NaN
                top = want.idx[1] == L.TOP
                assert top.any() and np.isnan(want.val[top]).any()


def test_relabelled_reference_matches_the_row_wise_oracle(orc):
    """Where the oracle's own row-wise evaluation fits (extents of a few hundred), the relabelled run is the same product."""
    for s in range(2000, 2060):
        c = _cases.mm_case(s, big=(s % 4 == 0))
        # scale vectors longer than their dimension are trimmed: the relabelling assumes they lie inside it
        sc = []
        for v, dim in ((c["si"], c["A"].shape[1 if c["tA"] == "T" else 0]), (c["sj"], None), (c["sk"], c["B"].shape[0 if c["tB"] == "T" else 1])):
            if v is not None and dim is not None:
                keep = v.idx[0] < dim
                v = O.Coo((dim,), [v.idx[0][keep]], v.val[keep], (0,))
            sc.append(v)
        args = (c["C"], sc[0], c["A"], c["tA"], sc[1], c["B"], c["tB"], sc[2], c["policy"], c["zero_nan"])
        assert _cases.same_coo(L.relabeled_mm(orc, *args), orc.multiply_mm(*args)), s


def test_merge_row_lengths_and_cancellation_inputs():
    """The inputs the GPU tests rely on: every row of op(A) exactly row_len entries long, index 2^31-1 in the roles asked for
    and nowhere else."""
    for ln in range(1, 9):
        A, B = L.mm_inputs(7 + ln, "ijk", row_len=ln)
        _, cnt = np.unique(A.idx[0], return_counts=True)
        assert set(cnt.tolist()) == {ln, 2} | ({ln} if ln == 2 else set())   # the three cancellation rows hold 2 each
    A, B = L.mm_inputs(3, "j")
    assert L.TOP in A.idx[1] or L.TOP in B.idx[0]
    assert L.TOP not in A.idx[0] and L.TOP not in B.idx[1]
    A, B = L.mm_inputs(3, "k")
    assert L.TOP in B.idx[1] and L.TOP not in A.idx[0] and L.TOP not in A.idx[1]
