"""An exact reference for the DP kernels that does not share code with the oracle: a plain int64 two-piece affine DP with ksw2's
conventions, and a scorer of CIGARs under the same scoring.  Test infrastructure only.

Conventions (those of ksw_extd2, ksw2_extd2_sse.c): target position t, query position j; a gap run of length l costs
min(q + l*e, q2 + l*e2); the first row and column are H(t,-1) = -min(q + (t+1)e, q2 + (t+1)e2), H(-1,j) likewise, H(-1,-1) = 0;
a pair with an N scores the matrix's N entry, and -e2 when that entry is 0 (e2 of the piece with the larger q+e, after the
pieces are ordered)."""
import numpy as np

NEG = -(1 << 40)


def _pieces(q, e, q2, e2):
    return (q, e, q2, e2) if q + e <= q2 + e2 else (q2, e2, q, e)


def _scores(mat, e2):
    mch, mis, nsc = int(mat[0]), int(mat[1]), int(mat[24])
    return mch, mis, (-e2 if nsc == 0 else nsc)


class KswRef:
    """H of every cell of a job (qlen x tlen, 0..4 codes), computed one anti-diagonal at a time.

    score: H(tlen-1, qlen-1); max: the largest H, at least 0 (ksw_extz_t.max starts at 0); mqe: max over t of H(t, qlen-1);
    mte: max over j of H(tlen-1, j).  H(t, j) is at(t, j)."""

    def __init__(self, q, t, mat, q_, e_, q2_, e2_):
        q = np.asarray(q, dtype=np.int64)
        t = np.asarray(t, dtype=np.int64)
        ql, tl = len(q), len(t)
        assert ql > 0 and tl > 0
        go, ge, go2, ge2 = _pieces(q_, e_, q2_, e2_)
        mch, mis, nsc = _scores(mat, ge2)
        self.qlen, self.tlen = ql, tl

        def border(l):  # H of a gap run of length l from the corner
            return -min(go + l * ge, go2 + l * ge2)

        qn, tn = q >= 4, t >= 4
        # Diagonal r holds the cells (t, r - t) for t in [A, B] = [max(-1, r-qlen+1), min(r+1, tlen-1)]: its cells and its border
        # cells (-1, r+1) and (r+1, -1).  P2 and P1 are diagonals r-2 and r-1 as (A, H, D1, D2, I1, I2); the gap states (D: runs
        # along the target, I: along the query) are NEG on the border, where ksw2 opens every gap from H.
        one = lambda v: np.array([v], np.int64)
        neg = one(NEG)
        P2 = (-1, one(0), neg, neg, neg, neg)                                           # r = -2: (-1, -1)
        P1 = (-1, np.array([border(1), border(1)], np.int64), *(np.full(2, NEG, np.int64),) * 4)  # r = -1: (-1, 0), (0, -1)
        self._diag = []
        for r in range(ql + tl - 1):
            lo, hi = max(0, r - ql + 1), min(r, tl - 1)
            ts = np.arange(lo, hi + 1)
            js = r - ts
            s = np.where(t[ts] == q[js], mch, mis)
            s = np.where(tn[ts] | qn[js], nsc, s)
            A1, H1, D1, D2, I1, I2 = P1
            k_up, k_left = ts - 1 - A1, ts - A1   # (t-1, j) and (t, j-1) in diagonal r-1
            up, left = H1[k_up], H1[k_left]
            d1 = np.maximum(up - go - ge, D1[k_up] - ge)
            d2 = np.maximum(up - go2 - ge2, D2[k_up] - ge2)
            i1 = np.maximum(left - go - ge, I1[k_left] - ge)
            i2 = np.maximum(left - go2 - ge2, I2[k_left] - ge2)
            h = np.maximum.reduce([P2[1][ts - 1 - P2[0]] + s, d1, d2, i1, i2])
            A, B = max(-1, r - ql + 1), min(r + 1, tl - 1)
            new = [np.full(B - A + 1, NEG, np.int64) for _ in range(5)]
            for a, v in zip(new, (h, d1, d2, i1, i2)):
                a[lo - A:hi - A + 1] = v
            if A == -1:
                new[0][0] = border(r + 2)       # (-1, r+1)
            if B == r + 1:
                new[0][-1] = border(r + 2)      # (r+1, -1)
            self._diag.append((lo, h.astype(np.int32)))
            P2, P1 = P1, (A, *new)
        self.score = self.at(tl - 1, ql - 1)
        self.max = max(0, max(int(h.max()) for _, h in self._diag))
        self.mqe = max(self.at(x, ql - 1) for x in range(tl))
        self.mte = max(self.at(tl - 1, j) for j in range(ql))

    def at(self, t, j):
        lo, h = self._diag[t + j]
        return int(h[t - lo])


def cigar_score(cigar, q, t, mat, q_, e_, q2_, e2_):
    """score of the alignment a CIGAR (ksw2 encoding: len << 4 | op, 0 M, 1 I, 2 D) describes from the start of q and t, and the
    numbers of query and target bases it spans"""
    go, ge, go2, ge2 = _pieces(q_, e_, q2_, e2_)
    mch, mis, nsc = _scores(mat, ge2)
    sc, i, k = 0, 0, 0
    for c in cigar:
        op, l = c & 0xf, c >> 4
        assert l > 0 and op in (0, 1, 2), cigar
        if op == 0:
            a, b = np.asarray(q[i:i + l], np.int64), np.asarray(t[k:k + l], np.int64)
            assert len(a) == l and len(b) == l, "the CIGAR runs past the end of a sequence"
            sc += int(np.where((a >= 4) | (b >= 4), nsc, np.where(a == b, mch, mis)).sum())
            i += l; k += l
        else:
            sc -= min(go + l * ge, go2 + l * ge2)
            if op == 1:
                i += l
            else:
                k += l
    return sc, i, k


def check_job(ez, q, t, mat, pen, flag, end_bonus, ref=None):
    """Asserts what the DP must give on a job whose band never clips, with z-drop off: score (global), max, mqe and mte
    (extension, exact mode) equal the reference DP's; H at (max_t, max_q) is max; the CIGAR spans the whole matrix, the max cell,
    or the query end when reach_end is set, and re-scores to score, max or mqe.  Returns the KswRef it used."""
    ref = ref or KswRef(q, t, mat, *pen)
    ql, tl = len(q), len(t)
    assert ez["zdropped"] == 0
    assert ez["score"] == ref.score, ("score", ez["score"], ref.score)
    exact = not (flag & 0x08)
    if exact:
        assert (ez["max"], ez["mqe"], ez["mte"]) == (ref.max, ref.mqe, ref.mte), ("max/mqe/mte", ez, ref.max, ref.mqe, ref.mte)
        if ez["max_t"] >= 0:
            assert ref.at(ez["max_t"], ez["max_q"]) == ez["max"], "H at (max_t, max_q) is not max"
        assert ref.at(ez["mqe_t"], ql - 1) == ez["mqe"]  # (mte_q is r - en with en rounded up to the SSE block: not a cell)
    if flag & 0x01:
        return ref
    cig = ez["cigar"]
    if flag & 0x80:  # REV_CIGAR: the ops from the end cell backwards
        cig = cig[::-1]
    if not (flag & 0x40):
        want_q, want_t, want = ql, tl, ref.score
    elif not exact:
        return ref
    elif ez["reach_end"]:
        assert ez["mqe"] + end_bonus > ez["max"]
        want_q, want_t, want = ql, ez["mqe_t"] + 1, ref.mqe
    elif ez["max_t"] >= 0:
        want_q, want_t, want = ez["max_q"] + 1, ez["max_t"] + 1, ref.max
    else:
        assert cig == []
        return ref
    sc, nq, nt = cigar_score(cig, q, t, mat, *pen)
    assert (nq, nt) == (want_q, want_t), ("CIGAR span", nq, nt, want_q, want_t)
    assert sc == want, ("CIGAR score", sc, want)
    return ref
