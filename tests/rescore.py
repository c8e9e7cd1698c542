"""Independent checks of an alignment's optimality, sharing no code with the oracle's or the
kernels' traceback (SURVEY.md 8c-A items 2-5):

* `rescore(ax, ay, scores)`: the score of a gapped pair of strings under TaxI2's six scores, gap
  runs typed end / internal by position exactly as Biopython types them;
* `best_score(x, y, scores)`: the optimum of the global alignment by a plain three-state
  dynamic programme (score only, ties irrelevant).

An emitted alignment is optimal iff rescore(...) == best_score(...); that pins everything about
it except WHICH co-optimal alignment was chosen."""
from __future__ import annotations

NEG = float("-inf")


def rescore(ax: str, ay: str, scores) -> float:
    match, mismatch, io, ie, eo, ee = (float(s) for s in scores)
    assert len(ax) == len(ay)
    nA = sum(c != "-" for c in ax)
    nB = sum(c != "-" for c in ay)
    i = j = 0            # characters of x / y consumed so far
    total = 0.0
    prev = None          # 'x' = previous column was a gap in x, 'y' = a gap in y, None = both present
    for a, b in zip(ax, ay):
        assert not (a == "-" and b == "-"), "column of two gaps"
        if a == "-":     # horizontal move: consumes a y character while x stands at row i
            end = i == 0 or i == nA
            total += (ee if end else ie) if prev == "x" else (eo if end else io)
            prev = "x"
            j += 1
        elif b == "-":   # vertical move: consumes an x character while y stands at column j
            end = j == 0 or j == nB
            total += (ee if end else ie) if prev == "y" else (eo if end else io)
            prev = "y"
            i += 1
        else:
            total += match if a == b else mismatch
            prev = None
            i += 1
            j += 1
    return total


def best_score(x: str, y: str, scores) -> float:
    """max over all global alignments; M / Ix (vertical) / Iy (horizontal) with Ix <-> Iy allowed."""
    match, mismatch, io, ie, eo, ee = (float(s) for s in scores)
    nA, nB = len(x), len(y)
    M = [[NEG] * (nB + 1) for _ in range(nA + 1)]
    X = [[NEG] * (nB + 1) for _ in range(nA + 1)]
    Y = [[NEG] * (nB + 1) for _ in range(nA + 1)]
    M[0][0] = 0.0
    for i in range(nA + 1):
        for j in range(nB + 1):
            if i > 0 and j > 0:
                s = match if x[i - 1] == y[j - 1] else mismatch
                M[i][j] = max(M[i - 1][j - 1], X[i - 1][j - 1], Y[i - 1][j - 1]) + s
            if i > 0:   # vertical: end gap in the first / last column
                o, e = (eo, ee) if j in (0, nB) else (io, ie)
                X[i][j] = max(M[i - 1][j] + o, X[i - 1][j] + e, Y[i - 1][j] + o)
            if j > 0:   # horizontal: end gap in the first / last row
                o, e = (eo, ee) if i in (0, nA) else (io, ie)
                Y[i][j] = max(M[i][j - 1] + o, X[i][j - 1] + o, Y[i][j - 1] + e)
    return max(M[nA][nB], X[nA][nB], Y[nA][nB])


def best_score_adjacent_gaps(x: str, y: str, scores) -> float:
    """max over the global alignments that put a vertical gap right next to a horizontal one (at
    least one Ix <-> Iy transition); -inf if there is none.  The packed kernel's recurrence drops
    those transitions, which is exact for a pair iff this stays strictly below best_score."""
    match, mismatch, io, ie, eo, ee = (float(s) for s in scores)
    nA, nB = len(x), len(y)
    # layer 0: no Ix <-> Iy transition yet, layer 1: at least one
    M = [[[NEG] * (nB + 1) for _ in range(nA + 1)] for _ in range(2)]
    X = [[[NEG] * (nB + 1) for _ in range(nA + 1)] for _ in range(2)]
    Y = [[[NEG] * (nB + 1) for _ in range(nA + 1)] for _ in range(2)]
    M[0][0][0] = 0.0
    for i in range(nA + 1):
        for j in range(nB + 1):
            for k in (0, 1):
                if i > 0 and j > 0:
                    s = match if x[i - 1] == y[j - 1] else mismatch
                    M[k][i][j] = max(M[k][i - 1][j - 1], X[k][i - 1][j - 1], Y[k][i - 1][j - 1]) + s
                if i > 0:
                    o, e = (eo, ee) if j in (0, nB) else (io, ie)
                    X[k][i][j] = max(M[k][i - 1][j] + o, X[k][i - 1][j] + e, Y[1][i - 1][j] + o if k else NEG, Y[0][i - 1][j] + o if k else NEG)
                if j > 0:
                    o, e = (eo, ee) if i in (0, nA) else (io, ie)
                    Y[k][i][j] = max(M[k][i][j - 1] + o, Y[k][i][j - 1] + e, X[1][i][j - 1] + o if k else NEG, X[0][i][j - 1] + o if k else NEG)
    return max(M[1][nA][nB], X[1][nA][nB], Y[1][nA][nB])
