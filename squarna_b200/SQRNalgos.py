"""The non-greedy structure builders of SQUARNA (Nussinov / Hungarian / Edmonds, SQRNalgos.py in the reference),
fed by the stems the GPU enumerates (sqrn_yield_stems_batch = AnnotateStems).  SURVEY.md 8(f)-2.  All three run on
the device when the caller has a library context (sqrn_nussinov_batch, csrc/sqrn_nussinov.cuh, DESIGN.md 3.8;
sqrn_hungarian_batch, csrc/sqrn_hungarian.cuh, 3.9; sqrn_edmonds_batch, csrc/sqrn_edmonds.cuh, 3.10); the functions
here are the specifications the device code reproduces pair for pair (tests/test_nussinov.py, tests/test_hungarian.py,
tests/test_edmonds.py) and the path of contexts without the device builders.  Results are pinned to the reference by
tests/golden/algos.json (tests/golden/make_golden.py algos).

Every function takes `stems` = [[pairs, length, score], ...] in AnnotateStems order and returns base pairs."""
import numpy as np


def _pair_scores(stems):
    """(v, w) -> stem score, in stem order (a pair belongs to one stem only)"""
    return {(v, w): stem[2] for stem in stems for (v, w) in stem[0]}


def _has_sep(seq, lo, hi, seps):
    return any(ch in seps for ch in seq[lo:hi])


def BackTrack(begin, end, K, minloop, seq, seps, partial=False):
    """pairs recorded in K, followed from the cell (begin, end) (SQRNalgos.py:1-41).  The reference walks the
    cells breadth first through a set; the pairs it returns are sorted, so the visiting order is free."""
    todo, found, seen = [(begin, end)], [], set()
    while todo:
        i, j = todo.pop()
        if (i, j) in seen:
            continue
        seen.add((i, j))
        k = K.get((i, j))
        if k is None:                                   # j unpaired: shrink from the right
            gap = (j - 1) - i
            if not partial and (gap > minloop or (gap > 0 and _has_sep(seq, i + 1, j - 1, seps))):
                todo.append((i, j - 1))
            continue
        found.append((k, j))
        left = (k - 1) - i                              # room before k
        if not partial and (left > minloop or (left > 0 and _has_sep(seq, i + 1, k - 1, seps))):
            todo.append((i, k - 1))
        inner = (j - 1) - (k + 1)                       # room inside (k, j)
        if inner > minloop or (inner > 0 and _has_sep(seq, k + 2, j - 1, seps)):
            todo.append((k + 1, j - 1))
    return sorted(found)


def Nussinov(seq, stems, N, seps, minloop=3, matrix=None):
    """minimum-energy nested structure over the stem pairs, energy of a pair = -(score of its stem)
    (SQRNalgos.py:44-93).  D[i, j] = best energy of i..j; for every j the partners k of j are tried in
    increasing k and the first strict minimum wins; a pair is taken when it is not worse than leaving j unpaired."""
    if matrix is None:
        energy = {bp: -sc for bp, sc in _pair_scores(stems).items()}
    else:
        energy = {(v, w): -matrix[v, w] for v in range(N - 1) for w in range(v + 1, N) if matrix[v, w] > 0}
    partners = [[] for _ in range(N)]                    # per j: its possible k in increasing order
    for (k, j) in sorted(energy):
        partners[j].append(k)
    part_arr = [np.array(p, dtype=np.int64) for p in partners]
    part_en = [np.array([energy[(k, j)] for k in partners[j]], dtype=np.float64) for j in range(N)]
    # one extra row / column of zeros stands for the cells the reference reads outside the triangle
    # (D[i, i-1], and D[0, -1] before it is written): they are all 0 when they are read
    D = np.zeros((N + 1, N + 1))
    K = {}
    for h in range(1, N):
        for i in range(N - h):
            j = i + h
            ks, es = part_arr[j], part_en[j]
            best_k, best = -1, 10 ** 9
            if len(ks):
                lo = np.searchsorted(ks, i)
                hi = np.searchsorted(ks, j - 1)            # k < j - 1
                if hi > lo:
                    kk = ks[lo:hi]
                    left = np.where(kk > i, D[i, kk - 1], 0.0)        # D[i, i-1] = 0
                    tot = left + D[kk + 1, j - 1] + es[lo:hi]
                    m = int(np.argmin(tot))                            # first minimum, as `<` keeps it
                    if tot[m] < best:
                        best_k, best = int(kk[m]), tot[m]
            if best <= D[i, j - 1]:
                K[(i, j)] = best_k
                D[i, j] = best
            else:
                D[i, j] = D[i, j - 1]
    return BackTrack(0, N - 1, K, minloop, seq, seps)


def _weighted_pairs(stems, power, matrix):
    """(v, w, weight) of every candidate pair, weight = score ** power: the pairs of the stems in stem order, or the
    positive upper-triangle cells of a score matrix in row-major order"""
    if matrix is not None:
        vs, ws = np.nonzero(np.triu(np.asarray(matrix) > 0, 1))
        return [(int(v), int(w), matrix[v, w] ** power) for v, w in zip(vs.tolist(), ws.tolist())]
    return [(v, w, sc ** power) for (v, w), sc in _pair_scores(stems).items()]


def Edmonds(stems, power=1.7, matrix=None):
    """maximum-weight matching of the graph whose edges are the stem pairs, weight = (stem score) ** 1.7
    (SQRNalgos.py:96-110); edges enter the graph in stem order, which is what ties are broken by"""
    from networkx import Graph, max_weight_matching
    graph = Graph()
    graph.add_weighted_edges_from(_weighted_pairs(stems, power, matrix))
    return sorted(max_weight_matching(graph))


def Hungarian(seq, stems, N, seps, minloop=3, power=1.7, matrix=None):
    """assignment problem on the symmetric N x N matrix of -(stem score) ** 1.7; a pair (k, l) is kept when the
    assignment is mutual, the cell is non-zero and the hairpin rule holds (SQRNalgos.py:113-136)"""
    from scipy.optimize import linear_sum_assignment
    if matrix is not None:
        cost = -(matrix ** power)
    else:
        cost = np.zeros((N, N))
        trip = _weighted_pairs(stems, power, None)
        if trip:
            vs, ws, wt = (np.array(x) for x in zip(*trip))
            cost[vs, ws] = -wt
            cost[ws, vs] = -wt
    rows, cols = linear_sum_assignment(cost)
    partner = np.full(N, -1, dtype=np.int64)
    partner[rows] = cols
    out = []
    for k in rows.tolist():                              # row order, as the reference's dict of the assignment
        l = int(partner[k])
        far_enough = k < l - minloop or (k < l and _has_sep(seq, k + 1, l, seps))
        if far_enough and partner[l] == k and cost[k, l] != 0:
            out.append((k, l))
    return out
