"""Exact output distributions of the three maze generators on small lattices (test infrastructure;
see oracle/__init__.py).

A memoized recursion over each generator's state gives the probability of every outcome
(start cell, spanning tree) of lib/maze_generation.py's processes, as oracle.generation restates them:

- r-prim: state = the tree so far (its cell set follows); a uniform frontier cell joins through a
  uniform in-tree neighbour.
- dfs: state = tree, current cell and parent map; a uniform unvisited neighbour, else back to the parent.
- prim&kill: state = tree, marked set and current cell; a uniform unmarked neighbour, else a restart
  from a uniform marked cell that still has an unmarked neighbour.

An outcome is one integer: start cell index (row-major) << n_edges | passage bits, passage k open
<=> bit k set, passages numbered as `lattice_edges` lists them.  `best_of_k` turns a generator's
distribution into the distribution of the maze best-of-k generation keeps.
"""
from __future__ import annotations

from functools import lru_cache

import numpy as np

# Two McClendon difficulties are the same score when they differ by at most TIE_REL relative: mathematically
# equal scores of different trees differ in the last bits only (sums run in another order), genuine
# differences between small mazes are >= 5e-4 relative.  Best-of-k keeps the FIRST candidate of the
# lowest score, so a candidate replaces the kept one only when it is lower by more than this.
TIE_REL = 1e-12


def same_score(a: float, b: float) -> bool:
    return abs(a - b) <= TIE_REL * max(abs(a), abs(b))


def best_candidate(scores) -> int:
    """Index of the candidate best-of-k keeps: the first one whose score no later candidate beats by
    more than TIE_REL (maze_generate_kernel's keep rule)."""
    best = 0
    for c in range(1, len(scores)):
        if scores[c] < scores[best] - TIE_REL * abs(scores[best]):
            best = c
    return best


def lattice_edges(nr: int, nc: int):
    """Cell pairs (row-major cell indices) of the lattice's passages in outcome-bit order: the
    horizontal ones (i, j)-(i, j+1) row by row, then the vertical ones (i, j)-(i+1, j)."""
    horiz = [(i * nc + j, i * nc + j + 1) for i in range(nr) for j in range(nc - 1)]
    vert = [(i * nc + j, (i + 1) * nc + j) for i in range(nr - 1) for j in range(nc)]
    return horiz + vert


def edge_weights(nr: int, nc: int):
    """int64 weights (2^bit) of the passage blocks of a bordered block grid: wE [nr, nc - 1] for
    grid[1::2, 2:-1:2], wS [nr - 1, nc] for grid[2:-1:2, 1::2]."""
    nh = nr * (nc - 1)
    wE = (np.int64(1) << np.arange(nh, dtype=np.int64)).reshape(nr, nc - 1)
    wS = (np.int64(1) << np.arange(nh, nh + (nr - 1) * nc, dtype=np.int64)).reshape(nr - 1, nc)
    return wE, wS


def n_edges(nr: int, nc: int) -> int:
    return nr * (nc - 1) + (nr - 1) * nc


def grid_outcome_id(grid, start) -> int:
    """Outcome of a bordered block grid with start block `start` (odd coordinates)."""
    g = np.asarray(grid)
    nr, nc = (g.shape[0] - 1) // 2, (g.shape[1] - 1) // 2
    wE, wS = edge_weights(nr, nc)
    bits = int(((g[1::2, 2:-1:2] != 0) * wE).sum() + ((g[2:-1:2, 1::2] != 0) * wS).sum())
    s = ((int(start[0]) - 1) // 2) * nc + (int(start[1]) - 1) // 2
    return (s << n_edges(nr, nc)) | bits


def walls_outcome_id(nr, nc, si, sj, E, S) -> int:
    """Outcome of wall planes as oracle.gen_stream.draw_walls returns them."""
    bits, k = 0, 0
    for i in range(nr):
        for j in range(nc - 1):
            bits |= ((E[i] >> j) & 1) << k
            k += 1
    for i in range(nr - 1):
        for j in range(nc):
            bits |= ((S[i] >> j) & 1) << k
            k += 1
    return ((si * nc + sj) << k) | bits


def outcome_grid(oid: int, nr: int, nc: int):
    """(start, grid) of an outcome: bordered block grid, cells and open passages 1, start in block coordinates."""
    ne = n_edges(nr, nc)
    g = np.zeros((2 * nr + 1, 2 * nc + 1), dtype=np.uint8)
    g[1::2, 1::2] = 1
    for k, (a, b) in enumerate(lattice_edges(nr, nc)):
        if (oid >> k) & 1:
            (i1, j1), (i2, j2) = divmod(a, nc), divmod(b, nc)
            g[i1 + i2 + 1, j1 + j2 + 1] = 1
    s = oid >> ne
    return (2 * (s // nc) + 1, 2 * (s % nc) + 1), g


def _adjacency(nr, nc):
    """Per cell: (neighbour, passage bit) in direction order up, down, left, right."""
    index = {e: k for k, e in enumerate(lattice_edges(nr, nc))}
    adj = []
    for c in range(nr * nc):
        i, j = divmod(c, nc)
        out = []
        for di, dj in ((-1, 0), (1, 0), (0, -1), (0, 1)):
            if 0 <= i + di < nr and 0 <= j + dj < nc:
                q = (i + di) * nc + j + dj
                out.append((q, index[(min(c, q), max(c, q))]))
        adj.append(tuple(out))
    return tuple(adj)


def _merge(out, sub, w):
    for k, v in sub.items():
        out[k] = out.get(k, 0.0) + w * v


def _rprim(adj, N, s):
    @lru_cache(maxsize=None)
    def rec(edges, inset):
        frontier = [c for c in range(N) if not (inset >> c) & 1 and any((inset >> q) & 1 for q, _ in adj[c])]
        if not frontier:
            return {edges: 1.0}
        out = {}
        for f in frontier:
            tree_nb = [k for q, k in adj[f] if (inset >> q) & 1]
            for k in tree_nb:
                _merge(out, rec(edges | (1 << k), inset | (1 << f)), 1.0 / (len(frontier) * len(tree_nb)))
        return out
    return rec(0, 1 << s)


def _dfs(adj, N, s):
    @lru_cache(maxsize=None)
    def rec(edges, vis, cur, parents):
        cand = [(q, k) for q, k in adj[cur] if not (vis >> q) & 1]
        if not cand:
            return {edges: 1.0} if cur == s else rec(edges, vis, dict(parents)[cur], parents)
        out = {}
        for q, k in cand:
            _merge(out, rec(edges | (1 << k), vis | (1 << q), q, tuple(sorted(parents + ((q, cur),)))), 1.0 / len(cand))
        return out
    return rec(0, 1 << s, s, ())


def _prim_and_kill(adj, N, s):
    full = (1 << N) - 1

    @lru_cache(maxsize=None)
    def rec(edges, marked, cur):
        cand = [(q, k) for q, k in adj[cur] if not (marked >> q) & 1]
        out = {}
        if cand:
            for q, k in cand:
                _merge(out, rec(edges | (1 << k), marked | (1 << q), q), 1.0 / len(cand))
            return out
        if marked == full:
            return {edges: 1.0}
        elig = [c for c in range(N) if (marked >> c) & 1 and any(not (marked >> q) & 1 for q, _ in adj[c])]
        for c in elig:
            _merge(out, rec(edges, marked, c), 1.0 / len(elig))
        return out
    return rec(0, 1 << s, s)


_ENUMERATORS = {"r-prim": _rprim, "dfs": _dfs, "prim&kill": _prim_and_kill}


@lru_cache(maxsize=None)
def _exact_outcomes(algo, nr, nc):
    adj, N, ne = _adjacency(nr, nc), nr * nc, n_edges(nr, nc)
    out = {}
    for s in range(N):   # lib/maze_generation.py:21: uniform start cell
        for edges, p in _ENUMERATORS[algo](adj, N, s).items():
            out[(s << ne) | edges] = p / N
    return out


def exact_outcomes(algo: str, nr: int, nc: int) -> dict:
    """{outcome id: probability} of generator `algo` on an nr x nc lattice, over all start cells."""
    return dict(_exact_outcomes(algo, int(nr), int(nc)))


def best_of_k(probs: dict, scores: dict, k: int) -> dict:
    """Distribution of the maze kept by best-of-k over i.i.d. draws from `probs`, keeping the lowest
    score with ties (same_score, chained over the sorted scores) going to the first draw:
    P(keep T) = P(T) / P(C) * (P(>= C)^k - P(> C)^k) for T in tie class C.  Any tie-break that does
    not look at which maze is which gives this same distribution."""
    ids = sorted(probs, key=lambda o: scores[o])
    classes, cur = [], [ids[0]]
    for o in ids[1:]:
        if same_score(scores[o], scores[cur[-1]]):
            cur.append(o)
        else:
            classes.append(cur)
            cur = [o]
    classes.append(cur)
    out = {}
    above = 1.0   # P(score >= class), walking from the lowest class up
    for cl in classes:
        pc = sum(probs[o] for o in cl)
        below_next = max(above - pc, 0.0)
        w = (above ** k - below_next ** k) / pc
        for o in cl:
            out[o] = probs[o] * w
        above = below_next
    return out


def chi_square(counts, probs: dict, min_expected: float = 5.0):
    """Pearson chi-square of observed outcome counts ({id: count}, or a dense array indexed by id) against
    `probs`.  Bins expected below `min_expected` are pooled into one (joined to the smallest regular bin
    if the pool is still too small).  Returns (p-value, count of draws outside the support)."""
    from scipy import stats

    if not isinstance(counts, dict):
        c = np.asarray(counts)
        nz = np.nonzero(c)[0]
        counts = dict(zip(nz.tolist(), c[nz].tolist()))
    n = sum(counts.values())
    outside = sum(v for o, v in counts.items() if o not in probs)
    ids = sorted(probs, key=lambda o: probs[o])
    exp = np.array([probs[o] * n for o in ids])
    obs = np.array([counts.get(o, 0) for o in ids], dtype=np.float64)
    small = exp < min_expected
    e, o = list(exp[~small]), list(obs[~small])
    if small.any():
        pe, po = exp[small].sum(), obs[small].sum()
        if pe < min_expected and e:
            e[0] += pe
            o[0] += po
        else:
            e.append(pe)
            o.append(po)
    e, o = np.array(e), np.array(o)
    if len(e) < 2:
        return 1.0, outside
    stat = float(((o - e) ** 2 / e).sum())
    return float(stats.chi2.sf(stat, len(e) - 1)), outside
