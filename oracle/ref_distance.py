"""Distance methods of the reference (Distance/), restated on the CPU.  TEST INFRASTRUCTURE ONLY.

pair_distance: DistanceEstimation::computeMatrix's inner step (Distance/DistanceEstimation.cpp) for one pair i < j: the two
sequences' columns are compressed on their own (TwoTreeLikelihood's site patterns), P comes from ref_models.pij_t, and the single
branch length is maximised over TwoTreeLikelihood's bounds [1e-6, 1e4].  The optimiser here is not the reference's (bpp-core is
not in the tree); parity is on the optimum: a dense log grid, then bounded Brent (scipy) in log t around the best grid point, then
(an interior optimum) the root of d lnL / dt near it by brentq, which pins t far below the sqrt(eps) that a search on lnL values
alone can resolve.
Conventions shared with the device: a pair whose every site involves a fully ambiguous code is flat and returns 1e-6 (the
reference's start value), an optimum on a bound returns the bound, and f_uv(t) <= 0 counts as lnL = -inf.

bionj: Gascuel's BIONJ (Mol. Biol. Evol. 14:685-695, 1997) as Bio++'s BioNJ runs it (Distance/BioNJ.cpp,
Distance/NeighborJoining.cpp): criterion S_i + S_j - (n - 2) D_ij maximised, first pair in row-major order on ties, variances
initialised to the distances.
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import brentq, minimize_scalar

from . import ref_models as rm

T_MIN, T_MAX = 1e-6, 1e4


def pair_counts(code_a, code_b, weights, n_codes):
    """TwoTreeLikelihood's compression of the pair's columns, as a [n_codes][n_codes] table of summed weights."""
    n = np.zeros((n_codes, n_codes), np.int64)
    np.add.at(n, (np.asarray(code_a, np.int64), np.asarray(code_b, np.int64)), np.asarray(weights, np.int64))
    return n


def pair_lnl(n, table, model: rm.Model, rates, probs, t):
    """lnL_ab(t) = sum_uv n[u][v] log f_uv(t), f_uv = sum_c p_c sum_x pi_x e_u(x) (P(r_c t) e_v)(x); -inf if some f <= 0."""
    E = np.asarray(table, float)
    F = np.zeros((E.shape[0], E.shape[0]))
    for r, p in zip(rates, probs):
        F += p * (E * model.freq[None, :]) @ rm.pij_t(model, r * t) @ E.T
    m = n > 0
    if np.any(F[m] <= 0):
        return -np.inf
    return float(np.sum(n[m] * np.log(F[m])))


def pair_derivatives(n, table, model: rm.Model, rates, probs, t):
    """(d lnL_ab / dt, d2 lnL_ab / dt2) from ref_models.dpij_dt / d2pij_dt2."""
    E = np.asarray(table, float)
    EP = E * model.freq[None, :]
    F, F1, F2 = (np.zeros((E.shape[0], E.shape[0])) for _ in range(3))
    for r, p in zip(rates, probs):
        F += p * EP @ rm.pij_t(model, r * t) @ E.T
        F1 += p * r * EP @ rm.dpij_dt(model, r * t) @ E.T
        F2 += p * r * r * EP @ rm.d2pij_dt2(model, r * t) @ E.T
    m = n > 0
    r1 = F1[m] / F[m]
    return float(np.sum(n[m] * r1)), float(np.sum(n[m] * (F2[m] / F[m] - r1 * r1)))


def pair_distance(code_a, code_b, weights, table, model: rm.Model, rates, probs, n_grid=201):
    """(distance, lnL at the distance) of one pair, code_a the root-side sequence."""
    E = np.asarray(table, float)
    n = pair_counts(code_a, code_b, weights, E.shape[0])
    amb = np.all(E == 1.0, axis=1)
    u, v = np.nonzero(n)
    if not np.any(~amb[u] & ~amb[v]):
        return T_MIN, pair_lnl(n, E, model, rates, probs, T_MIN)
    f = lambda t: pair_lnl(n, E, model, rates, probs, t)
    grid = np.exp(np.linspace(np.log(T_MIN), np.log(T_MAX), n_grid))
    grid[0], grid[-1] = T_MIN, T_MAX
    vals = np.array([f(t) for t in grid])
    ib = int(len(vals) - 1 - np.argmax(vals[::-1]))          # last maximum: a plateau at large t belongs to the upper bound
    lo, hi = np.log(grid[max(ib - 1, 0)]), np.log(grid[min(ib + 1, n_grid - 1)])
    res = minimize_scalar(lambda x: -f(np.exp(x)), bounds=(lo, hi), method="bounded", options={"xatol": 1e-13})
    tb = float(np.exp(res.x))
    cands = [(f(tb), tb), (vals[ib], grid[ib])]
    dl = lambda t: pair_derivatives(n, E, model, rates, probs, t)[0]
    a, b = tb * (1 - 1e-3), min(tb * (1 + 1e-3), T_MAX)
    root = None
    if T_MIN < a and np.isfinite(f(a)) and dl(a) > 0 > dl(b):
        tr = brentq(dl, a, b, xtol=1e-15 * tb, rtol=1e-15)
        root = (f(tr), tr)
        cands.append(root)
    if ib == 0:
        cands.append((vals[0], T_MIN))
    if ib == n_grid - 1:
        cands.append((vals[-1], T_MAX))
    best = max(c[0] for c in cands)
    bound = [c for c in cands if c[0] == best and c[1] in (T_MIN, T_MAX)]
    if bound:
        lnl, t = bound[0]
    elif root is not None and root[0] >= best - 1e-13 * abs(best):   # lnL values of points this close differ by rounding only
        lnl, t = root
    else:
        lnl, t = max(cands)
    return float(t), float(lnl)


def distance_matrix(codes, weights, table, model: rm.Model, rates, probs, pairs=None):
    """dist, lnl [L][L] for all pairs (or only `pairs`, a list of (a, b) with a < b; others left NaN)."""
    L = len(codes)
    dist = np.full((L, L), np.nan)
    lnl = np.full((L, L), np.nan)
    np.fill_diagonal(dist, 0.0)
    np.fill_diagonal(lnl, 0.0)
    for a, b in (pairs if pairs is not None else [(a, b) for a in range(L) for b in range(a + 1, L)]):
        d, l = pair_distance(codes[a], codes[b], weights, table, model, rates, probs)
        dist[a, b] = dist[b, a] = d
        lnl[a, b] = lnl[b, a] = l
    return dist, lnl


def bionj(D, names=None, rooted=False, positive_lengths=False):
    """Returns the tree as nested tuples: a leaf is its name, an internal node is [(child, length), ...]."""
    D = np.array(D, float)
    n = D.shape[0]
    names = [str(i) for i in range(n)] if names is None else list(names)
    V = D.copy()
    nodes = {i: names[i] for i in range(n)}
    active = list(range(n))
    clamp = (lambda x: max(x, 0.0)) if positive_lengths else (lambda x: x)
    while len(active) > (2 if rooted else 3):
        m = len(active)
        idx = np.array(active)
        sub = D[np.ix_(idx, idx)]
        S = np.array([sum(sub[i, k] for k in range(m)) for i in range(m)])   # id order, as the reference's loop
        crit = S[:, None] + S[None, :] - (m - 2) * sub
        crit[np.tril_indices(m)] = -np.inf
        k = int(np.argmax(crit))                                           # first maximum in row-major order
        i, j = active[k // m], active[k % m]
        ratio = (S[k // m] - S[k % m]) / (m - 2)
        di, dj = clamp(0.5 * (D[i, j] + ratio)), clamp(0.5 * (D[i, j] - ratio))
        if V[i, j] == 0:
            lam = 0.5
        else:
            lam = sum(V[j, x] - V[i, x] for x in active if x not in (i, j)) / (2 * (m - 2) * V[i, j]) + 0.5
        lam = min(max(lam, 0.0), 1.0)
        parent = [(nodes[i], di), (nodes[j], dj)]
        for x in active:
            if x in (i, j):
                continue
            d = clamp(lam * (D[i, x] - di) + (1 - lam) * (D[j, x] - dj))
            v = lam * V[i, x] + (1 - lam) * V[j, x] - lam * (1 - lam) * V[i, j]
            D[i, x] = D[x, i] = d
            V[i, x] = V[x, i] = v
        nodes[i] = parent
        active.remove(j)
        del nodes[j]
    if rooted:
        i, j = active
        return [(nodes[i], D[i, j] / 2), (nodes[j], D[i, j] / 2)]
    i, j, k = active
    return [(nodes[i], clamp(D[i, j] + D[i, k] - D[j, k]) / 2), (nodes[j], clamp(D[j, i] + D[j, k] - D[i, k]) / 2),
            (nodes[k], clamp(D[k, i] + D[k, j] - D[i, j]) / 2)]


def splits(tree):
    """{split: length} of a bionj() tree (see canonical_splits)."""
    out = {}
    allv = set()

    def walk(node):
        if not isinstance(node, list):
            allv.add(node)
            return frozenset([node])
        below = frozenset()
        for child, length in node:
            s = walk(child)
            out[s] = out.get(s, 0.0) + length
            below |= s
        return below

    walk(tree)
    return canonical_splits(out, frozenset(allv))


def canonical_splits(raw, leaves):
    """Splits keyed by the side that does not contain the smallest leaf name; lengths of the same split are added (the two
    branches at a bifurcating root form one edge)."""
    ref = min(leaves)
    out = {}
    for s, length in raw.items():
        key = s if ref not in s else leaves - s
        if len(key) == 0 or len(key) == len(leaves):
            continue
        out[key] = out.get(key, 0.0) + length
    return out
