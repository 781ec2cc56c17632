"""Stochastic mapping of event classes restated in numpy: the estimator of ChromEvol's ComputeChromosomeTransitionsExp
(Mayrose et al. 2010) as bppgpu_simulate_event_counts / bppgpu_expected_events define it (DESIGN §7b).

- ``chromosome_classes``: the generator's off-diagonal split into gain, loss, dupl, demi and baseNum, restating the loops of
  ChromosomeSubstitutionModel::updateQWith* (oracle.ref_models.chromosome) term by term.
- ``conditional_expectation`` (Van Loan) and ``conditional_expectation_fd`` (a complex-step difference of expm): the exact
  E[N_T | y -> x, t] = [int_0^t e^{sQ} Q_T e^{(t-s)Q} ds]_yx / P(t)_yx.
- ``simulate``: the path sampler and its tallies, bit for bit (Philox4x32-10 of oracle.ref_bootstrap).
- ``combine`` / ``exact_expected``: the per-branch expectations from the joint posteriors of
  oracle.ref_likelihood.marginal_posteriors."""
from __future__ import annotations

import math

import numpy as np
from scipy.linalg import expm

from oracle import ref_models as rm
from oracle.ref_bootstrap import philox4x32_10

CLASSES = ("gain", "loss", "dupl", "demi", "baseNum")
_2M53 = 2.0 ** -53


def chromosome_classes(min_chr, max_chr, gain=0.0, loss=0.0, dupl=0.0, demi=rm.IGNORE_PARAM, gain_r=rm.IGNORE_PARAM,
                       loss_r=rm.IGNORE_PARAM, dupl_r=rm.IGNORE_PARAM, base_num=rm.IGNORE_PARAM, base_num_r=rm.IGNORE_PARAM,
                       max_chr_range=0, rate_change="LINEAR"):
    """[5][n][n]: the contribution of each rate term of ChromosomeSubstitutionModel::update() to the class that produced it.
    A clamped duplication, demi-duplication or base-number jump stays in its own class; the two demi/2 targets at odd i are
    both demi.  Added in class order they give oracle.ref_models.chromosome's off-diagonal bit for bit."""
    IG = rm.IGNORE_PARAM
    n = max_chr - min_chr + 1
    R = np.zeros((5, n, n))

    def rate(i, const, lin):
        if const == IG and lin == IG:
            return 0.0
        total = lin if const == IG else const
        if lin == IG:
            return total
        if rate_change == "LINEAR":
            return total + lin * (i - 1)
        return total * math.exp(lin * (i - 1))

    demi_v = dupl if demi == rm.DEMI_EQUAL_DUPL else demi
    G, L, D, DM, B = range(5)
    for i in range(min_chr, max_chr + 1):
        r = i - min_chr
        if i + 1 <= max_chr:
            R[G, r, r + 1] += rate(i, gain, gain_r)
        if i - 1 >= min_chr:
            R[L, r, r - 1] += rate(i, loss, loss_r)
        if 2 * i <= max_chr:
            R[D, r, 2 * i - min_chr] += rate(i, dupl, dupl_r)
        elif i != max_chr:
            R[D, r, max_chr - min_chr] += rate(i, dupl, dupl_r)
        if demi_v != IG and i != max_chr:
            if i % 2 == 0 and int(i * 1.5) <= max_chr:
                R[DM, r, int(i * 1.5) - min_chr] += demi_v
            elif i % 2 != 0 and math.ceil(i * 1.5) <= max_chr:
                if i == 1:
                    R[DM, r, math.ceil(i * 1.5) - min_chr] += demi_v
                else:
                    R[DM, r, math.ceil(i * 1.5) - min_chr] += demi_v / 2
                    R[DM, r, math.floor(i * 1.5) - min_chr] += demi_v / 2
            else:
                R[DM, r, max_chr - min_chr] += demi_v
        if i < max_chr and base_num != IG:
            for j in range(i + 1, max_chr + 1):
                if j == max_chr:
                    if j - i <= max_chr_range:
                        R[B, r, j - min_chr] += base_num_r
                elif (j - i) % int(base_num) == 0 and j - i <= max_chr_range:
                    R[B, r, j - min_chr] += base_num_r
    return R


def class_sum(R):
    """sum over the classes in class order (the order the model adds its terms in)"""
    acc = np.zeros(R.shape[1:])
    for t in range(R.shape[0]):
        acc = acc + R[t]
    return acc


def generator(R):
    """Q with the off-diagonal sum_T R[T] and rows summing to 0"""
    Q = class_sum(R)
    np.fill_diagonal(Q, 0.0)
    np.fill_diagonal(Q, -Q.sum(axis=1))
    return Q


def transition_transversion(Q):
    """[2][4][4]: a nucleotide generator's off-diagonal split into transitions (A<->G, C<->T) and transversions"""
    ts = np.zeros((4, 4), bool)
    for a, b in ((0, 2), (2, 0), (1, 3), (3, 1)):
        ts[a, b] = True
    off = np.array(Q, float) * (1 - np.eye(4))
    return np.stack([np.where(ts, off, 0.0), np.where(ts, 0.0, off)])


def _integral(Q, QT, t):
    """int_0^t e^{sQ} Q_T e^{(t-s)Q} ds (upper-right block of expm(t [[Q, Q_T], [0, Q]]), Van Loan 1978) and P(t)"""
    n = Q.shape[0]
    M = np.zeros((2 * n, 2 * n))
    M[:n, :n] = Q
    M[n:, n:] = Q
    M[:n, n:] = QT
    E = expm(t * M)
    return E[:n, n:], E[:n, :n]


def conditional_expectation(Q, QT, t):
    """E[N_T | y -> x, t] [y][x] (Van Loan); nan where P(t)_yx = 0"""
    I, P = _integral(Q, QT, t)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(P > 0, I / np.where(P > 0, P, 1.0), np.nan)


def conditional_expectation_fd(Q, QT, t, h=1e-30):
    """the same from d/de expm(t (Q + e Q_T)) at e = 0, by a complex-step difference (Im expm(t (Q + i h Q_T)) / h: no
    subtraction, so small entries keep their digits)"""
    d = expm(t * (Q + 1j * h * QT)).imag / h
    P = expm(t * Q)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(P > 0, d / np.where(P > 0, P, 1.0), np.nan)


def conditional_variance(Q, QT, t):
    """Var[N_T | y -> x, t] [y][x]: E[N(N-1)] = 2 [block (1, 3) of expm(t [[Q, Q_T, 0], [0, Q, Q_T], [0, 0, Q]])]_yx / P_yx"""
    n = Q.shape[0]
    M = np.zeros((3 * n, 3 * n))
    for k in range(3):
        M[k * n:(k + 1) * n, k * n:(k + 1) * n] = Q
    M[:n, n:2 * n] = QT
    M[n:2 * n, 2 * n:] = QT
    E = expm(t * M)
    P, I1, I2 = E[:n, :n], E[:n, n:2 * n], E[:n, 2 * n:]
    with np.errstate(invalid="ignore", divide="ignore"):
        m1 = I1 / P
        return np.where(P > 0, 2 * I2 / P + m1 - m1 * m1, np.nan)


def _tables(R):
    """per state: running sums of its non-zero (class, target) entries, T-major and j ascending, padded with +inf; the class
    and target of each entry; the number of entries; r_i (the last running sum, or 0)"""
    T, S, _ = R.shape
    if not np.all(np.isfinite(R)) or np.any(R < 0) or np.any(R[:, np.arange(S), np.arange(S)] != 0):
        raise ValueError("class rates must be finite, >= 0 and 0 on the diagonal")
    rows = []
    for i in range(S):
        flat = R[:, i, :].ravel()                   # (T, j) in T-major order
        nz = np.nonzero(flat)[0]
        rows.append((np.cumsum(flat[nz]), nz // S, nz % S))
    w = max(1, max(len(c) for c, _, _ in rows))
    cum = np.full((S, w), np.inf)
    cls = np.zeros((S, w), np.int64)
    tgt = np.zeros((S, w), np.int64)
    nnz = np.zeros(S, np.int64)
    rate = np.zeros(S)
    for i, (c, t, j) in enumerate(rows):
        cum[i, :len(c)], cls[i, :len(c)], tgt[i, :len(c)], nnz[i] = c, t, j, len(c)
        rate[i] = c[-1] if len(c) else 0.0
    return cum, cls, tgt, nnz, rate


def simulate(R, lengths, n_sims, seed, first=0, starts=None):
    """The tallies of bppgpu_simulate_event_counts: (count [L][S][S] uint64, sum [L][S][S][T] uint64), all paths of all
    start states advanced in lockstep.  ``starts`` limits the start states simulated (the other rows stay 0)."""
    R = np.asarray(R, float)
    T, S, _ = R.shape
    lengths = np.asarray(lengths, float).ravel()
    ulen = np.unique(lengths)
    U = len(ulen)
    row_of = np.searchsorted(ulen, lengths)
    tmax = ulen[-1]
    cum, cls, tgt, nnz, rate = _tables(R)
    st = np.arange(S) if starts is None else np.asarray(starts, np.int64)
    P = len(st) * n_sims
    idx = np.arange(P, dtype=np.uint64)
    a = st[(idx % np.uint64(len(st))).astype(np.int64)]
    n = (np.uint64(first) + idx // np.uint64(len(st))).astype(np.uint64)
    s = a.copy()
    c = np.zeros((P, T), np.int64)
    row = np.zeros(P, np.int64)
    tau = np.zeros(P)
    live = np.ones(P, bool)
    dc = np.zeros((U + 1, S, S), np.int64)          # row U collects the subtractions past the last length
    ds = np.zeros((U + 1, S, S, T), np.int64)

    def add_run(m, r1):
        r0 = row[m]
        np.add.at(dc, (r0, a[m], s[m]), 1)
        np.add.at(dc, (r1, a[m], s[m]), -1)
        for t in range(T):
            np.add.at(ds, (r0, a[m], s[m], t), c[m, t])
            np.add.at(ds, (r1, a[m], s[m], t), -c[m, t])

    k = 0
    key = (seed & 0xFFFFFFFF, seed >> 32)
    while live.any():
        m = np.nonzero(live)[0]
        r = rate[s[m]]
        absorbed = r == 0.0
        if absorbed.any():
            done = m[absorbed]
            add_run(done, np.full(len(done), U))
            live[done] = False
            m, r = m[~absorbed], r[~absorbed]
        if len(m) == 0:
            break
        ctr = np.stack([n[m], a[m].astype(np.uint64), np.full(len(m), k, np.uint64), np.zeros(len(m), np.uint64)], axis=-1)
        x = philox4x32_10(ctr, key).astype(np.uint64)
        h1 = (x[:, 0] | (x[:, 1] << np.uint64(32))) >> np.uint64(11)
        h2 = (x[:, 2] | (x[:, 3] << np.uint64(32))) >> np.uint64(11)
        u1 = (h1 + np.uint64(1)).astype(np.float64) * _2M53
        tau[m] = tau[m] + -np.log(u1) / r
        over = tau[m] > tmax
        if over.any():
            done = m[over]
            add_run(done, np.full(len(done), U))
            live[done] = False
            m, r, h2 = m[~over], r[~over], h2[~over]
        if len(m):
            r1 = np.searchsorted(ulen, tau[m], side="left")
            moved = r1 > row[m]
            if moved.any():
                add_run(m[moved], r1[moved])
                row[m[moved]] = r1[moved]
            v = h2.astype(np.float64) * _2M53 * r
            sm = s[m]
            e = np.argmax(cum[sm] > v[:, None], axis=1)
            e = np.where(cum[sm, e] > v, e, nnz[sm] - 1)
            e = np.minimum(e, nnz[sm] - 1)
            c[m, cls[sm, e]] += 1
            s[m] = tgt[sm, e]
        k += 1
    count = np.cumsum(dc[:U], axis=0).astype(np.uint64)
    sums = np.cumsum(ds[:U], axis=0).astype(np.uint64)
    return count[row_of], sums[row_of]


def combine(count, sums, joints, weights):
    """(E [n_nodes][T], unreached [n_nodes]) of bppgpu_expected_events from tallies per node (count [n][S][S], sum
    [n][S][S][T], indexed by node id) and the joint posteriors {node: [N][S][S] (node state x, father state y)}; nodes absent
    from ``joints`` (the root) get 0."""
    nn, S = count.shape[0], count.shape[1]
    T = sums.shape[-1]
    w = np.asarray(weights, float)
    E = np.zeros((nn, T))
    un = np.zeros(nn)
    for b, J in joints.items():
        W = np.einsum("i,ixy->yx", w, J)             # [y][x]
        cnt = count[b].astype(np.float64)
        hit = count[b] > 0
        mean = np.where(hit[..., None], sums[b].astype(np.float64) / np.where(hit, cnt, 1.0)[..., None], 0.0)
        E[b] = np.einsum("yx,yxt->t", np.where(hit, W, 0.0), mean)
        un[b] = W[~hit].sum()
    return E, un


def exact_expected(Q, R, t_of_node, joints, weights):
    """the limit of ``combine``: sum_i w_i sum_{x,y} J[i][x][y] E[N_T | y -> x, t_b] (Van Loan)"""
    T = R.shape[0]
    w = np.asarray(weights, float)
    E = np.zeros((len(t_of_node), T))
    for b, J in joints.items():
        W = np.einsum("i,ixy->yx", w, J)
        for t in range(T):
            ce = conditional_expectation(Q, R[t], t_of_node[b])
            E[b, t] = np.where(W > 0, W * np.nan_to_num(ce), 0.0).sum()
    return E
