"""Fitch parsimony restated in numpy (Parsimony/DRTreeParsimonyScore.cpp: computeScoresFromArrays, testNNI, doNNI), the
double-recursive sets, the change of score of an NNI, the NNI search rule of DESIGN §7b, and an independent per-site Sankoff
programme (unit costs) for binary trees.  Trees are oracle.ref_tree.Node objects; tip sets are uint32 bitsets per pattern.

Node identity across NNIs: ``Node.id`` is kept by do_nni (as Bio++ keeps node ids); ``number`` assigns it once."""
from __future__ import annotations

import copy

import numpy as np

from oracle import ref_tree as rt


def code_sets(code_table):
    """Fitch set of each code: bit x iff code_table[code][x] > 0."""
    t = np.asarray(code_table, float)
    if t.shape[1] > 32:
        raise ValueError("more than 32 states")
    return np.array([sum(1 << x for x in range(t.shape[1]) if row[x] > 0) for row in t], np.uint32)


def leaf_sets(codes_by_name, code_table):
    """{leaf name: [N] uint32 sets} from {leaf name: [N] codes}."""
    s = code_sets(code_table)
    return {k: s[np.asarray(v, np.int64)] for k, v in codes_by_name.items()}


def number(root):
    """Persistent ids: post-order positions at the time of the call."""
    for i, n in enumerate(rt.postorder(root)):
        n.id = i
    return root


def _merge(a, b):
    """Fitch merge of two set arrays: (set, failed-intersection indicator)."""
    i = a & b
    fail = i == 0
    return np.where(fail, a | b, i), fail.astype(np.int64)


def up_sets(root, sets):
    """U[node] (dict by node object) and c[node] (per-pattern failure count of the subtree), sons merged in son order."""
    U, c = {}, {}
    for n in rt.postorder(root):
        if n.is_leaf():
            U[n] = sets[n.name]
            c[n] = np.zeros(len(U[n]), np.int64)
            continue
        b = U[n.sons[0]]
        cnt = sum(c[s] for s in n.sons)
        for s in n.sons[1:]:
            b, f = _merge(b, U[s])
            cnt = cnt + f
        U[n], c[n] = b, cnt
    return U, c


def site_scores(root, sets):
    return up_sets(root, sets)[1][root]


def score(root, sets, w):
    return int(np.dot(np.asarray(w, np.int64), site_scores(root, sets)))


def down_sets(root, U):
    """D[v] for every non-root node: the set of the rest of the tree seen from v, i.e. the merge (in son order) of D[father]
    (when the father is not the root) and U of v's siblings."""
    D = {}
    for n in reversed(rt.postorder(root)):
        for s in n.sons:
            parts = ([D[n]] if n.father is not None else []) + [U[o] for o in n.sons if o is not s]
            b = parts[0]
            for p in parts[1:]:
                b, _ = _merge(b, p)
            D[s] = b
    return D


def _m(P, Q, R, S):
    a, f1 = _merge(P, Q)
    b, f2 = _merge(R, S)
    _, f3 = _merge(a, b)
    return f1 + f2 + f3


def has_nni(v):
    return v.father is not None and v.father.father is not None


def uncle(v):
    f = v.father
    g = f.father
    pos = g.sons.index(f)
    return g.sons[0 if pos > 1 else 1 - pos]


def nni_delta(v, U, D, w):
    """testNNI(v) from the sets: sum_i w_i (m(C, B, A, X) - m(A, B, C, X)) on a binary tree with a three-son root."""
    f = v.father
    g = f.father
    u = uncle(v)
    A, C = U[v], U[u]
    B = U[[s for s in f.sons if s is not v][0]]
    X = U[[s for s in g.sons if s is not f and s is not u][0]] if g.father is None else D[g]
    return int(np.dot(np.asarray(w, np.int64), _m(C, B, A, X) - _m(A, B, C, X)))


def all_nni_deltas(root, sets, w):
    """{node: delta} for every node that has an NNI, and the current score."""
    U, c = up_sets(root, sets)
    D = down_sets(root, U)
    return {v: nni_delta(v, U, D, w) for v in rt.postorder(root) if has_nni(v)}, int(np.dot(np.asarray(w, np.int64), c[root]))


def do_nni(v):
    """doNNI: remove v and its uncle, append the uncle to v's father's sons and v to the grandfather's sons."""
    f = v.father
    g = f.father
    u = uncle(v)
    f.sons.remove(v)
    g.sons.remove(u)
    f.add_son(u)
    g.add_son(v)


def by_id(root):
    return {n.id: n for n in rt.postorder(root)}


def search(root, sets, w, max_rounds=10000):
    """The NNI search rule of DESIGN §7b.  Returns (final tree, [score before round 1, score after each accepted round])."""
    root = copy.deepcopy(root)
    deltas, cur = all_nni_deltas(root, sets, w)
    scores = [cur]
    for _ in range(max_rounds):
        pos = {n: i for i, n in enumerate(rt.postorder(root))}
        cand = sorted((d, pos[v], v) for v, d in deltas.items() if d < 0) if deltas else []
        if not cand:
            break
        taken, used = [], set()
        for d, _, v in cand:
            tri = {v.id, v.father.id, v.father.father.id}
            if tri & used:
                continue
            used |= tri
            taken.append(v.id)
        k = len(taken)
        while True:
            trial = copy.deepcopy(root)
            ids = by_id(trial)
            for i in taken[:k]:
                do_nni(ids[i])
            new = score(trial, sets, w)
            if new < cur or k == 1:
                break
            k //= 2
        assert new < cur, "a single improving NNI must lower the score"
        root, cur = trial, new
        scores.append(cur)
        deltas, _ = all_nni_deltas(root, sets, w)
    return root, scores


def sankoff(root, sets, n_states):
    """Per-pattern minimum number of changes (unit costs; a tip's set members cost 0, others are impossible) by the Sankoff
    dynamic programme: independent of Fitch, exact for any tree."""
    big = 1 << 40
    cost = {}
    states = np.arange(n_states)
    for n in rt.postorder(root):
        if n.is_leaf():
            s = sets[n.name]
            cost[n] = np.where((s[:, None] >> states[None, :].astype(np.uint32)) & 1, 0, big).astype(np.int64)
            continue
        tot = 0
        for s in n.sons:
            cs = cost[s]                                  # [N][S]
            best = cs.min(axis=1, keepdims=True) + 1      # change to any other state
            tot = tot + np.minimum(cs, best)              # min_y cs[y] + [x != y]
        cost[n] = tot
    return cost[root].min(axis=1)


def side_score(v, sets, w):
    """Weighted Fitch score of the tree on the father's side of the edge above v, rebuilt from scratch and rooted at v's
    father (the other side of the edge, scored on its own)."""
    def build(n, came_from):
        c = rt.Node(n.name)
        for m in n.sons + ([n.father] if n.father is not None else []):
            if m is not came_from:
                c.add_son(build(m, n))
        return c
    return score(build(v.father, v), sets, w)
