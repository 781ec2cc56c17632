"""The parsimony bootstrap restated in numpy (bppPars: SiteContainerTools::bootstrap, then a search per replicate, then
TreeTools::computeBootstrapValues): the replicate-weight sampler of bppgpu_bootstrap_weights bit for bit (Philox4x32-10 as
defined by Random123, Salmon et al. 2011), the bipartitions of a tree, and the support of each branch.  The replicate search
itself is oracle.ref_parsimony.search with a replicate's weights."""
from __future__ import annotations

import math

import numpy as np

from oracle import ref_tree as rt

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def philox4x32_10(ctr, key):
    """Philox4x32-10 of counters ctr [..., 4] under key (k0, k1): uint32 [..., 4]."""
    c = [np.asarray(ctr, np.uint64)[..., i] & _LO for i in range(4)]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for r in range(10):
        if r:
            k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
        p0, p1 = _M0 * c[0], _M1 * c[2]             # < 2^64: no wrap
        c = [(p1 >> _32) ^ c[1] ^ np.uint64(k0), p1 & _LO, (p0 >> _32) ^ c[3] ^ np.uint64(k1), p0 & _LO]
    return np.stack(c, axis=-1).astype(np.uint32)


def draws(n_sites, replicate, seed):
    """The n_sites sites replicate `replicate` draws: floor(u * n_sites / 2^64), u = x0 | x1 << 32 of counter (j lo, j hi,
    replicate, 0) under key (seed lo, seed hi)."""
    j = np.arange(n_sites, dtype=np.uint64)
    ctr = np.stack([j & _LO, j >> _32, np.full(n_sites, replicate, np.uint64), np.zeros(n_sites, np.uint64)], axis=-1)
    x = philox4x32_10(ctr, (seed & 0xFFFFFFFF, seed >> 32)).astype(np.uint64)
    n = np.uint64(n_sites)
    # multiply-high of the 64-bit u by n < 2^32, in 64-bit pieces: (x1 * n + (x0 * n >> 32)) >> 32
    return ((x[:, 1] * n + ((x[:, 0] * n) >> _32)) >> _32).astype(np.int64)


def bootstrap_weights(indices, n_patterns, n_replicates, seed, first=0):
    """[n_replicates][n_patterns] uint32: how often replicate first + r drew a site of each pattern."""
    idx = np.asarray(indices, np.int64)
    out = np.zeros((n_replicates, n_patterns), np.uint32)
    for r in range(n_replicates):
        out[r] = np.bincount(idx[draws(len(idx), first + r, seed)], minlength=n_patterns)
    return out


def bipartitions(root):
    """{node: split} for every non-root node of the tree: the leaves below the node's branch or the rest, whichever side
    does not hold the first leaf in sorted-name order, as a frozenset of names.  On a rooted tree the root's two branches
    give the same split."""
    names = sorted(l.name for l in rt.leaves(root))
    every, first = frozenset(names), names[0]
    below = {}
    out = {}
    for n in rt.postorder(root):
        below[n] = frozenset([n.name]) if n.is_leaf() else frozenset().union(*(below[s] for s in n.sons))
        if n.father is not None:
            out[n] = every - below[n] if first in below[n] else below[n]
    return out


def _round(x, digits):
    f = 10.0 ** digits
    return math.floor(x * f + 0.5) / f


def bootstrap_values(tree, trees, fmt=0):
    """TreeTools::computeBootstrapValues: {internal non-root node of `tree`: percentage of `trees` that contain its split},
    rounded half up to `fmt` decimals.  Leaf branches get none; a tree with another leaf set raises."""
    leaf_set = {l.name for l in rt.leaves(tree)}
    count = {}
    for t in trees:
        if {l.name for l in rt.leaves(t)} != leaf_set:
            raise ValueError("a replicate tree has another leaf set")
        for sp in set(bipartitions(t).values()):
            count[sp] = count.get(sp, 0) + 1
    return {n: _round(100.0 * count.get(sp, 0) / len(trees), fmt) for n, sp in bipartitions(tree).items() if not n.is_leaf()}
