"""Distinct tip-code combinations per subtree on the bench's DNA alignment (CPU only).

A node's conditional likelihood depends only on the tip codes below it, so a subtree with few tips has few distinct rows over
the whole alignment.  This script rebuilds the flagship workload's tree and tip codes (bench.py `dna_gtr_g4_1024x1M`: same
seeds, same 16 simulation blocks) and prints, per subtree size in tips, the number of internal nodes and the number of distinct
code combinations each one sees, plus the rows a walk evaluates today (internal nodes x patterns) against the sum of distinct
rows over all internal nodes.

    python tools/subtree_pattern_counts.py [patterns]      (default 1000000: the simulation takes ~10 min on one core)
"""
import json
import pathlib
import sys
import time

import numpy as np

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
from bpp_phyl_b200 import synth  # noqa: E402


def main():
    w = dict(S=4, C=4, taxa=1024, patterns=int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000, alpha=0.5, seed=20260102)
    rng = np.random.default_rng(w["seed"])
    tree = synth.random_tree(w["taxa"], rng, mean_brlen=0.05)
    es = synth.gtr()
    rates, _ = synth.gamma_rates(w["C"], w["alpha"])
    N, nblk = w["patterns"], 16
    t0 = time.time()
    codes = np.concatenate([synth.simulate_tip_codes(tree, es, rates, N // nblk, seed=w["seed"] + 7919 * (k + 1), device="cpu")
                            for k in range(nblk)], axis=1)
    print("simulated %s in %.1f s" % (codes.shape, time.time() - t0), file=sys.stderr)
    leaf_slot = {int(n): k for k, n in enumerate(tree.leaf_nodes)}
    ids, U, tips = {}, np.zeros(tree.nn, np.int64), np.zeros(tree.nn, np.int64)
    for n in range(tree.nn):            # node ids are in post-order: sons come first
        sons = tree.sons(n)
        if len(sons) == 0:
            ids[n] = codes[leaf_slot[n]].astype(np.int64)
            U[n], tips[n] = w["S"], 1
            continue
        key = ids[sons[0]]
        for s in sons[1:]:
            key = key * U[s] + ids[s]
        u, inv = np.unique(key, return_inverse=True)
        ids[n], U[n], tips[n] = inv.astype(np.int64), len(u), tips[sons].sum()
    internal = [n for n in range(tree.nn) if not tree.is_leaf[n]]
    by_tips = {}
    for n in internal:
        if tips[n] <= 4:
            by_tips.setdefault(int(tips[n]), []).append(int(U[n]))
    out = {"patterns": int(codes.shape[1]), "internal_nodes": len(internal),
           "subtrees": {"%d tips" % k: {"nodes": len(v), "distinct_min": min(v), "distinct_max": max(v)}
                        for k, v in sorted(by_tips.items())},
           "rows_evaluated_today": len(internal) * int(codes.shape[1]),
           "distinct_rows_all_internal": int(U[internal].sum())}
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
