"""Distinct tip-code combinations per subtree on the bench's DNA alignment (CPU only).

A node's conditional likelihood depends only on the tip codes below it, so a subtree with few tips has few distinct rows over
the whole alignment.  This script rebuilds the flagship workload's tree and tip codes (bench.py `dna_gtr_g4_1024x1M`: same
seeds, same 16 simulation blocks) and prints, per subtree size in tips, the number of internal nodes and the number of distinct
code combinations each one sees, plus the rows a walk evaluates today (internal nodes x patterns) against the sum of distinct
rows over all internal nodes.  It also counts the subtrees the DNA walk folds into wide tip tables (walk4c: cherries under a
binary father, three-tip subtrees -- a folded cherry and a tip under a binary node whose father is binary) and the flop per
(pattern, rate class) row of the walk program left over: 4 per product of two sons and 28 per contraction of an internal
son with its branch P (a tip, or a folded subtree, is a table gather).

    python tools/subtree_pattern_counts.py [patterns]      (default 1000000: the simulation takes ~10 min on one core)
"""
import json
import pathlib
import sys
import time

import numpy as np

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
from bpp_phyl_b200 import synth  # noqa: E402


def folded_programs(tree):
    """ops and flop per (pattern, class) row of the walk program: unfolded, with folded cherries, with folded cherries and
    three-tip subtrees (the planner's rule in engine.cu, at four codes: 16 pairs and 64 triples fit a one-byte row code)"""
    sons = [list(tree.sons(n)) for n in range(tree.nn)]
    tip = [len(s) == 0 for s in sons]
    binary = [len(s) == 2 for s in sons]
    cherry, three = [False] * tree.nn, [False] * tree.nn
    for f in range(tree.nn):
        if binary[f]:
            for n in sons[f]:
                cherry[n] = binary[n] and tip[sons[n][0]] and tip[sons[n][1]]
    for f in range(tree.nn):
        if binary[f]:
            for n in sons[f]:
                s = sons[n]
                three[n] = binary[n] and ((cherry[s[0]] and tip[s[1]]) or (tip[s[0]] and cherry[s[1]]))

    def program(folded):
        leafish = [tip[n] or folded[n] for n in range(tree.nn)]
        absorbed = [False] * tree.nn                 # ops inside a folded subtree
        for n in range(tree.nn - 1, -1, -1):       # fathers have larger ids
            for s in sons[n]:
                absorbed[s] = absorbed[n] or leafish[n]
        ops = [n for n in range(tree.nn) if not leafish[n] and not absorbed[n]]
        flop = sum(4 * (len(sons[n]) - 1) + 28 * sum(not leafish[s] for s in sons[n]) for n in ops)
        return {"ops": len(ops), "flop_per_row": flop}

    none = [False] * tree.nn
    return {"foldable_cherries": sum(cherry), "foldable_three_tip_subtrees": sum(three),
            "fathers_of_two_three_tip_subtrees": sum(1 for f in range(tree.nn) if binary[f] and all(three[s] for s in sons[f])),
            "unfolded": program(none), "cherries_folded": program(cherry),
            "cherries_and_three_tip_folded": program([cherry[n] or three[n] for n in range(tree.nn)])}


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
           "distinct_rows_all_internal": int(U[internal].sum()),
           "walk4c_folding": folded_programs(tree)}
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
