"""Fitch parsimony at the flagship workload's size (1024 taxa x 1M patterns, DNA simulated under GTR+Gamma4, and one 20-state
run): device time of a score call and of an all-NNI call, the bytes each moves over the measured HBM peak, a full NNI search
from the generating tree with 50 random NNIs applied, the oracle's time for one all-NNI pass at a subsample (labelled), and
exact agreement with the oracle on a sample of patterns at full size.

    python tools/bench_parsimony.py --out profiles/r5_parsimony_1024x1M.json

Needs a B200 (no fallback).  Writes only the --out file."""
from __future__ import annotations

import argparse
import copy
import json
import os
import pathlib
import subprocess
import sys
import time

for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):   # the oracle baseline is single-threaded
    os.environ[_v] = "1"
sys.dont_write_bytecode = True
ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

HBM_PEAK_GBS = 6543.0   # measured stream peak of one B200 (DESIGN §3)


def card_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def to_nodes(tree):
    """synth.Tree -> oracle Node objects; leaf names t<slot> (slot = row of simulate_tip_codes' output)"""
    from oracle import ref_tree as rt
    slot = {int(n): k for k, n in enumerate(tree.leaf_nodes)}
    nodes = [rt.Node("t%d" % slot[i] if tree.is_leaf[i] else None) for i in range(tree.nn)]
    for i in range(tree.nn):
        for s in tree.sons(i):
            nodes[i].add_son(nodes[int(s)])
    return nodes[tree.root]


def flat(root):
    from oracle import ref_tree as rt
    nodes = rt.postorder(root)
    idx = {n: i for i, n in enumerate(nodes)}
    off = np.zeros(len(nodes) + 1, np.int32)
    ch = []
    for i, n in enumerate(nodes):
        ch.extend(idx[s] for s in n.sons)
        off[i + 1] = len(ch)
    lr = np.array([int(n.name[1:]) if n.is_leaf() else -1 for n in nodes], np.int32)
    return nodes, (off, np.array(ch, np.int32), len(nodes) - 1, lr)


def pass_bytes(root, N, elem):
    """HBM bytes the passes need: score = tip sets read once, U written once and read once by the father, weights once;
    all-NNI = that plus, per non-root internal node f, four set reads (A0, A1, C, X) and the D[f] write when a son reads it,
    plus the weights once more (they stay in L2 across the edges)."""
    from oracle import ref_tree as rt
    nodes = rt.postorder(root)
    L = sum(n.is_leaf() for n in nodes)
    n_int = len(nodes) - L
    score = elem * N * (L + n_int + (n_int - 1)) + 4 * N
    pre_ops = n_int - 1
    d_writes = sum(1 for n in nodes if n.sons and n.father is not None and any(s.sons for s in n.sons))
    nni = score + elem * N * (4 * pre_ops + d_writes) + 4 * N
    return score, nni


def timed(p, topo, reps):
    s0 = p.score(*topo)
    d0, _ = p.nni_deltas(*topo)
    ts, tn = [], []
    for _ in range(reps):
        assert p.score(*topo) == s0
        ts.append(p.last_ms())
        d, _ = p.nni_deltas(*topo)
        assert np.array_equal(d, d0)
        tn.append(p.last_ms())
    return s0, d0, ts, tn


def search(p, root):
    """The search rule of DESIGN §7b with every score and NNI change from the device.  Returns (tree, scores, NNIs applied)."""
    from oracle import ref_parsimony as rpars
    from oracle import ref_tree as rt
    root = copy.deepcopy(root)
    nodes, topo = flat(root)
    delta, cur = p.nni_deltas(*topo)
    scores, applied = [cur], 0
    while True:
        cand = sorted((int(delta[i]), i) for i in range(len(nodes)) if delta[i] < 0)
        if not cand:
            break
        taken, used = [], set()
        for _, i in cand:
            v = nodes[i]
            tri = {v.id, v.father.id, v.father.father.id}
            if tri & used:
                continue
            used |= tri
            taken.append(v.id)
        k = len(taken)
        while True:
            trial = copy.deepcopy(root)
            ids = rpars.by_id(trial)
            for i in taken[:k]:
                rpars.do_nni(ids[i])
            _, ttopo = flat(trial)
            new = p.score(*ttopo)
            if new < cur or k == 1:
                break
            k //= 2
        assert new < cur
        root, cur = trial, new
        applied += k
        scores.append(cur)
        nodes, topo = flat(root)
        delta, _ = p.nni_deltas(*topo)
    return root, scores, applied


def run(label, tree, es, rates, n_sites, S, a, rng, res):
    from bpp_phyl_b200 import capi, synth
    from oracle import ref_parsimony as rpars
    from oracle import ref_tree as rt
    out = {"states": S, "taxa": tree.n_leaves, "patterns": n_sites}
    t0 = time.time()
    codes = synth.simulate_tip_codes(tree, es, rates, n_sites, seed=a.seed)      # [L][N] uint8 pinned, every site its own pattern
    out["simulate_s"] = time.time() - t0
    w = np.ones(n_sites, np.uint32)
    table = np.eye(S)
    elem = 1 if S <= 8 else 2 if S <= 16 else 4
    true = rpars.number(to_nodes(tree))
    _, topo = flat(true)
    t0 = time.perf_counter()
    p = capi.Parsimony(table, codes, w)
    out["create_s"] = time.perf_counter() - t0
    s0, d0, ts, tn = timed(p, topo, a.reps)
    sb, nb = pass_bytes(true, n_sites, elem)
    out.update({"score_generating_tree": s0, "score_ms": ts, "nni_ms": tn, "score_bytes": sb, "nni_bytes": nb,
                "score_hbm_fraction_best": sb / (min(ts) * 1e-3) / (HBM_PEAK_GBS * 1e9),
                "nni_hbm_fraction_best": nb / (min(tn) * 1e-3) / (HBM_PEAK_GBS * 1e9),
                "improving_nnis_at_generating_tree": int((d0 < 0).sum())})
    # exact agreement on a sample of patterns at full size: per-pattern scores, and every NNI change on the sample alone
    pick = np.sort(rng.choice(n_sites, size=a.check_patterns, replace=False))
    _, sc = p.score(*topo, site_scores=True)
    sets = rpars.leaf_sets({"t%d" % k: codes[k][pick] for k in range(tree.n_leaves)}, table)
    out["sample_patterns"] = int(len(pick))
    out["sample_site_scores_equal"] = bool(np.array_equal(sc[pick].astype(np.int64), rpars.site_scores(true, sets)))
    with capi.Parsimony(table, np.ascontiguousarray(codes[:, pick]), w[pick]) as ps:
        nodes, stopo = flat(true)
        d, s = ps.nni_deltas(*stopo)
        t0 = time.perf_counter()
        ref, cur = rpars.all_nni_deltas(true, sets, w[pick])
        out["oracle_all_nni_s_at_sample"] = time.perf_counter() - t0
        out["oracle_label"] = "numpy oracle, one all-NNI pass over the %d sampled patterns, single thread" % len(pick)
        out["sample_nni_equal"] = bool(s == cur and np.array_equal(d, np.array([ref.get(n, 0) for n in nodes], np.int64)))
    if a.search:
        start = copy.deepcopy(true)
        moved = 0
        while moved < 50:
            cand = [v for v in rt.postorder(start) if rpars.has_nni(v)]
            rpars.do_nni(cand[int(rng.integers(len(cand)))])
            moved += 1
        _, stopo = flat(start)
        s_start = p.score(*stopo)
        t0 = time.perf_counter()
        _, scores, applied = search(p, start)
        out["search"] = {"start": "generating tree with 50 random NNIs", "start_score": s_start, "rounds": len(scores) - 1,
                         "nnis_applied": applied, "wall_s": time.perf_counter() - t0, "final_score": scores[-1],
                         "generating_tree_score": s0, "scores": scores}
    p.close()
    res[label] = out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--taxa", type=int, default=1024)
    ap.add_argument("--sites", type=int, default=1 << 20)
    ap.add_argument("--protein-sites", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--check-patterns", type=int, default=4096)
    ap.add_argument("--no-search", dest="search", action="store_false")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()

    import __graft_entry__ as g
    g.build()
    from bpp_phyl_b200 import synth
    from oracle import ref_models as rm

    res = {"card": card_info(), "hbm_peak_gbs": HBM_PEAK_GBS}
    rng = np.random.default_rng(a.seed)
    tree = synth.random_tree(a.taxa, rng, mean_brlen=0.05)
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    r, _ = rm.gamma_rates(4, 0.5)
    es = {"Q": m.Q, "V": m.V, "Vinv": m.Vinv, "ev": m.ev_re, "pi": m.freq, "rate": m.rate}
    res["dna_model"] = "GTR(1.2,0.8,0.6,1.5,0.9; .3,.2,.25,.25)+Gamma4(0.5)"
    run("dna", tree, es, r, a.sites, 4, a, rng, res)
    if a.protein_sites:
        esp = synth.random_reversible(20, np.random.default_rng(a.seed + 1))
        res["protein_model"] = "random reversible 20-state model (synth.random_reversible, seed %d)+Gamma4(0.5)" % (a.seed + 1)
        run("protein", tree, esp, r, a.protein_sites, 20, a, rng, res)
    res["card_after"] = card_info()
    pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items()}))


if __name__ == "__main__":
    main()
