"""Fitch parsimony (bppgpu_parsimony_*: DRTreeParsimonyScore's score, per-site scores and testNNI for every node) and the NNI
search (the shim's OptimizationTools::optimizeTreeNNI), against oracle/ref_parsimony.py.

CPU: the oracle's Fitch score against its Sankoff programme, the per-edge identity of the double-recursive sets, every NNI's
change of score against rescoring from scratch, the search rule's invariants, and the shim compiling.  GPU: every integer
compared exactly with the oracle across set widths, code widths, weights, pattern counts, tree shapes and pattern blocks; the
NNI changes of score; error paths; memory kinds; and the shim end to end."""
import copy
import pathlib
import subprocess

import numpy as np
import pytest

import cases
from oracle import ref_models as rm
from oracle import ref_parsimony as rpars
from oracle import ref_tree as rt
from test_cpp_shim import compile_cpp

ROOT = pathlib.Path(__file__).resolve().parent.parent
HEAVY = (1, 127, 2 ** 31, 2 ** 32 - 1)


def _table(rng, S, n_amb=3, gap=False):
    """identity rows, a fully ambiguous row, n_amb random non-empty subsets; with gap, one more state (bit S-1) that only the
    last code has"""
    base = S - 1 if gap else S
    rows = [np.eye(S)[x] for x in range(base)]
    full = np.zeros(S)
    full[:base] = 1
    rows.append(full)
    for _ in range(n_amb):
        r = np.zeros(S)
        r[rng.choice(base, size=int(rng.integers(2, base + 1)), replace=False)] = 1
        rows.append(r)
    if gap:
        rows.append(np.eye(S)[S - 1])
    return np.array(rows)


def _codes(rng, L, N, K, dtype=np.uint8):
    return rng.integers(K, size=(L, N)).astype(dtype)


def _sets(codes, table, names):
    return rpars.leaf_sets({nm: codes[i] for i, nm in enumerate(names)}, table)


def _flat(root, row_of):
    nodes = rt.postorder(root)
    idx = {n: i for i, n in enumerate(nodes)}
    off = np.zeros(len(nodes) + 1, np.int32)
    ch = []
    for i, n in enumerate(nodes):
        ch.extend(idx[s] for s in n.sons)
        off[i + 1] = len(ch)
    leaf_row = np.array([row_of[n.name] if n.is_leaf() else -1 for n in nodes], np.int32)
    return nodes, (off, np.array(ch, np.int32), len(nodes) - 1, leaf_row)


def _tree(n, rng, rooted=False):
    return rt.random_tree(n, rng, rooted=rooted)


def _names(root):
    return [l.name for l in rt.leaves(root)]


def _multifurcate(root, rng, p=0.4):
    for n in rt.postorder(root):
        if n.father is not None and n.sons and rng.random() < p:
            f = n.father
            i = f.sons.index(n)
            f.sons[i:i + 1] = n.sons
            for s in n.sons:
                s.father = f
    return root


def _caterpillar(n):
    cur = rt.Node("t0")
    for k in range(1, n):
        p = rt.Node()
        p.add_son(cur)
        p.add_son(rt.Node("t%d" % k))
        cur = p
    return cur


# ---- CPU: the oracle against itself ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [4, 20])
def test_oracle_fitch_equals_sankoff(S):
    rng = np.random.default_rng(S)
    for n in (4, 7, 13, 40):
        root = _tree(n, rng)
        table = _table(rng, S)
        codes = _codes(rng, n, 200, len(table))
        sets = _sets(codes, table, _names(root))
        assert np.array_equal(rpars.site_scores(root, sets), rpars.sankoff(root, sets, S))


def test_oracle_every_edge_gives_the_total():
    rng = np.random.default_rng(5)
    for n in (4, 9, 25):
        root = _tree(n, rng)
        table = _table(rng, 4)
        sets = _sets(_codes(rng, n, 150, len(table)), table, _names(root))
        w = rng.integers(1, 50, size=150)
        U, c = rpars.up_sets(root, sets)
        D = rpars.down_sets(root, U)
        total = rpars.score(root, sets, w)
        for v in rt.postorder(root)[:-1]:
            s_up = int(np.dot(w, c[v]))
            s_down = rpars.side_score(v, sets, w)
            assert s_up + s_down + int(np.dot(w, (U[v] & D[v]) == 0)) == total


def test_oracle_delta_equals_rescoring():
    rng = np.random.default_rng(6)
    for n, S in ((5, 4), (12, 4), (30, 20)):
        root = rpars.number(_tree(n, rng))
        table = _table(rng, S)
        sets = _sets(_codes(rng, n, 120, len(table)), table, _names(root))
        w = rng.integers(1, 9, size=120)
        deltas, cur = rpars.all_nni_deltas(root, sets, w)
        assert len(deltas) == 2 * (n - 3)
        for v, d in deltas.items():
            t = copy.deepcopy(root)
            rpars.do_nni(rpars.by_id(t)[v.id])
            assert rpars.score(t, sets, w) - cur == d


def test_oracle_search_rounds_decrease_and_end_at_a_local_optimum():
    rng = np.random.default_rng(7)
    root = rpars.number(_tree(30, rng))
    table = _table(rng, 4)
    sets = _sets(_codes(rng, 30, 300, len(table)), table, _names(root))
    w = rng.integers(1, 5, size=300)
    final, scores = rpars.search(root, sets, w)
    assert len(scores) > 1 and all(b < a for a, b in zip(scores, scores[1:]))
    deltas, cur = rpars.all_nni_deltas(final, sets, w)
    assert cur == scores[-1] and min(deltas.values()) >= 0


def test_shim_compiles_with_parsimony_header(built_lib):
    compile_cpp("test_parsimony", built_lib)


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
def _check_score(root, codes, table, w, max_bytes=0):
    from bpp_phyl_b200 import capi
    names = ["t%d" % i for i in range(codes.shape[0])]
    sets = _sets(codes, table, names)
    _, topo = _flat(root, {nm: i for i, nm in enumerate(names)})
    with capi.Parsimony(table, codes, w, max_bytes=max_bytes) as p:
        s, sc = p.score(*topo, site_scores=True)
    ref = rpars.site_scores(root, sets)
    assert np.array_equal(sc.astype(np.int64), ref)
    assert s == int(np.dot(np.asarray(w, np.int64), ref))


@pytest.mark.gpu
@pytest.mark.parametrize("S", [4, 8, 9, 16, 17, 20, 32])
@pytest.mark.parametrize("N", [1, 31, 33, 4099])
def test_score_matches_oracle_set_widths(built_lib, S, N):
    rng = np.random.default_rng(S * 10007 + N)
    root = _tree(23, rng)
    table = _table(rng, S, n_amb=5)
    codes = _codes(rng, 23, N, len(table))
    w = rng.choice(HEAVY, size=N).astype(np.uint32)
    _check_score(root, codes, table, w)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["rooted", "multifurcating", "caterpillar500", "two_taxa", "star"])
@pytest.mark.parametrize("code_dtype", [np.uint8, np.uint16])
def test_score_matches_oracle_tree_shapes(built_lib, shape, code_dtype):
    rng = np.random.default_rng(11)
    if shape == "rooted":
        root = _tree(40, rng, rooted=True)
    elif shape == "multifurcating":
        root = _multifurcate(_tree(60, rng), rng)
        assert max(len(n.sons) for n in rt.postorder(root)) > 3
    elif shape == "caterpillar500":
        root = _caterpillar(500)
    elif shape == "two_taxa":
        root = rt.parse_newick("(t0,t1);")
    else:
        root = rt.parse_newick("(t0,t1,t2,t3,t4);")
    L = len(_names(root))
    table = _table(rng, 4, n_amb=6, gap=False)
    codes = _codes(rng, L, 777, len(table), code_dtype)
    w = rng.integers(1, 1000, size=777).astype(np.uint32)
    _check_score(root, codes, table, w)


@pytest.mark.gpu
def test_score_include_gaps_and_heavy_weights(built_lib):
    rng = np.random.default_rng(12)
    root = _tree(50, rng)
    table = _table(rng, 5, n_amb=4, gap=True)        # DNA + a gap bit of its own
    codes = _codes(rng, 50, 2000, len(table))
    w = rng.choice(HEAVY, size=2000).astype(np.uint32)
    _check_score(root, codes, table, w)


@pytest.mark.gpu
@pytest.mark.parametrize("max_bytes", [1, 64 * 97, 100000])
def test_pattern_blocks_add_up(built_lib, max_bytes):
    """max_bytes forces many pattern blocks (one pattern each at 1 byte); totals, per-pattern scores and NNI changes stay exact"""
    from bpp_phyl_b200 import capi
    rng = np.random.default_rng(13)
    root = rpars.number(_tree(40, rng))
    table = _table(rng, 20, n_amb=4)
    N = 3001
    codes = _codes(rng, 40, N, len(table))
    w = rng.choice(HEAVY, size=N).astype(np.uint32)
    _check_score(root, codes, table, w, max_bytes=max_bytes)
    _check_nni(root, codes, table, w, max_bytes=max_bytes)


def _check_nni(root, codes, table, w, max_bytes=0):
    from bpp_phyl_b200 import capi
    names = ["t%d" % i for i in range(codes.shape[0])]
    sets = _sets(codes, table, names)
    nodes, topo = _flat(root, {nm: i for i, nm in enumerate(names)})
    with capi.Parsimony(table, codes, w, max_bytes=max_bytes) as p:
        delta, s = p.nni_deltas(*topo)
    ref, cur = rpars.all_nni_deltas(root, sets, w)
    assert s == cur
    want = np.array([ref.get(n, 0) for n in nodes], np.int64)
    assert np.array_equal(delta, want)
    return delta


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5, 6, 17, 64, 300])
@pytest.mark.parametrize("S", [4, 20])
def test_nni_deltas_match_oracle(built_lib, n, S):
    rng = np.random.default_rng(n * 31 + S)
    root = _tree(n, rng)
    table = _table(rng, S, n_amb=3)
    N = 2500
    codes = _codes(rng, n, N, len(table))
    w = rng.choice(HEAVY, size=N).astype(np.uint32)
    _check_nni(root, codes, table, w)


@pytest.mark.gpu
def test_nni_deltas_match_oracle_1024_taxa_100k_patterns(built_lib):
    """simulated DNA (so that most NNIs are not ties), 1024 taxa x 100k patterns"""
    r, p = rm.gamma_rates(4, 0.5)
    c = cases.make_case(1024, 100000, rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25)), r, p, seed=14, ambiguity=0.02,
                        compress=False)
    root = c.flat.root_node
    names = c.flat.leaf_names
    codes = np.stack([c.codes_by_leaf[l] for l in c.flat.leaf_ids])
    row = {nm: int(nm[1:]) for nm in names}
    ordered = np.empty_like(codes)
    for i, nm in enumerate(names):
        ordered[row[nm]] = codes[i]
    delta = _check_nni(root, ordered, c.table, np.asarray(c.weights, np.uint32))
    assert (delta > 0).any()


@pytest.mark.gpu
def test_error_paths(built_lib):
    from bpp_phyl_b200 import capi
    rng = np.random.default_rng(15)
    codes = _codes(rng, 4, 10, 4)
    w = np.ones(10, np.uint32)
    creates = [
        lambda: capi.Parsimony(np.eye(33), codes, w),                                 # 33 bits
        lambda: capi.Parsimony(np.eye(4), np.full((4, 10), 4, np.uint8), w),          # code >= n_codes
        lambda: capi.Parsimony(np.vstack([np.eye(4), np.zeros((1, 4))]), codes, w),   # empty code row
        lambda: capi.Parsimony(np.eye(4), codes[:1], w),                              # one sequence
    ]
    for f in creates:
        with pytest.raises(capi.BppGpuError) as e:
            f()
        assert e.value.code == capi.E_INVALID
    root = rt.parse_newick("((t0,t1),t2,t3);")
    nodes, (off, ch, r, lr) = _flat(root, {"t%d" % i: i for i in range(4)})
    with capi.Parsimony(np.eye(4), codes, w) as p:
        assert p.score(off, ch, r, lr) >= 0
        bad = [
            (off, ch, r, np.where(lr == 1, 0, lr)),                   # two leaves, one row
            (off, ch, r, np.where(lr == 1, 4, lr)),                   # row out of range
            (off, np.where(ch == 0, 1, ch), r, lr),                   # node 1 reached twice, node 0 never
            (off, ch, 0, lr),                                         # root is a leaf
            (off, ch, len(lr), lr),                                   # root out of range
        ]
        for topo in bad:
            with pytest.raises(capi.BppGpuError) as e:
                p.score(*topo)
            assert e.value.code == capi.E_INVALID
    star = rt.parse_newick("(t0,t1,(t2,t3,t4));")
    codes5 = _codes(rng, 5, 10, 4)
    with capi.Parsimony(np.eye(4), codes5, w) as p:
        _, topo = _flat(star, {"t%d" % i: i for i in range(5)})
        assert p.score(*topo) >= 0
        with pytest.raises(capi.BppGpuError) as e:
            p.nni_deltas(*topo)
        assert e.value.code == capi.E_INVALID


@pytest.mark.gpu
def test_memory_kinds_pageable_pinned_device(built_lib):
    import torch
    from bpp_phyl_b200 import capi
    rng = np.random.default_rng(16)
    L, n_sites = 24, 20000
    cols = rng.integers(6, size=(n_sites, L)).astype(np.uint8)
    cols[: n_sites // 2] = cols[0]
    table = _table(rng, 4, n_amb=1)
    ps, wt, ix, tip = capi.site_patterns_device(cols)
    root = _tree(L, rng)
    _, topo = _flat(root, {"t%d" % i: i for i in range(L)})
    res = []
    with capi.Parsimony(table, np.ascontiguousarray(tip), wt) as p:
        res.append((p.score(*topo, site_scores=True), p.nni_deltas(*topo)))
    pc = torch.from_numpy(np.ascontiguousarray(tip)).pin_memory()
    pw = torch.from_numpy(np.ascontiguousarray(wt).view(np.int32)).pin_memory()
    with capi.Parsimony(table, pc.data_ptr(), pw.data_ptr(), n_leaves=L, n_patterns=len(wt), code_bytes=1) as p:
        res.append((p.score(*topo, site_scores=True), p.nni_deltas(*topo)))
    dcols = torch.from_numpy(cols).cuda()
    d_ps = torch.empty(n_sites, dtype=torch.int64, device="cuda")
    d_wt = torch.empty(n_sites, dtype=torch.int32, device="cuda")
    d_ix = torch.empty(n_sites, dtype=torch.int64, device="cuda")
    d_tip = torch.empty(n_sites * L, dtype=torch.uint8, device="cuda")
    npat = capi.site_patterns_device_raw(dcols.data_ptr(), n_sites, L, d_ps.data_ptr(), d_wt.data_ptr(), d_ix.data_ptr(),
                                         d_tip.data_ptr())
    assert npat == len(wt)
    with capi.Parsimony(table, d_tip.data_ptr(), d_wt.data_ptr(), n_leaves=L, n_patterns=npat, code_bytes=1) as p:
        res.append((p.score(*topo, site_scores=True), p.nni_deltas(*topo)))
    for (s, sc), (d, s2) in res[1:]:
        assert s == res[0][0][0] and np.array_equal(sc, res[0][0][1])
        assert s2 == res[0][1][1] and np.array_equal(d, res[0][1][0])
    sets = _sets(np.asarray(tip), table, ["t%d" % i for i in range(L)])
    assert res[0][0][0] == rpars.score(root, sets, np.asarray(wt))


def _parse_scores(lines, key):
    return [int(x) for l in lines if l.startswith(key + " ") for x in l.split()[1:]]


@pytest.mark.gpu
def test_shim_bionj_parsimony_nni_search(built_lib, tmp_path):
    """DistanceEstimation -> BioNJ -> DRTreeParsimonyScore -> optimizeTreeNNI on DNA simulated down a 60-taxon tree: the
    sequence of scores equals the oracle's run of the same rule from the same start, no NNI improves the final tree, and the
    final score is not above the generating tree's."""
    rng = np.random.default_rng(17)
    r, p = rm.gamma_rates(4, 0.5)
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    true = rt.random_tree(60, rng, mean_brlen=0.08)
    flat = rt.FlatTree(copy.deepcopy(true))
    tips = cases.simulate_tips(flat, m, r, 600, rng)
    seqs = {nm: "".join("ACGT"[x] for x in tips[i]) for i, nm in enumerate(flat.leaf_names)}
    seqs["t3"] = "N" + seqs["t3"][1:]                       # ambiguity codes
    seqs["t4"] = seqs["t4"][:5] + "R-" + seqs["t4"][7:]
    f = tmp_path / "aln.txt"
    f.write_text("".join("%s %s\n" % kv for kv in seqs.items()))
    exe = compile_cpp("test_parsimony", built_lib)
    out = subprocess.check_output([str(exe), "search", str(f), rt.to_newick(true)], text=True)
    lines = out.splitlines()
    start = rt.parse_newick([l for l in lines if l.startswith("START ")][0][6:])
    rounds = _parse_scores(lines, "ROUND")
    min_test = _parse_scores(lines, "MIN_TEST_NNI")[0]
    true_score = _parse_scores(lines, "TRUE")[0]
    chars = {"A": 1, "C": 2, "G": 4, "T": 8, "N": 15, "R": 5, "-": 15}
    sets = {nm: np.array([chars[ch] for ch in s], np.uint32) for nm, s in seqs.items()}
    w = np.ones(600, np.int64)
    _, ref_rounds = rpars.search(rpars.number(rt.unroot(start) if len(start.sons) == 2 else start), sets, w)
    assert rounds == ref_rounds
    assert len(rounds) > 1 and min_test >= 0
    assert rounds[-1] <= true_score == rpars.score(true, sets, w)
    assert _parse_scores(lines, "SITE_SUM")[0] == rounds[-1]
