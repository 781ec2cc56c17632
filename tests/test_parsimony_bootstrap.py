"""The parsimony bootstrap: replicate weights drawn on the device (bppgpu_bootstrap_weights), the replicate-batched Fitch
passes (bppgpu_parsimony_score_replicates / _nni_replicates), the shim's DRTreeParsimonyBootstrap with its lockstep NNI search,
and bootstrap support values, against oracle/ref_bootstrap.py and oracle/ref_parsimony.py.

CPU: the oracle's Philox4x32-10 against the Random123 known answers, the oracle's sampler and supports on hand-built trees,
the shim compiling, and no CPU fallback.  GPU: everything compared exactly."""
import copy
import subprocess

import numpy as np
import pytest

import cases
from oracle import ref_bootstrap as rb
from oracle import ref_models as rm
from oracle import ref_parsimony as rpars
from oracle import ref_tree as rt
from test_cpp_shim import compile_cpp
from test_parsimony import HEAVY, _codes, _flat, _sets, _table

CHARS = {"A": 1, "C": 2, "G": 4, "T": 8, "N": 15, "R": 5, "-": 15}


def _newick(n):
    return "(" + ",".join(_newick(s) for s in n.sons) + ")" if n.sons else n.name


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_oracle_philox_known_answers(ctr, key, want):
    assert tuple(int(x) for x in rb.philox4x32_10(ctr, key)) == want


def test_oracle_sampler_rows_and_chunks():
    idx = np.arange(1000) % 37
    w = rb.bootstrap_weights(idx, 37, 10, 2 ** 40 + 5)
    assert (w.sum(axis=1) == 1000).all()
    assert np.array_equal(w[4:7], rb.bootstrap_weights(idx, 37, 3, 2 ** 40 + 5, first=4))
    assert not np.array_equal(w[0], w[1])


def _support(tree, trees, fmt=0):
    """{frozenset split: value} of the internal branches of `tree`"""
    bp = rb.bipartitions(tree)
    return {bp[n]: v for n, v in rb.bootstrap_values(tree, trees, fmt).items()}


def test_oracle_supports_on_hand_built_trees():
    a = rt.parse_newick("((t0,t1),(t2,t3),(t4,t5));")
    b = rt.parse_newick("((t0,t2),(t1,t3),(t4,t5));")
    c = rt.parse_newick("((t0,t3),(t2,t1),(t5,t4));")
    assert set(_support(a, [copy.deepcopy(a)] * 4).values()) == {100.0}
    s0 = _support(a, [a, b, c])
    assert s0[frozenset({"t2", "t3"})] == 33.0 and s0[frozenset({"t4", "t5"})] == 100.0
    assert _support(a, [a, b, c], 2)[frozenset({"t2", "t3"})] == 33.33
    # son order and rooting do not change a support
    a_rev = rt.parse_newick("((t5,t4),(t3,t2),(t1,t0));")
    a_rooted = rt.parse_newick("(((t0,t1),(t2,t3)),(t4,t5));")
    c_rooted = rt.parse_newick("((t3,t0),((t2,t1),(t5,t4)));")
    for main in (a_rev, a_rooted):
        assert _support(main, [a, b, c_rooted], 2) == {k: v for k, v in _support(a, [a, b, c], 2).items()
                                                      if k in set(rb.bipartitions(main).values())}
    root_vals = [v for n, v in rb.bootstrap_values(a_rooted, [a, b, c]).items() if n.father is a_rooted]
    assert root_vals == [100.0, 100.0]
    with pytest.raises(ValueError):
        rb.bootstrap_values(a, [rt.parse_newick("((t0,t1),(t2,t3),(t4,t6));")])


def test_shim_compiles_with_bootstrap(built_lib):
    compile_cpp("test_parsimony_bootstrap", built_lib)


def test_shim_support_values_on_hand_built_trees(built_lib):
    """the shim's BipartitionList / computeBootstrapValues (host code) against the oracle: unrooted, reordered and rooted main
    trees, a rooted replicate tree, formats 0 and 2, and the throw for another leaf set"""
    exe = compile_cpp("test_parsimony_bootstrap", built_lib)
    reps = ["((t0,t1),(t2,t3),(t4,t5));", "((t0,t2),(t1,t3),(t4,t5));", "((t3,t0),((t2,t1),(t5,t4)));"]
    mains = ["((t0,t1),(t2,t3),(t4,t5));", "((t5,t4),(t3,t2),(t1,t0));", "(((t0,t1),(t2,t3)),(t4,t5));",
             "((t4,(t5,(t1,t0))),(t3,t2));"]
    for m in mains:
        for fmt in (0, 2):
            out = subprocess.check_output([str(exe), "values", m, str(fmt)] + reps, text=True).splitlines()
            got = [(frozenset(l.split()[2].split(",")), float(l.split()[1])) for l in out]
            main = rt.parse_newick(m)
            bp = rb.bipartitions(main)
            vals = rb.bootstrap_values(main, [rt.parse_newick(r) for r in reps], fmt)
            assert got == [(bp[n], vals[n]) for n in rt.postorder(main) if n in vals]
    out = subprocess.check_output([str(exe), "values", mains[0], "0", "((t0,t1),(t2,t3),(t4,t6));"], text=True)
    assert out.startswith("THROWS ") and "leaf set" in out


def test_no_cpu_fallback_for_the_sampler(built_lib):
    from bpp_phyl_b200 import capi
    if capi.device_count() > 0:
        pytest.skip("a GPU is visible here")
    with pytest.raises(capi.BppGpuError) as e:
        capi.bootstrap_weights(np.arange(10), 10, 2, 1)
    assert e.value.code == capi.E_CUDA


# ---- GPU: the sampler ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("seed, n_sites, N, first, R", [
    (0, 1, 1, 0, 3), (1, 1000, 1, 0, 2), (7, 1, 5, 9, 4), (12345, 5000, 700, 0, 16), (2 ** 63 + 11, 4099, 4099, 1000, 8),
    (2 ** 32 - 1, 20000, 3000, 2 ** 32 - 5, 5),
])
def test_sampler_equals_oracle(built_lib, seed, n_sites, N, first, R):
    from bpp_phyl_b200 import capi
    rng = np.random.default_rng(n_sites + N)
    idx = np.sort(rng.integers(N, size=n_sites)) if N < n_sites else np.arange(n_sites) % N
    if N <= n_sites:
        idx[:N] = np.arange(N)                       # every pattern has a site
    w = capi.bootstrap_weights(idx, N, R, seed, first=first)
    assert np.array_equal(w, rb.bootstrap_weights(idx, N, R, seed, first=first))
    assert (w.sum(axis=1, dtype=np.int64) == n_sites).all()
    parts = [capi.bootstrap_weights(idx, N, k, seed, first=first + a) for a, k in ((0, 1), (1, R - 2), (R - 1, 1)) if k > 0]
    assert np.array_equal(np.concatenate(parts), w)


@pytest.mark.gpu
def test_sampler_memory_kinds(built_lib):
    import torch
    from bpp_phyl_b200 import capi
    rng = np.random.default_rng(3)
    n_sites, N, R, seed = 30000, 900, 6, 77
    idx = rng.integers(N, size=n_sites).astype(np.int64)
    ref = rb.bootstrap_weights(idx, N, R, seed)
    kinds = {"pageable": torch.from_numpy(idx.copy()), "pinned": torch.from_numpy(idx.copy()).pin_memory(),
             "device": torch.from_numpy(idx.copy()).cuda()}
    for ki, ti in kinds.items():
        for ko in ("numpy", "pinned", "device"):
            out = (np.zeros((R, N), np.uint32) if ko == "numpy" else
                   torch.zeros((R, N), dtype=torch.int32).pin_memory() if ko == "pinned" else
                   torch.zeros((R, N), dtype=torch.int32, device="cuda"))
            capi.bootstrap_weights(ti, N, R, seed, out=out)
            got = out if ko == "numpy" else out.cpu().numpy().view(np.uint32)
            assert np.array_equal(got, ref), (ki, ko)


@pytest.mark.gpu
def test_sampler_error_paths(built_lib):
    from bpp_phyl_b200 import capi
    idx = np.arange(10)
    bad = [
        lambda: capi.bootstrap_weights(np.zeros(0, np.int64), 1, 1, 0, n_sites=0),      # no sites
        lambda: capi.bootstrap_weights(idx, 10, 1, 0, n_sites=2 ** 32),                  # n_sites >= 2^32 (checked first)
        lambda: capi.bootstrap_weights(np.r_[idx, 10], 10, 1, 0),                         # index = n_patterns
        lambda: capi.bootstrap_weights(np.r_[-1, idx], 10, 1, 0),                         # negative index
        lambda: capi.bootstrap_weights(idx, 10, 0, 0),                                    # no replicate
        lambda: capi.bootstrap_weights(idx, 10, 2, 0, first=2 ** 32 - 1),                 # replicate index >= 2^32
    ]
    for f in bad:
        with pytest.raises(capi.BppGpuError) as e:
            f()
        assert e.value.code == capi.E_INVALID


@pytest.mark.gpu
def test_sampler_chi_square(built_lib):
    """identity indices, fixed seed: per-site draw counts over 400 replicates of 2000 sites against the uniform law"""
    from scipy import stats
    from bpp_phyl_b200 import capi
    n, R = 2000, 400
    counts = capi.bootstrap_weights(np.arange(n), n, R, 20261022).sum(axis=0, dtype=np.int64)
    exp = R                                     # n * R draws over n sites
    chi2 = float(((counts - exp) ** 2 / exp).sum())
    assert stats.chi2.sf(chi2, n - 1) > 1e-6


# ---- GPU: replicate-batched passes -----------------------------------------------------------------------------------------------
def _check_batch(S, N, E, n_taxa=20, R=5, max_bytes=0, seed=0):
    from bpp_phyl_b200 import capi
    rng = np.random.default_rng(seed + S * 1009 + N * 7 + E)
    table = _table(rng, S, n_amb=3)
    codes = _codes(rng, n_taxa, N, len(table))
    names = ["t%d" % i for i in range(n_taxa)]
    sets = _sets(codes, table, names)
    row = {nm: i for i, nm in enumerate(names)}
    W = rng.choice(HEAVY, size=(R, N)).astype(np.uint32)
    own = rng.integers(1, 100, size=N).astype(np.uint32)
    roots = [rt.random_tree(n_taxa, rng) for _ in range(E)]
    flats = [_flat(r, row) for r in roots]
    rep = rng.integers(R, size=E).astype(np.int32)
    if E > 1:
        rep[1] = rep[0]                                   # a repeated replicate id
    with capi.Parsimony(table, codes, own, max_bytes=max_bytes) as p:
        p.set_replicate_weights(W)
        s, sc = p.score_replicates(rep, [f[1] for f in flats], site_scores=True)
        d, s2 = p.nni_replicates(rep, [f[1] for f in flats])
        # the handle's own weights are untouched
        assert p.score(*flats[0][1]) == rpars.score(roots[0], sets, own)
        d_own, s_own = p.nni_deltas(*flats[0][1])
    ref_own, cur_own = rpars.all_nni_deltas(roots[0], sets, own)
    assert s_own == cur_own and np.array_equal(d_own, [ref_own.get(n, 0) for n in flats[0][0]])
    assert np.array_equal(s, s2)
    singles = {}
    for e in range(E):
        nodes, topo = flats[e]
        w = W[rep[e]]
        assert np.array_equal(sc[e].astype(np.int64), rpars.site_scores(roots[e], sets))
        ref, cur = rpars.all_nni_deltas(roots[e], sets, w)
        assert s[e] == cur
        assert np.array_equal(d[e], np.array([ref.get(n, 0) for n in nodes], np.int64))
        if e < 3:    # the single-replicate calls on a handle built with this replicate's weights
            if rep[e] not in singles:
                singles[rep[e]] = capi.Parsimony(table, codes, w, max_bytes=max_bytes)
            ps = singles[rep[e]]
            assert ps.score(*topo) == s[e]
            assert np.array_equal(ps.nni_deltas(*topo)[0], d[e])
    for ps in singles.values():
        ps.close()


@pytest.mark.gpu
@pytest.mark.parametrize("S", [4, 20, 32])
@pytest.mark.parametrize("N", [1, 33, 4099])
@pytest.mark.parametrize("E", [1, 3, 64])
def test_batched_passes_equal_single_calls_and_oracle(built_lib, S, N, E):
    _check_batch(S, N, E)


@pytest.mark.gpu
@pytest.mark.parametrize("max_bytes", [1, 3000, 200000])
def test_batched_pattern_blocks_add_up(built_lib, max_bytes):
    _check_batch(4, 3001, 7, n_taxa=30, max_bytes=max_bytes, seed=1)


@pytest.mark.gpu
def test_device_resident_and_drawn_replicate_weights(built_lib):
    import torch
    from bpp_phyl_b200 import capi
    rng = np.random.default_rng(21)
    L, n_sites = 12, 3000
    cols = rng.integers(4, size=(n_sites, L)).astype(np.uint8)
    cols[: n_sites // 3] = cols[0]
    _, wt, ix, tip = capi.site_patterns_device(cols)
    N, R, seed = len(wt), 9, 4242
    table = np.eye(4)
    root = rt.random_tree(L, rng)
    _, topo = _flat(root, {"t%d" % i: i for i in range(L)})
    dw = torch.zeros((R, N), dtype=torch.int32, device="cuda")
    capi.bootstrap_weights(torch.from_numpy(ix).cuda(), N, R, seed, out=dw)
    sets = _sets(np.asarray(tip), table, ["t%d" % i for i in range(L)])
    want = [rpars.score(root, sets, w) for w in rb.bootstrap_weights(ix, N, R, seed)]
    with capi.Parsimony(table, np.ascontiguousarray(tip), wt) as p:
        p.set_replicate_weights(dw)                                           # device to device
        assert list(p.score_replicates(np.arange(R), [topo] * R)) == want
        p.draw_replicate_weights(ix, R, seed)                                 # drawn in place
        assert list(p.score_replicates(np.arange(R), [topo] * R)) == want
        p.set_replicate_weights(np.zeros((0, N), np.uint32))                  # freed
        with pytest.raises(capi.BppGpuError) as e:
            p.score_replicates([0], [topo])
        assert e.value.code == capi.E_INVALID


@pytest.mark.gpu
def test_batched_error_paths(built_lib):
    from bpp_phyl_b200 import capi
    rng = np.random.default_rng(22)
    codes = _codes(rng, 5, 10, 4)
    row = {"t%d" % i: i for i in range(5)}
    good = _flat(rt.random_tree(5, rng), row)[1]
    star = _flat(rt.parse_newick("(t0,t1,(t2,t3,t4));"), row)[1]
    rooted = _flat(rt.parse_newick("((t0,t1,t2),(t3,t4));"), row)[1]     # as many nodes as `good`, but no NNI scoring
    twice = (good[0], good[1], good[2], np.where(good[3] == 1, 0, good[3]))
    with capi.Parsimony(np.eye(4), codes, np.ones(10, np.uint32)) as p:
        p.set_replicate_weights(np.ones((2, 10), np.uint32))
        assert p.score_replicates([0, 1], [good, good]).tolist() == [p.score(*good)] * 2
        cases_ = [
            (lambda: p.score_replicates([0, 2], [good, good]), "entry 1"),          # replicate out of range
            (lambda: p.score_replicates([0, -1], [good, good]), "entry 1"),
            (lambda: p.score_replicates([0, 0, 1], [good, good, twice]), "entry 2"),  # two leaves, one row
            (lambda: p.nni_replicates([1, 0], [good, rooted]), "entry 1"),         # not binary
        ]
        for f, where in cases_:
            with pytest.raises(capi.BppGpuError) as e:
                f()
            assert e.value.code == capi.E_INVALID and where in str(e.value)
        assert p.score_replicates([1], [star]).tolist() == [p.score(*star)]   # scoring takes a multifurcation


# ---- GPU: the shim ---------------------------------------------------------------------------------------------------------------
def _simulate(rng, true, n_sites):
    r, p = rm.gamma_rates(4, 0.5)
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    flat = rt.FlatTree(copy.deepcopy(true))
    tips = cases.simulate_tips(flat, m, r, n_sites, rng)
    return {nm: "".join("ACGT"[x] for x in tips[i]) for i, nm in enumerate(flat.leaf_names)}


def _write(tmp_path, seqs):
    f = tmp_path / "aln.txt"
    f.write_text("".join("%s %s\n" % kv for kv in seqs.items()))
    return f


@pytest.mark.gpu
def test_shim_lockstep_search_equals_oracle(built_lib, tmp_path):
    """R = 24 replicates of 36 taxa x 400 sites: every replicate's scores and final tree equal ref_parsimony.search from the
    same start with the oracle's weights, and a second run prints the same"""
    rng = np.random.default_rng(24)
    n_sites, R, seed = 400, 24, 987654321
    true = rt.random_tree(36, rng, mean_brlen=0.1)
    seqs = _simulate(rng, true, n_sites)
    seqs["t3"] = "N" + seqs["t3"][1:]
    seqs["t4"] = seqs["t4"][:5] + "R-" + seqs["t4"][7:]
    start = rt.random_tree(36, rng)
    exe = compile_cpp("test_parsimony_bootstrap", built_lib)
    args = [str(exe), "lockstep", str(_write(tmp_path, seqs)), _newick(start) + ";", str(R), str(seed)]
    out = subprocess.check_output(args, text=True)
    assert subprocess.check_output(args, text=True) == out
    lines = out.splitlines()
    sets = {nm: np.array([CHARS[c] for c in s], np.uint32) for nm, s in seqs.items()}
    W = rb.bootstrap_weights(np.arange(n_sites), n_sites, R, seed)     # one pattern per site: the same totals
    moved = 0
    for r in range(R):
        final, scores = rpars.search(rpars.number(copy.deepcopy(start)), sets, W[r].astype(np.int64))
        assert [int(x) for x in lines[[l.split()[:2] for l in lines].index(["SCORES", str(r)])].split()[2:]] == scores
        assert "TREE %d %s;" % (r, _newick(final)) in lines
        assert "WEIGHT_SUM %d %d" % (r, n_sites) in lines
        moved += len(scores) > 1
        if r == 3:
            assert "ALONE 3 " + " ".join(map(str, scores)) in lines
    assert moved > R // 2


@pytest.mark.gpu
def test_shim_bionj_search_bootstrap_supports(built_lib, tmp_path):
    """alignment -> DistanceEstimation -> BioNJ -> optimizeTreeNNI -> DRTreeParsimonyBootstrap (R = 50) -> lockstep search ->
    computeBootstrapValues: from the printed start, the oracle's searches and bootstrap_values give the same support for
    every branch; the generating tree's splits on long branches get at least 90"""
    rng = np.random.default_rng(23)
    n_sites, R, seed = 800, 50, 99
    true = rt.random_tree(16, rng, mean_brlen=0.05)
    long_ = []
    for i, n in enumerate(n for n in rt.postorder(true) if n.sons and n.father is not None):
        n.length = 0.15 if i % 2 == 0 else 0.004
        if i % 2 == 0:
            long_.append(n)
    seqs = _simulate(rng, true, n_sites)
    exe = compile_cpp("test_parsimony_bootstrap", built_lib)
    lines = subprocess.check_output([str(exe), "support", str(_write(tmp_path, seqs)), str(R), str(seed)], text=True).splitlines()
    start = rt.parse_newick([l for l in lines if l.startswith("START ")][0][6:])
    sets = {nm: np.array([CHARS[c] for c in s], np.uint32) for nm, s in seqs.items()}
    main, _ = rpars.search(rpars.number(start), sets, np.ones(n_sites, np.int64))
    assert "MAIN %s;" % _newick(main) in lines
    W = rb.bootstrap_weights(np.arange(n_sites), n_sites, R, seed)
    trees = [rpars.search(main, sets, W[r].astype(np.int64))[0] for r in range(R)]
    want = {sp: v for sp, v in _support(main, trees, 2).items()}
    got = {frozenset(l.split()[2].split(",")): float(l.split()[1]) for l in lines if l.startswith("SUPPORT ")}
    assert got == want
    bt = rb.bipartitions(true)
    for n in long_:
        assert got[bt[n]] >= 90
    assert min(got.values()) < 100

