"""Pairwise ML distances (bppgpu_pairwise_distances: DistanceEstimation::computeMatrix with one TwoTreeLikelihood per pair) and
BIONJ (the shim's BioNJ), against oracle/ref_distance.py.

CPU: the oracle against the JC69 closed form and the branch-length bounds; the shim's BioNJ against the numpy BIONJ on random
matrices and on additive metrics; the shim compiles with distance.hpp.  GPU: joint code counts bit-exact against numpy, distances
and lnL against the oracle, bounds, run-to-run identity, memory kinds, error paths, and the shim end to end."""
import pathlib
import subprocess

import numpy as np
import pytest

import cases
from oracle import ref_distance as rd
from oracle import ref_models as rm
from oracle import ref_patterns as rp
from oracle import ref_tree as rt
from test_cpp_shim import compile_cpp

ROOT = pathlib.Path(__file__).resolve().parent.parent


def _jc(p):
    return -0.75 * np.log(1 - 4 * p / 3)


def _mutate(rng, a, frac, S=4):
    b = a.copy()
    flip = rng.random(len(a)) < frac
    b[flip] = (b[flip] + rng.integers(1, S, size=int(flip.sum()))) % S
    return b


# ---- CPU -------------------------------------------------------------------------------------------------------------------------
def test_oracle_jc69_closed_form():
    rng = np.random.default_rng(3)
    for N, frac in ((40, 0.1), (500, 0.3), (2000, 0.55)):
        a = rng.integers(4, size=N)
        b = _mutate(rng, a, frac)
        p = np.mean(a != b)
        d, _ = rd.pair_distance(a, b, np.ones(N), np.eye(4), rm.jc69(), [1.0], [1.0])
        assert abs(d - _jc(p)) <= 1e-12 * _jc(p), (d, _jc(p))


def test_oracle_bounds():
    rng = np.random.default_rng(4)
    a = rng.integers(4, size=300)
    r, p = rm.gamma_rates(4, 0.5)
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    assert rd.pair_distance(a, a, np.ones(300), np.eye(4), m, r, p)[0] == 1e-6
    assert rd.pair_distance(a, (a + 1) % 4, np.ones(300), np.eye(4), m, r, p)[0] == 1e4


def _newick_splits(text):
    root = rt.parse_newick(text)
    raw, names = {}, set()

    def walk(n):
        if n.is_leaf():
            names.add(n.name)
            s = frozenset([n.name])
        else:
            s = frozenset().union(*[walk(c) for c in n.sons])
        if n.father is not None:
            raw[s] = raw.get(s, 0.0) + n.length
        return s

    walk(root)
    return rd.canonical_splits(raw, frozenset(names))


def _shim_bionj(exe, D, names, tmp_path, rooted=False, positive=False):
    f = tmp_path / "matrix.txt"
    with open(f, "w") as fh:
        fh.write("%d\n" % len(names))
        for i, nm in enumerate(names):
            fh.write(nm + " " + " ".join("%.17g" % x for x in D[i]) + "\n")
    out = subprocess.check_output([str(exe), "bionj", str(f), "1" if rooted else "0", "1" if positive else "0"], text=True)
    return _newick_splits(out.split("TREE ")[1].split("\n")[0])


def _assert_same_splits(a, b, tol):
    assert set(a) == set(b)
    for s in a:
        assert abs(a[s] - b[s]) <= tol * max(1.0, abs(b[s])), (sorted(s), a[s], b[s])


@pytest.mark.parametrize("rooted,positive", [(False, False), (True, False), (False, True)])
def test_shim_bionj_matches_numpy_bionj(built_lib, tmp_path, rooted, positive):
    exe = compile_cpp("test_distance", built_lib)
    rng = np.random.default_rng(5)
    for n in (2, 3, 4, 9, 40):
        if n < 3 and not rooted:
            continue
        X = rng.random((n, n))
        D = X + X.T
        np.fill_diagonal(D, 0.0)
        names = ["t%d" % i for i in range(n)]
        ref = rd.splits(rd.bionj(D, names, rooted=rooted, positive_lengths=positive))
        _assert_same_splits(_shim_bionj(exe, D, names, tmp_path, rooted, positive), ref, 1e-12)


def test_shim_bionj_rejects_a_matrix_without_finite_criteria(built_lib, tmp_path):
    exe = compile_cpp("test_distance", built_lib)
    D = np.full((5, 5), np.nan)
    np.fill_diagonal(D, 0.0)
    f = tmp_path / "matrix.txt"
    f.write_text("5\n" + "".join("t%d " % i + " ".join("%.17g" % x for x in D[i]) + "\n" for i in range(5)))
    r = subprocess.run([str(exe), "bionj", str(f)], capture_output=True, text=True)
    assert r.returncode == 1 and "finite criterion" in r.stderr, (r.returncode, r.stdout, r.stderr)


def _path_metric(root):
    leaves = rt.leaves(root)
    names = [l.name for l in leaves]
    # distance from every leaf by a walk over the undirected tree
    adj = {}
    nodes = rt.postorder(root)
    for n in nodes:
        for s in n.sons:
            adj.setdefault(id(n), []).append((s, s.length))
            adj.setdefault(id(s), []).append((n, s.length))
    D = np.zeros((len(leaves), len(leaves)))
    pos = {id(l): k for k, l in enumerate(leaves)}
    for i, l in enumerate(leaves):
        stack, seen = [(l, 0.0)], {id(l)}
        while stack:
            n, d = stack.pop()
            if id(n) in pos:
                D[i, pos[id(n)]] = d
            for m, w in adj.get(id(n), []):
                if id(m) not in seen:
                    seen.add(id(m))
                    stack.append((m, d + w))
    return D, names


def test_additive_metric_recovers_the_tree(built_lib, tmp_path):
    exe = compile_cpp("test_distance", built_lib)
    rng = np.random.default_rng(6)
    root = rt.random_tree(50, rng, mean_brlen=0.1)
    D, names = _path_metric(root)
    truth = _newick_splits(rt.to_newick(root))
    _assert_same_splits(rd.splits(rd.bionj(D, names)), truth, 1e-10)
    _assert_same_splits(_shim_bionj(exe, D, names, tmp_path), truth, 1e-10)


def test_shim_compiles_with_distance_header(built_lib):
    compile_cpp("test_distance", built_lib)


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
def _model(name):
    r4, p4 = rm.gamma_rates(4, 0.5)
    return {"GTR": (rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25)), r4, p4), "LG08": (rm.lg08(), r4, p4),
            "YN98": (rm.yn98(2.0, 0.3), [1.0], [1.0]), "JC69": (rm.jc69(), [1.0], [1.0])}[name]


def _gpu(codes, w, table, m, r, p, **kw):
    from bpp_phyl_b200 import capi
    return capi.pairwise_distances(codes, w, table, cases.to_model_desc(m), m.freq, r, p, **kw)


def _numpy_counts(codes, w, K):
    L = codes.shape[0]
    out = np.zeros((L * (L - 1) // 2, K, K), np.int64)
    k = 0
    for a in range(L):
        for b in range(a + 1, L):
            np.add.at(out[k], (codes[a].astype(np.int64), codes[b].astype(np.int64)), w.astype(np.int64))
            k += 1
    return out


def _weights(rng, N):
    w = rng.choice(np.array([1, 127, 128, 255], np.uint32), size=N)
    w[::97] = 10 ** 6                                             # split into 7875 virtual columns each
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("L", [2, 3, 17, 130])
@pytest.mark.parametrize("N", [1, 31, 33, 4099])
def test_counts_bit_exact_k4(built_lib, L, N):
    rng = np.random.default_rng(L * 10007 + N)
    codes = rng.integers(4, size=(L, N)).astype(np.uint8)
    w = _weights(rng, N)
    m, r, p = _model("GTR")
    _, _, cnt = _gpu(codes, w, np.eye(4), m, r, p, counts=True)
    assert np.array_equal(cnt.astype(np.int64), _numpy_counts(codes, w, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("weights", [[0, 200], [0, 128] * 16 + [5, 0, 200, 0, 254] * 7 + [255, 0, 0] * 3])
def test_counts_zero_and_heavy_weights(built_lib, weights):
    # zero weights and weights above 127 in equal numbers: as many virtual columns as patterns, yet column j is not pattern j
    w = np.array(weights, np.uint32)
    assert sum((int(x) + 126) // 127 for x in w) == len(w)
    rng = np.random.default_rng(len(w))
    codes = rng.integers(4, size=(5, len(w))).astype(np.uint8)
    m, r, p = _model("GTR")
    _, _, cnt = _gpu(codes, w, np.eye(4), m, r, p, counts=True)
    assert np.array_equal(cnt.astype(np.int64), _numpy_counts(codes, w, 4))


IUPAC_CHARS, IUPAC_TABLE = rp.init_value_table(rp.DNA_STATES, rp.DNA_ALIASES)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["K6_ambiguity", "K21_iupac", "K21_iupac_code_bytes_2", "K128_pair_blocks"])
def test_counts_bit_exact_alphabets(built_lib, kind):
    rng = np.random.default_rng(11)
    m, r, p = _model("GTR")
    if kind == "K6_ambiguity":
        c = cases.make_case(17, 800, m, r, p, seed=3, ambiguity=0.2)
        codes = np.stack([c.codes_by_leaf[l] for l in c.flat.leaf_ids])
        w, table = np.asarray(c.weights, np.uint32), c.table
    elif kind.startswith("K21"):
        L, N = 33, 999
        codes = rng.integers(len(IUPAC_CHARS), size=(L, N))
        codes = codes.astype(np.uint16 if kind.endswith("2") else np.uint8)
        w, table = _weights(rng, N), IUPAC_TABLE
    else:
        # 130 sequences x 128 codes: 8385 pairs x 64 KB of counts exceed the device's count budget, so the pairs run in blocks
        L, N = 130, 300
        table = (rng.random((128, 4)) < 0.5).astype(float)
        table[table.sum(1) == 0, 0] = 1.0
        codes = rng.integers(128, size=(L, N)).astype(np.uint8)
        w = _weights(rng, N)
    _, _, cnt = _gpu(codes, w, table, m, r, p, counts=True)
    K = table.shape[0]
    if kind == "K128_pair_blocks":
        k = 0
        for a in range(L):
            for b in range(a + 1, L):
                ref = np.bincount(codes[a].astype(np.int64) * K + codes[b], weights=w.astype(np.float64), minlength=K * K)
                assert np.array_equal(cnt[k].ravel().astype(np.float64), ref), (a, b)
                k += 1
    else:
        assert np.array_equal(cnt.astype(np.int64), _numpy_counts(codes, w, K))


def _check_against_oracle(dist, lnl, codes, w, table, m, r, p, pairs=None):
    L = codes.shape[0]
    pairs = pairs if pairs is not None else [(a, b) for a in range(L) for b in range(a + 1, L)]
    E = np.asarray(table, float)
    checked_t = 0
    for a, b in pairs:
        t_ref, l_ref = rd.pair_distance(codes[a], codes[b], w, table, m, r, p)
        assert dist[a, b] == dist[b, a]
        # (a flat pair of all-ambiguous rows has lnL = 0 up to rounding of f = 1)
        assert abs(lnl[a, b] - l_ref) <= 1e-10 * max(abs(l_ref), 1.0), (a, b, lnl[a, b], l_ref)
        if rd.T_MIN * 1.01 < t_ref < rd.T_MAX / 1.01:
            n = rd.pair_counts(codes[a], codes[b], w, E.shape[0])
            _, d2 = rd.pair_derivatives(n, E, m, r, p, t_ref)
            if t_ref * t_ref * abs(d2) >= 1.0:
                assert abs(dist[a, b] - t_ref) <= 1e-6 * t_ref, (a, b, dist[a, b], t_ref)
                checked_t += 1
        else:
            assert dist[a, b] == t_ref, (a, b, dist[a, b], t_ref)
    return checked_t


@pytest.mark.gpu
@pytest.mark.parametrize("name,L,N", [("GTR", 64, 400), ("LG08", 20, 300), ("YN98", 10, 200)])
def test_distances_match_oracle(built_lib, name, L, N):
    m, r, p = _model(name)
    c = cases.make_case(L, N, m, r, p, seed=7, mean_brlen=0.1)
    codes = np.stack([c.codes_by_leaf[l] for l in c.flat.leaf_ids])
    w = np.asarray(c.weights, np.uint32)
    dist, lnl = _gpu(codes, w, c.table, m, r, p)
    assert np.all(np.diag(dist) == 0)
    checked = _check_against_oracle(dist, lnl, codes, w, c.table, m, r, p)
    assert checked >= (L * (L - 1) // 2) // 4


@pytest.mark.gpu
def test_jc69_equals_closed_form(built_lib):
    rng = np.random.default_rng(8)
    N, L = 3000, 12
    base = rng.integers(4, size=N)
    codes = np.stack([_mutate(rng, base, f) for f in np.linspace(0.02, 0.6, L)]).astype(np.uint8)
    m, r, p = _model("JC69")
    dist, _ = _gpu(codes, np.ones(N, np.uint32), np.eye(4), m, r, p)
    for a in range(L):
        for b in range(a + 1, L):
            pd = np.mean(codes[a] != codes[b])
            assert abs(dist[a, b] - _jc(pd)) <= 1e-9 * _jc(pd), (a, b, dist[a, b], _jc(pd))


@pytest.mark.gpu
def test_bounds_and_special_rows(built_lib):
    rng = np.random.default_rng(9)
    N = 500
    a = rng.integers(4, size=N)
    n_row = np.full(N, IUPAC_CHARS.index("N"))
    codes = np.stack([a, a, (a + 1) % 4, n_row, n_row]).astype(np.uint8)
    m, r, p = _model("GTR")
    dist, lnl = _gpu(codes, np.ones(N, np.uint32), IUPAC_TABLE, m, r, p)
    assert dist[0, 1] == 1e-6                 # identical
    assert dist[0, 2] == 1e4 and dist[1, 2] == 1e4   # different at every site
    assert dist[0, 3] == 1e-6 and dist[3, 4] == 1e-6  # all-N rows: flat
    _check_against_oracle(dist, lnl, codes, np.ones(N, np.uint32), IUPAC_TABLE, m, r, p)


@pytest.mark.gpu
def test_run_to_run_identical(built_lib):
    m, r, p = _model("GTR")
    c = cases.make_case(40, 3000, m, r, p, seed=10, ambiguity=0.05)
    codes = np.stack([c.codes_by_leaf[l] for l in c.flat.leaf_ids])
    w = np.asarray(c.weights, np.uint32)
    d1, l1, c1 = _gpu(codes, w, c.table, m, r, p, counts=True)
    d2, l2, c2 = _gpu(codes, w, c.table, m, r, p, counts=True)
    assert np.array_equal(d1, d2) and np.array_equal(l1, l2) and np.array_equal(c1, c2)


@pytest.mark.gpu
def test_memory_kinds_pageable_pinned_device(built_lib):
    import torch
    from bpp_phyl_b200 import capi
    m, r, p = _model("GTR")
    rng = np.random.default_rng(12)
    L, n_sites = 24, 20000
    cols = rng.integers(4, size=(n_sites, L)).astype(np.uint8)
    cols[: n_sites // 2] = cols[0]                      # heavy patterns: weights above 127
    ps, wt, ix, tip = capi.site_patterns_device(cols)
    pageable = _gpu(np.ascontiguousarray(tip), wt, np.eye(4), m, r, p, counts=True)
    pinned_codes = torch.from_numpy(np.ascontiguousarray(tip)).pin_memory()
    pinned_w = torch.from_numpy(np.ascontiguousarray(wt).view(np.int32)).pin_memory()
    pinned = _gpu(pinned_codes.data_ptr(), pinned_w.data_ptr(), np.eye(4), m, r, p, counts=True, n_leaves=L,
                  n_patterns=len(wt), code_bytes=1)
    # device-resident: site_patterns_device writes its tip codes straight into device buffers
    dcols = torch.from_numpy(cols).cuda()
    d_ps = torch.empty(n_sites, dtype=torch.int64, device="cuda")
    d_wt = torch.empty(n_sites, dtype=torch.int32, device="cuda")
    d_ix = torch.empty(n_sites, dtype=torch.int64, device="cuda")
    d_tip = torch.empty(n_sites * L, dtype=torch.uint8, device="cuda")
    npat = capi.site_patterns_device_raw(dcols.data_ptr(), n_sites, L, d_ps.data_ptr(), d_wt.data_ptr(), d_ix.data_ptr(),
                                         d_tip.data_ptr())
    assert npat == len(wt)
    device = _gpu(d_tip.data_ptr(), d_wt.data_ptr(), np.eye(4), m, r, p, counts=True, n_leaves=L, n_patterns=npat,
                  code_bytes=1)
    for x, y in zip(pageable, pinned):
        assert np.array_equal(x, y)
    for x, y in zip(pageable, device):
        assert np.array_equal(x, y)
    assert np.array_equal(pageable[2].astype(np.int64), _numpy_counts(np.asarray(tip), np.asarray(wt), 4))


@pytest.mark.gpu
def test_error_paths(built_lib):
    from bpp_phyl_b200 import capi
    m, r, p = _model("GTR")
    codes = np.zeros((4, 10), np.uint8)
    w = np.ones(10, np.uint32)
    # a diagonalizable, non-singular descriptor whose spectrum has a complex pair (rotation block on states 2, 3)
    cplx = capi.model_desc(4, capi.MODEL_DIAGONALIZABLE | capi.MODEL_NONSINGULAR, V=np.eye(4), Vinv=np.eye(4),
                           ev_re=[0.0, -1.0, -0.5, -0.5], ev_im=[0.0, 0.0, 0.3, -0.3])
    cases_ = [
        lambda: capi.pairwise_distances(codes, w, np.eye(4), cplx, np.full(4, 0.25), [1.0], [1.0]),
        lambda: _gpu(codes, w, np.ones((129, 4)), m, r, p),
        lambda: _gpu(codes[:1], w, np.eye(4), m, r, p),
        lambda: _gpu(codes, np.full(10, 2 ** 31 // 10 + 1, np.uint32), np.eye(4), m, r, p),
        lambda: _gpu(np.full((4, 10), 4, np.uint8), w, np.eye(4), m, r, p),
    ]
    for f in cases_:
        with pytest.raises(capi.BppGpuError) as e:
            f()
        assert e.value.code == capi.E_INVALID


@pytest.mark.gpu
def test_shim_distance_estimation_bionj_and_newton(built_lib):
    exe = compile_cpp("test_distance", built_lib)
    out = subprocess.check_output([str(exe), "estimate"], text=True)
    lines = out.splitlines()
    rows = [l.split()[1:] for l in lines if l.startswith("DIST ")]
    names = [r[0] for r in rows]
    D = np.array([[float(x) for x in r[1:]] for r in rows])
    seqs = {"A": "AAATGGCTGTGCACGTC", "B": "GACTGGATCTGCACGTC", "C": "CTCTGGATGTGCACGTG", "D": "AAATGGCGGTGCGCCTA"}
    r, p = rm.gamma_rates(4, 1.0)
    m = rm.t92(3.0, 0.5)
    chars, table = rp.init_value_table(rp.DNA_STATES, rp.DNA_ALIASES)
    codes = np.array([[chars.index(ch) for ch in seqs[nm]] for nm in names])
    ref, _ = rd.distance_matrix(codes, np.ones(codes.shape[1]), table, m, r, p)
    np.testing.assert_allclose(D, ref, rtol=1e-6, atol=0)
    tree = [l for l in lines if l.startswith("TREE ")][0][5:]
    assert sorted(l.name for l in rt.leaves(rt.parse_newick(tree))) == sorted(seqs)
    start = float([l for l in lines if l.startswith("START ")][0].split()[1])
    final = float([l for l in lines if l.startswith("FINAL ")][0].split()[1])
    assert np.isfinite(start) and final <= start + 1e-9
