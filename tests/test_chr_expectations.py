"""Expected numbers of events per branch and class by stochastic mapping (ComputeChromosomeTransitionsExp; DESIGN §7b):
the class split, the exact conditional expectations and the numpy sampler on the CPU; on the device the tallies of
bppgpu_simulate_event_counts against the sampler bit for bit, identities that hold path by path, convergence to the exact
values, bppgpu_expected_events against the oracle's combination, its error paths, and the shim end to end."""
import json
import subprocess

import numpy as np
import pytest

import cases
from oracle import ref_likelihood as rl
from oracle import ref_mapping as mp
from oracle import ref_models as rm
from oracle import ref_tree as rt
from test_cpp_shim import compile_cpp

IG = rm.IGNORE_PARAM
# (name, min, max, kwargs of rm.chromosome): the shim prints the same sets (tests/cpp/test_chr_expectations.cpp, "split")
SPLIT_CASES = [
    ("linear", 1, 30, dict(gain=0.7, loss=0.4, dupl=0.2, demi=0.1, gain_r=0.03, loss_r=0.02, dupl_r=0.01)),
    ("exp", 1, 30, dict(gain=0.7, loss=0.4, dupl=0.2, demi=0.1, gain_r=0.03, loss_r=-0.02, dupl_r=0.01, rate_change="EXP")),
    ("demi_equal_dupl", 3, 12, dict(gain=0.5, loss=0.3, dupl=0.8, demi=rm.DEMI_EQUAL_DUPL)),
    ("demi_ignored", 3, 12, dict(gain=0.5, loss=0.3, dupl=0.8, demi=IG)),
    ("base_number", 1, 40, dict(gain=0.6, loss=0.5, dupl=0.3, demi=0.2, base_num=4, base_num_r=0.35, max_chr_range=13)),
    ("clamped", 3, 12, dict(gain=0.9, loss=0.2, dupl=1.1, demi=0.7, base_num=3, base_num_r=0.25, max_chr_range=20)),
]
# the five-taxon ChromEvol case of test_zz_chr_optimizer: its branch lengths, with a zero and a tied length added
FIVE_TAXON = "(((a:0.3,b:0.2):0.4,c:0.5):0.1,(d:0.3,e:0.6):0.2);"
LENGTHS = [0.3, 0.2, 0.4, 0.5, 0.1, 0.3, 0.6, 0.2, 0.0, 0.6]


def _offdiag(Q):
    return np.asarray(Q, float) * (1 - np.eye(Q.shape[0]))


@pytest.mark.parametrize("name,lo,hi,kw", SPLIT_CASES, ids=[c[0] for c in SPLIT_CASES])
def test_class_split_adds_up_to_the_generator(name, lo, hi, kw):
    """The five class matrices, added in class order, are the generator's off-diagonal bit for bit; diagonals are 0."""
    R = mp.chromosome_classes(lo, hi, **kw)
    Q = rm.chromosome(lo, hi, **kw).Q
    assert np.all(R[:, np.arange(R.shape[1]), np.arange(R.shape[1])] == 0)
    np.testing.assert_array_equal(_offdiag(mp.class_sum(R)), _offdiag(Q))
    if name == "clamped":          # dupl, demi and base-number jumps clamped to the maximum keep their class
        n = hi - lo + 1
        assert R[2, n - 2, n - 1] > 0 and R[3, n - 3, n - 1] > 0 and R[4, n - 2, n - 1] > 0
    if name == "linear":           # odd i > 1: two demi targets at demi / 2
        i = 5
        assert R[3, i - lo, 7 - lo] == R[3, i - lo, 8 - lo] == 0.05


def test_shim_class_split_equals_the_oracle(built_lib):
    """ChromosomeSubstitutionModel::getTypeRates (host build) against the oracle's split, bit for bit, and the shim's own
    generator against the sum of its classes."""
    exe = compile_cpp("test_chr_expectations", built_lib)
    doc = json.loads(subprocess.run([str(exe), "split"], capture_output=True, text=True, check=True, timeout=120).stdout)
    for name, lo, hi, kw in SPLIT_CASES:
        n = hi - lo + 1
        R = np.array(doc[name]["R"]).reshape(5, n, n)
        np.testing.assert_array_equal(R, mp.chromosome_classes(lo, hi, **kw), err_msg=name)
        np.testing.assert_array_equal(_offdiag(mp.class_sum(R)), _offdiag(np.array(doc[name]["Q"]).reshape(n, n)), err_msg=name)


def _chr_model(S=30):
    return mp.chromosome_classes(1, S, gain=0.7, loss=0.4, dupl=0.2, demi=0.1, base_num=3, base_num_r=0.15, max_chr_range=6)


def _gtr_split():
    return mp.transition_transversion(rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25)).Q)


@pytest.mark.parametrize("t", [0.05, 0.6, 2.0])
def test_van_loan_equals_the_derivative_of_expm(t):
    R = _chr_model(12)
    Q = mp.generator(R)
    for T in range(5):
        a, b = mp.conditional_expectation(Q, R[T], t), mp.conditional_expectation_fd(Q, R[T], t)
        ok = np.isfinite(a) & (expm_p(Q, t) > 1e-12)
        np.testing.assert_allclose(b[ok], a[ok], rtol=1e-7, atol=1e-12)


def expm_p(Q, t):
    from scipy.linalg import expm
    return expm(t * Q)


def test_gain_minus_loss_is_the_net_change():
    """Gain/loss only: every path from y to x has gains - losses = x - y, so the conditional expectations differ by x - y."""
    R = mp.chromosome_classes(1, 15, gain=0.8, loss=0.6)[:2]
    Q = mp.generator(R)
    for t in (0.1, 0.7, 1.5):
        d = mp.conditional_expectation(Q, R[0], t) - mp.conditional_expectation(Q, R[1], t)
        P = expm_p(Q, t)
        y, x = np.nonzero(P > 1e-300)
        np.testing.assert_allclose(d[y, x], (x - y).astype(float), rtol=0, atol=1e-10)


def test_numpy_sampler_converges_to_the_exact_conditional_means():
    """At a fixed seed the sampler's conditional means are within 5 standard errors (exact variance) of Van Loan wherever at
    least 200 paths end in the cell and at least 10 events are expected there, and the end-state frequencies within 5 binomial
    SE of P(t) where n P >= 10."""
    R = _gtr_split()
    Q = mp.generator(R)
    lengths = [0.05, 0.4, 1.3]
    n = 40000
    cnt, sums = mp.simulate(R, lengths, n, seed=12345)
    _check_convergence(R, Q, lengths, n, cnt, sums, min_count=200)


def _check_convergence(R, Q, lengths, n, cnt, sums, min_count):
    checked = 0
    for b, t in enumerate(lengths):
        P = expm_p(Q, t)
        freq = cnt[b] / n
        big = n * P >= 10
        se = np.sqrt(P * (1 - P) / n)
        assert np.all(np.abs(freq - P)[big] <= 5 * se[big]), b
        for T in range(R.shape[0]):
            m = mp.conditional_expectation(Q, R[T], t)
            v = mp.conditional_variance(Q, R[T], t)
            # the normal approximation: enough paths, and enough expected events (a cell whose mean is 3e-6 and that sees one
            # event in 5 000 paths is a Poisson outlier, not a bias)
            sel = (cnt[b] >= min_count) & (cnt[b] * np.nan_to_num(m) >= 10)
            got = sums[b][..., T][sel] / cnt[b][sel]
            se_m = np.sqrt(np.maximum(v[sel], 0) / cnt[b][sel])
            assert np.all(np.abs(got - m[sel]) <= 5 * se_m + 1e-12), (b, T, np.max(np.abs(got - m[sel]) / (se_m + 1e-300)))
            checked += int(sel.sum())
    assert checked > 0


# ---- device -------------------------------------------------------------------------------------------------------------
def _capi():
    from bpp_phyl_b200 import capi
    return capi


def _assert_tallies_equal(got, want, what):
    """exact equality; any mismatch is listed (cell and both values) rather than tolerated"""
    bad = np.argwhere(got != want)
    assert len(bad) == 0, "%s: %d mismatched tallies, first %s: device %s, oracle %s" % (
        what, len(bad), bad[:5].tolist(), [int(got[tuple(i)]) for i in bad[:5]], [int(want[tuple(i)]) for i in bad[:5]])


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["chromosome", "gtr_ts_tv"])
@pytest.mark.parametrize("n_sims,seed,first", [(1, 7, 0), (1000, 2 ** 63 + 12345, 0), (1000, 99, 2 ** 32 - 1000), (1, 5, 2 ** 32 - 1)])
def test_device_tallies_equal_the_oracle_sampler(built_lib, model, n_sims, seed, first):
    capi = _capi()
    R = _chr_model() if model == "chromosome" else _gtr_split()
    cnt, sums = capi.simulate_event_counts(R, LENGTHS, n_sims, seed, first=first)
    want_c, want_s = mp.simulate(R, LENGTHS, n_sims, seed, first=first)
    _assert_tallies_equal(cnt, want_c, "count")
    _assert_tallies_equal(sums, want_s, "sum")
    np.testing.assert_array_equal(cnt.sum(axis=2), n_sims)
    np.testing.assert_array_equal(cnt[8], np.eye(R.shape[1], dtype=np.uint64) * n_sims)     # length 0: no event yet
    np.testing.assert_array_equal(cnt[6], cnt[9])                                          # tied lengths


@pytest.mark.gpu
def test_device_tallies_memory_kinds_chunks_and_repeatability(built_lib):
    """Pinned and device outputs equal host ones; chunks of paths add up to one call; two runs are bit-identical."""
    import torch
    capi = _capi()
    R = _chr_model()
    S, L, n, seed = R.shape[1], len(LENGTHS), 3000, 424242
    c1, s1 = capi.simulate_event_counts(R, LENGTHS, n, seed)
    c2, s2 = capi.simulate_event_counts(R, LENGTHS, n, seed)
    np.testing.assert_array_equal(c1, c2)
    np.testing.assert_array_equal(s1, s2)
    acc_c, acc_s = np.zeros_like(c1), np.zeros_like(s1)
    for f, k in ((0, 1000), (1000, 1), (1001, 1999)):
        c, s = capi.simulate_event_counts(R, LENGTHS, k, seed, first=f)
        acc_c += c
        acc_s += s
    np.testing.assert_array_equal(acc_c, c1)
    np.testing.assert_array_equal(acc_s, s1)
    dc = torch.zeros((L, S, S), dtype=torch.int64, device="cuda")
    ds = torch.zeros((L, S, S, 5), dtype=torch.int64, device="cuda")
    capi.simulate_event_counts(R, LENGTHS, n, seed, count=dc, sum=ds)
    np.testing.assert_array_equal(dc.cpu().numpy().view(np.uint64), c1)
    np.testing.assert_array_equal(ds.cpu().numpy().view(np.uint64), s1)
    pc = torch.zeros((L, S, S), dtype=torch.int64).pin_memory()
    ps = torch.zeros((L, S, S, 5), dtype=torch.int64).pin_memory()
    capi.simulate_event_counts(R, LENGTHS, n, seed, count=pc, sum=ps)
    np.testing.assert_array_equal(pc.numpy().view(np.uint64), c1)
    np.testing.assert_array_equal(ps.numpy().view(np.uint64), s1)


@pytest.mark.gpu
def test_path_identities_at_a_million_paths(built_lib):
    """n_sims = 2^20: every start state's paths end somewhere (sum_j count = n_sims), and under a gain/loss-only model
    sum_gain - sum_loss = (j - a) count in every cell, path by path."""
    capi = _capi()
    n = 2 ** 20
    R = mp.chromosome_classes(1, 30, gain=0.9, loss=0.7)[:2]
    cnt, sums = capi.simulate_event_counts(R, LENGTHS, n, 2024)
    np.testing.assert_array_equal(cnt.sum(axis=2), n)
    S = R.shape[1]
    net = (np.arange(S)[None, :] - np.arange(S)[:, None]).astype(np.int64)
    diff = sums[..., 0].astype(np.int64) - sums[..., 1].astype(np.int64)
    np.testing.assert_array_equal(diff, net[None] * cnt.astype(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["chromosome", "gtr_ts_tv"])
def test_device_tallies_converge_to_the_exact_values(built_lib, model):
    """n_sims = 2^20, fixed seed: conditional means within 5 SE (exact variance) of Van Loan where count >= 1000 and at least
    10 events are expected, end-state frequencies within 5 binomial SE of P(t) where n P >= 10."""
    capi = _capi()
    R = _chr_model() if model == "chromosome" else _gtr_split()
    Q = mp.generator(R)
    lengths = [0.1, 0.3, 0.6, 1.0]
    n = 2 ** 20
    cnt, sums = capi.simulate_event_counts(R, lengths, n, 77)
    _check_convergence(R, Q, lengths, n, cnt, sums, min_count=1000)


def _five_taxon_engine_case(R):
    flat = rt.FlatTree(rt.parse_newick(FIVE_TAXON), check_rooted=False)
    counts = {"a": 7, "b": 8, "c": 14, "d": 9, "e": None}
    S = R.shape[1]
    ch = cases.Case()
    ch.flat, ch.rates, ch.probs = flat, np.ones(1), np.ones(1)
    ch.table, ch.N, ch.weights = np.vstack([np.eye(S), np.ones((1, S))]), 1, np.ones(1, np.uint32)
    ch.codes_by_leaf = {lid: np.array([S if counts[flat.nodes[lid].name] is None else counts[flat.nodes[lid].name] - 1], np.uint8)
                        for lid in flat.leaf_ids}
    ch.code_dtype = np.uint8
    m = rm.chromosome(1, S, gain=0.7, loss=0.4, dupl=0.2, demi=0.1, base_num=3, base_num_r=0.15, max_chr_range=6)
    ch.model = m
    ch.root_freqs = np.random.default_rng(8).dirichlet(np.ones(S))
    return ch, m


def _expected_tolerance(Q, R, t_of_node, joints, weights, n, unreached):
    """5 standard errors of the estimator (exact per-cell variances, counts taken as n P) plus the unreached mass times the
    largest conditional mean of the branch"""
    tol = np.zeros((len(t_of_node), R.shape[0]))
    for b, J in joints.items():
        W = np.einsum("i,ixy->yx", np.asarray(weights, float), J)
        P = expm_p(Q, t_of_node[b])
        for T in range(R.shape[0]):
            v = np.nan_to_num(mp.conditional_variance(Q, R[T], t_of_node[b]))
            m = np.nan_to_num(mp.conditional_expectation(Q, R[T], t_of_node[b]))
            reach = P * n >= 1
            se = np.sqrt(np.sum(np.where(reach, W * W * np.maximum(v, 0) / np.where(reach, P * n, 1), 0)))
            tol[b, T] = 5 * se + unreached[b] * m.max() + 1e-12
    return tol


@pytest.mark.gpu
def test_expected_events_against_the_oracle_combination(built_lib):
    """expected_events equals the oracle's combination of the device's own tallies (same seed, one length per node) with the
    oracle's joint posteriors to 1e-12, unreached too; it is within simulation tolerance of the exact expectation; the root's
    row is 0."""
    capi = _capi()
    R = _chr_model()
    ch, m = _five_taxon_engine_case(R)
    flat = ch.flat
    res = cases.oracle_eval(ch, want_d1=True)
    n, seed = 2 ** 17, 31337
    with cases.make_engine(ch, flags=capi.FLAG_KEEP_CLVS) as e:
        e.eval(capi.EVAL_LNL | capi.EVAL_D1)
        ex, un = e.expected_events(R, n, seed)
        ex2, un2 = e.expected_events(R, n, seed)
        sim_ms, comb_ms = capi.expected_events_timing()
    np.testing.assert_array_equal(ex, ex2)
    np.testing.assert_array_equal(un, un2)
    assert sim_ms > 0 and comb_ms > 0
    t_of_node = m.rate * (np.asarray(flat.brlen, float) * ch.rates[0])
    t_of_node[flat.root] = 0.0
    cnt, sums = capi.simulate_event_counts(R, t_of_node, n, seed)
    joints = {b: rl.marginal_posteriors(flat, res, res.P, b, ch.probs)[1] for b in range(flat.n_nodes) if b != flat.root}
    want, want_un = mp.combine(cnt, sums, joints, ch.weights)
    np.testing.assert_allclose(ex, want, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(un, want_un, rtol=1e-12, atol=1e-15)
    assert np.all(ex[flat.root] == 0) and un[flat.root] == 0
    exact = mp.exact_expected(mp.generator(R), R, t_of_node, joints, ch.weights)
    tol = _expected_tolerance(mp.generator(R), R, t_of_node, joints, ch.weights, n, un)
    assert np.all(np.abs(ex - exact) <= tol), np.max(np.abs(ex - exact) / tol)


@pytest.mark.gpu
def test_event_mapping_error_paths(built_lib):
    capi = _capi()
    R = _gtr_split()

    def rejects(code, fn, text):
        with pytest.raises(capi.BppGpuError) as ei:
            fn()
        assert ei.value.code == code and text in str(ei.value), str(ei.value)

    for bad, text in ((-1e-3, "finite and >= 0"), (np.nan, "finite and >= 0"), (np.inf, "finite and >= 0")):
        Rb = R.copy()
        Rb[1, 0, 1] = bad
        rejects(capi.E_INVALID, lambda: capi.simulate_event_counts(Rb, [0.1], 10, 1), text)
    Rd = R.copy()
    Rd[0, 2, 2] = 0.5
    rejects(capi.E_INVALID, lambda: capi.simulate_event_counts(Rd, [0.1], 10, 1), "diagonal")
    rejects(capi.E_INVALID, lambda: capi.simulate_event_counts(R, [0.1], 0, 1), "n_sims >= 1")
    rejects(capi.E_INVALID, lambda: capi.simulate_event_counts(R, [0.1], 2, 1, first=2 ** 32 - 1), "2^32 - 1")
    rejects(capi.E_INVALID, lambda: capi.simulate_event_counts(R, [-0.1], 2, 1), "lengths must be finite")
    rejects(capi.E_INVALID, lambda: capi.simulate_event_counts(np.zeros((9, 4, 4)), [0.1], 2, 1), "event classes")

    c1 = cases.make_case(6, 80, rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25)), *rm.constant_rate(), seed=3, rooted=True,
                         compress=False)                      # 80 patterns: the table route, not the batched-points one
    with cases.make_engine(c1) as e:                          # DNA walk without kept CLVs
        e.eval(capi.EVAL_LNL)
        rejects(capi.E_STATE, lambda: e.expected_events(R, 10, 1), "KEEP_CLVS")
    Rc = _chr_model()
    ch, _ = _five_taxon_engine_case(Rc)
    with cases.make_engine(ch, flags=capi.FLAG_KEEP_CLVS) as e:
        rejects(capi.E_STATE, lambda: e.expected_events(Rc, 10, 1), "no evaluation")
        e.eval(capi.EVAL_LNL)
        rejects(capi.E_STATE, lambda: e.expected_events(Rc, 10, 1), "derivatives")
        e.eval(capi.EVAL_LNL | capi.EVAL_D1)
        rejects(capi.E_INVALID, lambda: e.expected_events(Rc, 0, 1), "n_sims >= 1")
        Rn = Rc.copy()
        Rn[0, 0, 1] = -1.0
        rejects(capi.E_INVALID, lambda: e.expected_events(Rn, 10, 1), "finite and >= 0")
    with cases.make_engine(ch, flags=capi.FLAG_KEEP_CLVS, n_points=2, n_models=1) as e:   # one pattern, two points: batched path
        e.eval(capi.EVAL_LNL)                                     # (which has no derivative pass)
        rejects(capi.E_STATE, lambda: e.expected_events(Rc, 10, 1), "batched-points")
    r, p = rm.gamma_rates(2, 0.5)
    c2 = cases.make_case(6, 20, rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25)), r, p, seed=3, rooted=True)
    with cases.make_engine(c2, flags=capi.FLAG_KEEP_CLVS) as e:
        e.eval(capi.EVAL_LNL | capi.EVAL_D1)
        rejects(capi.E_INVALID, lambda: e.expected_events(R, 10, 1), "one rate class")
    with cases.make_engine(c1, flags=capi.FLAG_KEEP_CLVS, n_models=2) as e:
        md = cases.to_model_desc(c1.model)
        e._model_holders.append(md)
        e.set_model(1, md)
        slots = np.zeros(c1.flat.n_nodes, np.int32)
        slots[0] = 1
        e.set_branch_models(0, slots)
        e.eval(capi.EVAL_LNL | capi.EVAL_D1)
        rejects(capi.E_INVALID, lambda: e.expected_events(R, 10, 1), "different model slots")
    with cases.make_engine(c1, flags=capi.FLAG_KEEP_CLVS, n_points=2) as e:
        e.eval(capi.EVAL_LNL | capi.EVAL_D1)
        errs = []
        for p in (0, 1):
            try:
                e.expected_events(R, 10, 1, point=p)
            except capi.BppGpuError as x:
                errs.append(x)
        assert len(errs) == 1 and errs[0].code == capi.E_STATE and "resident" in str(errs[0]), errs


@pytest.mark.gpu
def test_compute_chromosome_transitions_exp_through_the_shim(built_lib):
    """Five-taxon ChromEvol case: DRNonHomogeneousTreeLikelihood -> MarginalNonRevAncestralStateReconstruction ->
    ComputeChromosomeTransitionsExp (1e5 paths).  The class's values equal the likelihood's own bppgpu_expected_events call
    with the same seed exactly, and the oracle's exact expectation within simulation tolerance."""
    exe = compile_cpp("test_chr_expectations", built_lib)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    vals = {f[0]: float(f[1]) for f in (line.split() for line in r.stdout.splitlines()) if len(f) == 2}
    assert vals["ABI_MISMATCHES"] == 0
    R = _chr_model()
    ch, m = _five_taxon_engine_case(R)
    ch.root_freqs = m.freq
    res = cases.oracle_eval(ch, want_d1=True, weighted_root=True)
    assert abs(vals["LNL"] - res.lnl) <= 1e-9 * abs(res.lnl)
    flat = ch.flat
    joints = {b: rl.marginal_posteriors(flat, res, res.P, b, ch.probs)[1] for b in range(flat.n_nodes) if b != flat.root}
    t_of_node = np.asarray(flat.brlen, float).copy()
    t_of_node[flat.root] = 0.0
    Q = mp.generator(R)
    exact = mp.exact_expected(Q, R, t_of_node, joints, ch.weights)
    ex = np.array([[vals["EXP_%d_%d" % (b, t)] for t in range(5)] for b in range(flat.n_nodes)])
    un = np.array([vals["UNREACHED_%d" % b] for b in range(flat.n_nodes)])
    tol = _expected_tolerance(Q, R, t_of_node, joints, ch.weights, 100000, un)
    assert np.all(np.abs(ex - exact) <= tol), np.max(np.abs(ex - exact) / tol)
    assert np.all(ex[flat.root] == 0)
    for t in range(5):
        assert abs(vals["TOTAL_%d" % t] - ex[:, t].sum()) <= 1e-12 * max(1.0, abs(ex[:, t].sum()))
