"""The oracle against every known-answer value the reference's own tests hold for the path
(SURVEY.md section 8c).  CPU only."""
import numpy as np
import pytest

from oracle import ref_likelihood as rl
from oracle import ref_models as rm
from oracle import ref_patterns as rp
from oracle import ref_tree as rt
import cases

# test/test_likelihood.cpp:91-108
TREE1 = "((A:0.01, B:0.02):0.03,C:0.01,D:0.1);"
SEQS1 = {"A": "AAATGGCTGTGCACGTC", "B": "GACTGGATCTGCACGTC", "C": "CTCTGGATGTGCACGTG", "D": "AAATGGCGGTGCGCCTA"}
GOLD1 = 85.030942031997312824
# test/test_likelihood_clock.cpp:99-115
TREE2 = "(((A:0.01, B:0.01):0.02,C:0.03):0.01,D:0.04);"
SEQS2 = {"A": "AAATGGCTGTGCACGTC", "B": "AACTGGATCTGCATGTC", "C": "ATCTGGACGTGCACGTG", "D": "CAACGGGAGTGCGCCTA"}
GOLD2 = 94.3957


def case1():
    r, p = rm.gamma_rates(4, 1.0)
    return cases.case_from_alignment(TREE1, SEQS1, rm.t92(3.0, 0.5), r, p)


def test_gamma_class_means():
    r, p = rm.gamma_rates(4, 1.0)
    np.testing.assert_allclose(r, [0.13695378, 0.47675186, 1.0, 2.38629436], atol=5e-9)
    np.testing.assert_allclose(p, 0.25)


def test_pattern_order_matches_survey_appendix_c():
    c = case1()
    assert [u.decode() for u in c.patterns] == ["AAAG", "AATA", "ACCA", "AGCA", "CAAC", "CCCC", "CCGA", "GCGG",
                                                "GGGC", "GGGG", "TTTG", "TTTT"]
    assert int(c.weights.sum()) == 17
    # indices_: site -> pattern reproduces every original column
    flat = c.flat
    cols = rp.columns_from_sequences([SEQS1[n] for n in flat.leaf_names])
    assert [c.patterns[i] for i in c.site_index] == cols


def test_golden_dr_class_value():
    c = case1()
    for scaled in (False, True):
        res = cases.oracle_eval(c, scaled=scaled)
        assert abs(-res.lnl - GOLD1) < 1e-9, (-res.lnl, GOLD1)


def test_golden_r_class_value_recursive_patterns():
    """R classes: per-subtree compression + per-site sum (RHomogeneousTreeLikelihood.cpp:162-176)."""
    r, p = rm.gamma_rates(4, 1.0)
    m = rm.t92(3.0, 0.5)
    flat = rt.FlatTree(rt.parse_newick(TREE1))
    rec = rp.recursive_patterns(flat, SEQS1)
    chars, table = rp.init_value_table(rp.DNA_STATES, rp.DNA_ALIASES)
    tip_codes = {lid: rp.encode_columns(rec["cols"][lid], chars)[0] for lid in flat.leaf_ids}
    P, _, _ = rm.transition_tables(m, flat.brlen, r)
    clv, ex, _ = rl.prune(flat, tip_codes, table, P, 4, links=rec["links"])
    lnl, _ = rl.loglik_R(clv, ex, m.freq, p, rec["root_links"])
    assert abs(-lnl - GOLD1) < 1e-9


def test_golden_hky85_equals_t92():
    """BASELINE.json config 1 says HKY85; the test uses T92(theta=.5) = HKY85(kappa=3, pi=1/4) (SURVEY finding 4)."""
    r, p = rm.gamma_rates(4, 1.0)
    c = cases.case_from_alignment(TREE1, SEQS1, rm.hky85(3.0), r, p)
    assert abs(-cases.oracle_eval(c).lnl - GOLD1) < 1e-9


def test_golden_clock_rooted_constant_rate():
    r, p = rm.constant_rate()
    c = cases.case_from_alignment(TREE2, SEQS2, rm.t92(3.0, 0.5), r, p, check_rooted=False)
    assert len(c.flat.children[c.flat.root]) == 2
    assert abs(-cases.oracle_eval(c).lnl - GOLD2) < 1e-4        # the reference prints 6 digits


def test_r_vs_dr_derivatives_identity():
    """test/test_likelihood.cpp:124-135: d1 from the single and the double recursion agree to 1e-6."""
    c = case1()
    res = cases.oracle_eval(c, want_d1=True, want_d2=True, scaled=False)
    for b in range(c.flat.n_nodes - 1):
        d1r = rl.r_derivative(c.flat, c.codes_by_leaf, c.table, res.P, res.dP, 4, c.root_freqs, c.probs,
                              c.weights.astype(float), b, order=1)
        d2r = rl.r_derivative(c.flat, c.codes_by_leaf, c.table, res.P, res.dP, 4, c.root_freqs, c.probs,
                              c.weights.astype(float), b, order=2, d2P=res.d2P)
        assert abs(d1r - res.d1[b]) < 1e-6
        assert abs(d2r - res.d2[b]) < 1e-6 * max(1.0, abs(d2r))


def test_derivatives_vs_finite_differences():
    c = case1()
    res = cases.oracle_eval(c, want_d1=True, want_d2=True)
    h = 1e-5
    for b in range(c.flat.n_nodes - 1):
        bl = c.flat.brlen.copy()
        bl[b] += h
        fp = -cases.oracle_eval(c, brlen=bl).lnl
        bl[b] -= 2 * h
        fm = -cases.oracle_eval(c, brlen=bl).lnl
        f0 = -res.lnl
        assert abs((fp - fm) / (2 * h) - res.d1[b]) < 1e-5 * max(1, abs(res.d1[b]))
        assert abs((fp - 2 * f0 + fm) / h ** 2 - res.d2[b]) < 2e-3 * max(1, abs(res.d2[b]))


def test_grantham_table_against_grantham_s_formula_and_gy94_structure():
    """The restated Grantham (1974) table (GY94's index; bpp-seq is not under /root/reference) against the paper's own formula
    D = 50.723 sqrt(1.833 dc^2 + 0.1018 dp^2 + 0.000399 dv^2) from composition, polarity and volume: every entry within rounding
    except the two entries the published table is known to carry off-formula (Asn-Glu 42, Asp-Trp 181).  GY94 itself: V -> inf
    gives YN98 with omega = 1, small V suppresses radical changes most, frequencies are the codon frequencies."""
    import math
    d = rm.grantham_matrix()
    assert len(d) == 400 and d["L", "I"] == 5 and d["C", "W"] == 215 and d["S", "R"] == 110
    for a in rm.GRANTHAM_ORDER:
        for b in rm.GRANTHAM_ORDER:
            (ca, pa, va), (cb, pb, vb) = rm.GRANTHAM_PROPERTIES[a], rm.GRANTHAM_PROPERTIES[b]
            f = 50.723 * math.sqrt(1.833 * (ca - cb) ** 2 + 0.1018 * (pa - pb) ** 2 + 0.000399 * (va - vb) ** 2)
            if {a, b} in ({"N", "E"}, {"D", "W"}):
                assert abs(f - d[a, b]) < 10
            else:
                assert abs(f - d[a, b]) <= 1.01, (a, b, f, d[a, b])
    big, yn = rm.gy94(2.0, 1e12), rm.yn98(2.0, 1.0)
    np.testing.assert_allclose(big.Q, yn.Q, atol=1e-10)
    m = rm.gy94(2.0, 50.0)
    aa = rm.standard_genetic_code()
    i, j_cons, j_rad = 16 * 3 + 4 * 3 + 3, 16 * 3 + 4 * 3 + 1, 16 * 3 + 4 * 2 + 3        # TTT(F) -> TTC(F) syn, -> TGT(C) radical
    assert aa[i] == "F" and aa[j_cons] == "F" and aa[j_rad] == "C"
    assert m.Q[i, j_rad] / m.Q[i, j_cons] == pytest.approx(math.exp(-205 / 50.0) / 2.0, rel=1e-12)   # transversion vs transition(kappa=2)
    F = m.freq[:, None] * m.Q
    np.testing.assert_allclose(F, F.T, atol=1e-14)


@pytest.mark.parametrize("name", ["gtr", "lg08", "yn98", "gy94", "chromosome"])
def test_pt_family_against_scipy_expm(name):
    from scipy.linalg import expm
    m = {"gtr": lambda: rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25)),
         "lg08": rm.lg08,
         "yn98": lambda: rm.yn98(2.0, 0.3), "gy94": lambda: rm.gy94(2.0, 50.0),
         "chromosome": lambda: rm.chromosome(1, 30, gain=0.7, loss=0.4, dupl=0.2, demi=rm.DEMI_EQUAL_DUPL)}[name]()
    for t in (1e-6, 0.05, 0.7, 3.0):
        E = expm(m.Q * m.rate * t)
        P = rm.pij_t(m, t)
        tol = 1e-10 if name != "chromosome" else 1e-8
        np.testing.assert_allclose(P, np.where(m.chromosome & (E < 0), rm.VERY_TINY, E), atol=tol)
        np.testing.assert_allclose(P.sum(axis=1), 1.0, atol=1e-9)
        if not m.chromosome:
            np.testing.assert_allclose(rm.dpij_dt(m, t), m.rate * m.Q @ E, atol=1e-9)
            np.testing.assert_allclose(rm.d2pij_dt2(m, t), m.rate ** 2 * m.Q @ m.Q @ E, atol=1e-8)


def test_reversible_models_detailed_balance_and_normalisation():
    for m in (rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25)), rm.lg08(), rm.yn98(2.0, 0.3)):
        F = m.freq[:, None] * m.Q
        np.testing.assert_allclose(F, F.T, atol=1e-14)
        assert abs(-np.dot(np.diag(m.Q), m.freq) - 1.0) < 1e-12


@pytest.mark.parametrize("S,mk", [(4, lambda: rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))),
                                  (20, rm.lg08)])
def test_pruning_against_brute_force(S, mk):
    """Sum over all internal-state assignments on a 4-taxon tree (2 internal nodes)."""
    m = mk()
    rates, probs = rm.gamma_rates(2, 0.7)
    c = cases.make_case(4, 3, m, rates, probs, seed=5, random_tips=True)
    res = cases.oracle_eval(c, scaled=False)
    for i in range(c.N):
        L = 0.0
        for ci, r in enumerate(rates):
            Pc = {n: rm.pij_t(m, c.flat.brlen[n] * r) for n in range(c.flat.n_nodes - 1)}
            tips = {l: c.table[c.codes_by_leaf[l][i]] for l in c.flat.leaf_ids}
            L += probs[ci] * rl.brute_force_site(c.flat, tips, Pc, c.root_freqs)
        assert abs(np.log(L) - res.site_lnl[i]) < 1e-12 * abs(np.log(L)) + 1e-13


def test_scaled_equals_unscaled_where_finite_and_survives_underflow():
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    rates, probs = rm.gamma_rates(4, 0.5)
    c = cases.make_case(40, 30, m, rates, probs, seed=3)
    a = cases.oracle_eval(c, scaled=False)
    b = cases.oracle_eval(c, scaled=True)
    assert abs(a.lnl - b.lnl) <= 1e-12 * abs(a.lnl)
    big = cases.make_case(700, 4, m, rates, probs, seed=4, random_tips=True, mean_brlen=0.5)
    assert not np.isfinite(cases.oracle_eval(big, scaled=False).lnl)      # the reference would return -inf
    s = cases.oracle_eval(big, scaled=True)
    assert np.isfinite(s.lnl) and s.SR_exp.max() > 256


def test_posterior_probabilities_against_brute_force_enumeration():
    """likelihood_at_node / posterior_probabilities (the restatement of computeLikelihoodAtNode_ and
    DRTreeLikelihoodTools.cpp:46-119) equal the marginals obtained by enumerating every assignment of the internal states."""
    import itertools
    import cases
    from oracle import ref_likelihood as rl
    r, p = rm.gamma_rates(2, 0.7)
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    c = cases.make_case(5, 6, m, r, p, seed=5, compress=False, ambiguity=0.1)
    res = cases.oracle_eval(c, want_d1=True)
    flat, S = c.flat, 4
    internals = [n for n in range(flat.n_nodes) if not flat.is_leaf[n]]
    for i in (0, 2, 5):
        tot = {n: np.zeros((len(r), S)) for n in internals}
        for cc in range(len(r)):
            for states in itertools.product(range(S), repeat=len(internals)):
                st = dict(zip(internals, states))
                pr = c.root_freqs[st[flat.root]]
                for n in range(flat.n_nodes - 1):
                    f = int(flat.parent[n])
                    if flat.is_leaf[n]:
                        pr *= (res.P[n][cc][st[f]] * c.table[c.codes_by_leaf[n][i]]).sum()
                    else:
                        pr *= res.P[n][cc][st[f]][st[n]]
                for n in internals:
                    tot[n][cc, st[n]] += pr
        for n in internals:
            post = rl.posterior_probabilities(flat, res, res.P, n, c.probs)
            np.testing.assert_allclose(post[i], tot[n] / tot[n].sum(), rtol=1e-12, atol=1e-16)
            A, E = rl.likelihood_at_node(flat, res, res.P, n)
            np.testing.assert_allclose(np.ldexp(A[i], -E[i][:, None]), tot[n], rtol=1e-12, atol=1e-300)
    # leaves: the reference's formula uses the leaf likelihoods alone
    leaf = flat.leaf_ids[0]
    post = rl.posterior_probabilities(flat, res, res.P, leaf, c.probs, c.codes_by_leaf, c.table)
    np.testing.assert_allclose(post.sum(axis=(1, 2)), 1.0, rtol=1e-14)


def test_root_reparametrisation_derivatives_against_finite_differences():
    """root_reparam_derivatives (BrLenRoot / RootPosition, DRNonHomogeneousTreeLikelihood.cpp:445-478, :576-867): first order equals
    the reference's combination of the two root branches' derivatives, both orders equal central differences of -lnL; with
    a reversible model and stationary root frequencies the root position is not identifiable (pulley principle): zero derivative."""
    import cases
    from oracle import ref_likelihood as rl
    r, p = rm.gamma_rates(3, 0.7)
    m = rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))
    c = cases.make_case(7, 40, m, r, p, seed=11, rooted=True, ambiguity=0.05, mean_brlen=0.2)
    res = cases.oracle_eval(c, want_d1=True, want_d2=True)
    g = rl.root_reparam_derivatives(c.flat, res, res.P, res.dP, res.d2P, c.probs, c.weights)
    assert abs(g["d1_pos"]) < 1e-10 and abs(g["d2_pos"]) < 1e-10
    c.root_freqs = np.array([.1, .4, .3, .2])
    res = cases.oracle_eval(c, want_d1=True, want_d2=True)
    g = rl.root_reparam_derivatives(c.flat, res, res.P, res.dP, res.d2P, c.probs, c.weights)
    r1, r2, L, pos = g["root1"], g["root2"], g["length"], g["pos"]
    assert abs(g["d1_len"] - (pos * res.d1[r1] + (1 - pos) * res.d1[r2])) < 1e-9        # :445-463
    assert abs(g["d1_pos"] - L * (res.d1[r1] - res.d1[r2])) < 1e-9                      # :464-478

    def nll(length, q):
        bl = np.array(c.flat.brlen)
        bl[r1], bl[r2] = length * q, length * (1 - q)
        return -cases.oracle_eval(c, brlen=bl).lnl
    h, f0 = 1e-5, nll(L, pos)
    assert abs((nll(L + h, pos) - nll(L - h, pos)) / (2 * h) - g["d1_len"]) < 1e-6
    assert abs((nll(L, pos + h) - nll(L, pos - h)) / (2 * h) - g["d1_pos"]) < 1e-6
    assert abs((nll(L + h, pos) - 2 * f0 + nll(L - h, pos)) / h ** 2 - g["d2_len"]) < 2e-3 * abs(g["d2_len"])
    assert abs((nll(L, pos + h) - 2 * f0 + nll(L, pos - h)) / h ** 2 - g["d2_pos"]) < 2e-3 * abs(g["d2_pos"])


def test_marginal_nonrev_posteriors_one_pass_equals_reference_s_pass_form_and_enumeration():
    """MarginalNonRevAncestralStateReconstruction (fork): the one-pass restatement (ordinary prefix arrays) equals the
    reference's S-pass algorithm restated literally (prefix pass conditional on every root state,
    DRNonHomogeneousTreeLikelihood.cpp:1026-1162 + MarginalNonRev...cpp:10-136) and, independently, the node and
    (node, father) marginals obtained by enumerating every assignment of the internal states.  Non-reversible model
    (chromosome gains / losses / duplications), non-stationary root frequencies, rooted tree: nothing cancels."""
    import itertools
    import cases
    from oracle import ref_likelihood as rl
    r, p = rm.gamma_rates(2, 0.7)
    m = rm.chromosome(1, 5, gain=0.9, loss=0.4, dupl=0.3)
    S = m.size
    c = cases.make_case(5, 4, m, r, p, seed=17, rooted=True, compress=False, mean_brlen=0.3)
    c.root_freqs = np.array([.1, .3, .2, .25, .15])
    res = cases.oracle_eval(c, want_d1=True, scaled=False)
    flat = c.flat
    post_ref, joint_ref = rl.marginal_posteriors_by_root_state(flat, res, res.P, c.probs)
    for n in range(flat.n_nodes):
        post, joint = rl.marginal_posteriors(flat, res, res.P, n, c.probs)
        np.testing.assert_allclose(post, post_ref[n], rtol=1e-12, atol=1e-16)
        np.testing.assert_allclose(post.sum(axis=1), 1.0, rtol=1e-12)
        if n != flat.root:
            np.testing.assert_allclose(joint, joint_ref[n], rtol=1e-12, atol=1e-16)
    # the scaled arrays (what the device holds) give the same posteriors
    res_s = cases.oracle_eval(c, want_d1=True, scaled=True)
    for n in range(flat.n_nodes):
        np.testing.assert_allclose(rl.marginal_posteriors(flat, res_s, res_s.P, n, c.probs)[0], post_ref[n], rtol=1e-12, atol=1e-16)
    # brute force: P(node = x, father = y | data) by enumeration of the internal states
    internals = [n for n in range(flat.n_nodes) if not flat.is_leaf[n]]
    for i in (0, 3):
        tot = {n: np.zeros((S, S)) for n in range(flat.n_nodes) if n != flat.root}
        rootm = np.zeros(S)
        for cc in range(len(r)):
            for states in itertools.product(range(S), repeat=len(internals)):
                st = dict(zip(internals, states))
                pr = c.probs[cc] * c.root_freqs[st[flat.root]]
                leaf_terms = {}
                for n in range(flat.n_nodes - 1):
                    f = int(flat.parent[n])
                    if flat.is_leaf[n]:
                        leaf_terms[n] = res.P[n][cc][st[f]] * c.table[c.codes_by_leaf[n][i]]     # over the leaf's state x
                        pr *= leaf_terms[n].sum()
                    else:
                        pr *= res.P[n][cc][st[f]][st[n]]
                rootm[st[flat.root]] += pr
                for n in tot:
                    f = int(flat.parent[n])
                    if flat.is_leaf[n]:
                        s = leaf_terms[n].sum()
                        if s > 0:
                            tot[n][:, st[f]] += pr * leaf_terms[n] / s
                    else:
                        tot[n][st[n], st[f]] += pr
        L = rootm.sum()
        np.testing.assert_allclose(rl.marginal_posteriors(flat, res, res.P, flat.root, c.probs)[0][i], rootm / L, rtol=1e-11)
        for n in tot:
            np.testing.assert_allclose(joint_ref[n][i], tot[n] / L, rtol=1e-10, atol=1e-16)


def test_ml_joint_reconstruction_against_enumeration():
    """ml_joint_reconstruction (the restatement of MLAncestralStateReconstruction's max-product recursion and trace back): the
    assignment it returns has the largest joint probability among ALL assignments of the internal states, and the root array's
    maximum is that probability.  One rate class (the reference assumes it), non-reversible model, free root frequencies."""
    import itertools
    import cases
    from oracle import ref_likelihood as rl
    r, p = rm.constant_rate()
    m = rm.chromosome(1, 5, gain=0.9, loss=0.4, dupl=0.3)
    S = m.size
    c = cases.make_case(6, 5, m, r, p, seed=29, rooted=True, compress=False, mean_brlen=0.4)
    c.root_freqs = np.array([.1, .3, .2, .25, .15])
    res = cases.oracle_eval(c)
    flat = c.flat
    states, Lroot = rl.ml_joint_reconstruction(flat, c.codes_by_leaf, c.table, res.P, c.root_freqs)
    internals = [n for n in range(flat.n_nodes) if not flat.is_leaf[n]]
    for i in range(c.N):
        def joint(st):
            pr = c.root_freqs[st[flat.root]]
            for n in range(flat.n_nodes - 1):
                f = int(flat.parent[n])
                pr *= res.P[n][0][st[f]][st[n]]
            return pr
        obs = {l: int(c.codes_by_leaf[l][i]) for l in flat.leaf_ids}
        assert all(v < S for v in obs.values())                      # no ambiguity in this case
        best = max(joint({**obs, **dict(zip(internals, s))}) for s in itertools.product(range(S), repeat=len(internals)))
        got = joint({n: int(states[n][i]) for n in range(flat.n_nodes)})
        assert all(states[l][i] == obs[l] for l in flat.leaf_ids)
        assert abs(got - best) <= 1e-13 * best
        assert abs(Lroot[i, 0].max() - best) <= 1e-13 * best


def _relax_case():
    import cases
    from oracle import ref_patterns as rp
    from oracle import ref_tree as rt
    cod_states = [a + b + c_ for a in "ACGT" for b in "ACGT" for c_ in "ACGT"]
    flat = rt.FlatTree(rt.parse_newick("(((A:0.01, B:0.01):0.02,C:0.03):0.01,D:0.04);"), check_rooted=False)
    seqs = {"A": "AAATGGCTGTGCACGTCT", "B": "AACTGGATCTGCATGTCT", "C": "ATCTGGACGTGCACGTGT", "D": "CAACGGGAGTGCGCCTAT"}
    uniq, w, idx = rp.global_patterns(seqs, flat.leaf_names, width=3)
    codes = rp.encode_columns(uniq, cod_states, width=3)
    c = cases.Case()
    c.flat, c.rates, c.probs = flat, np.ones(1), np.ones(1)
    c.table, c.N, c.weights = np.eye(64), len(uniq), w
    c.codes_by_leaf = {lid: codes[k] for k, lid in enumerate(flat.leaf_ids)}
    c.code_dtype = codes.dtype
    return c


def _mixture_minus_lnl(c, paths, probs):
    """sum over the sites of -log sum_k p_k L_k(site); paths[k] = (models, slot_of_node) of component k"""
    import cases
    site = []
    for models, slots in paths:
        c.root_freqs = np.asarray(models[0].freq)
        site.append(cases.oracle_eval_nh(c, models, slots, nh_form=False).site_lnl)
    mixed = np.log(np.sum(np.asarray(probs)[:, None] * np.exp(np.asarray(site)), axis=0))
    return -float(np.sum(c.weights * mixed))


def test_relax_equals_m2_when_k_is_one_and_partitions_do_not_matter():
    """The assertions of test/test_relax.cpp:104-141 on the oracle: RELAX(kappa=2, p=0.1, omega1=1, omega2=2, k=1, theta1=0.5,
    theta2=0.8) on any partition of the branches into two model groups gives the likelihood of YNGP_M2(kappa=2, omega0=0.1,
    omega2=2, theta1=0.5, theta2=0.8); with k != 1 on one group it does not."""
    c = _relax_case()
    nn = c.flat.n_nodes
    m2, p2 = rm.yngp_m2(2.0, 0.1, 2.0, 0.5, 0.8)
    np.testing.assert_allclose(p2, [0.5, 0.4, 0.1])
    assert abs(float(np.dot(p2, [m.rate for m in m2])) - 1.0) < 1e-14
    # equal synonymous rates across the components (the point of the homogenisation)
    syn = [m.rate * m.Q[2, 0] for m in m2]
    assert max(syn) - min(syn) < 1e-15
    ref = _mixture_minus_lnl(c, [([m], np.zeros(nn, np.int64)) for m in m2], p2)
    r1, pr = rm.relax(2.0, 0.1, 1.0, 2.0, 1.0, 0.5, 0.8)
    for group0 in ([0], [1, 2, 3, 4, 5]):                                      # model1.nodes_id of the two partitions
        slots = np.array([0 if n in group0 else 1 for n in range(nn)])
        v = _mixture_minus_lnl(c, [([a, b], slots) for a, b in zip(r1, r1)], pr)
        assert abs(v - ref) < 1e-9
    r2, _ = rm.relax(2.0, 0.1, 1.0, 2.0, 0.3, 0.5, 0.8)
    slots = np.array([0 if n == 0 else 1 for n in range(nn)])
    v = _mixture_minus_lnl(c, [([a, b], slots) for a, b in zip(r2, r1)], pr)
    assert abs(v - ref) > 1e-4


def test_lg08_tables_are_the_reference_s_own_numbers():
    """The committed LG08 tables (oracle/lg08_data.py and the shim's lg08_data.inc) against the assignment lists the reference
    includes (Model/Protein/__LG08ExchangeabilityCode, __LG08FrequenciesCode; LG08.cpp:53-62), stored entry by entry in
    tests/golden/lg08_reference.json."""
    import json
    import pathlib
    import re
    from oracle.lg08_data import LG08_FREQ, LG08_LOWER
    gold = json.loads((pathlib.Path(__file__).resolve().parent / "golden" / "lg08_reference.json").read_text())
    ex = np.zeros((20, 20))
    for i, j, v in gold["exchangeabilities"]:
        ex[i, j] = ex[j, i] = v
    fr = np.array(gold["frequencies"])
    assert len(gold["exchangeabilities"]) == 190 and np.count_nonzero(ex - np.diag(np.diag(ex))) == 380 and len(fr) == 20
    for i in range(1, 20):
        assert list(ex[i, :i]) == list(LG08_LOWER[i - 1])
    assert list(fr) == list(LG08_FREQ)
    inc = (pathlib.Path(__file__).resolve().parent.parent / "bpp_phyl_b200" / "host" / "lg08_data.inc").read_text()
    nums = [float(x) for x in re.findall(r"(?<![\w.])\d+\.\d+(?:[eE][+-]?\d+)?", inc.split("LG08_LOWER[190]")[1])]
    assert nums[:190] == [ex[i, j] for i in range(1, 20) for j in range(i)] and nums[190:210] == list(fr)
    # the exchangeabilities and frequencies define the generator the oracle builds
    m = rm.lg08()
    np.testing.assert_allclose(m.freq, fr / fr.sum(), rtol=1e-12)


def test_chromosome_pijt_rows_sum_to_one_like_test_chr_model():
    """test/test_chr_model.cpp:100-114,141,152-168: ChromosomeSubstitutionModel(1..25; gain 2, loss 1, dupl 3, demi 1.3) -- every row
    of getPij_t sums to 1 within 1e-4 for the tree's branch lengths (the tree file is not in the repository: a spread of lengths),
    through the eigen path and through the model's own Taylor rule, and the two agree within the rule's 1e-4 test."""
    m = rm.chromosome(1, 25, gain=2.0, loss=1.0, dupl=3.0, demi=1.3)
    for t in (1e-6, 0.003, 0.05, 0.3, 1.0, 3.6):
        P = rm.pij_t(m, t)
        assert np.all(np.abs(P.sum(axis=1) - 1.0) <= 1e-4)
        assert P.min() >= 0.0 and P.max() <= 1.0
        T = rm._chr_pij_t(m, t, False)
        assert np.all(np.abs(T.sum(axis=1) - 1.0) <= 1e-4)
        assert np.abs(T - P).max() <= 2e-4


def test_t92_generator_and_closed_form_transition_probabilities():
    """The oracle's generic route for T92 (generator -> eigen-decomposition -> V exp(D t) V^-1) against the reference's analytic T92:
    generator and normalisation r_ (Model/Nucleotide/T92.cpp:81-116) and the closed-form getPij_t (:355-386) with its t-derivatives
    (getdPij_dt / getd2Pij_dt2 differentiate the same expressions), for several kappa, theta, t and a model rate != 1."""
    for kappa, theta in ((3.0, 0.5), (0.7, 0.2), (8.0, 0.83)):
        pi = np.array([(1 - theta) / 2, theta / 2, theta / 2, (1 - theta) / 2])
        k = (kappa + 1.0) / 2.0
        r = 2.0 / (1.0 + 2.0 * theta * kappa - 2.0 * theta * theta * kappa)
        G = np.zeros((4, 4))
        G[0, 0] = G[3, 3] = -(1.0 + theta * kappa) / 2
        G[1, 1] = G[2, 2] = -(1.0 + (1.0 - theta) * kappa) / 2
        G[1, 0] = G[3, 0] = G[0, 3] = G[2, 3] = (1.0 - theta) / 2
        G[0, 1] = G[2, 1] = G[1, 2] = G[3, 2] = theta / 2
        G[2, 0] = G[1, 3] = kappa * (1.0 - theta) / 2
        G[3, 1] = G[0, 2] = kappa * theta / 2
        m = rm.t92(kappa, theta)
        np.testing.assert_allclose(m.Q, G * r, rtol=0, atol=1e-14)
        np.testing.assert_allclose(m.freq, pi, rtol=0, atol=1e-15)
        for rate in (1.0, 0.37):
            m.rate = rate
            for t in (1e-6, 0.01, 0.3, 2.5):
                def closed(order):
                    s = rate * r                                     # l_ = rate_ * r_ * d
                    e1 = (-s) ** order * np.exp(-s * t)
                    e2 = (-k * s) ** order * np.exp(-k * s * t)
                    one = 1.0 if order == 0 else 0.0
                    P = np.empty((4, 4))
                    P[0] = [pi[0] * (one + e1) + theta * e2, pi[1] * (one - e1), pi[2] * (one + e1) - theta * e2, pi[3] * (one - e1)]
                    P[1] = [pi[0] * (one - e1), pi[1] * (one + e1) + (1 - theta) * e2, pi[2] * (one - e1), pi[3] * (one + e1) - (1 - theta) * e2]
                    P[2] = [pi[0] * (one + e1) - (1 - theta) * e2, pi[1] * (one - e1), pi[2] * (one + e1) + (1 - theta) * e2, pi[3] * (one - e1)]
                    P[3] = [pi[0] * (one - e1), pi[1] * (one + e1) - theta * e2, pi[2] * (one - e1), pi[3] * (one + e1) + theta * e2]
                    return P
                np.testing.assert_allclose(rm.pij_t(m, t), closed(0), rtol=0, atol=2e-15)
                np.testing.assert_allclose(rm.dpij_dt(m, t), closed(1), rtol=0, atol=2e-14 * (1 + kappa))
                np.testing.assert_allclose(rm.d2pij_dt2(m, t), closed(2), rtol=0, atol=2e-13 * (1 + kappa) ** 2)


def test_gtr_generator_is_the_reference_s_exchangeability_formula():
    """GTR::updateMatrices (Model/Nucleotide/GTR.cpp:84-124): exchangeabilities / p_ with p_ = 2(a piC piT + b piA piT + c piG piT +
    d piA piC + e piC piG + piA piG), generator = exchangeability x pi (AbstractReversibleSubstitutionModel::updateMatrices,
    AbstractSubstitutionModel.cpp:694-703): one expected substitution per unit time.  The benchmark's cfg2 model."""
    a, b, c, d, e = 1.2, 0.8, 0.6, 1.5, 0.9
    pi = np.array([.3, .2, .25, .25])
    pA, pC, pG, pT = pi
    p = 2 * (a * pC * pT + b * pA * pT + c * pG * pT + d * pA * pC + e * pC * pG + pA * pG)
    ex = np.zeros((4, 4))
    ex[0, 0] = (-b * pT - pG - d * pC) / (pA * p)
    ex[1, 0] = ex[0, 1] = d / p
    ex[2, 0] = ex[0, 2] = 1 / p
    ex[3, 0] = ex[0, 3] = b / p
    ex[1, 1] = (-a * pT - e * pG - d * pA) / (pC * p)
    ex[1, 2] = ex[2, 1] = e / p
    ex[1, 3] = ex[3, 1] = a / p
    ex[2, 2] = (-c * pT - e * pC - pA) / (pG * p)
    ex[2, 3] = ex[3, 2] = c / p
    ex[3, 3] = (-c * pG - a * pC - b * pA) / (pT * p)
    Q = ex * pi[None, :]
    m = rm.gtr(a, b, c, d, e, tuple(pi))
    np.testing.assert_allclose(m.Q, Q, rtol=0, atol=1e-15)
    assert abs(-(pi * np.diag(Q)).sum() - 1.0) < 1e-15 and np.abs(Q.sum(axis=1)).max() < 1e-15


def test_hky85_generator_and_closed_form_transition_probabilities():
    """HKY85 (BASELINE configs[0]): generator and normalisation (Model/Nucleotide/HKY85.cpp:80-125) and the closed-form getPij_t
    (:351-383) with unequal base frequencies, against the oracle's generic eigen route."""
    kappa = 2.7
    pi = np.array([.31, .19, .22, .28])
    pA, pC, pG, pT = pi
    pR, pY = pA + pG, pT + pC
    k1, k2 = kappa * pY + pR, kappa * pR + pY
    G = np.array([[0, pC, kappa * pG, pT], [pA, 0, pG, kappa * pT], [kappa * pA, pC, 0, pT], [pA, kappa * pC, pG, 0]], float)
    np.fill_diagonal(G, -G.sum(axis=1))
    r = 1.0 / (2.0 * (pA * pC + pC * pG + pA * pT + pG * pT + kappa * (pC * pT + pA * pG)))
    m = rm.hky85(kappa, tuple(pi))
    np.testing.assert_allclose(m.Q, G * r, rtol=0, atol=1e-15)
    for t in (1e-6, 0.02, 0.4, 3.0):
        l = r * t
        e1, e22, e21 = np.exp(-l), np.exp(-k2 * l), np.exp(-k1 * l)
        P = np.empty((4, 4))
        P[0] = [pA * (1 + pY / pR * e1) + pG / pR * e22, pC * (1 - e1), pG * (1 + pY / pR * e1) - pG / pR * e22, pT * (1 - e1)]
        P[1] = [pA * (1 - e1), pC * (1 + pR / pY * e1) + pT / pY * e21, pG * (1 - e1), pT * (1 + pR / pY * e1) - pT / pY * e21]
        P[2] = [pA * (1 + pY / pR * e1) - pA / pR * e22, pC * (1 - e1), pG * (1 + pY / pR * e1) + pA / pR * e22, pT * (1 - e1)]
        P[3] = [pA * (1 - e1), pC * (1 + pR / pY * e1) - pC / pY * e21, pG * (1 - e1), pT * (1 + pR / pY * e1) + pC / pY * e21]
        np.testing.assert_allclose(rm.pij_t(m, t), P, rtol=0, atol=3e-15)


def test_bench_parameter_points_keep_every_draw_on_the_reference_s_route():
    """bench.py's chromosome workload (synth.chromosome_points): nothing is redrawn; every point carries the route the reference
    takes for it (ChromosomeSubstitutionModel.cpp:686-767: eigen form when V can be inverted and one eigenvalue is null, Taylor series
    otherwise) -- the same decision the oracle's update_matrices makes -- and eigen-route points reproduce their generator up to
    `resid`.  `well_conditioned_only` is the round-1 sample (eigen route, resid <= 1e-9)."""
    from bpp_phyl_b200 import synth
    pts = synth.chromosome_points(36, 40, seed=11, workers=2)
    assert len(pts) == 40
    routes = {p["route"] for p in pts}
    assert routes <= {"eigen", "series"}
    for p in pts:
        Q = p["Q"]
        assert np.allclose(Q.sum(axis=1), 0.0, atol=1e-12)
        if p["route"] == "eigen":
            n = len(Q)
            D = np.diag(p["ev"])
            for k in range(n - 1):
                if p["ev_im"][k] > 0:
                    D[k, k + 1], D[k + 1, k] = p["ev_im"][k], -p["ev_im"][k]
            rec = np.abs(p["V"] @ D @ p["Vinv"] - Q).max() / np.abs(Q).max()
            assert rec <= max(10 * p["resid"], 1e-6 * (p["resid"] > 1e-9) + 1e-12) or rec <= 1e-9   # (one eigenvalue was set to exactly 0)
            assert int((np.abs(p["ev"]) + np.abs(p["ev_im"]) == 0).sum()) >= 1
            gain, loss, dupl, demi = p["params"]
            m = rm.chromosome(1, n, gain=gain, loss=loss, dupl=dupl, demi=demi)
            if p["resid"] <= 1e-9:
                assert m.nonsingular                          # the oracle takes the eigen route for every well-conditioned point
        else:
            assert not np.isfinite(p["resid"])
    good = synth.chromosome_points(36, 12, seed=11, workers=2, well_conditioned_only=True)
    assert len(good) == 12 and all(p["route"] == "eigen" and p["resid"] <= 1e-9 for p in good)
