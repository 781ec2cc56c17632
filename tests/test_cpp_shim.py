"""The C++ host shim (bpp_phyl_b200/host/bppgpu_shim.hpp: the reference's class surface above the C ABI).

CPU part: the shim compiles, and its host-side pieces (rate classes, generators + host eigen-decomposition, tree
flattening, site patterns) agree with the oracle.  GPU part: tests/cpp/test_likelihood.cpp -- the reference's own
test_likelihood.cpp / test_likelihood_clock.cpp rewritten against the shim -- exits 0, and the values it prints for
the other state spaces match the oracle."""
import json
import os
import pathlib
import subprocess

import numpy as np
import pytest

import cases
from oracle import ref_models as rm
from oracle import ref_patterns as rp
from oracle import ref_tree as rt

ROOT = pathlib.Path(__file__).resolve().parent.parent
BUILD = ROOT / "tests" / "cpp" / "_build"


def compile_cpp(name, built_lib):
    BUILD.mkdir(exist_ok=True)
    src = ROOT / "tests" / "cpp" / (name + ".cpp")
    exe = BUILD / name
    hdrs = [h for h in (ROOT / "bpp_phyl_b200" / "host").rglob("*") if h.is_file()] + [ROOT / "include" / "bppgpu.h"]
    lib = ROOT / "bpp_phyl_b200" / "lib"
    if not exe.exists() or exe.stat().st_mtime < max([src.stat().st_mtime] + [h.stat().st_mtime for h in hdrs]):
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-Wno-unused", "-I", str(ROOT), "-o", str(exe), str(src),
                               "-L", str(lib), "-lbppgpu", "-Wl,-rpath," + str(lib)])
    return exe


@pytest.fixture(scope="module")
def host_doc(built_lib, tmp_path_factory):
    exe = compile_cpp("shim_host", built_lib)
    # the file readers' inputs go to a directory of this run, not to a /tmp shared with other users
    env = dict(os.environ, BPPGPU_TEST_TMP=str(tmp_path_factory.mktemp("shim_io")))
    return json.loads(subprocess.check_output([str(exe)], env=env))


def test_shim_and_reference_style_test_compile(built_lib):
    compile_cpp("test_likelihood", built_lib)


def test_gamma_rate_classes(host_doc):
    for key, (n, a) in {"gamma_4_1": (4, 1.0), "gamma_4_0.5": (4, 0.5), "gamma_8_2.3": (8, 2.3), "gamma_1_0.7": (1, 0.7)}.items():
        np.testing.assert_allclose(host_doc[key], rm.gamma_rates(n, a)[0], rtol=1e-13)


def test_file_readers_newick_fasta_phylip_chrfasta(host_doc):
    """SURVEY 8f-4, second half: Newick (multi-line, comments, text after the first ';' ignored -- Io/Newick.cpp:69-92), Fasta
    (names up to the end of the line, lower case, multi-line), sequential Phylip, the fork's chrFasta (one count per taxon)."""
    d = host_doc
    assert d["IO_tree_leaves"] == 4 and d["IO_tree_nodes"] == 6 and abs(d["IO_tree_len"] - 0.17) < 1e-15
    assert d["IO_fasta_n"] == 4 and d["IO_fasta_sites"] == 12 and d["IO_fasta_name0"] == "A first" and d["IO_fasta_B7"] == "T"
    assert d["IO_phylip_n"] == 2 and d["IO_phylip_B5"] == "C"
    assert d["IO_chr_n"] == 3 and d["IO_chr_b"] == "14" and d["IO_chr_e"] == "X"
    assert d["IO_missing_throws"] == 1


def _block_diag(re, im):
    n = len(re)
    D = np.zeros((n, n))
    i = 0
    while i < n:
        if im[i] != 0:
            D[i, i] = D[i + 1, i + 1] = re[i]
            D[i, i + 1], D[i + 1, i] = im[i], -im[i]
            i += 2
        else:
            D[i, i] = re[i]
            i += 1
    return D


@pytest.mark.parametrize("key", ["T92", "GTR", "LG08", "YN98", "GY94", "CHR_REAL", "CHR_COMPLEX", "CHR_SINGULAR"])
def test_models_generator_and_eigensystem(host_doc, key):
    m = {"T92": lambda: rm.t92(3.0, 0.5), "GTR": lambda: rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25)), "LG08": rm.lg08,
         "YN98": lambda: rm.yn98(2.0, 0.3), "GY94": lambda: rm.gy94(2.0, 50.0),
         "CHR_REAL": lambda: rm.chromosome(1, 40, gain=0.7, loss=0.4, dupl=0.2, demi=rm.DEMI_EQUAL_DUPL),
         "CHR_COMPLEX": lambda: rm.chromosome(1, 25, gain=1.5, loss=0.1, dupl=0.9, demi=0.4, gain_r=0.05),
         "CHR_SINGULAR": lambda: rm.chromosome(1, 20, gain=0.5, loss=0.0, dupl=0.0)}[key]()
    c = host_doc[key]
    Q = np.array(c["Q"])
    np.testing.assert_allclose(Q, m.Q, rtol=0, atol=1e-14 * np.abs(m.Q).max())          # generator: same numbers
    np.testing.assert_allclose(c["freq"], m.freq, rtol=0, atol=1e-15)
    assert bool(c["nonsingular"]) == m.nonsingular and bool(c["diagonalizable"]) == m.diagonalizable
    if c["nonsingular"]:
        # only V f(D) V^-1 matters (SURVEY appendix B): the shim's eigen form must reproduce the generator
        V, Vi = np.array(c["V"]), np.array(c["Vinv"])
        R = V @ _block_diag(c["re"], c["im"]) @ Vi
        assert np.abs(R - Q).max() <= 1e-10 * np.abs(Q).max()
        np.testing.assert_allclose(np.sort(c["re"]), np.sort(m.ev_re), rtol=0, atol=1e-10 * np.abs(Q).max())


def test_omega_mixtures_and_model_set_parameters_host_side(host_doc):
    """YNGP_M2 / RELAX sub-model rates and probabilities (host logic of the shim) equal the oracle's restatement of
    YNGP_M2.cpp:134-146 / RELAX.cpp:176-218; SubstitutionModelSet naming, aliasing and root frequency set."""
    m2, p2 = rm.yngp_m2(2.0, 0.1, 2.0, 0.5, 0.8)
    np.testing.assert_allclose(host_doc["M2_rates"], [m.rate for m in m2], rtol=1e-10)
    np.testing.assert_allclose(host_doc["M2_probs"], p2, rtol=0, atol=1e-15)
    np.testing.assert_allclose(host_doc["M2_Q_AAG_AAA"], [m.Q[2, 0] for m in m2], rtol=1e-10)
    rx, _ = rm.relax(2.0, 0.1, 1.0, 2.0, 2.0, 0.5, 0.8)
    np.testing.assert_allclose(host_doc["RELAX_k2_rates"], [m.rate for m in rx], rtol=1e-10)
    assert host_doc["NHSET_kappas"] == [5.0] * 6
    assert host_doc["NHSET_thetas"] == [0.5, 0.5, 0.5, 0.7, 0.5, 0.5]
    np.testing.assert_allclose(host_doc["NHSET_rootfreqs"], [0.4, 0.1, 0.1, 0.4], rtol=0, atol=1e-15)
    assert host_doc["NHSET_nparams"] == 1 + 1 + 6            # GC.theta, the shared kappa, six thetas


def test_batched_brent_line_searches_host_side(host_doc):
    """BatchedBrent (SURVEY 8f-1: every point's probe of a line search in ONE batched evaluation) on five analytic, non-smooth,
    coupled 2-d functions: every searched point ends at a local minimum of its own function along both coordinates (checked
    against scipy on the same function), never above its start; the point left inactive does not move; the number of batched
    evaluations is that of the slowest point, not the sum over the points."""
    from scipy.optimize import minimize_scalar
    a = [0.5, 3.0, 7.5, 20.0, 99.0]
    b = [1.0, 0.2, 42.0, 5.5, 0.01]
    f = lambda k, x, y: (x - a[k]) ** 2 + 0.5 * (y - b[k]) ** 4 + 0.3 * np.sin(0.05 * x * y) + abs(x - 2 * a[k])
    X, Y, V, S = host_doc["BRENT_x"], host_doc["BRENT_y"], host_doc["BRENT_val"], host_doc["BRENT_start"]
    for k in range(5):
        assert abs(V[k] - f(k, X[k], Y[k])) <= 1e-12 * max(1.0, abs(V[k]))
        if k == 3:
            assert X[k] == 10.0 and Y[k] == 10.0 and V[k] == S[k]
            continue
        assert V[k] <= S[k]
        # coordinate-wise optimality: nothing better nearby along x or along y
        for d in (1e-3, 1e-2, 0.1):
            for sx, sy in ((d, 0), (-d, 0), (0, d), (0, -d)):
                x, y = min(max(X[k] + sx, 1e-10), 100.0), min(max(Y[k] + sy, 1e-10), 100.0)
                assert f(k, x, y) >= V[k] - 1e-5, (k, sx, sy)
        best_x = minimize_scalar(lambda x: f(k, x, Y[k]), bounds=(1e-10, 100.0), method="bounded", options={"xatol": 1e-10})
        assert V[k] <= best_x.fun + 1e-5 or abs(X[k] - best_x.x) > 1e-3      # same basin -> same value
    assert host_doc["BRENT_calls"] == host_doc["BRENT_batch_evals"] + 1
    assert host_doc["BRENT_batch_evals"] < 24 * 80                             # 24 searches, each bounded by its slowest point


def test_alias_init_values(host_doc):
    assert host_doc["init_R"] == [1, 0, 1, 0]          # R = A or G


def test_tree_flattening_matches_oracle(host_doc):
    flat = rt.FlatTree(rt.parse_newick("(((A:0.01, B:0.01):0.02,C:0.03):0.01,(D:0.04,E:0.05):0.06);"))
    got = host_doc["unrooted_postorder"]
    assert len(got) == flat.n_nodes
    for i, (name, length, father) in enumerate(got):
        assert (name or None) == flat.nodes[i].name
        assert father == flat.parent[i]
        if i < flat.n_nodes - 1:
            assert abs(length - flat.brlen[i]) < 1e-15
    assert host_doc["leaves"] == flat.leaf_names


def test_site_patterns_through_the_shim(host_doc):
    seqs = {"A": "AAATGGCTGTGCACGTC", "B": "GACTGGATCTGCACGTC", "C": "CTCTGGATGTGCACGTG", "D": "AAATGGCGGTGCGCCTA"}
    _, w, idx = rp.global_patterns(seqs, ["A", "B", "C", "D"])
    assert host_doc["pattern_weights"] == list(map(int, w))
    assert host_doc["pattern_indices"] == list(map(int, idx))
    cod = {"A": "AAATGGCTGTGCACGTCTTGGAAA", "B": "AACTGGATCTGCATGTCTTGGAAC", "C": "ATCTGGACGTGCACGTGTTGGATC", "D": "CAACGGGAGTGCGCCTATCGGCAA"}
    _, w, idx = rp.global_patterns(cod, ["A", "B", "C", "D"], width=3)       # three-letter states (codons)
    assert host_doc["codon_pattern_weights"] == list(map(int, w)) and sum(w) == 8 and len(w) == 6
    assert host_doc["codon_pattern_indices"] == list(map(int, idx))


@pytest.mark.gpu
def test_reference_likelihood_tests_through_the_shim(built_lib):
    exe = compile_cpp("test_likelihood", built_lib)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    vals = {}
    derivs = {}
    nh_derivs = {}
    for line in r.stdout.splitlines():
        f = line.split()
        if len(f) == 2 and f[0].isupper() or (len(f) == 2 and "_" in f[0]):
            try:
                vals[f[0]] = float(f[1])
            except ValueError:
                pass
        if len(f) == 4 and f[0] == "LG08_G4_d":
            derivs[f[1]] = (float(f[2]), float(f[3]))
        if len(f) == 4 and f[0] == "NH_T92_G4_d":
            nh_derivs[f[1]] = (float(f[2]), float(f[3]))
    assert abs(vals["R_T92_G4"] - 85.030942031997312824) < 1e-9
    assert abs(vals["DR_T92_G4"] - 85.030942031997312824) < 1e-9
    assert abs(vals["CLOCK_T92_CONST"] - 94.3957) < 1e-4
    # protein: LG08 + Gamma4(0.7) with ambiguity characters, value and both derivatives against the oracle
    r4, p4 = rm.gamma_rates(4, 0.7)
    c = cases.case_from_alignment("((a:0.1,b:0.2):0.05,(c:0.3,d:0.02):0.07,e:0.15);",
                                  {"a": "ARNDCQEGHILKMFPSTWYVAAX", "b": "ARNDCQEGHILKMFPSTWYVLK-", "c": "ARNECQDGHLIKMFPTSWYVAKB",
                                   "d": "GRNDCQEGHILRMYPSTWFVAAZ", "e": "ARNDCQEGHVLKMFPSTWYIVAA"}, rm.lg08(), r4, p4,
                                  states=rp.PROTEIN_STATES, aliases=rp.PROTEIN_ALIASES)
    res = cases.oracle_eval(c, want_d1=True, want_d2=True)
    assert abs(vals["LG08_G4"] + res.lnl) <= 1e-9 * abs(res.lnl)
    for b in range(c.flat.n_nodes - 1):
        d1, d2 = derivs["BrLen%d" % b]
        assert abs(d1 - res.d1[b]) <= 1e-8 * max(1, abs(res.d1[b]))
        assert abs(d2 - res.d2[b]) <= 1e-8 * max(1, abs(res.d2[b]))
    # codon: YN98(kappa 2, omega 0.3), constant rate
    cod_states = [a + b + c_ for a in "ACGT" for b in "ACGT" for c_ in "ACGT"]
    flat = rt.FlatTree(rt.parse_newick("((a:0.1,b:0.2):0.05,c:0.3,d:0.02);"))
    seqs = {"a": "ATGGCTAAATTTGGGCCC", "b": "ATGGCCAAATTCGGGCCA", "c": "ATGGCTAAGTTTGGACCC", "d": "ATGTCTAAATTTGGGCCC"}
    uniq, w, idx = rp.global_patterns(seqs, flat.leaf_names, width=3)
    codes = rp.encode_columns(uniq, cod_states, width=3)
    cc = cases.Case()
    m = rm.yn98(2.0, 0.3)
    cc.flat, cc.model, cc.rates, cc.probs = flat, m, np.ones(1), np.ones(1)
    cc.table, cc.N, cc.weights = np.eye(64), len(uniq), w
    cc.codes_by_leaf = {lid: codes[k] for k, lid in enumerate(flat.leaf_ids)}
    cc.root_freqs = m.freq
    res = cases.oracle_eval(cc)
    assert abs(vals["YN98_CONST"] + res.lnl) <= 1e-9 * abs(res.lnl)
    assert vals["MASR_ERR"] <= 1e-12 and int(vals["MASR_NNODES"]) == 6
    # posterior rate of each site / best rate class (AbstractDiscreteRatesAcrossSitesTreeLikelihood.cpp:201-248) against the oracle
    rg4, pg4 = rm.gamma_rates(4, 1.0)
    cg = cases.case_from_alignment("((A:0.01, B:0.02):0.03,C:0.01,D:0.1);",
                                   {"A": "AAATGGCTGTGCACGTC", "B": "GACTGGATCTGCACGTC", "C": "CTCTGGATGTGCACGTG", "D": "AAATGGCGGTGCGCCTA"},
                                   rm.t92(3.0, 0.5), rg4, pg4)
    rg = cases.oracle_eval(cg)
    root = cg.flat.root
    S_ic = np.ldexp(np.einsum("icx,x->ic", rg.lower[root], cg.root_freqs), -rg.lexp[root])
    post = S_ic * np.asarray(pg4)[None, :]
    post /= post.sum(axis=1, keepdims=True)
    for site in range(17):
        k = cg.site_index[site]
        assert abs(vals["POSTRATE_%d" % site] - float(post[k] @ np.asarray(rg4))) <= 1e-12, site
        assert int(vals["MAXCLASS_%d" % site]) == int(np.argmax(S_ic[k])), site
    assert vals["DRAS_ERR"] <= 1e-12
    # clock class (test/test_likelihood_clock.cpp): start = the unconstrained value, optimum = the reference's 71.2657, both by
    # evaluation at the stored argmin and by a descent run through the shim on the device
    import json
    clock = json.loads((ROOT / "tests" / "golden" / "clock_optimum.json").read_text())
    assert abs(vals["CLOCK_INIT"] - 94.3957) < 5e-5 and abs(vals["CLOCK_TOTALHEIGHT"] - 0.04) < 1e-12 and int(vals["CLOCK_NPARAMS"]) == 3
    assert abs(vals["CLOCK_OPTIMUM"] - clock["oracle_minus_lnl"]) <= 1e-9 * clock["oracle_minus_lnl"]
    assert abs(vals["CLOCK_OPTIMUM"] - clock["reference_minus_lnl"]) <= 1e-4
    assert abs(vals["CLOCK_DESCENT"] - clock["reference_minus_lnl"]) <= 1e-4 and vals["CLOCK_DESCENT"] >= vals["CLOCK_OPTIMUM"] - 1e-7
    # non-homogeneous model set (test/test_likelihood_nh.cpp's construction): one T92 per branch, kappa shared, GC root frequencies
    r1, p1 = rm.gamma_rates(4, 1.0)
    seqs_nh = {"A": "ATGTTATCCCGTCGAATCATATGGAATCGTCTAGAACTCA", "B": "ATGGTATCTCGCCTAATCATGTGGCATCGTCAAAAAATCA",
               "C": "TTGGTGTGTCCCTTAATCGTGTGGTATCGTCCGGATATAG", "D": "ATGGAATCTCCCCTATTCAAGTGGTAACGTCTAGAAATAA",
               "E": "CTGGTATCTCCCATTATCATGTGCTATAGTCGAAAAACAA", "F": "ATGGTTTCTCCCCTAATAGTTCGGCAACGTCAAGACATCA"}
    cn = cases.case_from_alignment("(((A:0.1, B:0.2):0.3,C:0.1):0.2,(D:0.3,(E:0.2,F:0.05):0.1):0.1);", seqs_nh, rm.t92(3.0, 0.5),
                                   r1, p1, check_rooted=False)
    nb = cn.flat.n_nodes - 1
    assert int(vals["NH_NMODELS"]) == nb == 10 and int(vals["NH_NPARAMS"]) == 1 + 1 + nb      # GC.theta, kappa_1, ten thetas
    thetas = [0.15 + 0.07 * i for i in range(nb)]
    cn.root_freqs = np.array([.25, .25, .25, .25])
    resn = cases.oracle_eval_nh(cn, [rm.t92(3.0, th) for th in thetas], np.arange(nb + 1) % nb, want_d1=True, want_d2=True)
    assert abs(vals["NH_DR_T92_G4"] + resn.lnl) <= 1e-9 * abs(resn.lnl)
    assert abs(vals["NH_R_T92_G4"] + resn.lnl) <= 1e-9 * abs(resn.lnl)
    for b in range(nb):
        d1, d2 = nh_derivs["BrLen%d" % b]
        assert abs(d1 - resn.d1[b]) <= 1e-8 * max(1, abs(resn.d1[b])), b
        assert abs(d2 - resn.d2[b]) <= 1e-8 * max(1, abs(resn.d2[b])), b
    thetas[2] = 0.6
    cn.root_freqs = np.array([.35, .15, .15, .35])
    resn = cases.oracle_eval_nh(cn, [rm.t92(2.0, th) for th in thetas], np.arange(nb + 1) % nb)
    assert abs(vals["NH_DR_T92_G4_MOVED"] + resn.lnl) <= 1e-9 * abs(resn.lnl)
    assert vals["NH_KAPPA_7"] == 2.0
    # chromosome: one character, weighted root frequencies, unknown count at one tip
    flat = rt.FlatTree(rt.parse_newick("(((a:0.3,b:0.2):0.4,c:0.5):0.1,(d:0.3,e:0.6):0.2);"), check_rooted=False)
    m = rm.chromosome(1, 30, gain=0.7, loss=0.4, dupl=0.2, demi=rm.DEMI_EQUAL_DUPL)
    table = np.vstack([np.eye(30), np.ones((1, 30))])
    counts = {"a": 7, "b": 8, "c": 14, "d": 9, "e": None}
    ch = cases.Case()
    ch.flat, ch.model, ch.rates, ch.probs = flat, m, np.ones(1), np.ones(1)
    ch.table, ch.N, ch.weights = table, 1, np.ones(1, np.uint32)
    ch.codes_by_leaf = {lid: np.array([30 if counts[flat.nodes[lid].name] is None else counts[flat.nodes[lid].name] - 1], np.uint8)
                        for lid in flat.leaf_ids}
    ch.root_freqs = m.freq
    res = cases.oracle_eval(ch, weighted_root=True)
    assert abs(vals["CHR_WEIGHTED"] + res.lnl) <= 1e-9 * abs(res.lnl)
    # MarginalNonRevAncestralStateReconstruction on that likelihood: best state and its posterior at every node
    from oracle import ref_likelihood as rl
    res_m = cases.oracle_eval(ch, weighted_root=True, want_d1=True)
    for n in range(flat.n_nodes):
        post, _ = rl.marginal_posteriors(flat, res_m, res_m.P, n, ch.probs)
        assert int(vals["CHR_ANC_%d" % n]) == int(np.argmax(post[0])), n
        assert abs(vals["CHR_POSTMAX_%d" % n] - post[0].max()) <= 1e-9, n
    ml_states, ml_root = rl.ml_joint_reconstruction(flat, ch.codes_by_leaf, ch.table, res_m.P, res_m.root_freqs)
    for n in range(flat.n_nodes):
        assert int(vals["CHR_ML_%d" % n]) == int(ml_states[n][0]), n
    assert abs(vals["CHR_ML_BEST"] - np.log(ml_root[0, 0].max())) <= 1e-10
    assert vals["CHR_MARG_SUM_ERR"] <= 1e-10 and vals["CHR_MARG_JOINT_ERR"] <= 1e-12 and vals["CHR_MARG_FATHER_ERR"] <= 1e-10
    # batched front-end (LikelihoodPointBatch): five parameter points in one device evaluation, each against the oracle
    pts = [(0.7, 0.4, 0.2, 0.1), (1.1, 0.4, 0.2, 0.05), (0.2, 1.3, 0.6, 0.3), (2.0, 2.0, 0.01, 0.4), (0.05, 0.05, 0.9, 0.0)]
    for k, (g, l, du, de) in enumerate(pts):
        mk = rm.chromosome(1, 30, gain=g, loss=l, dupl=du, demi=de)
        ch.model, ch.root_freqs = mk, mk.freq
        rk = cases.oracle_eval(ch, weighted_root=True)
        assert abs(vals["CHR_BATCH_%d" % k] + rk.lnl) <= 1e-9 * abs(rk.lnl), k
    assert vals["CHR_BATCH_MAXREL"] <= 1e-12 and vals["CHR_BATCH_PROBE_REL"] <= 1e-12
    # mixture of sub-models: L_site = sum_k p_k L_k,site (RHomogeneousMixedTreeLikelihood.cpp:191-212)
    seqs1 = {"A": "AAATGGCTGTGCACGTC", "B": "GACTGGATCTGCACGTC", "C": "CTCTGGATGTGCACGTG", "D": "AAATGGCGGTGCGCCTA"}
    rg, pg = rm.gamma_rates(4, 1.0)
    site_l = []
    for kappa in (1.0, 3.0, 8.0):
        ck = cases.case_from_alignment("((A:0.01, B:0.02):0.03,C:0.01,D:0.1);", seqs1, rm.t92(kappa, 0.5), rg, pg)
        site_l.append(cases.oracle_eval(ck).site_lnl)
    mixed = np.log(0.2 * np.exp(site_l[0]) + 0.5 * np.exp(site_l[1]) + 0.3 * np.exp(site_l[2]))
    expect = -float(np.sum(ck.weights * mixed))
    assert abs(vals["MIXED_T92_G4"] - expect) <= 1e-9 * abs(expect)
    assert abs(vals["MIXED_DEGENERATE"] - 85.030942031997312824) < 1e-9


def oracle_pseudo_newton(c, tol=1e-6, max_correction=10, max_steps=200):
    """PseudoNewtonOptimizer::doStep (Likelihood/PseudoNewtonOptimizer.cpp:100-193, CG disabled) on the ORACLE's -lnL and its
    branch derivatives: the trajectory the shim's optimiser must follow on the device."""
    from oracle import ref_tree as rt
    nb = c.flat.n_nodes - 1

    def evaluate(bl, derivs):
        res = cases.oracle_eval(c, brlen=np.concatenate([bl, [0.0]]), want_d1=derivs, want_d2=derivs)
        return -res.lnl, (res.d1, res.d2) if derivs else None
    x = np.asarray(c.flat.brlen[:nb], float).copy()
    cur, (d1, d2) = evaluate(x, True)
    values = [cur]
    for _ in range(max_steps):
        with np.errstate(divide="ignore", invalid="ignore"):
            mv = np.where(d2 == 0, 0.0, np.where(d2 < 0, -d1 / d2, d1 / d2))
        mv = np.where(np.isnan(mv), 0.0, mv)
        new = np.clip(x - mv, rt.MIN_BRLEN, rt.MAX_BRLEN)
        mv = x - new
        val, _ = evaluate(new, False)
        count = 0
        while count < max_correction and (val > cur + tol or np.isnan(val)):
            mv = mv / 2
            new = np.clip(x - mv, rt.MIN_BRLEN, rt.MAX_BRLEN)
            val, _ = evaluate(new, False)
            count += 1
        prev = cur
        if val > cur + tol:
            val = cur
        else:
            x, cur = new, val
            _, (d1, d2) = evaluate(x, True)
        values.append(val)
        if abs(cur - prev) < tol:
            break
    return values, x


@pytest.mark.gpu
def test_pseudo_newton_branch_lengths_follow_the_oracle_trajectory(built_lib):
    """SURVEY 8f-1: the reference's Newton-Raphson branch-length optimiser on top of the device's d1 / d2 (all branches from one
    evaluation per step).  Same start, same rule => the same sequence of -lnL values as the oracle-driven run, step by step."""
    exe = compile_cpp("test_newton", built_lib)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    vals = {f[0]: float(f[1]) for f in (line.split() for line in r.stdout.splitlines()) if len(f) == 2}
    r4, p4 = rm.gamma_rates(4, 1.0)
    dna = cases.case_from_alignment("((A:0.01, B:0.02):0.03,C:0.01,D:0.1);",
                                    {"A": "AAATGGCTGTGCACGTC", "B": "GACTGGATCTGCACGTC", "C": "CTCTGGATGTGCACGTG", "D": "AAATGGCGGTGCGCCTA"},
                                    rm.t92(3.0, 0.5), r4, p4)
    r7, p7 = rm.gamma_rates(4, 0.7)
    prot = cases.case_from_alignment("((a:0.1,b:0.2):0.05,(c:0.3,d:0.02):0.07,e:0.15);",
                                     {"a": "ARNDCQEGHILKMFPSTWYVAAX", "b": "ARNDCQEGHILKMFPSTWYVLK-", "c": "ARNECQDGHLIKMFPTSWYVAKB",
                                      "d": "GRNDCQEGHILRMYPSTWFVAAZ", "e": "ARNDCQEGHVLKMFPSTWYIVAA"}, rm.lg08(), r7, p7,
                                     states=rp.PROTEIN_STATES, aliases=rp.PROTEIN_ALIASES)
    for tag, c in (("PN_T92", dna), ("PN_LG08", prot)):
        values, x = oracle_pseudo_newton(c)
        assert abs(vals[tag + "_START"] - values[0]) <= 1e-9 * values[0]
        assert int(vals[tag + "_NSTEPS"]) == len(values) - 1, tag
        for k, v in enumerate(values[1:]):
            assert abs(vals["%s_STEP_%d" % (tag, k)] - v) <= 1e-7 * abs(v), (tag, k)
        assert vals[tag + "_FINAL"] < vals[tag + "_START"] - 1.0            # it did optimise
        for b in range(len(x)):
            assert abs(vals["%s_BrLen%d" % (tag, b)] - x[b]) <= 1e-5 * max(1.0, x[b]), (tag, b)


@pytest.mark.gpu
def test_relax_and_yngp_m2_through_the_shim(built_lib):
    """test/test_relax.cpp's three equalities through the shim on the device (RNonHomogeneousMixedTreeLikelihood: every site path is a
    point of one engine, K x M model slots, one branch -> slot map per point), and every value against the oracle's mixture."""
    import test_oracle_golden as tog
    exe = compile_cpp("test_relax", built_lib)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    vals = {f[0]: float(f[1]) for f in (line.split() for line in r.stdout.splitlines()) if len(f) == 2}
    c = tog._relax_case()
    nn = c.flat.n_nodes
    m2, p2 = rm.yngp_m2(2.0, 0.1, 2.0, 0.5, 0.8)
    for k in range(3):
        assert abs(vals["M2_RATE_%d" % k] - m2[k].rate) <= 1e-10 * m2[k].rate
        assert abs(vals["M2_PROB_%d" % k] - p2[k]) <= 1e-15
    ref = tog._mixture_minus_lnl(c, [([m], np.zeros(nn, np.int64)) for m in m2], p2)
    for key in ("M2", "RELAX_PARTITION_A", "RELAX_PARTITION_B"):
        assert abs(-vals[key] - ref) <= 1e-9 * ref, key
    m2b, _ = rm.yngp_m2(2.0, 0.01, 4.0, 0.5, 0.8)
    slots = np.array([1 if n == 0 else 0 for n in range(nn)])                # model 2 (k = 2) on node 0
    ref2 = tog._mixture_minus_lnl(c, [([a, b], slots) for a, b in zip(m2, m2b)], p2)
    for key in ("RELAX_K2", "DOUBLE_M2"):
        assert abs(-vals[key] - ref2) <= 1e-9 * ref2, key
    assert abs(ref - ref2) > 1e-4


@pytest.mark.gpu
def test_dr_homogeneous_mixed_tree_likelihood_through_the_shim(built_lib):
    """DRHomogeneousMixedTreeLikelihood (SURVEY 8f-3 names R and DR): YNGP_M2 on test_relax's data.  Value = the R class's = the
    oracle's mixture; derivatives = the reference's own combination of the sub-likelihoods' RELATIVE per-site arrays
    (DRHomogeneousMixedTreeLikelihood.cpp:399-508), rebuilt from the oracle's dL / d2L arrays; a branch move, a model move."""
    import test_oracle_golden as tog
    import cases
    exe = compile_cpp("test_dr_mixed", built_lib)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    vals = {f[0]: float(f[1]) for f in (line.split() for line in r.stdout.splitlines()) if len(f) == 2}
    c = tog._relax_case()
    nn = c.flat.n_nodes

    def oracle(models, probs, brlen=None):
        res = []
        for m in models:
            c.model, c.root_freqs = m, np.asarray(m.freq)
            res.append(cases.oracle_eval(c, want_d1=True, want_d2=True, brlen=brlen))
        mixed = np.log(np.sum(np.asarray(probs)[:, None] * np.exp(np.asarray([q.site_lnl for q in res])), axis=0))
        d1, d2 = {}, {}
        for b in range(nn - 1):
            x = sum(p * q.dL[b] for p, q in zip(probs, res))
            x2 = sum(p * q.d2L[b] for p, q in zip(probs, res))
            d1[b] = -float(np.sum(c.weights * x))
            d2[b] = -float(np.sum(c.weights * (x2 - x * x)))
        return -float(np.sum(c.weights * mixed)), mixed, d1, d2

    m2, p2 = rm.yngp_m2(2.0, 0.1, 2.0, 0.5, 0.8)
    v, mixed, d1, d2 = oracle(m2, p2)
    assert abs(vals["DRM_VALUE"] - v) <= 1e-9 * v and abs(vals["RM_VALUE"] - v) <= 1e-9 * v
    assert int(vals["DRM_NBRANCH"]) == nn - 1
    for b in range(nn - 1):
        assert abs(vals["DRM_D1_%d" % b] - d1[b]) <= 1e-8 * max(1.0, abs(d1[b])), b
        assert abs(vals["DRM_D2_%d" % b] - d2[b]) <= 1e-7 * max(1.0, abs(d2[b])), b
    for i, k in enumerate(c.site_index if hasattr(c, "site_index") else range(c.N)):
        pass
    bl = c.flat.brlen.copy()
    bl[1] = 0.2
    v2, _, d1b, _ = oracle(m2, p2, brlen=bl)
    assert abs(vals["DRM_VALUE_MOVED"] - v2) <= 1e-9 * v2
    assert abs(vals["DRM_D1_MOVED_1"] - d1b[1]) <= 1e-8 * max(1.0, abs(d1b[1]))
    m3, p3 = rm.yngp_m2(2.0, 0.3, 2.0, 0.5, 0.8)
    v3, _, _, _ = oracle(m3, p3, brlen=bl)
    assert abs(vals["DRM_VALUE_OMEGA"] - v3) <= 1e-9 * v3
    assert int(vals["DRM_MODEL_DERIV_THROWS"]) == 1
