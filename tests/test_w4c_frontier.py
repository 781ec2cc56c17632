"""Folded cherries in the DNA walk (walk4c_kernel): a cherry whose father is binary is evaluated once per code pair in the
table pass and read by its father as a wide tip.  The table rows are computed with the walk's own arithmetic, so the
log-likelihoods must equal those of the unfolded program (BPPGPU_W4C_FRONTIER=0) bit for bit.  Needs a B200: -m gpu."""
import numpy as np
import pytest

import cases
from oracle import ref_models as rm

pytestmark = pytest.mark.gpu

REL = 1e-9


def gtr():
    return rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))


def _run(monkeypatch, c, frontier, pt=None):
    from bpp_phyl_b200 import capi
    monkeypatch.setenv("BPPGPU_W4C_FRONTIER", frontier)
    if pt is None:
        monkeypatch.delenv("BPPGPU_WALK4_PT", raising=False)
    else:
        monkeypatch.setenv("BPPGPU_WALK4_PT", str(pt))
    with cases.make_engine(c) as e:
        lnl, _, _ = e.eval(capi.EVAL_LNL)
        return lnl[0], e.site_lnl().copy(), e.stats()


def _check(monkeypatch, c, folded, pt=None):
    """folded: whether the case has foldable cherries (cherries with a binary father, alphabet of at most 8 codes)."""
    lnl0, site0, st0 = _run(monkeypatch, c, "0", pt)
    lnl1, site1, st1 = _run(monkeypatch, c, "1", pt)
    assert st0["path"] == st1["path"] == 1
    assert st0["w4c_frontier_nodes"] == 0
    assert (st1["w4c_frontier_nodes"] > 0) == folded, st1["w4c_frontier_nodes"]
    assert lnl1 == lnl0
    np.testing.assert_array_equal(site1, site0)
    res = cases.oracle_eval(c)
    assert abs(lnl1 - res.lnl) <= REL * abs(res.lnl), (lnl1, res.lnl)
    return st1


def _four_codes(c):
    """the bench's alphabet: the four plain states only (16 code pairs)"""
    assert all(int(v.max()) < 4 for v in c.codes_by_leaf.values())
    c.table = c.table[:4]
    return c


@pytest.mark.parametrize("ncat", [1, 4])
@pytest.mark.parametrize("pt", [1, 2, 4])
@pytest.mark.parametrize("rooted", [False, True])
def test_random_trees_four_codes(monkeypatch, ncat, pt, rooted):
    r, p = rm.gamma_rates(ncat, 0.5) if ncat > 1 else rm.constant_rate()
    c = _four_codes(cases.make_case(200, 333, gtr(), r, p, seed=90 + ncat, rooted=rooted))
    st = _check(monkeypatch, c, True, pt)
    assert st["w4c_frontier_nodes"] >= 20


@pytest.mark.parametrize("ncat", [1, 4])
def test_ambiguity_alphabet_below_the_cap(monkeypatch, ncat):
    """six codes (four states, N, a two-state ambiguity): 36 code pairs; with four classes two folded cherries under one
    father would outgrow the table chunk, so such a father keeps one of them unfolded"""
    r, p = rm.gamma_rates(ncat, 0.5) if ncat > 1 else rm.constant_rate()
    for ntaxa, nsites, seed in ((64, 700, 91), (9, 130, 92)):
        c = cases.make_case(ntaxa, nsites, gtr(), r, p, seed=seed, ambiguity=0.05)
        assert c.table.shape[0] == 6
        _check(monkeypatch, c, True)


def test_ambiguity_alphabet_above_the_cap(monkeypatch):
    """the IUPAC alphabet (21 codes, 441 pairs) folds nothing"""
    r, p = rm.gamma_rates(4, 0.5)
    c = cases.case_from_alignment("((A:0.1,B:0.2):0.05,((C:0.3,D:0.05):0.02,E:0.01):0.1);",
                                  {"A": "ACGTNACG", "B": "ACGTRACC", "C": "AGGT-TCG", "D": "ACCTYACG", "E": "TCGTAACG"},
                                  gtr(), r, p, check_rooted=False)
    assert c.table.shape[0] > 8
    _check(monkeypatch, c, False)


def test_multifurcations(monkeypatch):
    """cherries under a binary father fold; cherries under the three-son root or a four-son node do not; a three-tip
    node is no cherry"""
    r, p = rm.gamma_rates(4, 0.5)
    nwk = "(((A:0.1,B:0.2):0.05,(C:0.1,D:0.3):0.1):0.02,((E:0.1,F:0.2):0.1,(G:0.1,H:0.1):0.2,I:0.1,J:0.2):0.1,(K:0.1,L:0.1,M:0.2):0.3);"
    rng = np.random.default_rng(93)
    seqs = {n: "".join("ACGT"[k] for k in rng.integers(4, size=157)) for n in "ABCDEFGHIJKLM"}
    c = _four_codes(cases.case_from_alignment(nwk, seqs, gtr(), r, p))
    st = _check(monkeypatch, c, True)
    assert st["w4c_frontier_nodes"] == 2


@pytest.mark.parametrize("pt", [1, 4])
def test_tree_of_cherries(monkeypatch, pt):
    """rooted trees made of cherries only: the root of the first reads two wide tips"""
    r, p = rm.gamma_rates(4, 0.5)
    rng = np.random.default_rng(94)
    for nwk, nfold in (("((A:0.1,B:0.2):0.05,(C:0.1,D:0.3):0.1);", 2),
                       ("(((A:0.1,B:0.2):0.05,(C:0.1,D:0.3):0.1):0.1,((E:0.2,F:0.1):0.1,(G:0.05,H:0.4):0.2):0.1);", 4)):
        names = sorted(set(ch for ch in nwk if ch.isalpha()))
        seqs = {n: "".join("ACGT"[k] for k in rng.integers(4, size=301)) for n in names}
        c = _four_codes(cases.case_from_alignment(nwk, seqs, gtr(), r, p, check_rooted=False))
        st = _check(monkeypatch, c, True, pt)
        assert st["w4c_frontier_nodes"] == nfold


def test_cherry_rows_rescaled(monkeypatch):
    """a fifth code whose tip vector is 1e-150 everywhere: a cherry row with that code is ~1e-150 (~1e-300 with two) and is
    rescaled inside the table pass; the exponent travels with the row"""
    r, p = rm.gamma_rates(4, 0.5)
    c = _four_codes(cases.make_case(64, 300, gtr(), r, p, seed=95))
    c.table = np.vstack([c.table, np.full((1, 4), 1e-150)])
    rng = np.random.default_rng(95)
    for lid in c.codes_by_leaf:
        v = c.codes_by_leaf[lid]
        c.codes_by_leaf[lid] = np.where(rng.random(v.shape) < 0.2, 4, v).astype(v.dtype)
    _check(monkeypatch, c, True)


@pytest.mark.parametrize("ncat", [1, 4])
def test_underflowing_sites_large_tree(monkeypatch, ncat):
    """700 taxa, random tips, long branches: site likelihoods far below 1e-308, rescaled many times along the walk"""
    r, p = rm.gamma_rates(ncat, 0.5) if ncat > 1 else rm.constant_rate()
    c = _four_codes(cases.make_case(700, 130, gtr(), r, p, seed=96, random_tips=True, mean_brlen=0.5))
    res = cases.oracle_eval(c)
    assert res.site_lnl.max() < np.log(1e-308)
    _check(monkeypatch, c, True)
