"""Folded three-tip subtrees in the DNA walk (walk4c_kernel): a binary node under a binary father whose sons are a folded
cherry and a tip is evaluated once per triple of tip codes in the table pass (ncodes^3 rows, at most 64) and read by its
father as a wide tip.  The rows are computed with the walk's own arithmetic, so lnL and the site log-likelihoods must equal
those of the unfolded program (BPPGPU_W4C_FRONTIER=0) bit for bit.  One rate class per CTA: the class terms of a pattern
meet in the root reduction of the block's last CTA.  Needs a B200: -m gpu."""
import numpy as np
import pytest

import cases
from oracle import ref_models as rm

pytestmark = pytest.mark.gpu

REL = 1e-9


def gtr():
    return rm.gtr(1.2, 0.8, 0.6, 1.5, 0.9, (.3, .2, .25, .25))


def rates(ncat):
    return rm.gamma_rates(ncat, 0.5) if ncat > 1 else rm.constant_rate()


def _four_codes(c):
    """the bench's alphabet: the four plain states only (64 code triples)"""
    assert all(int(v.max()) < 4 for v in c.codes_by_leaf.values())
    c.table = c.table[:4]
    return c


def expected_folds(c, ncodes):
    """(folded cherries, folded three-tip subtrees) by the rule of the planner, from the tree alone"""
    off, ch = c.flat.csr()
    off, ch = np.asarray(off), np.asarray(ch)
    nn = len(off) - 1
    sons = [list(ch[off[n]:off[n + 1]]) for n in range(nn)]
    tip = [len(s) == 0 for s in sons]
    cherry, three = [False] * nn, [False] * nn
    if ncodes ** 2 > 64:
        return 0, 0
    for f in range(nn):
        if len(sons[f]) == 2:
            for n in sons[f]:
                cherry[n] = len(sons[n]) == 2 and tip[sons[n][0]] and tip[sons[n][1]]
    if ncodes ** 3 <= 64:
        for f in range(nn):
            if len(sons[f]) == 2:
                for n in sons[f]:
                    s = sons[n]
                    three[n] = len(s) == 2 and ((cherry[s[0]] and tip[s[1]]) or (tip[s[0]] and cherry[s[1]]))
    return sum(cherry), sum(three)


def _run(monkeypatch, c, frontier, pt=None, env=None):
    from bpp_phyl_b200 import capi
    monkeypatch.setenv("BPPGPU_W4C_FRONTIER", frontier)
    if pt is None:
        monkeypatch.delenv("BPPGPU_WALK4_PT", raising=False)
    else:
        monkeypatch.setenv("BPPGPU_WALK4_PT", str(pt))
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    with cases.make_engine(c) as e:
        lnl, _, _ = e.eval(capi.EVAL_LNL)
        return lnl[0], e.site_lnl().copy(), e.stats()


def _check(monkeypatch, c, pt=None, env=None):
    """default folding against the unfolded program (bit for bit) and the oracle (1e-9); the fold counters against the tree"""
    lnl0, site0, st0 = _run(monkeypatch, c, "0", pt, env)
    lnl1, site1, st1 = _run(monkeypatch, c, "1", pt, env)
    assert st0["path"] == st1["path"] == 1
    assert st0["w4c_frontier_nodes"] == st0["w4c_three_tip_nodes"] == 0
    assert (st1["w4c_frontier_nodes"], st1["w4c_three_tip_nodes"]) == expected_folds(c, c.table.shape[0])
    assert lnl1 == lnl0
    np.testing.assert_array_equal(site1, site0)
    res = cases.oracle_eval(c)
    assert abs(lnl1 - res.lnl) <= REL * abs(res.lnl), (lnl1, res.lnl)
    np.testing.assert_allclose(site1, res.site_lnl, rtol=REL, atol=0)
    return st1


def _alignment(nwk, nsites, seed, ncat=4):
    r, p = rates(ncat)
    rng = np.random.default_rng(seed)
    names = sorted(set(ch for ch in nwk if ch.isalpha()))
    seqs = {n: "".join("ACGT"[k] for k in rng.integers(4, size=nsites)) for n in names}
    return _four_codes(cases.case_from_alignment(nwk, seqs, gtr(), r, p, check_rooted=False))


@pytest.mark.parametrize("ncat", [1, 2, 4, 8])
@pytest.mark.parametrize("pt", [1, 2, 4])
@pytest.mark.parametrize("rooted", [False, True])
def test_random_trees(monkeypatch, ncat, pt, rooted):
    r, p = rates(ncat)
    c = _four_codes(cases.make_case(200, 777, gtr(), r, p, seed=110 + ncat, rooted=rooted))
    st = _check(monkeypatch, c, pt)
    assert st["w4c_three_tip_nodes"] >= 10


def test_caterpillar(monkeypatch):
    """a caterpillar has exactly one three-tip subtree: ((A,B),C)"""
    c = _alignment("((((((A:0.1,B:0.2):0.05,C:0.1):0.1,D:0.2):0.1,E:0.05):0.2,F:0.1):0.1,G:0.3);", 401, 111)
    st = _check(monkeypatch, c)
    assert (st["w4c_frontier_nodes"], st["w4c_three_tip_nodes"]) == (1, 1)


@pytest.mark.parametrize("pt", [1, 4])
def test_father_of_two_three_tip_subtrees(monkeypatch, pt):
    """the root reads two three-tip tables (one with its tip first, one with its tip second); in the second tree a
    binary father reads one three-tip table next to a cherry table"""
    for nwk, folds in (("((C:0.3,(A:0.1,B:0.2):0.05):0.1,((D:0.1,E:0.3):0.1,F:0.2):0.2);", (2, 2)),
                       ("(((C:0.3,(A:0.1,B:0.2):0.05):0.1,(G:0.1,H:0.1):0.3):0.1,((D:0.1,E:0.3):0.1,F:0.2):0.2);", (3, 2))):
        c = _alignment(nwk, 513, 112)
        st = _check(monkeypatch, c, pt)
        assert (st["w4c_frontier_nodes"], st["w4c_three_tip_nodes"]) == folds


@pytest.mark.parametrize("ncat", [1, 4])
def test_five_codes_fold_cherries_only(monkeypatch, ncat):
    """four states and N: 25 code pairs fold, 125 code triples do not fit a one-byte row code"""
    r, p = rates(ncat)
    c = _four_codes(cases.make_case(150, 600, gtr(), r, p, seed=113, rooted=True))
    c.table = np.vstack([np.eye(4), np.ones((1, 4))])
    rng = np.random.default_rng(113)
    for lid in c.codes_by_leaf:
        v = c.codes_by_leaf[lid]
        c.codes_by_leaf[lid] = np.where(rng.random(v.shape) < 0.1, 4, v).astype(v.dtype)
    st = _check(monkeypatch, c)
    assert st["w4c_frontier_nodes"] > 0 and st["w4c_three_tip_nodes"] == 0


def test_three_tip_rows_rescaled(monkeypatch):
    """code 3's tip vector scaled to 1e-150: a three-tip row with that code three times is ~1e-450, rescaled inside the
    table pass both in the cherry row and after the product with the tip term; the exponents travel with the row"""
    r, p = rates(4)
    c = _four_codes(cases.make_case(64, 500, gtr(), r, p, seed=114, random_tips=True))
    c.table = c.table.copy()
    c.table[3] *= 1e-150
    st = _check(monkeypatch, c)
    assert st["w4c_three_tip_nodes"] > 0


@pytest.mark.parametrize("ncat", [1, 4])
def test_underflowing_sites_large_tree(monkeypatch, ncat):
    """700 taxa, random tips, long branches: site likelihoods far below 1e-308, rescaled many times along the walk"""
    r, p = rates(ncat)
    c = _four_codes(cases.make_case(700, 130, gtr(), r, p, seed=115, random_tips=True, mean_brlen=0.5))
    assert cases.oracle_eval(c).site_lnl.max() < np.log(1e-308)
    _check(monkeypatch, c)


@pytest.mark.parametrize("nsites", [1, 37, 511, 1500])
def test_ragged_pattern_counts(monkeypatch, nsites):
    """pattern counts below one block of PPC = NW 32 PT patterns and not a multiple of it"""
    r, p = rates(4)
    c = _four_codes(cases.make_case(90, nsites, gtr(), r, p, seed=116, random_tips=True))
    for pt in (1, 4):
        _check(monkeypatch, c, pt)


def test_two_segments(monkeypatch):
    """a split launch plan: full waves at PT = 4, the remainder at PT = 1 -- the second launch's partials and blocks start
    where the first one's end"""
    r, p = rates(4)
    c = _four_codes(cases.make_case(24, 60000, gtr(), r, p, seed=117, random_tips=True))
    assert c.N > 50000
    _check(monkeypatch, c, env={"BPPGPU_WALK4_PLAN": "split:1:0"})
