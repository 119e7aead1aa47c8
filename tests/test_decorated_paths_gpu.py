"""Decorated p-values of whole path lists on the device (gcre_exec_decorated_paths): splits formed from the resident gene rows,
non-stratified and stratified exact modes, checked against
  * gcre_exec_decorated_exact on the same splits packed by the host (non-stratified: bit for bit),
  * exact rational arithmetic (Fraction / math.comb convolution over the strata) - shares nothing with the kernels,
  * the host implementation (decorated.decorated_pvalues_for_path) on the top-K lists of a GPU replay, and the join's own scores.
Tolerances: 1e-12 relative against rationals, 1e-11 against the host (gammaln-based); counts and the f64 score bit-exact."""
from fractions import Fraction
from math import comb

import numpy as np
import pytest

from geneticscre_b200 import _lib, decorated, schedule, synth

pytestmark = pytest.mark.gpu

LEVELS = ("2", "3", "4", "5")


def make_exec(engine, method, nc, nt, vt, iters=1):
    ex = engine.JoinExec("method1" if method == 1 else "method2", nc, nt, iters)
    ex.setValueTable(vt)
    return ex


def gene_set(ex, rows):
    ps = ex.createPathSet(rows.shape[0])
    ps.load_bits(np.ascontiguousarray(synth.pack_bits(rows)))
    return ps


def host_splits(rows, genes, signs, L, method):
    """(pos1, neg1, pos2, neg2) of a path's splits in the order of decorated_pvalues_for_path."""
    r = rows[genes[:L]]
    s = np.asarray(signs[:L])
    pos, neg = r.copy(), np.zeros_like(r)
    if method == 2:
        neg[s == -1] = r[s == -1]
        pos[s == -1] = False
    out = [(pos[:j].any(0), neg[:j].any(0), pos[j], neg[j]) for j in range(1, L)]
    out += [(pos[j:].any(0), neg[j:].any(0), pos[j - 1], neg[j - 1]) for j in range(L - 1, 0, -1)]
    return out


def random_paths(rng, n_genes, count, lengths=(1, 2, 3, 4, 5)):
    L = rng.choice(lengths, size=count).astype(np.int32)
    genes = rng.integers(0, n_genes, size=(count, 5)).astype(np.int32)
    signs = np.where(rng.random((count, 5)) < 0.5, 1, -1).astype(np.int32)
    signs[:, 0] = 1
    return genes, signs, L


def hyp(good, bad, k):
    tot = comb(good + bad, k)
    return {x: Fraction(comb(good, x) * comb(bad, k - x), tot) for x in range(max(0, k - bad), min(k, good) + 1)}


def exact_stratified(pos1, neg1, pos2, neg2, nc, nt, method, vt, strata):
    """The stratified exact limit in rationals: per stratum the positive draw, then the negative draw from what it left."""
    n = nc + nt
    is_case = np.arange(n) < nc
    p2, n2 = pos2 & ~pos1, neg2 & ~neg1
    cp1, tp1 = int((pos1 & is_case).sum()), int((pos1 & ~is_case).sum())
    cn1, tn1 = int((neg1 & ~is_case).sum()), int((neg1 & is_case).sum())
    free = ~(pos1 | neg1)
    J = {(0, 0): Fraction(1)}
    TP = TN = 0
    for g in dict.fromkeys(strata.tolist()):
        m = strata == g
        c, d = int((free & m & is_case).sum()), int((free & m & ~is_case).sum())
        kp, kn = int((p2 & free & m).sum()), int((n2 & free & m).sum())
        TP += kp
        TN += kn
        gj = {(x, y): px * py for x, px in hyp(c, d, kp).items() for y, py in hyp(d - (kp - x), c - x, kn).items()}
        out = {}
        for (a, b), pa in J.items():
            for (x, y), pg in gj.items():
                out[(a + x, b + y)] = out.get((a + x, b + y), 0) + pa * pg
        J = out

    def sc(a, tp, b, tn):
        if method == 1:
            return vt[cp1 + a + cn1 + b, tp1 + (tp - a) + tn1 + (tn - b)]
        return vt[cp1 + a, tp1 + (tp - a)] + vt[cn1 + b, tn1 + (tn - b)]

    score = sc(int((p2 & is_case).sum()), int(p2.sum()), int((n2 & ~is_case).sum()), int(n2.sum()))
    return float(sum(v for (a, b), v in J.items() if sc(a, TP, b, TN) >= score)), float(score)


def assert_same(dev, host, rel):
    assert len(dev) == len(host)
    for d, h in zip(dev, host):
        assert (d["direction"], d["subpath1"], d["subpath2"]) == (h["direction"], h["subpath1"], h["subpath2"])
        assert (d["cases1"], d["controls1"], d["cases2"], d["controls2"]) == (h["cases1"], h["controls1"], h["cases2"], h["controls2"])
        assert d["score"] == h["score"]
        assert abs(d["decorated_pvalue"] - h["decorated_pvalue"]) <= rel * max(h["decorated_pvalue"], 1e-300), (d, h)


def bits_of(res):
    return [(r["decorated_pvalue"], r["score"], r["cases1"], r["controls1"], r["cases2"], r["controls2"]) for p in res for r in p]


@pytest.mark.parametrize("method", [1, 2])
def test_non_stratified_equals_the_packed_split_call_bit_for_bit(engine, method):
    nc, nt = 700, 650
    n = nc + nt
    rng = np.random.default_rng(3)
    rows = rng.random((30, n)) < rng.uniform(0.005, 0.08, size=(30, 1))
    vt = synth.make_value_table(nc, nt) if method == 2 else synth.make_test_table(n, n, 3)
    ex = make_exec(engine, method, nc, nt, vt)
    gs = gene_set(ex, rows)
    genes, signs, L = random_paths(rng, 30, 60)
    genes[0, :3], signs[0, :3], L[0] = [4, 9, 4], [1, 1, -1], 3  # a cyclic path: one gene twice, with opposite signs
    dev = decorated.decorated_pvalues_device(ex, gs, genes, signs, L)
    splits = [sp for i in range(len(L)) for sp in host_splits(rows, genes[i], signs[i], L[i], method)]
    ref = decorated.decorated_exact_device(ex, splits)
    flat = [r for p in dev for r in p]
    assert len(flat) == len(ref) == sum(2 * (int(x) - 1) for x in L)
    for d, r in zip(flat, ref):
        assert (d["decorated_pvalue"], d["score"], d["cases1"], d["controls1"], d["cases2"], d["controls2"]) == \
            (r.decorated_pvalue, r.score, r.cases1, r.controls1, r.cases2, r.controls2)
    assert all(len(p) == 0 for p, x in zip(dev, L) if x == 1)


@pytest.mark.parametrize("method", [1, 2])
@pytest.mark.parametrize("nc,nt,n_strata,n_paths", [(37, 44, 3, 6), (37, 44, 7, 6), (1500, 1700, 16, 1)])
def test_stratified_matches_exact_rational_arithmetic(engine, method, nc, nt, n_strata, n_paths):
    n = nc + nt
    rng = np.random.default_rng(17 + n_strata)
    dens = 0.15 if n < 100 else 0.02
    rows = rng.random((8, n)) < dens
    vt = synth.make_value_table(nc, nt) if method == 2 else synth.make_test_table(n, n, 3)
    strata = rng.integers(0, n_strata, n)
    ex = make_exec(engine, method, nc, nt, vt)
    ex.setPermutationStrata(strata)
    gs = gene_set(ex, rows)
    genes, signs, L = random_paths(rng, 8, n_paths, lengths=(3,) if n > 100 else (2, 3, 4, 5))
    if n > 100:
        genes[0, :3], signs[0, :3] = [0, 1, 2], [1, -1, -1]
    dev = decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=True)
    checked = 0
    for i in range(n_paths):
        sps = host_splits(rows, genes[i], signs[i], L[i], method)
        if n > 100:
            sps, got = sps[-2:], dev[i][-2:]  # the two backward splits: a Fraction evaluation at this size takes seconds
        else:
            got = dev[i]
        for sp, d in zip(sps, got):
            want_p, want_s = exact_stratified(*sp, nc, nt, method, vt, strata)
            assert d["score"] == want_s
            assert abs(d["decorated_pvalue"] - want_p) <= 1e-12 * max(want_p, 1e-300), (d, want_p)
            checked += 1
    assert checked >= 2


@pytest.fixture(scope="module")
def replay(engine):
    """GPU replay of levels 2-5 on a 3,200-patient workload: per method the exec, its gene rows and every level's top-K."""
    w = synth.make_workload(1500, 1700, 120, 500, 16, seed=31, max_path_length=5, real_table=True, max_freq=0.08, zero_frac=0.2)
    out = {}
    for method in (1, 2):
        ex = engine.JoinExec("method1" if method == 1 else "method2", w.n_cases, w.n_ctrls, w.n_perms)
        ex.top_k = 12
        ex.setValueTable(w.value_table)
        ex.setPermutedMasks(w.perm_masks)
        res, _ = schedule.replay_levels(ex, engine.UidRelSet, w, 5)
        gs = ex.createPathSet(w.gene_bits.shape[0])
        gs.load_bits(w.gene_bits)
        out[method] = (ex, gs, {lv: [s for s in res[lv].scores if s.src >= 0] for lv in LEVELS})
    return w, out


@pytest.mark.parametrize("method", [1, 2])
@pytest.mark.parametrize("stratified", [False, True])
def test_top_k_lists_match_the_host(replay, method, stratified):
    w, per = replay
    ex, gs, scores = per[method]
    n = w.n_patients
    rows = synth.unpack_bits(w.gene_bits, n).astype(bool)
    strata = np.random.default_rng(5).integers(0, 16, n) if stratified else None
    ex.setPermutationStrata(strata)
    try:
        for lv in LEVELS:
            sc = scores[lv]
            genes, signs, L = synth.path_genes(w.net, lv, [s.src for s in sc], [s.trg for s in sc])
            if lv == "3":  # a hand-made cyclic path: gene a, then b, then a again with the opposite sign
                genes = np.vstack([genes, [[5, 7, 5, 0, 0]]]).astype(np.int32)
                signs = np.vstack([signs, [[1, 1, -1, 0, 0]]]).astype(np.int32)
                L = np.append(L, 3).astype(np.int32)
            dev = decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=stratified)
            for i in range(len(L)):
                host = decorated.decorated_pvalues_for_path(rows[genes[i, :L[i]]], signs[i, :L[i]], w.n_cases, w.n_ctrls, method,
                                                            w.value_table, strata=strata)
                assert_same(dev[i], host, 1e-11)
    finally:
        ex.setPermutationStrata(None)


@pytest.mark.parametrize("method", [1, 2])
def test_whole_path_split_reproduces_the_join(replay, method):
    """The last forward split of every top-K path scores exactly what the join scored, with the join's cases / controls."""
    w, per = replay
    ex, gs, scores = per[method]
    for stratified in (False, True):
        for lv in LEVELS:
            sc = scores[lv]
            assert sc
            genes, signs, L = synth.path_genes(w.net, lv, [s.src for s in sc], [s.trg for s in sc])
            dev = decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=stratified)
            for s, d, x in zip(sc, dev, L):
                last = d[x - 2]
                assert last["direction"] == "Forward" and last["subpath2"] == x - 1
                assert last["score"] == s.score
                assert (last["cases1"] + last["cases2"], last["controls1"] + last["controls2"]) == (s.cases, s.ctrls)


def test_strata_labels_only_matter_as_a_partition(engine):
    nc, nt = 800, 900
    n = nc + nt
    rng = np.random.default_rng(8)
    rows = rng.random((12, n)) < 0.04
    vt = synth.make_value_table(nc, nt)
    ex = make_exec(engine, 2, nc, nt, vt)
    gs = gene_set(ex, rows)
    genes, signs, L = random_paths(rng, 12, 20, lengths=(2, 3, 4, 5))
    strata = rng.integers(0, 9, n)
    ex.setPermutationStrata(strata)
    a = bits_of(decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=True))
    ex.setPermutationStrata(strata * 37 - 1000)  # other labels, same partition and order of first appearance
    b = bits_of(decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=True))
    assert a == b
    # one stratum: the setting of no strata, and the host with every patient labelled 0
    ex.setPermutationStrata(np.full(n, 4))
    one = decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=True)
    ex.setPermutationStrata(None)
    assert bits_of(one) == bits_of(decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=True))
    for i in range(len(L)):
        host = decorated.decorated_pvalues_for_path(rows[genes[i, :L[i]]], signs[i, :L[i]], nc, nt, 2, vt, strata=np.zeros(n))
        assert_same(one[i], host, 1e-11)


def test_repeated_calls_give_identical_bits(engine):
    nc, nt = 900, 1000
    n = nc + nt
    rng = np.random.default_rng(9)
    rows = rng.random((15, n)) < 0.05
    ex = make_exec(engine, 2, nc, nt, synth.make_value_table(nc, nt))
    gs = gene_set(ex, rows)
    genes, signs, L = random_paths(rng, 15, 40)
    ex.setPermutationStrata(rng.integers(0, 12, n))
    for stratified in (False, True):
        a = bits_of(decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=stratified))
        b = bits_of(decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=stratified))
        assert a == b


@pytest.mark.parametrize("stratified", [False, True])
def test_chunked_list_equals_paths_one_at_a_time(engine, monkeypatch, stratified):
    nc, nt = 600, 640
    n = nc + nt
    rng = np.random.default_rng(10)
    rows = rng.random((10, n)) < 0.06
    ex = make_exec(engine, 2, nc, nt, synth.make_value_table(nc, nt))
    gs = gene_set(ex, rows)
    genes, signs, L = random_paths(rng, 10, 25, lengths=(2, 3, 4, 5))
    ex.setPermutationStrata(rng.integers(0, 6, n))
    one = [decorated.decorated_pvalues_device(ex, gs, genes[i:i + 1], signs[i:i + 1], L[i:i + 1], stratified=stratified)[0] for i in range(len(L))]
    # a budget of a few splits' scratch: the list runs as many chunks (and a split larger than the budget alone)
    monkeypatch.setenv("GCRE_TEST_DECORATED_SCRATCH", str(60_000 if not stratified else 3_000))
    many = decorated.decorated_pvalues_device(ex, gs, genes, signs, L, stratified=stratified)
    assert bits_of(many) == bits_of(one)


def test_errors(engine):
    nc, nt = 40, 50
    n = nc + nt
    rows = np.random.default_rng(1).random((6, n)) < 0.2
    ex = engine.JoinExec("method2", nc, nt, 1)
    gs = gene_set(ex, rows)
    g = np.array([[0, 1, 2, 0, 0]], np.int32)
    s = np.array([[1, -1, 1, 0, 0]], np.int32)
    L = np.array([3], np.int32)
    with pytest.raises(_lib.GcreAssertion):  # no value table
        decorated.decorated_pvalues_device(ex, gs, g, s, L)
    ex.setValueTable(synth.make_value_table(nc, nt))
    assert decorated.decorated_pvalues_device(ex, gs, g[:0], s[:0], L[:0]) == []
    other = engine.JoinExec("method2", nc, nt, 1)
    other.setValueTable(synth.make_value_table(nc, nt))
    with pytest.raises(_lib.GcreError) as e:  # the gene rows of another exec
        decorated.decorated_pvalues_device(other, gs, g, s, L)
    assert e.value.status == _lib.GCRE_ERR_ARG
    with pytest.raises(_lib.GcreError) as e:  # a method-2 sign that is not +-1
        decorated.decorated_pvalues_device(ex, gs, g, np.array([[1, 0, 1, 0, 0]], np.int32), L)
    assert e.value.status == _lib.GCRE_ERR_ARG
    with pytest.raises(_lib.GcreOutOfRange):  # a gene index outside the set
        decorated.decorated_pvalues_device(ex, gs, np.array([[0, 6, 2, 0, 0]], np.int32), s, L)
    with pytest.raises(_lib.GcreOutOfRange):
        decorated.decorated_pvalues_device(ex, gs, np.array([[0, -1, 2, 0, 0]], np.int32), s, L)
    for bad_len in (0, 6):  # a length outside 1..5
        with pytest.raises(_lib.GcreOutOfRange):
            decorated.decorated_pvalues_device(ex, gs, g, s, np.array([bad_len], np.int32))
    # method 1 ignores the signs
    ex1 = make_exec(engine, 1, nc, nt, synth.make_test_table(n, n, 3))
    gs1 = gene_set(ex1, rows)
    a = decorated.decorated_pvalues_device(ex1, gs1, g, np.array([[1, 0, 7, 0, 0]], np.int32), L)
    assert bits_of([a[0]]) == bits_of(decorated.decorated_pvalues_device(ex1, gs1, g, s, L))


def test_a_stratum_exactly_filled_by_the_added_gene(engine):
    """The boundary of R's sample() check: the added gene's carriers are every free patient of a stratum.  A path's added gene
    sits in one part only and only its free carriers are redrawn, so a path never asks for more than a stratum holds: neither
    the device nor the host refuses, and they agree.  (The host's ValueError needs positive and negative carriers added at once,
    which no path split has.)"""
    nc, nt = 30, 30
    n = nc + nt
    strata = np.repeat([0, 1, 2], 20)
    rows = np.zeros((3, n), bool)
    rows[0, 20:30] = True                   # gene 0 covers half of stratum 1
    rows[1, 30:40] = True                   # gene 1: the other half, its free patients
    rows[2, ::7] = True
    ex = make_exec(engine, 2, nc, nt, synth.make_value_table(nc, nt))
    ex.setPermutationStrata(strata)
    gs = gene_set(ex, rows)
    for sg in ([1, 1, 1], [1, -1, 1], [1, -1, -1]):
        g, s, L = np.array([[0, 1, 2, 0, 0]], np.int32), np.array([sg + [0, 0]], np.int32), np.array([3], np.int32)
        dev = decorated.decorated_pvalues_device(ex, gs, g, s, L, stratified=True)
        host = decorated.decorated_pvalues_for_path(rows, sg, nc, nt, 2, synth.make_value_table(nc, nt), strata=strata)
        assert_same(dev[0], host, 1e-11)
