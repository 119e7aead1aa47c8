"""Grouping of equal upstream rows in score-only sparse joins (gcre_capi.cu: group_upstream_rows): one representative of rows with
equal bits and index entries is scored and its candidates are appended for the others.  Bit-exact against the CPU oracle and
against the same join without grouping, on cohorts with many empty genes (so many paths3 rows repeat each other).
GCRE_TEST_DEDUP=1 groups joins of any size; GCRE_TEST_DEDUP_COLLIDE=1 leaves the fingerprints out of the grouping keys, so only the
word-for-word compare keeps unequal rows apart."""
import numpy as np
import pytest

import helpers
from geneticscre_b200 import _lib, synth

pytestmark = pytest.mark.gpu


def sparse_exec(engine):
    class Exec(engine.JoinExec):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.kernel = _lib.KERNEL_SPARSE

    return Exec


def _workload(nc, nt, g, e, perms, seed):
    return synth.make_workload(nc, nt, g, e, perms, seed=seed, max_path_length=4, real_table=True, max_freq=0.08, zero_frac=0.7)


SHAPES = [
    # n_cases, n_ctrls, genes, edges, perms, top_k
    (64, 64, 80, 400, 1000, 5),
    (257, 300, 200, 900, 1000, 70),   # top_k > 64: prefix launch and host threshold, no self-tightening slots
    (100, 93, 150, 700, 100, 10),     # <= 512 permutations: the split-carrier kernels
]


@pytest.mark.parametrize("collide", [False, True])
@pytest.mark.parametrize("small_plan", [False, True])
@pytest.mark.parametrize("tail", ["0", "1"])
@pytest.mark.parametrize("method", ["method1", "method2"])
@pytest.mark.parametrize("shape", SHAPES)
def test_grouped_level4(engine, oracles, shape, method, tail, small_plan, collide, monkeypatch):
    nc, nt, g, e, perms, top_k = shape
    w = _workload(nc, nt, g, e, perms, seed=4100 + nc + perms)
    monkeypatch.setenv("GCRE_TEST_TAIL", tail)
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", "0")
    if small_plan:
        monkeypatch.setenv("GCRE_TEST_SMALL_PLAN", "1")
    want, _, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 4, top_k)
    monkeypatch.setenv("GCRE_TEST_DEDUP", "0")
    plain, _, _ = helpers.run_schedule(sparse_exec(engine), engine.UidRelSet, w, method, 4, top_k)
    monkeypatch.setenv("GCRE_TEST_DEDUP", "1")
    if collide:
        monkeypatch.setenv("GCRE_TEST_DEDUP_COLLIDE", "1")
    got, _, _ = helpers.run_schedule(sparse_exec(engine), engine.UidRelSet, w, method, 4, top_k)
    for lvl in want:
        what = f"{method} {shape} tail={tail} small={small_plan} collide={collide} L{lvl}"
        helpers.assert_same_results(got[lvl], want[lvl], what=what)
        helpers.assert_same_results(got[lvl], plain[lvl], what=what)
        assert plain[lvl].info["dedup_rows"] == 0
    assert got["4"].info["dedup_rows"] > 0, "the workload was built to repeat rows"


def _level4_direct(engine, w, method, top_k, mutate=None, uid_range=None):
    """levels 1a, 2, 3 on the engine, then `mutate(ex, p3)` and level 4; returns the level-4 result and the rows it read"""
    ex = sparse_exec(engine)(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    lv, didx = w.net.levels, w.net.data_idx
    u = {k: engine.UidRelSet(lv[k].path_length, lv[k].src, lv[k].trg, lv[k].count, lv[k].location, lv[k].signs) for k in ("1a", "2", "3", "4")}
    d1 = ex.createPathSet(w.net.n_genes)
    d1.load_bits(w.gene_bits)
    p1 = ex.createPathSet(lv["1a"].n_pairs)
    ex.join(u["1a"], ex.createPathSet(lv["1a"].n_uids), d1.select(didx["1a"]), p1)
    p2 = ex.createPathSet(lv["2"].n_pairs)
    ex.join(u["2"], p1, d1.select(didx["2"]), p2)
    p3 = ex.createPathSet(lv["3"].n_pairs)
    ex.join(u["3"], p2, d1.select(didx["3"]), p3)
    if mutate is not None:
        mutate(ex, p3)
    r = ex.join(u["4"], p3, p2, ex.createPathSet(0), uid_range=uid_range)
    return r, p3.to_numpy(), p2.to_numpy()


@pytest.mark.parametrize("method", ["method1", "method2"])
def test_row_rewritten_after_keep_join(engine, method, monkeypatch):
    """a paths3 row set after the level-3 join leaves the set without fingerprints: level 4 is not grouped (a stale fingerprint
    would group the rewritten row with its old twin and give it the twin's scores), and equals the join without grouping"""
    w = _workload(64, 64, 80, 400, 1000, seed=4300)

    def rewrite(ex, p3):
        rows = p3.to_numpy()
        _, first, counts = np.unique(rows, axis=0, return_index=True, return_counts=True)
        k = int(np.nonzero(counts > 1)[0][0])
        twin = [i for i in range(rows.shape[0]) if i != first[k] and np.array_equal(rows[i], rows[first[k]])][0]
        new = rows[twin].copy()
        new[0] ^= np.uint64(1)
        p3.set(twin, new)

    monkeypatch.setenv("GCRE_TEST_DEDUP", "1")
    got, _, _ = _level4_direct(engine, w, method, 5, mutate=rewrite)
    assert got.info["dedup_rows"] == 0
    monkeypatch.setenv("GCRE_TEST_DEDUP", "0")
    want, _, _ = _level4_direct(engine, w, method, 5, mutate=rewrite)
    helpers.assert_same_results(got, want, what=f"{method} rewritten row")


@pytest.mark.parametrize("method", ["method1", "method2"])
def test_uid_range_shard(engine, method, monkeypatch):
    """row shards group within their own rows; the shards' merged top-K and maxima equal the whole join without grouping"""
    w = _workload(257, 300, 200, 900, 1000, seed=4400)
    n4 = w.net.levels["4"].n_uids
    monkeypatch.setenv("GCRE_TEST_DEDUP", "0")
    whole, _, _ = _level4_direct(engine, w, method, 12)
    monkeypatch.setenv("GCRE_TEST_DEDUP", "1")
    cut = n4 // 3
    parts = [_level4_direct(engine, w, method, 12, uid_range=rng)[0] for rng in ((0, cut), (cut, n4))]
    assert sum(p.info["dedup_rows"] for p in parts) > 0
    assert np.array_equal(np.maximum(parts[0].permuted_scores, parts[1].permuted_scores), whole.permuted_scores)
    merged = sorted([s for p in parts for s in p.scores if s.src >= 0], key=lambda s: (-s.score, s.src, s.trg))[:12]
    ref = sorted([s for s in whole.scores if s.src >= 0], key=lambda s: (-s.score, s.src, s.trg))
    assert [(s.score, s.src, s.trg, s.cases, s.ctrls) for s in merged] == [(s.score, s.src, s.trg, s.cases, s.ctrls) for s in ref]


@pytest.mark.parametrize("top_k", [3, 70])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_ties_with_members(engine, oracles, method, top_k, monkeypatch):
    """K-th place shared by a representative and its members: a cohort where most genes are empty scores many pairs equally"""
    monkeypatch.setenv("GCRE_TEST_SMALL_PLAN", "1")
    w = synth.make_workload(40, 40, 60, 400, 1000, seed=4500, max_path_length=4, real_table=True, max_freq=0.05, zero_frac=0.85)
    want, _, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 4, top_k)
    monkeypatch.setenv("GCRE_TEST_DEDUP", "0")
    plain, _, _ = helpers.run_schedule(sparse_exec(engine), engine.UidRelSet, w, method, 4, top_k)
    monkeypatch.setenv("GCRE_TEST_DEDUP", "1")
    got, _, _ = helpers.run_schedule(sparse_exec(engine), engine.UidRelSet, w, method, 4, top_k)
    assert got["4"].info["dedup_rows"] > 0
    if top_k == 70:  # (at K = 3 this cohort's K-th score is not tied)
        ks = [s.score for s in want["4"].scores if s.src >= 0]
        assert len(ks) == top_k and ks.count(ks[0]) > 1, "the K-th score is shared"
    helpers.assert_same_results(got["4"], want["4"], what=f"{method} top_k={top_k}")
    helpers.assert_same_results(got["4"], plain["4"], what=f"{method} top_k={top_k}")


@pytest.mark.parametrize("method", ["method1", "method2"])
def test_cached_grouping_follows_the_rows(engine, method, monkeypatch):
    """a resident join index keeps its grouping between joins; it is rebuilt (or dropped) whenever the upstream rows change:
    a row set, the rows rewritten by a new level-3 join, or only a shard of them rewritten"""
    monkeypatch.setenv("GCRE_TEST_DEDUP", "1")
    w = _workload(64, 64, 80, 400, 1000, seed=4600)
    lv, didx = w.net.levels, w.net.data_idx
    ex = sparse_exec(engine)(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = 6
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    u = {k: engine.UidRelSet(lv[k].path_length, lv[k].src, lv[k].trg, lv[k].count, lv[k].location, lv[k].signs).make_resident(ex)
         for k in ("1a", "2", "3", "4")}
    d1 = ex.createPathSet(w.net.n_genes)
    d1.load_bits(w.gene_bits)
    p1 = ex.createPathSet(lv["1a"].n_pairs)
    ex.join(u["1a"], ex.createPathSet(lv["1a"].n_uids), d1.select(didx["1a"]), p1)
    p2 = ex.createPathSet(lv["2"].n_pairs)
    ex.join(u["2"], p1, d1.select(didx["2"]), p2)
    p3 = ex.createPathSet(lv["3"].n_pairs)
    sel3 = d1.select(didx["3"])
    ex.join(u["3"], p2, sel3, p3)

    def level4_both():
        got = ex.join(u["4"], p3, p2, ex.createPathSet(0))
        monkeypatch.setenv("GCRE_TEST_DEDUP", "0")
        want = ex.join(u["4"], p3, p2, ex.createPathSet(0))
        monkeypatch.setenv("GCRE_TEST_DEDUP", "1")
        helpers.assert_same_results(got, want, what=method)
        return got

    assert level4_both().info["dedup_rows"] > 0
    assert level4_both().info["dedup_rows"] > 0  # the cached grouping
    rows = p3.to_numpy()
    _, first, counts = np.unique(rows, axis=0, return_index=True, return_counts=True)
    k = int(np.nonzero(counts > 1)[0][0])
    twin = [i for i in range(rows.shape[0]) if i != first[k] and np.array_equal(rows[i], rows[first[k]])][0]
    new = rows[twin].copy()
    new[0] ^= np.uint64(1)
    p3.set(twin, new)
    assert level4_both().info["dedup_rows"] == 0  # no fingerprints after the write
    ex.join(u["3"], p2, sel3, p3)  # rewritten in full: fingerprints again, and the old twin is a twin again
    assert level4_both().info["dedup_rows"] > 0
    half = lv["3"].n_uids // 2
    ex.join(u["3"], p2, sel3, p3, uid_range=(half, lv["3"].n_uids))  # a shard of the rows rewritten
    level4_both()
