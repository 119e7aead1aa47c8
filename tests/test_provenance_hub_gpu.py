"""Provenance passes (record_rows_kernel, tail_eligible_kernel: one warp per work unit) on a network with one hub gene of 3,000
out-edges: its level-2 row and the level-3 / level-4 rows that end in it span many work units each.  The tail form must be taken
and exact when every pair is eligible, and not taken - the join still exact - when one pair of a hub row is not.  More than
1,024 permutations make the running-maxima kernels flush their maxima in the middle of a launch as well as at its end."""
import numpy as np
import pytest

import helpers
from geneticscre_b200 import synth
from test_tail_gene_gpu import _uids, sparse_exec

pytestmark = pytest.mark.gpu

HUB, HUB_OUT = 0, 3000
N_GENES, N_CASES, N_CTRLS, TOP_K = 3200, 70, 63, 8


@pytest.fixture(autouse=True)
def _knobs(monkeypatch):
    monkeypatch.setenv("GCRE_TEST_TAIL", "1")
    monkeypatch.setenv("GCRE_TEST_NO_SPLIT", "1")  # (<= 512 permutations would otherwise run the split-carrier kernels)
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", "0")
    monkeypatch.setenv("GCRE_SC_PTS", "0")


def hub_workload(perms, seed):
    """a sparse random network plus gene HUB with HUB_OUT out-edges and three in-edges"""
    rng = np.random.default_rng(seed)
    src = np.concatenate([rng.integers(1, N_GENES, 6000), np.full(HUB_OUT, HUB), rng.choice(np.arange(1, N_GENES), 3, replace=False)])
    trg = np.concatenate([rng.integers(1, N_GENES, 6000), np.arange(1, HUB_OUT + 1), np.full(3, HUB)])
    e = np.unique(np.stack([src, trg], axis=1)[src != trg], axis=0)  # unique, sorted by (src, trg)
    sign = np.where(rng.random(e.shape[0]) < 0.7, 1, -1)
    net = synth.network_from_edges(N_GENES, e[:, 0], e[:, 1], sign, max_path_length=4)
    bits = synth.make_cohort_bits(N_CASES + N_CTRLS, N_GENES, seed + 2, max_freq=0.12, zero_frac=0.3)
    masks = synth.make_perm_masks(N_CASES, N_CTRLS, perms, seed + 3)
    w = synth.Workload(N_CASES, N_CTRLS, perms, bits, np.ascontiguousarray(bits[net.ents2]), masks,
                       synth.make_value_table(N_CASES, N_CTRLS), net)
    lv = w.net.levels
    assert lv["2"].count[HUB] == HUB_OUT and (lv["4"].count == HUB_OUT).sum() >= 1
    return w


@pytest.mark.parametrize("thr", ["0", "1"])
@pytest.mark.parametrize("perms", [257, 2100])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_hub_schedule_tail_form(engine, oracles, method, perms, thr, monkeypatch):
    monkeypatch.setenv("GCRE_THR", thr)
    w = hub_workload(perms, seed=5100 + perms)
    want, kept_want, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 4, TOP_K)
    got, kept, _ = helpers.run_schedule(sparse_exec(engine), engine.UidRelSet, w, method, 4, TOP_K)
    for k in kept_want:
        assert np.array_equal(kept[k], kept_want[k]), f"kept {k} differs"
    for lvl in want:
        helpers.assert_same_results(got[lvl], want[lvl], what=f"{method} p{perms} THR={thr} L{lvl}")
    assert got["4"].info["tail_form"]


@pytest.mark.parametrize("method", ["method1", "method2"])
def test_hub_one_ineligible_pair(engine, oracles, method):
    """One level-4 hub row shifted by one partner: its last pair's partner starts at another gene, so the join runs without the
    tail form, and exactly"""
    w = hub_workload(1025, seed=5200)
    lv, didx = w.net.levels, w.net.data_idx
    ex = sparse_exec(engine)(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = TOP_K
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    d1 = ex.createPathSet(w.net.n_genes)
    d1.load_bits(w.gene_bits)
    p1 = ex.createPathSet(lv["1a"].n_pairs)
    ex.join(_uids(engine, lv["1a"]), ex.createPathSet(lv["1a"].n_uids), d1.select(didx["1a"]), p1)
    p2 = ex.createPathSet(lv["2"].n_pairs)
    ex.join(_uids(engine, lv["2"]), p1, d1.select(didx["2"]), p2)
    p3 = ex.createPathSet(lv["3"].n_pairs)
    ex.join(_uids(engine, lv["3"]), p2, d1.select(didx["3"]), p3)

    l4 = lv["4"]
    assert ex.join(_uids(engine, l4), p3, p2, ex.createPathSet(0)).info["tail_form"]
    location = l4.location.copy()
    row = int(np.nonzero(l4.count == HUB_OUT)[0][0])
    location[row] += 1  # the hub's edges are rows [0, HUB_OUT) of paths2; row HUB_OUT starts gene 1's
    assert w.net.edges_src[location[row] + HUB_OUT - 1] != HUB
    got = ex.join(_uids(engine, l4, location), p3, p2, ex.createPathSet(0))
    assert not got.info["tail_form"]

    o = oracles.OracleExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    o.top_k = TOP_K
    o.setValueTable(w.value_table)
    o.setPermutedMasks(w.perm_masks)
    o0, o1 = o.createPathSet(p3.size), o.createPathSet(p2.size)
    o0.rows[:] = p3.to_numpy()
    o1.rows[:] = p2.to_numpy()
    want = o.join(_uids(oracles, l4, location), o0, o1, o.createPathSet(0))
    helpers.assert_same_results(got, want, what=f"{method} one ineligible pair")
