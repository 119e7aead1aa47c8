"""Tail form of the pre-counted sparse kernel (join_sparse.cuh): a level-4 pair scored through the data1 row of the one gene its
partner adds.  Bit-exact against the CPU oracle when it runs, exact and NOT taken whenever the engine cannot know where the rows
came from, and exact on the row-sharded (multi-GPU) path.  GCRE_TEST_TAIL=1 takes the form on joins of any size."""
import gc

import numpy as np
import pytest

import helpers
from geneticscre_b200 import _lib, synth
from test_join_gpu import SHAPES

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _tail_on(monkeypatch):
    monkeypatch.setenv("GCRE_TEST_TAIL", "1")
    monkeypatch.setenv("GCRE_TEST_NO_SPLIT", "1")  # (<= 512 permutations would otherwise run the split-carrier kernels)
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", "0")
    monkeypatch.setenv("GCRE_SC_PTS", "0")


def sparse_exec(engine, kernel=_lib.KERNEL_SPARSE):
    class Exec(engine.JoinExec):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.kernel = kernel

    return Exec


@pytest.mark.parametrize("thr", ["0", "1"])
@pytest.mark.parametrize("method", ["method1", "method2"])
@pytest.mark.parametrize("shape", SHAPES)
def test_schedule_tail_form(engine, oracles, method, shape, thr, monkeypatch):
    monkeypatch.setenv("GCRE_THR", thr)
    nc, nt, g, e, perms, top_k = shape
    w = synth.make_workload(nc, nt, g, e, perms, seed=1000 + nc + perms, max_path_length=5, real_table=(nc % 2 == 0),
                            max_freq=0.12, zero_frac=0.3)
    want, kept_want, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 5, top_k)
    got, kept, _ = helpers.run_schedule(sparse_exec(engine), engine.UidRelSet, w, method, 5, top_k)
    for k in kept_want:
        assert np.array_equal(kept[k], kept_want[k]), f"kept {k} differs"
    for lvl in want:
        helpers.assert_same_results(got[lvl], want[lvl], what=f"{method} {shape} THR={thr} L{lvl}")
        assert got[lvl].info["tail_form"] == (lvl == "4" and w.net.levels[lvl].n_pairs > 0), f"L{lvl}"
        if got[lvl].info["tail_form"]:
            assert not got[lvl].info["precounted"] and got[lvl].info["thresholded"] == (thr == "1")


def _uids(api, level, location=None, signs=None):
    return api.UidRelSet(level.path_length, level.src, level.trg, level.count, level.location if location is None else location,
                         level.signs if signs is None else signs)


def _level4(engine, oracles, w, method, top_k, variant):
    """levels 1a, 2, 3 on the engine, then whatever `variant` does to the level-4 operands, then level 4 on the engine and - on
    the operands the engine holds at that point - on the oracle"""
    ex = sparse_exec(engine)(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    lv, didx = w.net.levels, w.net.data_idx
    d1 = ex.createPathSet(w.net.n_genes)
    d1.load_bits(w.gene_bits)
    p1 = ex.createPathSet(lv["1a"].n_pairs)
    ex.join(_uids(engine, lv["1a"]), ex.createPathSet(lv["1a"].n_uids), d1.select(didx["1a"]), p1)
    p2 = ex.createPathSet(lv["2"].n_pairs)
    ex.join(_uids(engine, lv["2"]), p1, d1.select(didx["2"]), p2)
    p3 = ex.createPathSet(lv["3"].n_pairs)
    ex.join(_uids(engine, lv["3"]), p2, d1.select(didx["3"]), p3)

    l4 = lv["4"]
    location, signs, partner = l4.location, l4.signs, p2
    rng = np.random.default_rng(7)
    live = np.nonzero(l4.count > 0)[0]
    if variant == "shuffled":  # partner rows no longer follow the network
        location = l4.location.copy()
        location[live] = rng.integers(0, p2.size - l4.count[live] + 1).astype(np.uint32)
    elif variant == "signs":  # method 2: some pairs join the partner's first gene into the other half
        signs = l4.signs.copy()
        signs[::5] *= -1
    elif variant == "bits":  # a partner set the engine did not build
        partner = ex.createPathSet(p2.size)
        partner.load_bits(p2.to_numpy()[:, : synth.words_for(w.n_patients)])
    elif variant == "reload":  # data1 rewritten (with other rows) after paths2 / paths3 were built from it
        d1.load_bits(np.roll(w.gene_bits, 1, axis=0))
    elif variant == "set_row":  # one paths2 row read by the join gains carriers through the row setter
        r = int(l4.location[live[0]])
        row = p2[r]
        row[: synth.words_for(w.n_patients)] |= w.gene_bits[(int(didx["2"][r]) + 1) % w.net.n_genes]
        p2.set(r, row)
    elif variant == "destroyed":
        del d1
        gc.collect()
    uid4 = _uids(engine, l4, location, signs)
    got = ex.join(uid4, p3, partner, ex.createPathSet(0))

    o = oracles.OracleExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    o.top_k = top_k
    o.setValueTable(w.value_table)
    o.setPermutedMasks(w.perm_masks)
    o0, o1 = o.createPathSet(p3.size), o.createPathSet(partner.size)
    o0.rows[:] = p3.to_numpy()
    o1.rows[:] = partner.to_numpy()
    want = o.join(_uids(oracles, l4, location, signs), o0, o1, o.createPathSet(0))
    return got, want


FALLBACKS = ["shuffled", "bits", "reload", "set_row", "destroyed"]


@pytest.mark.parametrize("variant", ["none"] + FALLBACKS + ["signs"])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_tail_form_only_with_known_provenance(engine, oracles, method, variant):
    """The form runs only when the engine knows every level-4 partner adds one gene of a live, unchanged data1; otherwise the
    join runs as before.  Either way the result is exact."""
    if variant == "signs" and method == "method1":
        pytest.skip("method 1 has no orientation")
    w = synth.make_workload(257, 300, 200, 800, 257, seed=4244, max_path_length=4, real_table=True, max_freq=0.12, zero_frac=0.3)
    got, want = _level4(engine, oracles, w, method, 8, variant)
    helpers.assert_same_results(got, want, what=f"{method} {variant}")
    assert got.info["tail_form"] == (variant == "none")
    assert got.info["pairs"] > 0


@pytest.mark.parametrize("method", ["method1", "method2"])
def test_row_shards_match_whole_join(engine, oracles, method):
    """The row-sharded multi-GPU path: each shard builds only its slice of paths3 (level 3 over a range of its upstream rows)
    and scores level 4 over exactly those rows; merged, the shards give the whole join."""
    nc, nt, g, e, perms, top_k = SHAPES[4]
    w = synth.make_workload(nc, nt, g, e, perms, seed=4245, max_path_length=4, real_table=True, max_freq=0.12, zero_frac=0.3)
    want, _, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 4, top_k)
    ex = sparse_exec(engine)(method, nc, nt, perms)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    lv, didx = w.net.levels, w.net.data_idx
    d1 = ex.createPathSet(w.net.n_genes)
    d1.load_bits(w.gene_bits)
    p1 = ex.createPathSet(lv["1a"].n_pairs)
    ex.join(_uids(engine, lv["1a"]), ex.createPathSet(lv["1a"].n_uids), d1.select(didx["1a"]), p1)
    p2 = ex.createPathSet(lv["2"].n_pairs)
    ex.join(_uids(engine, lv["2"]), p1, d1.select(didx["2"]), p2)
    u3, u4 = _uids(engine, lv["3"]), _uids(engine, lv["4"])
    prefix3 = np.concatenate([[0], np.cumsum(lv["3"].count.astype(np.int64))])
    bounds = [0, lv["3"].n_uids // 3, (2 * lv["3"].n_uids) // 3, lv["3"].n_uids]
    scores, perm = [], np.zeros(perms)
    for a, b in zip(bounds[:-1], bounds[1:]):
        p3 = ex.createPathSet(lv["3"].n_pairs)
        ex.join(u3, p2, d1.select(didx["3"]), p3, uid_range=(a, b))
        r = ex.join(u4, p3, p2, ex.createPathSet(0), uid_range=(int(prefix3[a]), int(prefix3[b])))
        assert r.info["tail_form"]
        scores.append(r.scores)
        perm = np.maximum(perm, np.asarray(r.permuted_scores))
    got = want["4"].__class__(engine.merge_topk(scores, top_k), perm)
    helpers.assert_same_results(got, want["4"], what=f"{method} sharded L4")
