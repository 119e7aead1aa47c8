"""Pre-counted KEEP joins through a selection's base set (join_sparse.cuh): level 3's partners are copies of data1's gene rows, so
a level-3 pair is scored through the data1 row and data1's pre-counted table, and the kept rows take the final counts along.
Bit-exact against the CPU oracle with the form forced on and off; the counts it emits are the ones level 4 would otherwise walk;
the form is not taken when the engine cannot know the partner rows are still their base rows.

GCRE_PRECOUNT_MAX_MB=1 lets data1's table (a few hundred gene rows) fit and keeps a table of the partner copy itself (over a
thousand rows) out, so with GCRE_TEST_PRECOUNT=1 a level-3 join reports `precounted` exactly when it ran through the base set."""
import numpy as np
import pytest

import helpers
from geneticscre_b200 import synth
from test_join_gpu import SHAPES
from test_tail_gene_gpu import _uids, sparse_exec

pytestmark = pytest.mark.gpu

FORMS = [pytest.param("0", id="delta"), pytest.param("1", id="selection")]
BUDGET_MB = 1


@pytest.fixture(autouse=True)
def _knobs(monkeypatch):
    monkeypatch.setenv("GCRE_TEST_NO_SPLIT", "1")  # (<= 512 permutations would otherwise run the split-carrier kernels)
    monkeypatch.setenv("GCRE_SC_PTS", "0")
    monkeypatch.setenv("GCRE_TEST_TAIL", "1")  # level 4 reads level 3's rows through their provenance, as in the benchmark
    monkeypatch.setenv("GCRE_PRECOUNT_MAX_MB", str(BUDGET_MB))


def _workload(shape, seed, length=4):
    nc, nt, g, e, perms, top_k = shape
    w = synth.make_workload(nc, nt, g, e, perms, seed=seed, max_path_length=length, real_table=True, max_freq=0.12, zero_frac=0.3)
    return w, top_k


def _table_bytes(rows, method, perms):
    return rows * (1 if method == "method1" else 2) * ((perms + 1023) // 1024) * 2048


def _check_budget(w, method):
    """the premise of the module docstring"""
    budget = BUDGET_MB << 20
    assert _table_bytes(w.net.n_genes, method, w.n_perms) <= budget < _table_bytes(w.net.levels["3"].n_pairs, method, w.n_perms)


def _engine_exec(engine, w, method, top_k):
    ex = sparse_exec(engine)(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    return ex


def _oracle_join(oracles, w, method, top_k, level, rows0, rows1):
    o = oracles.OracleExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    o.top_k = top_k
    o.setValueTable(w.value_table)
    o.setPermutedMasks(w.perm_masks)
    o0, o1 = o.createPathSet(rows0.shape[0]), o.createPathSet(rows1.shape[0])
    o0.rows[:] = rows0
    o1.rows[:] = rows1
    keep = o.createPathSet(w.net.levels[level].n_pairs if level == "3" else 0)
    return o.join(_uids(oracles, w.net.levels[level]), o0, o1, keep), keep.rows


@pytest.mark.parametrize("thr", ["0", "1"])
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("method", ["method1", "method2"])
@pytest.mark.parametrize("shape", [SHAPES[2], SHAPES[4], SHAPES[5]], ids=["p129", "p257", "p40"])
def test_schedule(engine, oracles, method, form, thr, shape, monkeypatch):
    """The full five-level schedule: kept rows of every level and all results, both look-up stages"""
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", form)
    monkeypatch.setenv("GCRE_THR", thr)
    w, top_k = _workload(shape, 1000 + shape[0] + shape[4], length=5)
    want, kept_want, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 5, top_k)
    got, kept, _ = helpers.run_schedule(sparse_exec(engine), engine.UidRelSet, w, method, 5, top_k)
    for k in kept_want:
        assert np.array_equal(kept[k], kept_want[k]), f"kept {k} differs"
    for lvl in want:
        helpers.assert_same_results(got[lvl], want[lvl], what=f"{method} {shape} {form} THR={thr} L{lvl}")
    for lvl in ("1a", "2", "3"):  # the KEEP joins whose partners are selections of data1
        if w.net.levels[lvl].n_pairs > 0:
            assert got[lvl].info["precounted"] == (form == "1"), f"L{lvl}"
            assert not got[lvl].info["tail_form"], f"L{lvl}"


def _levels_1_to_3(engine, w, method, top_k, uid_range=None):
    ex = _engine_exec(engine, w, method, top_k)
    lv, didx = w.net.levels, w.net.data_idx
    d1 = ex.createPathSet(w.net.n_genes)
    d1.load_bits(w.gene_bits)
    p1 = ex.createPathSet(lv["1a"].n_pairs)
    ex.join(_uids(engine, lv["1a"]), ex.createPathSet(lv["1a"].n_uids), d1.select(didx["1a"]), p1)
    p2 = ex.createPathSet(lv["2"].n_pairs)
    ex.join(_uids(engine, lv["2"]), p1, d1.select(didx["2"]), p2)
    p3 = ex.createPathSet(lv["3"].n_pairs)
    r3 = ex.join(_uids(engine, lv["3"]), p2, d1.select(didx["3"]), p3, uid_range=uid_range)
    return ex, d1, p2, p3, r3


@pytest.mark.parametrize("thr", ["0", "1"])
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_emitted_counts_match_walked_counts(engine, oracles, method, form, thr, monkeypatch):
    """Level 4 with its base counts loaded from the tables level 3 emitted, against level 4 over the same rows copied into a
    set that carries no tables (its base counts walked from carrier lists): identical, and equal to the oracle"""
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", form)
    monkeypatch.setenv("GCRE_THR", thr)
    w, top_k = _workload(SHAPES[4], 4301)
    _check_budget(w, method)
    ex, d1, p2, p3, r3 = _levels_1_to_3(engine, w, method, top_k)
    assert r3.info["precounted"] == (form == "1")
    u4 = _uids(engine, w.net.levels["4"])
    from_tables = ex.join(u4, p3, p2, ex.createPathSet(0))
    assert from_tables.info["tail_form"]
    copy3 = p3.select(np.arange(p3.size, dtype=np.int32))
    walked = ex.join(u4, copy3, p2, ex.createPathSet(0))
    helpers.assert_same_results(from_tables, walked, what=f"{method} {form} emitted vs walked")
    want, _ = _oracle_join(oracles, w, method, top_k, "4", p3.to_numpy(), p2.to_numpy())
    helpers.assert_same_results(from_tables, want, what=f"{method} {form} L4")


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_row_shards(engine, oracles, method, form, monkeypatch):
    """Row-sharded level 3 (each shard writes and emits only its slice) followed by level 4 over that slice, merged"""
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", form)
    w, top_k = _workload(SHAPES[4], 4302)
    _check_budget(w, method)
    want, _, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 4, top_k)
    lv = w.net.levels
    prefix3 = np.concatenate([[0], np.cumsum(lv["3"].count.astype(np.int64))])
    bounds = [0, lv["3"].n_uids // 3, (2 * lv["3"].n_uids) // 3, lv["3"].n_uids]
    scores, perm = [], np.zeros(w.n_perms)
    for a, b in zip(bounds[:-1], bounds[1:]):
        ex, d1, p2, p3, r3 = _levels_1_to_3(engine, w, method, top_k, uid_range=(a, b))
        assert r3.info["precounted"] == (form == "1" and prefix3[b] > prefix3[a])
        r = ex.join(_uids(engine, lv["4"]), p3, p2, ex.createPathSet(0), uid_range=(int(prefix3[a]), int(prefix3[b])))
        scores.append(r.scores)
        perm = np.maximum(perm, np.asarray(r.permuted_scores))
    got = want["4"].__class__(engine.merge_topk(scores, top_k), perm)
    helpers.assert_same_results(got, want["4"], what=f"{method} {form} sharded L4")


@pytest.mark.parametrize("hook", ["GCRE_TEST_SMALL_PLAN", "GCRE_TEST_WIDE_CARRIERS"])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_plan_and_carrier_width(engine, oracles, method, hook, monkeypatch):
    """The budget-overflow redo of the launch plan (every launch size shrunk) and u32 carrier indices"""
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", "1")
    monkeypatch.setenv(hook, "1")
    w, top_k = _workload(SHAPES[4], 4303, length=5)
    want, kept_want, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 5, top_k)
    got, kept, _ = helpers.run_schedule(sparse_exec(engine), engine.UidRelSet, w, method, 5, top_k)
    for k in kept_want:
        assert np.array_equal(kept[k], kept_want[k]), f"kept {k} differs"
    for lvl in want:
        helpers.assert_same_results(got[lvl], want[lvl], what=f"{method} {hook} L{lvl}")
    assert got["3"].info["precounted"]


@pytest.mark.parametrize("variant", ["none", "reload", "set_row", "bits"])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_only_with_live_selection(engine, oracles, method, variant, monkeypatch):
    """The form needs the partner rows to still be their base rows: data1 reloaded or one of its rows rewritten after the
    selection was taken, or a partner set loaded from bits with no selection behind it, run the delta form - exactly"""
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", "1")
    w, top_k = _workload(SHAPES[4], 4304)
    _check_budget(w, method)
    ex = _engine_exec(engine, w, method, top_k)
    lv, didx = w.net.levels, w.net.data_idx
    d1 = ex.createPathSet(w.net.n_genes)
    d1.load_bits(w.gene_bits)
    p1 = ex.createPathSet(lv["1a"].n_pairs)
    ex.join(_uids(engine, lv["1a"]), ex.createPathSet(lv["1a"].n_uids), d1.select(didx["1a"]), p1)
    p2 = ex.createPathSet(lv["2"].n_pairs)
    ex.join(_uids(engine, lv["2"]), p1, d1.select(didx["2"]), p2)
    partner = d1.select(didx["3"])
    if variant == "reload":  # the same content, written again: the engine cannot tell
        d1.load_bits(w.gene_bits)
    elif variant == "set_row":
        g = int(didx["3"][0])
        d1.set(g, d1[g])
    elif variant == "bits":
        rows = partner.to_numpy()
        partner = ex.createPathSet(rows.shape[0])
        if method == "method1":
            partner.load_bits(rows)
        else:
            for k in range(rows.shape[0]):
                partner.set(k, rows[k])
    p3 = ex.createPathSet(lv["3"].n_pairs)
    got = ex.join(_uids(engine, lv["3"]), p2, partner, p3)
    assert got.info["precounted"] == (variant == "none")
    want, kept_want = _oracle_join(oracles, w, method, top_k, "3", p2.to_numpy(), partner.to_numpy())
    helpers.assert_same_results(got, want, what=f"{method} {variant} L3")
    assert np.array_equal(p3.to_numpy(), kept_want)
    # and level 4 over those rows (counts emitted by whichever form ran)
    got4 = ex.join(_uids(engine, lv["4"]), p3, p2, ex.createPathSet(0))
    want4, _ = _oracle_join(oracles, w, method, top_k, "4", p3.to_numpy(), p2.to_numpy())
    helpers.assert_same_results(got4, want4, what=f"{method} {variant} L4")
