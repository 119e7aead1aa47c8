"""State the engine derives from a path set's rows, the exec's masks and its value table, checked after every mutation.

Between calls the engine keeps, per path set, its recorded largest half-row (``max_half_pop``, which sizes the carrier lists and
the anti-diagonal value tables), carrier lists, emitted and pre-count tables and provenance entries; per exec, the patient-major
masks, the anti-diagonal tables and a grow-only identity row map.  Each sequence here lets a join cache some of that state, then
applies one mutation (rows set or loaded, a selection, the object being the result of another KEEP join, new masks, a new value
table), then runs a second join that reads the mutated object in one role (upstream operand, partner, base of a selection,
tail-form provenance holder, result).  After every step every set is checked against numpy (``check_state``):
    recorded max_half_pop is -1 (unknown) or >= the true largest half-row popcount,
    carrier lists, when built, equal the ones the rows give and fit in the entries allocated,
    a count table marked current equals the counts of its rows under the exec's current masks.
The second join is compared bit for bit with a fresh CPU oracle built from the current contents of every operand, and its
info flags show that the intended kernel form ran.  A cohort above 1,024 patients makes a bound that is too small show up in
the results: at n <= 1,024 the anti-diagonal tables cover every total whatever the bound says."""
import numpy as np
import pytest

import helpers
import test_count_tables_gpu as ct
from geneticscre_b200 import _lib, synth

pytestmark = pytest.mark.gpu

ENV_KEYS = ("GCRE_TEST_NO_SPLIT", "GCRE_TEST_PRECOUNT", "GCRE_THR", "GCRE_SC_PTS", "GCRE_TEST_WIDE_CARRIERS", "GCRE_TEST_SMALL_PLAN",
            "GCRE_TEST_TAIL", "GCRE_TEST_VIEW_EXACT", "GCRE_TEST_EMIT")
# form -> (environment, expected info of the second join); the sparse forms of test_count_tables_gpu plus three more
FORMS = {k: (dict(env, GCRE_TEST_TAIL="0"), info) for k, (env, info, _) in ct.FORMS.items()}
FORMS["tail"] = ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_SC_PTS": "0", "GCRE_TEST_TAIL": "1"}, {"tail_form": True, "precounted": False})
FORMS["view_exact"] = ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_TEST_TAIL": "0", "GCRE_TEST_VIEW_EXACT": "1"},
                       {"precounted": False, "split_carrier": False})
FORMS["dense"] = ({"GCRE_TEST_TAIL": "0"}, {"kernel": _lib.KERNEL_DENSE})
# cohorts: "big" is above the anti-diagonal tables' 1,024-carrier floor and its level-3 rows pass 1,024 carriers
COHORTS = {"big": dict(nc=1300, nt=1700, genes=50, edges=110, max_freq=0.55, zero_frac=0.2),
           "small": dict(nc=60, nt=68, genes=60, edges=150, max_freq=0.15, zero_frac=0.2)}


# ---- references ---------------------------------------------------------------------------------------------------------
def half_pops(rows, m, w64):
    return np.stack([np.bitwise_count(h).sum(axis=1) for h in ct._halves(rows, m, w64)], axis=1) if rows.shape[0] else np.zeros((0, m), np.int64)


def max_half_pop(rows, m, w64):
    return int(half_pops(rows, m, w64).max()) if rows.shape[0] else 0


def check_state(ex, sets, what):
    """the invariants of every set's derived state (module docstring), against numpy on the rows, masks and table as they are"""
    masks = ex.getPermutedMasks()
    n, w64 = ex.num_cases + ex.num_ctrls, ex.w64
    for name, ps in sets.items():
        if ps.size == 0:
            continue
        tag = f"{what}: {name}"
        rows = ps.to_numpy()
        b = ps.debug_bounds()
        true = max_half_pop(rows, ex.m, w64)
        assert b["max_half_pop"] == -1 or b["max_half_pop"] >= true, f"{tag}: recorded max_half_pop {b['max_half_pop']} < true {true}"
        view = ps.debug_view()
        if view["lists"] is not None:
            used = int(view["lists"]["off"][-1])
            assert b["allocated"] >= used, f"{tag}: carrier lists use {used} entries, {b['allocated']} allocated"
            ct.check_lists(ps, n, ex.num_cases, ex.m, what=tag)
        else:
            assert b["allocated"] == 0, tag
        t = view["table"]
        if t is not None and t["current"]:
            ct.check_table(ps, masks, ex.m, ex.num_cases, lo=t["lo"], hi=t["hi"], what=f"{tag} table")


def check_diag(ex, res_rows, what):
    """the anti-diagonal tables cover every joined half-row total of a KEEP join's rows"""
    cap, t = ex.debug_diag_cap(), max_half_pop(res_rows, ex.m, ex.w64)
    assert cap >= t, f"{what}: anti-diagonal tables cover {cap} carriers, a joined half-row has {t}"


def oracle_exec(oracles, ex):
    """a fresh oracle with the exec's current masks and table"""
    o = oracles.OracleExec(ex.method, ex.num_cases, ex.num_ctrls, ex.iters_requested)
    o.top_k = ex.top_k
    o.setValueTable(ex.getValueTable())
    o.setPermutedMasks(ex.getPermutedMasks())
    return o


def oracle_join(oracles, ex, level, p0, p1, keep):
    """(joined_res, result rows or None) of the whole join on the operands' current rows"""
    o = oracle_exec(oracles, ex)
    r0, r1 = p0.to_numpy(), p1.to_numpy()
    o0, o1 = o.createPathSet(r0.shape[0]), o.createPathSet(r1.shape[0])
    o0.rows[:], o1.rows[:] = r0, r1
    res = o.createPathSet(level.n_pairs if keep else 0)
    want = o.join(ct.uids(oracles, level), o0, o1, res)
    return want, (res.rows if keep else None)


def place_rows(level, joined, prev, uid_range=None, path_idx=None):
    """result rows of a KEEP join over uids [a, b) whose pair rows go to path_idx (default: running sums), others as in prev"""
    prefix = np.concatenate([[0], np.cumsum(np.maximum(level.count.astype(np.int64), 0))])
    dst = prefix if path_idx is None else np.asarray(path_idx, np.int64)
    a, b = (0, level.n_uids) if uid_range is None else uid_range
    out = prev.copy()
    for u in range(a, b):
        c = int(max(level.count[u], 0))
        out[dst[u]:dst[u] + c] = joined[prefix[u]:prefix[u] + c]
    return out


def assert_form(info, form, what, **override):
    for k, v in dict(FORMS[form][1], **override).items():
        assert info[k] == v, f"{what}: info[{k}] = {info[k]}, want {v}"


# ---- set-up ---------------------------------------------------------------------------------------------------------------
def set_form(monkeypatch, form):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in FORMS[form][0].items():
        monkeypatch.setenv(k, v)


def make_case(engine, monkeypatch, form, perms, cohort, method, seed, test_table=False):
    """the environment of `form` (read when the exec is created), the exec, and levels 1a, 2, 3 kept"""
    set_form(monkeypatch, form)
    c = COHORTS[cohort]
    w = ct.workload(c["nc"], c["nt"], perms, seed=seed, genes=c["genes"], edges=c["edges"], max_freq=c["max_freq"], zero_frac=c["zero_frac"])
    ex = ct.make_exec(engine, w, method, table=synth.make_test_table(w.n_cases, w.n_ctrls, seed=seed) if test_table else None)
    if form == "dense":
        ex.kernel = _lib.KERNEL_DENSE
    d1, out = ct.run_keep_levels(engine, ex, w, partner_from_bits=form.startswith("pc_bits"))
    sets = {"d1": d1, "p1": out["1a"][0], "p2": out["2"][0], "p3": out["3"][0]}
    if cohort == "big":  # joined half-rows past the anti-diagonal tables' floor
        assert max_half_pop(sets["p3"].to_numpy(), ex.m, ex.w64) > 1024
    return w, ex, sets


def dense_bits(n, rows, seed, max_freq=0.45):
    return synth.make_cohort_bits(n, rows, seed=seed, max_freq=max_freq, zero_frac=0.0)


def shard(level, k=1, parts=3):
    return (level.n_uids * k) // parts, (level.n_uids * (k + 1)) // parts


def written_rows(level, uid_range):
    """bool[n_pairs]: the result rows a prefix KEEP join over uids [a, b) writes"""
    prefix = np.concatenate([[0], np.cumsum(np.maximum(level.count.astype(np.int64), 0))])
    out = np.zeros(level.n_pairs, dtype=bool)
    out[prefix[uid_range[0]]:prefix[uid_range[1]]] = True
    return out


# ---- mutations --------------------------------------------------------------------------------------------------------------
ROW_MUTATIONS = ("set", "load", "load_bits", "load_device")
KEEP_MUTATIONS = ("keep_full", "keep_shard", "keep_two_shards", "keep_nonprefix")
EXEC_MUTATIONS = ("set_masks", "set_cases", "gen_masks", "gen_masks_strata", "set_table", "set_table_device", "gen_table")
SELECT_MUTATIONS = ("select_before", "select_after")


def mutate_rows(ex, ps, mutation, seed, keep_alive):
    """rewrite ps's rows (denser than a kept row) through one of the setters; returns the rows it must now hold"""
    import torch

    n, w64, m = ex.num_cases + ex.num_ctrls, ex.w64, ex.m
    want = ps.to_numpy()
    if mutation == "set":  # a few rows gain carriers, in both halves
        rows = np.random.default_rng(seed).choice(ps.size, size=min(5, ps.size), replace=False)
        extra = dense_bits(n, len(rows) * m, seed).reshape(len(rows), m * w64)
        for r, e in zip(rows, extra):
            want[r] |= e
            ps.set(int(r), want[r])
        return want
    bits = dense_bits(n, ps.size, seed)
    want[:] = 0
    want[:, :w64] = bits
    if mutation == "load":
        ps.load(np.unpackbits(bits.view(np.uint8), axis=1, bitorder="little")[:, :n].astype(np.int32))
    elif mutation == "load_bits":
        ps.load_bits(bits)
    else:
        t = torch.from_numpy(bits.view(np.int64)).cuda()
        torch.cuda.synchronize()
        keep_alive.append(t)  # read on the exec's stream by the next join
        ps.load_bits_device(t.data_ptr(), ps.size, w64)
    return want


def mutate_exec(ex, mutation, seed, keep_alive):
    import torch

    nc, nt, n = ex.num_cases, ex.num_ctrls, ex.num_cases + ex.num_ctrls
    before_masks, before_table = ex.getPermutedMasks(), ex.getValueTable()
    if mutation == "set_masks":
        masks = synth.make_perm_masks(nc, nt, ex.iters_requested, seed=seed)
        ex.setPermutedMasks(masks)
        assert np.array_equal(ex.getPermutedMasks(), masks)
    elif mutation == "set_cases":
        masks = synth.make_perm_masks(nc, nt, ex.iters_requested, seed=seed)
        bits = np.unpackbits(masks.view(np.uint8), axis=1, bitorder="little")[:, :n].astype(bool)
        ex.setPermutedCases((bits == (np.arange(n) < nc)[None, :]).astype(np.int32))
        assert np.array_equal(ex.getPermutedMasks(), masks)
    elif mutation in ("gen_masks", "gen_masks_strata"):
        ex.setPermutationStrata(np.random.default_rng(seed).integers(0, 3, n) if mutation == "gen_masks_strata" else None)
        ex.generatePermutedMasks(seed=seed, first_perm=3)
    elif mutation == "set_table":
        table = synth.make_test_table(nc, nt, seed=seed)
        ex.setValueTable(table)
        assert np.array_equal(ex.getValueTable(), table)
    elif mutation == "set_table_device":
        table = synth.make_test_table(nc, nt, seed=seed)
        t = torch.from_numpy(table).cuda()
        torch.cuda.synchronize()
        keep_alive.append(t)
        ex.setValueTableDevice(t.data_ptr(), nc + 1, nt + 1)
        assert np.array_equal(ex.getValueTable(), table)
    elif mutation == "gen_table":  # the exec started from a test table
        ex.generateValueTable()
    if mutation in ("set_masks", "set_cases", "gen_masks", "gen_masks_strata"):
        assert not np.array_equal(ex.getPermutedMasks(), before_masks), mutation
    else:
        assert not np.array_equal(ex.getValueTable(), before_table), mutation


def mutate_by_keep(engine, oracles, ex, w, sets, name, mutation, seed):
    """rewrite sets[name] (paths2 or paths3) as the result of its level's KEEP join over partners from denser gene rows: the
    whole join, the middle third of its uids, two thirds in turn (different partners), or a shard whose pair rows are placed
    in reverse uid order (not the running sums).  Returns the rows it must now hold."""
    lvl = {"p2": "2", "p3": "3"}[name]
    level = w.net.levels[lvl]
    up = sets[{"p2": "p1", "p3": "p2"}[name]]
    target = sets[name]
    n = w.n_patients
    prev = target.to_numpy()
    steps = {"keep_full": [(None, seed)], "keep_shard": [(shard(level), seed)], "keep_nonprefix": [(shard(level), seed)],
             "keep_two_shards": [(shard(level, 0), seed), (shard(level, 2), seed + 1)]}[mutation]
    path_idx = None
    if mutation == "keep_nonprefix":
        c = np.maximum(level.count.astype(np.int64), 0)
        path_idx = np.cumsum(c[::-1])[::-1] - c  # uid u's rows after those of every later uid
    for rng, s in steps:
        dense = ex.createPathSet(w.net.n_genes)
        dense.load_bits(dense_bits(n, w.net.n_genes, s, max_freq=0.35))
        part = dense.select(w.net.data_idx[lvl])
        u = engine.UidRelSet(level.path_length, level.src, level.trg, level.count, level.location, level.signs, path_idx=path_idx)
        ex.join(u, up, part, target, uid_range=rng)
        _, joined = oracle_join(oracles, ex, level, up, part, keep=True)
        prev = place_rows(level, joined, prev, rng, path_idx)
    return prev


# ---- roles: the second join ------------------------------------------------------------------------------------------------
# role -> (the object mutated, the second join's level, (upstream, partner, result) of that join)
ROLES = {
    "upstream": ("p2", "3", ("p2", "sel3", "fresh")),   # paths2 as the upstream operand of level 3 (its emitted counts)
    "partner": ("p2", "4", ("p3", "p2", None)),          # paths2 as level 4's partner (pre-count table)
    "sel_base": ("d1", "3", ("p2", "sel3", "fresh")),    # data1 as the base of level 3's selection partner
    "tail": ("p3", "4", ("p3", "p2", None)),             # paths3 as level 4's upstream with tail provenance
    "result": ("p3", "3", ("p2", "sel3", "p3")),         # paths3 as level 3's result again
}

CASES = [
    # rows rewritten through the setters and loaders
    ("set", "upstream", "delta", 1025, "big", "method1"),
    ("set", "partner", "selection", 1025, "big", "method2"),
    ("set", "tail", "tail", 33, "small", "method2"),
    ("set", "result", "dense", 33, "big", "method1"),
    ("load", "upstream", "split", 300, "big", "method2"),
    ("load", "sel_base", "selection", 33, "big", "method1"),
    ("load_bits", "upstream", "selection_thr", 33, "small", "method1"),
    ("load_bits", "partner", "pc_bits", 1025, "small", "method2"),
    ("load_bits", "tail", "tail", 1025, "big", "method1"),
    ("load_device", "upstream", "split_pts", 100, "small", "method2"),
    ("load_device", "sel_base", "view_exact", 1025, "big", "method2"),
    # selections taken before and after their base is rewritten
    ("select_before", "sel_base", "selection", 1025, "big", "method2"),
    ("select_before", "sel_base", "split", 100, "small", "method1"),
    ("select_after", "sel_base", "selection_wide", 33, "small", "method1"),
    ("select_after", "sel_base", "delta_wide", 1025, "big", "method2"),
    # the result of another KEEP join
    ("keep_full", "upstream", "split", 100, "big", "method1"),
    ("keep_full", "result", "split", 300, "small", "method2"),
    ("keep_shard", "upstream", "delta", 1025, "big", "method2"),
    ("keep_shard", "partner", "selection", 33, "big", "method1"),
    ("keep_shard", "result", "view_exact", 33, "big", "method2"),
    ("keep_two_shards", "upstream", "split_wide", 300, "big", "method1"),
    ("keep_two_shards", "result", "selection", 1025, "small", "method2"),
    ("keep_nonprefix", "upstream", "selection", 33, "big", "method2"),
    ("keep_nonprefix", "partner", "delta_thr", 1025, "big", "method1"),
    # new permutation masks
    ("set_masks", "upstream", "split", 300, "big", "method1"),
    ("set_masks", "partner", "selection", 1025, "big", "method2"),
    ("set_masks", "tail", "tail", 1025, "small", "method1"),
    ("set_cases", "upstream", "delta", 33, "big", "method2"),
    ("set_cases", "sel_base", "selection", 1025, "small", "method1"),
    ("gen_masks", "sel_base", "selection", 33, "big", "method2"),
    ("gen_masks", "upstream", "split_pts", 100, "small", "method1"),
    ("gen_masks_strata", "upstream", "split", 300, "big", "method2"),
    ("gen_masks_strata", "partner", "selection_thr", 1025, "big", "method1"),
    # a new value table
    ("set_table", "upstream", "delta_thr", 1025, "big", "method1"),
    ("set_table", "result", "dense", 1025, "small", "method2"),
    ("set_table_device", "upstream", "split", 100, "big", "method2"),
    ("set_table_device", "tail", "tail", 33, "big", "method2"),
    ("gen_table", "partner", "selection", 1025, "big", "method1"),
    ("gen_table", "tail", "tail", 1025, "big", "method2"),
    ("gen_table", "upstream", "selection_small_plan", 33, "small", "method2"),
]


def _case_id(c):
    return "-".join(str(x) for x in c)


@pytest.mark.parametrize("mutation,role,form,perms,cohort,method", [pytest.param(*c, id=_case_id(c)) for c in CASES])
def test_mutation_then_join(engine, oracles, mutation, role, form, perms, cohort, method, monkeypatch):
    seed = 8000 + perms + len(mutation) * 31 + len(role) * 7 + (1 if method == "method2" else 0)
    what = _case_id((mutation, role, form, perms, cohort, method))
    w, ex, sets = make_case(engine, monkeypatch, form, perms, cohort, method, seed, test_table=(mutation == "gen_table"))
    lv, didx = w.net.levels, w.net.data_idx
    target, lvl, (s0, s1, sr) = ROLES[role]
    if role in ("partner", "tail"):  # the state the second join reads: level 4 once (pre-count table, provenance checks)
        ex.join(ct.uids(engine, lv["4"]), sets["p3"], sets["p2"], ex.createPathSet(0))
    check_state(ex, sets, f"{what} before")

    keep_alive = []
    sel3 = sets["d1"].select(didx["3"]) if mutation == "select_before" else None
    if mutation in ROW_MUTATIONS:
        want_rows = mutate_rows(ex, sets[target], mutation, seed, keep_alive)
        assert np.array_equal(sets[target].to_numpy(), want_rows), f"{what}: rows after {mutation}"
    elif mutation in SELECT_MUTATIONS:
        sets["d1"].load_bits(np.roll(dense_bits(w.n_patients, w.net.n_genes, seed), 1, axis=0))
    elif mutation in KEEP_MUTATIONS:
        want_rows = mutate_by_keep(engine, oracles, ex, w, sets, target, mutation, seed)
        assert np.array_equal(sets[target].to_numpy(), want_rows), f"{what}: rows after {mutation}"
    else:
        mutate_exec(ex, mutation, seed, keep_alive)
    if sel3 is None:
        sel3 = sets["d1"].select(didx["3"])
    sets["sel3"] = sel3
    check_state(ex, sets, f"{what} after {mutation}")  # the bounds hold before any join reads the mutated set

    level = lv[lvl]
    p0, p1 = sets[s0], sets[s1]
    res = ex.createPathSet(level.n_pairs) if sr == "fresh" else ex.createPathSet(0) if sr is None else sets[sr]
    keep = res.size > 0
    want, want_rows = oracle_join(oracles, ex, level, p0, p1, keep)  # before the join: the result may be an operand's rows
    got = ex.join(ct.uids(engine, level), p0, p1, res)
    assert got.info["pairs"] == level.n_pairs > 0, what
    if role == "tail":  # the form runs only while paths3's provenance holds: rows rewritten through a setter drop it
        assert_form(got.info, form, what, tail_form=mutation not in ROW_MUTATIONS)
    else:
        assert_form(got.info, form, what)
    helpers.assert_same_results(got, want, what=what)
    if keep:
        rows = res.to_numpy()
        assert np.array_equal(rows, want_rows), f"{what}: kept rows differ"
        check_diag(ex, rows, what)
        sets["res"] = res
    check_state(ex, sets, f"{what} after the second join")


# ---- the identity row map, shards into fresh sets ------------------------------------------------------------------------
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_identity_map_grows(engine, oracles, method, monkeypatch):
    """Pre-counted joins whose partners are their own rows (a set loaded from bits, not a selection) read the exec's row map:
    first through a small partner set, then a larger one, then the small one again"""
    set_form(monkeypatch, "pc_bits")
    nc, nt, perms = 257, 300, 1025
    n = nc + nt
    ex = ct.make_exec(engine, ct.workload(nc, nt, perms, seed=8500), method)
    m, w64 = ex.m, ex.w64
    rng = np.random.default_rng(8500)
    for k, rows in enumerate((40, 700, 40)):
        partner = ex.createPathSet(rows)
        bits = dense_bits(n, rows * m, 8500 + k, max_freq=0.2).reshape(rows, m * w64)
        if m == 1:
            partner.load_bits(bits)
        else:
            for r in range(rows):
                partner.set(r, bits[r])
        n_up = 30
        up = ex.createPathSet(n_up)
        up.load_bits(dense_bits(n, n_up, 8600 + k, max_freq=0.2))
        count = rng.integers(1, rows // n_up + 8, n_up).astype(np.int32)
        loc = rng.integers(0, rows - count + 1).astype(np.uint32)
        signs = np.where(rng.random(max(rows, n_up)) < 0.5, 1, -1).astype(np.int32)
        args = (4, np.arange(n_up), np.arange(n_up), count, loc, signs)
        got = ex.join(engine.UidRelSet(*args), up, partner, ex.createPathSet(0))
        assert got.info["precounted"], (method, rows)
        o = oracle_exec(oracles, ex)
        o0, o1 = o.createPathSet(n_up), o.createPathSet(rows)
        o0.rows[:], o1.rows[:] = up.to_numpy(), partner.to_numpy()
        want = o.join(oracles.UidRelSet(*args), o0, o1, o.createPathSet(0))
        helpers.assert_same_results(got, want, what=f"{method} partner of {rows} rows")
        check_state(ex, {"up": up, "partner": partner}, f"{method} partner of {rows} rows")


@pytest.mark.parametrize("form,perms", [("delta", 1025), ("selection", 33), ("split", 300), ("dense", 1025)])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_shard_into_a_fresh_set(engine, oracles, form, perms, method, monkeypatch):
    """A row shard of level 3 into a fresh set: its rows are the whole join's, every other row reads back zero, and the set's
    bound covers them (the next level reads it)"""
    seed = 8700 + perms
    w, ex, sets = make_case(engine, monkeypatch, form, perms, "big", method, seed)
    lv, didx = w.net.levels, w.net.data_idx
    l3 = lv["3"]
    res = ex.createPathSet(l3.n_pairs)
    rng = shard(l3)
    p2, sel = sets["p2"], sets["d1"].select(didx["3"])
    ex.join(ct.uids(engine, l3), p2, sel, res, uid_range=rng)
    _, joined = oracle_join(oracles, ex, l3, p2, sel, keep=True)
    want_rows = place_rows(l3, joined, np.zeros_like(joined), rng)
    assert np.array_equal(res.to_numpy(), want_rows), f"{form} {method}: shard rows"
    sets["res"] = res
    check_state(ex, sets, f"{form} {method} after the shard")
    check_diag(ex, want_rows, f"{form} {method} shard")
    got = ex.join(ct.uids(engine, lv["4"]), res, p2, ex.createPathSet(0))
    assert_form(got.info, form, f"{form} {method} L4")
    want, _ = oracle_join(oracles, ex, lv["4"], res, p2, keep=False)
    helpers.assert_same_results(got, want, what=f"{form} {method} L4 over the shard")


# ---- a set loaded with dense rows, then rewritten by a row shard of sparser rows ----------------------------------------------
@pytest.mark.parametrize("form,perms", [("delta", 1025), ("selection", 33), ("split", 300)])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_dense_set_rewritten_by_a_row_shard(engine, oracles, form, perms, method, monkeypatch):
    """The rows outside the shard keep their dense carriers: the set's recorded bound must stay unknown (or cover them), or the
    next join sizes its carrier lists and anti-diagonal tables for the shard's sparser rows"""
    seed = 8900 + perms
    w, ex, sets = make_case(engine, monkeypatch, form, perms, "big", method, seed)
    lv, didx = w.net.levels, w.net.data_idx
    l3 = lv["3"]
    r3 = ex.createPathSet(l3.n_pairs)
    dense = dense_bits(w.n_patients, r3.size, seed, max_freq=0.9)
    r3.load_bits(dense)
    prev = r3.to_numpy()
    rng = shard(l3)
    p2, sel = sets["p2"], sets["d1"].select(didx["3"])
    ex.join(ct.uids(engine, l3), p2, sel, r3, uid_range=rng)
    rows = r3.to_numpy()
    true = max_half_pop(rows, ex.m, ex.w64)
    written = max_half_pop(rows[written_rows(l3, rng)], ex.m, ex.w64)
    assert true > written, "the rows outside the shard must be the densest"
    bound = r3.debug_bounds()["max_half_pop"]
    assert bound == -1 or bound >= true, f"{form} {method}: recorded max_half_pop {bound} < true {true} (shard rows: {written})"
    _, joined = oracle_join(oracles, ex, l3, p2, sel, keep=True)
    assert np.array_equal(rows, place_rows(l3, joined, prev, rng)), f"{form} {method}: rows after the shard"
    sets["r3"] = r3
    check_state(ex, sets, f"{form} {method} after the shard")
    got = ex.join(ct.uids(engine, lv["4"]), r3, p2, ex.createPathSet(0))
    assert_form(got.info, form, f"{form} {method} L4")
    want, _ = oracle_join(oracles, ex, lv["4"], r3, p2, keep=False)
    helpers.assert_same_results(got, want, what=f"{form} {method} L4 over the rewritten set")
    check_state(ex, sets, f"{form} {method} after level 4")
