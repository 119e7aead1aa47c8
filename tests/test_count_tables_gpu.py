"""The sparse kernels' intermediate state, read back and checked directly (PathSet.debug_view): the count tables KEEP joins emit
for their rows, the pre-count tables of partner sets, the carrier lists, and - through joins that hold exactly one pair - the
per-pair values of score-only joins.

The join outputs (top-K, per-permutation maxima) hide most count errors: a permutation's maximum comes from one of a few extreme
rows.  Here every entry is compared with an exact numpy reference computed from the set's rows and the exec's permutation masks:
    count[row][h][r] = popcount(half h of row & case mask of permutation r),  len = popcount(half),  ncase = its carriers < n_cases.
Test hooks pick the kernel form (GCRE_TEST_NO_SPLIT, GCRE_TEST_PRECOUNT, GCRE_THR, GCRE_SC_PTS, GCRE_TEST_WIDE_CARRIERS,
GCRE_TEST_SMALL_PLAN, GCRE_TEST_TAIL, GCRE_TEST_EMIT); each test asserts from the join's info that the intended form ran."""
import zlib

import numpy as np
import pytest

import helpers
from geneticscre_b200 import _lib, synth

pytestmark = pytest.mark.gpu

NONE = np.uint32(0xFFFFFFFF)


# ---- exact references -------------------------------------------------------------------------------------------------
def _halves(rows, m, w64):
    return [np.ascontiguousarray(rows[:, h * w64:(h + 1) * w64]) for h in range(m)]


def ref_counts(rows, masks, m, n_cases):
    """rows uint64[R][m * w64] (unpadded), masks uint64[P][w64] -> counts int64[R][m][P], len / ncase int64[R][m]"""
    w64 = masks.shape[1]
    case_words = synth.pack_bits(np.arange(w64 * 64)[None, :] < n_cases)[0]
    cnt = np.zeros((rows.shape[0], m, masks.shape[0]), dtype=np.int64)
    ln = np.zeros((rows.shape[0], m), dtype=np.int64)
    nc = np.zeros_like(ln)
    for h, half in enumerate(_halves(rows, m, w64)):
        ln[:, h] = np.bitwise_count(half).sum(axis=1)
        nc[:, h] = np.bitwise_count(half & case_words[None, :]).sum(axis=1)
        for r0 in range(0, rows.shape[0], 64):
            blk = half[r0:r0 + 64]
            cnt[r0:r0 + 64, h, :] = np.bitwise_count(blk[:, None, :] & masks[None, :, :]).sum(axis=2)
    return cnt, ln, nc


def check_table(ps, masks, m, n_cases, lo=None, hi=None, layout=None, what=""):
    """the set's count table holds rows [lo, hi) (default: all) and every entry equals the reference"""
    view = ps.debug_view()
    t = view["table"]
    assert t is not None, f"{what}: no count table"
    assert t["current"], f"{what}: table not current"
    lo = 0 if lo is None else lo
    hi = ps.size if hi is None else hi
    assert (t["lo"], t["hi"]) == (lo, hi), f"{what}: table rows [{t['lo']}, {t['hi']}), want [{lo}, {hi})"
    if layout is not None:
        assert t["layout"] == layout, f"{what}: layout {t['layout']}, want {layout}"
    rows = ps.to_numpy()[lo:hi]
    cnt, ln, nc = ref_counts(rows, masks, m, n_cases)
    assert t["counts"].shape == cnt.shape, what
    bad = np.argwhere(t["counts"].astype(np.int64) != cnt)
    assert bad.size == 0, f"{what}: {len(bad)} counts differ, first [row, half, perm] {bad[:6].tolist()}"
    assert np.array_equal(t["len"].astype(np.int64), ln), f"{what}: len differs"
    assert np.array_equal(t["ncase"].astype(np.int64), nc), f"{what}: ncase differs"
    return t


def check_lists(ps, n, n_cases, m, bits=None, what=""):
    """carrier lists against np.nonzero per half (of `bits`, default the set's rows): ascending, padded to 8 with the sentinel n,
    starts on 8-entry (16-byte) boundaries, ncase the prefix below n_cases"""
    lists = ps.debug_view()["lists"]
    assert lists is not None, f"{what}: no carrier lists"
    w64 = synth.words_for(n)
    rows = ps.to_numpy() if bits is None else bits
    off, car = lists["off"].astype(np.int64), lists["car"]
    assert off[0] == 0 and np.all(off % 8 == 0) and np.all(np.diff(off) >= 0), what
    for r in range(ps.size):
        for h, half in enumerate(_halves(rows[r:r + 1], m, w64)):
            want = np.nonzero(np.unpackbits(half.view(np.uint8), bitorder="little")[:n])[0]
            item = r * m + h
            seg = car[off[item]:off[item + 1]]
            k = want.shape[0]
            assert lists["len"][r, h] == k, f"{what}: row {r} half {h}: len {lists['len'][r, h]}, want {k}"
            assert seg.shape[0] == (k + 7) // 8 * 8, f"{what}: row {r} half {h}: list of {seg.shape[0]} entries for {k} carriers"
            assert np.array_equal(seg[:k], want), f"{what}: row {r} half {h}: carriers differ"
            assert np.all(seg[k:] == n), f"{what}: row {r} half {h}: padding is not the sentinel"
            assert lists["ncase"][r, h] == np.count_nonzero(want < n_cases), f"{what}: row {r} half {h}: ncase"


# ---- engine set-up --------------------------------------------------------------------------------------------------
def make_exec(engine, w, method, top_k=5, table=None):
    ex = engine.JoinExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.kernel = _lib.KERNEL_SPARSE
    ex.top_k = top_k
    ex.setValueTable(w.value_table if table is None else table)
    ex.setPermutedMasks(w.perm_masks)
    return ex


def uids(api, level, count=None, location=None):
    return api.UidRelSet(level.path_length, level.src, level.trg, level.count if count is None else count,
                         level.location if location is None else location, level.signs)


def run_keep_levels(engine, ex, w, partner_from_bits=False, uid_range3=None):
    """levels 1a, 2, 3 (the KEEP joins of the schedule) -> data1, {level: (result set, info)}"""
    lv, didx = w.net.levels, w.net.data_idx
    d1 = ex.createPathSet(w.net.n_genes)
    d1.load_bits(w.gene_bits)

    def partner(level):
        sel = d1.select(didx[level])
        if not partner_from_bits:
            return sel
        ps = ex.createPathSet(sel.size)  # the same rows, no selection behind them
        ps.load_bits(sel.to_numpy()[:, : synth.words_for(w.n_patients)])
        return ps

    out = {}
    p0 = ex.createPathSet(lv["1a"].n_uids)
    for name in ("1a", "2", "3"):
        res = ex.createPathSet(lv[name].n_pairs)
        rng = uid_range3 if name == "3" else None
        r = ex.join(uids(engine, lv[name]), p0, partner(name), res, uid_range=rng)
        out[name] = (res, r.info)
        p0 = res
    return d1, out


def workload(nc, nt, perms, seed, genes=120, edges=300, max_freq=0.12, zero_frac=0.3, length=5, real_table=True):
    return synth.make_workload(nc, nt, genes, edges, perms, seed=seed, max_path_length=length, real_table=real_table, max_freq=max_freq,
                               zero_frac=zero_frac)


# ---- 1. emitted tables of every KEEP join ---------------------------------------------------------------------------------
# form -> (environment, expected info, layout: "c16" = the 1,024-permutation image, "sc" = split carriers)
FORMS = {
    "delta": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_THR": "0"}, {"precounted": False, "split_carrier": False, "thresholded": False}, "c16"),
    "delta_thr": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_THR": "1"}, {"precounted": False, "split_carrier": False, "thresholded": True}, "c16"),
    "selection": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "1", "GCRE_THR": "0"}, {"precounted": True, "split_carrier": False, "thresholded": False}, "c16"),
    "selection_thr": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "1", "GCRE_THR": "1"}, {"precounted": True, "split_carrier": False, "thresholded": True}, "c16"),
    "pc_bits": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "1", "GCRE_THR": "0"}, {"precounted": True, "split_carrier": False}, "c16"),
    "pc_bits_thr": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "1", "GCRE_THR": "1"}, {"precounted": True, "split_carrier": False, "thresholded": True}, "c16"),
    "split": ({"GCRE_SC_PTS": "0"}, {"precounted": False, "split_carrier": True, "shared_masks": False}, "sc"),
    "split_pts": ({"GCRE_SC_PTS": "1"}, {"precounted": False, "split_carrier": True, "shared_masks": True}, "sc"),
    "delta_wide": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_TEST_WIDE_CARRIERS": "1"}, {"precounted": False, "split_carrier": False}, "c16"),
    "selection_wide": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "1", "GCRE_TEST_WIDE_CARRIERS": "1"}, {"precounted": True}, "c16"),
    "split_wide": ({"GCRE_SC_PTS": "0", "GCRE_TEST_WIDE_CARRIERS": "1"}, {"split_carrier": True}, "sc"),
    "selection_small_plan": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "1", "GCRE_TEST_SMALL_PLAN": "1"}, {"precounted": True}, "c16"),
}
PERMS_C16 = [1, 31, 32, 33, 129, 512, 513, 1024, 1025, 2100]
PERMS_SC = [1, 31, 32, 33, 128, 129, 257, 512]
# cohorts: n % 64 == 0 (W64 = 2), W64 = 9 (odd, padded to 10)
COHORTS = {"n128": (64, 64), "n557": (257, 300)}


def _sc_words(perms):
    return 4 if perms <= 128 else 8 if perms <= 256 else 16


def _cases():
    out = []
    for form, (_, _, layout) in FORMS.items():
        perms = PERMS_SC if layout == "sc" else PERMS_C16
        if form == "split_pts":
            perms = [1, 33, 128]
        elif form.endswith(("_wide", "_small_plan")) or form == "pc_bits_thr":
            perms = [33, 1025] if layout == "c16" else [129]
        for i, p in enumerate(perms):
            cohort = "n557" if i % 2 else "n128"
            if form == "split_pts":
                cohort = "n128"
            method = "method2" if (i // 2) % 2 == 0 else "method1"
            out.append(pytest.param(form, p, cohort, method, id=f"{form}-p{p}-{cohort}-{method}"))
    # both methods at the 1,024-permutation block boundary
    for form in ("delta", "selection", "selection_thr"):
        out.append(pytest.param(form, 1025, "n557", "method1", id=f"{form}-p1025-n557-method1-b"))
    out.append(pytest.param("split", 512, "n557", "method2", id="split-p512-n557-method2-b"))
    return out


def _set_form(monkeypatch, form):
    env, _, _ = FORMS[form]
    for k in ("GCRE_TEST_NO_SPLIT", "GCRE_TEST_PRECOUNT", "GCRE_THR", "GCRE_SC_PTS", "GCRE_TEST_WIDE_CARRIERS", "GCRE_TEST_SMALL_PLAN"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _assert_form(info, form, what):
    for k, v in FORMS[form][1].items():
        assert info[k] == v, f"{what}: info[{k}] = {info[k]}, want {v}"


@pytest.mark.parametrize("form,perms,cohort,method", _cases())
def test_emitted_tables(engine, form, perms, cohort, method, monkeypatch):
    """Levels 1a, 2 and 3: the table each KEEP join emits for its rows, every row, half and permutation"""
    _set_form(monkeypatch, form)
    nc, nt = COHORTS[cohort]
    w = workload(nc, nt, perms, seed=7100 + perms + nc)
    ex = make_exec(engine, w, method)
    m = ex.m
    _, out = run_keep_levels(engine, ex, w, partner_from_bits=form.startswith("pc_bits"))
    masks = ex.getPermutedMasks()
    layout = _sc_words(ex.iterations) if FORMS[form][2] == "sc" else 0
    for name, (res, info) in out.items():
        what = f"{form} p{perms} {cohort} {method} L{name}"
        if res.size == 0:
            continue
        _assert_form(info, form, what)
        check_table(res, masks, m, w.n_cases, layout=layout, what=what)


@pytest.mark.parametrize("form", ["delta", "selection", "split"])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_common_variant_tables(engine, form, method, monkeypatch):
    """Rows with more than 240 and more than 400 carriers per half: the bit planes flush mid-list and the filter queue drains
    several times per half"""
    _set_form(monkeypatch, form)
    perms = 300 if form == "split" else 1025
    w = workload(500, 600, perms, seed=7200, genes=50, edges=110, max_freq=0.45, zero_frac=0.1, length=3)
    ex = make_exec(engine, w, method)
    _, out = run_keep_levels(engine, ex, w)
    res3 = out["3"][0]
    rows = res3.to_numpy()
    w64 = synth.words_for(w.n_patients)
    assert max(np.bitwise_count(h).sum(axis=1).max() for h in _halves(rows, ex.m, w64)) > 400
    masks = ex.getPermutedMasks()
    for name, (res, info) in out.items():
        _assert_form(info, form, f"{form} {method} L{name}")
        check_table(res, masks, ex.m, w.n_cases, what=f"{form} {method} L{name}")


@pytest.mark.parametrize("form", ["delta", "selection", "split"])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_row_sharded_keep(engine, form, method, monkeypatch):
    """Level 3 over the middle third of its upstream rows: the table holds exactly that shard's result rows"""
    _set_form(monkeypatch, form)
    perms = 129 if form == "split" else 1025
    w = workload(257, 300, perms, seed=7300)
    ex = make_exec(engine, w, method)
    l3 = w.net.levels["3"]
    a, b = l3.n_uids // 3, (2 * l3.n_uids) // 3
    prefix = np.concatenate([[0], np.cumsum(l3.count.astype(np.int64))])
    _, out = run_keep_levels(engine, ex, w, uid_range3=(a, b))
    res, info = out["3"]
    _assert_form(info, form, f"{form} {method} shard")
    assert prefix[b] > prefix[a]
    check_table(res, ex.getPermutedMasks(), ex.m, w.n_cases, lo=int(prefix[a]), hi=int(prefix[b]), what=f"{form} {method} shard")


@pytest.mark.parametrize("method", ["method1", "method2"])
def test_precount_table_of_a_sharded_set(engine, oracles, method, monkeypatch):
    """A set whose emitted table holds one shard's rows is then a pre-counted partner (level 5 over paths3): its table must
    be rebuilt for every row, not taken as it is"""
    _set_form(monkeypatch, "selection")
    monkeypatch.setenv("GCRE_TEST_TAIL", "0")
    w = workload(257, 300, 1025, seed=7350)
    ex = make_exec(engine, w, method)
    l3, l5 = w.net.levels["3"], w.net.levels["5"]
    a, b = l3.n_uids // 3, (2 * l3.n_uids) // 3
    _, out = run_keep_levels(engine, ex, w, uid_range3=(a, b))
    p3 = out["3"][0]
    got = ex.join(uids(engine, l5), p3, p3, ex.createPathSet(0))
    assert got.info["precounted"]
    check_table(p3, ex.getPermutedMasks(), ex.m, w.n_cases, what=f"{method} paths3 after level 5")
    o = oracles.OracleExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    o.top_k = ex.top_k
    o.setValueTable(w.value_table)
    o.setPermutedMasks(w.perm_masks)
    o3 = o.createPathSet(p3.size)
    o3.rows[:] = p3.to_numpy()
    want = o.join(uids(oracles, l5), o3, o3, o.createPathSet(0))
    helpers.assert_same_results(got, want, what=f"{method} L5 over a sharded paths3")


def test_no_table_without_emit(engine, monkeypatch):
    _set_form(monkeypatch, "delta")
    monkeypatch.setenv("GCRE_TEST_EMIT", "0")
    w = workload(64, 64, 33, seed=7400)
    ex = make_exec(engine, w, "method2")
    _, out = run_keep_levels(engine, ex, w)
    for name, (res, _) in out.items():
        assert res.debug_view()["table"] is None, name


# ---- 2. pre-count tables and carrier lists ---------------------------------------------------------------------------------
@pytest.mark.parametrize("perms", [33, 1025])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_precount_table_follows_the_masks(engine, method, perms, monkeypatch):
    """data1's pre-count table after the joins that built it; stale once new masks are generated; rebuilt for them by the next
    join, whose emitted table follows the new masks too"""
    _set_form(monkeypatch, "selection")
    w = workload(257, 300, perms, seed=7500 + perms)
    ex = make_exec(engine, w, method)
    d1, out = run_keep_levels(engine, ex, w)
    assert out["3"][1]["precounted"]
    masks = ex.getPermutedMasks()
    check_table(d1, masks, ex.m, w.n_cases, layout=0, what="data1")
    check_lists(d1, w.n_patients, w.n_cases, ex.m, what="data1 lists")
    ex.generatePermutedMasks(seed=99, first_perm=5)
    assert not d1.debug_view()["table"]["current"]
    assert not out["3"][0].debug_view()["table"]["current"]
    new_masks = ex.getPermutedMasks()
    assert not np.array_equal(new_masks, masks)
    lv = w.net.levels
    res = ex.createPathSet(lv["3"].n_pairs)
    r = ex.join(uids(engine, lv["3"]), out["2"][0], d1.select(w.net.data_idx["3"]), res)
    assert r.info["precounted"]
    check_table(d1, new_masks, ex.m, w.n_cases, layout=0, what="data1 rebuilt")
    check_table(res, new_masks, ex.m, w.n_cases, layout=0, what="level 3 under new masks")


@pytest.mark.parametrize("wide", ["0", "1"])
@pytest.mark.parametrize("method", ["method1", "method2"])
@pytest.mark.parametrize("n_cases,n_ctrls", [(64, 64), (70, 33), (257, 300)])
def test_carrier_lists_with_dirty_bits(engine, method, n_cases, n_ctrls, wide, monkeypatch):
    """Lists of a partner set loaded with bits set at and beyond n: those bits are not carriers"""
    _set_form(monkeypatch, "delta")
    if wide == "1":
        monkeypatch.setenv("GCRE_TEST_WIDE_CARRIERS", "1")
    n = n_cases + n_ctrls
    w64 = synth.words_for(n)
    rng = np.random.default_rng(n + int(wide))
    rows = 40
    bits = synth.make_cohort_bits(n, rows, seed=n, max_freq=0.3, zero_frac=0.2)
    clean = bits.copy()
    dirty = bits.copy()
    if n % 64:
        dirty[:, -1] |= ~np.uint64((1 << (n % 64)) - 1)  # every bit at or beyond n
    masks = synth.make_perm_masks(n_cases, n_ctrls, 40, seed=3)
    ex = engine.JoinExec(method, n_cases, n_ctrls, 40)
    ex.kernel = _lib.KERNEL_SPARSE
    ex.setValueTable(synth.make_value_table(n_cases, n_ctrls))
    ex.setPermutedMasks(masks)
    partner = ex.createPathSet(rows)
    if method == "method1":
        partner.load_bits(dirty)
    else:
        for r in range(rows):  # [pos | neg], both halves dirty
            partner.set(r, np.concatenate([dirty[r], dirty[(r + 7) % rows]]))
        clean = np.concatenate([clean, clean[(np.arange(rows) + 7) % rows]], axis=1)
    up = ex.createPathSet(rows)
    u = engine.UidRelSet(2, np.arange(rows), np.arange(rows), np.ones(rows), np.arange(rows, dtype=np.uint32), np.ones(rows))
    ex.join(u, up, partner, ex.createPathSet(0))
    check_lists(partner, n, n_cases, ex.m, bits=clean, what=f"{method} n={n} wide={wide}")
    assert np.array_equal(partner.to_numpy(), clean)


# ---- 3. hand-built unit: runs of empty partners ------------------------------------------------------------------------------
@pytest.mark.parametrize("form", ["delta", "delta_thr", "pc_bits", "pc_bits_thr", "split"])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_runs_of_empty_partners(engine, form, method, monkeypatch):
    """Partners that add no carrier to their upstream row (zero rows, subsets of it) in runs between ones that do, oriented
    both ways: a partner skipped as empty emits the base's counts"""
    _set_form(monkeypatch, form)
    nc, nt, perms = 70, 63, (100 if form == "split" else 1025)
    n, w64 = nc + nt, synth.words_for(nc + nt)
    rng = np.random.default_rng(11)
    m = 1 if method == "method1" else 2
    n_up, per = 6, 24
    # method 2 upstream rows [A, A | B]: a partner whose halves are subsets of A adds nothing in either orientation
    a_bits = synth.make_cohort_bits(n, n_up, seed=5, max_freq=0.3, zero_frac=0.0)
    up_bits = a_bits if m == 1 else np.concatenate([a_bits, a_bits | synth.make_cohort_bits(n, n_up, seed=6, max_freq=0.2, zero_frac=0.0)], axis=1)
    partners = np.zeros((n_up * per, m * w64), dtype=np.uint64)
    for u in range(n_up):
        for j in range(per):
            kind = j % 6  # 0, 5: new carriers; 1, 2: zero rows; 3, 4: subsets of the upstream row
            if kind in (0, 5):
                partners[u * per + j] = synth.make_cohort_bits(n, m, seed=100 * u + j, max_freq=0.2, zero_frac=0.0).reshape(-1)
            elif kind in (3, 4):
                keep = rng.integers(0, 2**63, size=m * w64, dtype=np.uint64)
                partners[u * per + j] = np.tile(a_bits[u], m) & keep
    signs = np.where(rng.random(n_up * per) < 0.5, 1, -1).astype(np.int32)
    masks = synth.make_perm_masks(nc, nt, perms, seed=9)
    ex = engine.JoinExec(method, nc, nt, perms)
    ex.kernel = _lib.KERNEL_SPARSE
    ex.setValueTable(synth.make_value_table(nc, nt))
    ex.setPermutedMasks(masks)
    p0, p1 = ex.createPathSet(n_up), ex.createPathSet(n_up * per)
    for r in range(n_up):
        p0.set(r, up_bits[r])
    for r in range(n_up * per):
        p1.set(r, partners[r])
    count = np.full(n_up, per, dtype=np.int32)
    loc = (np.arange(n_up) * per).astype(np.uint32)
    u = engine.UidRelSet(2, np.arange(n_up), np.arange(n_up), count, loc, signs)
    res = ex.createPathSet(n_up * per)
    r = ex.join(u, p0, p1, res)
    _assert_form(r.info, form, f"{form} {method}")
    check_table(res, ex.getPermutedMasks(), m, nc, what=f"{form} {method}")


# ---- 4. per-pair values of score-only joins ------------------------------------------------------------------------------------
PAIR_FORMS = {
    "delta": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_THR": "0", "GCRE_TEST_TAIL": "0"}, {"precounted": False, "tail_form": False, "thresholded": False, "split_carrier": False}),
    "pc": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "1", "GCRE_THR": "0", "GCRE_TEST_TAIL": "0"}, {"precounted": True, "tail_form": False, "thresholded": False}),
    "tail": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_THR": "0", "GCRE_TEST_TAIL": "1"}, {"tail_form": True, "thresholded": False}),
    "thr": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_THR": "1", "GCRE_TEST_TAIL": "0"}, {"precounted": False, "thresholded": True}),
    "pc_thr": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "1", "GCRE_THR": "1", "GCRE_TEST_TAIL": "0"}, {"precounted": True, "thresholded": True}),
    "tail_thr": ({"GCRE_TEST_NO_SPLIT": "1", "GCRE_TEST_PRECOUNT": "0", "GCRE_THR": "1", "GCRE_TEST_TAIL": "1"}, {"tail_form": True, "thresholded": True}),
    "split": ({"GCRE_SC_PTS": "0", "GCRE_TEST_PRECOUNT": "0", "GCRE_TEST_TAIL": "0"}, {"split_carrier": True}),
}
PAIRS_PER_LEVEL = 30


def _one_pair_uids(api, level, u, j):
    """the level's UidRelSet with every uid emptied (count 0, location -1) except uid u, which keeps its j-th partner only"""
    count = np.zeros_like(level.count)
    location = np.full_like(level.location, NONE)
    count[u] = 1
    location[u] = level.location[u] + j
    return uids(api, level, count, location)


def _sample_pairs(level, k, rng):
    live = np.nonzero(level.count > 0)[0]
    us = rng.choice(live, size=min(k, live.shape[0]), replace=False)
    return [(int(u), int(rng.integers(0, level.count[u]))) for u in us]


@pytest.mark.parametrize("table", ["real", "test", "injective"])
@pytest.mark.parametrize("form", list(PAIR_FORMS))
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_single_pair_joins(engine, oracles, method, form, table, monkeypatch):
    """Joins that hold one pair: the permutation maxima are that pair's own values, compared bit for bit with the oracle (and,
    with vt[x][y] = x + 1, with the pair's exact counts)"""
    if table == "injective" and method == "method2":
        pytest.skip("the injective table reads back counts through method 1's single look-up")
    env, want_info = PAIR_FORMS[form]
    for k in ("GCRE_TEST_NO_SPLIT", "GCRE_SC_PTS"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    perms = 257 if form == "split" else 1025
    w = workload(257, 300, perms, seed=7600 + perms, genes=150, edges=420, real_table=True)
    if table == "test":
        vt = synth.make_test_table(w.n_cases, w.n_ctrls, seed=5)
    elif table == "injective":
        vt = np.repeat(np.arange(1, w.n_cases + 2, dtype=np.float64)[:, None], w.n_ctrls + 1, axis=1)
    else:
        vt = w.value_table
    ex = make_exec(engine, w, method, table=vt)
    lv = w.net.levels
    # kept sets built with the tail and pre-count hooks off (the engine's own choice of form)
    with monkeypatch.context() as mp:
        for k in ("GCRE_TEST_PRECOUNT", "GCRE_THR", "GCRE_TEST_TAIL"):
            mp.delenv(k, raising=False)
        d1, out = run_keep_levels(engine, ex, w)
    p2, p3 = out["2"][0], out["3"][0]
    d2 = ex.createPathSet(w.gene_bits2.shape[0])
    d2.load_bits(w.gene_bits2)
    sets = {"1b": (ex.createPathSet(lv["1b"].n_uids), d2.select(w.net.data_idx["1b"])), "4": (p3, p2), "5": (p3, p3)}
    levels = ["4"] if form.startswith("tail") else ["1b", "4", "5"]

    o = oracles.OracleExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    o.setValueTable(vt)
    o.setPermutedMasks(ex.getPermutedMasks())
    masks = ex.getPermutedMasks()
    rng = np.random.default_rng(zlib.crc32(f"{method} {form} {table}".encode()))
    zero = ex.createPathSet(0)
    w64 = synth.words_for(w.n_patients)
    for name in levels:
        level = lv[name]
        s0, s1 = sets[name]
        r0, r1 = s0.to_numpy(), s1.to_numpy()
        o0, o1 = o.createPathSet(r0.shape[0]), o.createPathSet(r1.shape[0])
        o0.rows[:], o1.rows[:] = r0, r1
        for u, j in _sample_pairs(level, PAIRS_PER_LEVEL, rng):
            what = f"{method} {form} {table} L{name} uid {u} partner {j}"
            got = ex.join(_one_pair_uids(engine, level, u, j), s0, s1, zero)
            assert got.info["pairs"] == 1, what
            for k, v in want_info.items():
                assert got.info[k] == v, f"{what}: info[{k}] = {got.info[k]}, want {v}"
            want = o.join(_one_pair_uids(oracles, level, u, j), o0, o1, o.createPathSet(0))
            helpers.assert_same_results(got, want, what=what)
            if table == "injective":
                joined = r0[u] | r1[int(level.location[u]) + j]
                cnt, _, _ = ref_counts(joined[None, :w64], masks, 1, w.n_cases)
                assert np.array_equal(np.asarray(got.permuted_scores) - 1.0, cnt[0, 0].astype(np.float64)), what
