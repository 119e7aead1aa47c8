"""Seeded permutation masks made on the device (gcre_exec_generate_permuted_masks, csrc/perm_gen.cuh): bit for bit the numpy
restatement synth.make_perm_masks_philox at every shape edge, strata included; the level schedule against generated masks equals
the schedule against the same masks uploaded from the host and the CPU oracle under every kernel form; count tables kept from
older masks are never reused; batched generation equals one exec holding every permutation; the C++ class layer, on one GPU
and on two."""
import os
import subprocess

import numpy as np
import pytest

import helpers
from geneticscre_b200 import _lib, schedule, synth
from test_join_gpu import KERNELS, SHAPES, _precount_mode  # noqa: F401  (_precount_mode: the env knobs of each kernel form)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRATA_LIMIT = 1024
SEED = 0x9E3779B97F4A7C15


class _Tail(int):
    """KERNEL_SPARSE with the tail form of the level-4 join forced on (GCRE_TEST_TAIL=1, one-word-per-lane kernel)."""


FORMS = KERNELS + [pytest.param(_Tail(_lib.KERNEL_SPARSE), id="sparse_tail")]


def _form_env(kernel, monkeypatch):
    if isinstance(kernel, _Tail):
        monkeypatch.setenv("GCRE_TEST_TAIL", "1")
        monkeypatch.setenv("GCRE_TEST_NO_SPLIT", "1")


def labels_for(n, kind, seed=0):
    """kind distinct, arbitrary int32 labels over n patients (None: no strata)"""
    if kind is None:
        return None
    rng = np.random.default_rng(seed + kind)
    values = rng.choice(np.arange(-5 * kind, 5 * kind, dtype=np.int64), size=kind, replace=False).astype(np.int32)
    return values[rng.permutation(np.arange(n) % kind)]


def check_counts(masks, nc, n, labels):
    case = np.unpackbits(masks.view(np.uint8), axis=1, bitorder="little")
    assert not case[:, n:].any(), "bits at patient indices >= n"
    case = case[:, :n].astype(bool)
    lab = np.zeros(n, np.int32) if labels is None else labels
    for g in np.unique(lab):
        sel = lab == g
        assert (case[:, sel].sum(1) == sel[:nc].sum()).all(), f"stratum {g} lost its case count"


# (n_cases, n_ctrls) x iterations x strata x first_perm: every n with several iteration counts, strata and first_perm
# cycling over their values; fewer permutations at the large sizes
FIRSTS = [0, 2**32 - 3, 2**40]
GRID = [((1, 1), (1, 100, 1025)), ((30, 33), (128, 1000, 4096)), ((32, 32), (1, 1025, 4096)), ((1, 64), (100, 128)),
        ((70, 130), (1, 100, 128, 1000, 1025, 4096)), ((5000, 5000), (1000, 4096)), ((30000, 35537), (1, 100)),
        ((50000, 50000), (128, 1025))]
CASES = []
for (_nc, _nt), _iters_list in GRID:
    for _iters in _iters_list:
        _kinds = [k for k in (None, 2, 37, STRATA_LIMIT) if k is None or k <= _nc + _nt]
        _s, _f = _kinds[len(CASES) % len(_kinds)], len(CASES) % 3
        CASES.append(pytest.param(_nc, _nt, _iters, _s, FIRSTS[_f], id=f"n{_nc + _nt}-i{_iters}-s{_s}-f{_f}"))
CASES += [pytest.param(5000, 5000, 1000, STRATA_LIMIT, FIRSTS[2], id="n10000-i1000-s1024-f2"),
          pytest.param(50000, 50000, 128, STRATA_LIMIT, FIRSTS[1], id="n100000-i128-s1024-f1")]


@pytest.mark.parametrize("nc,nt,iters,strata,first", CASES)
def test_device_masks_match_restatement(engine, nc, nt, iters, strata, first):
    n = nc + nt
    labels = labels_for(n, strata)
    ex = engine.JoinExec("method1", nc, nt, iters)
    if labels is not None:
        ex.setPermutationStrata(labels)
    ex.generatePermutedMasks(SEED, first)
    got = ex.getPermutedMasks()
    assert got.shape == (iters, synth.words_for(n))
    check_counts(got, nc, n, labels)
    if iters * n <= 4_000_000:
        rows = [(0, iters)]
    else:  # both ends of the exec, the restatement computes any range of permutations directly
        rows = [(0, 16), (iters // 2, 8), (iters - 16, 16)] if iters > 32 else [(0, iters)]
    for r0, cnt in rows:
        want = synth.make_perm_masks_philox(nc, nt, cnt, SEED, first_perm=first + r0, strata=labels)
        bad = np.nonzero((got[r0 : r0 + cnt] != want).any(axis=1))[0]
        assert bad.size == 0, f"rows {r0 + bad[:8]} differ"


def test_strata_setting_rules(engine):
    nc, nt = 600, 700
    n = nc + nt
    ex = engine.JoinExec("method2", nc, nt, 33)
    labels = labels_for(n, 37)
    ex.setPermutationStrata(labels)
    ex.generatePermutedMasks(7, 5)
    want = synth.make_perm_masks_philox(nc, nt, 33, 7, first_perm=5, strata=labels)
    assert np.array_equal(ex.getPermutedMasks(), want)
    ex.setPermutationStrata(np.arange(n) % 3)
    assert np.array_equal(ex.getPermutedMasks(), want), "setting strata must not change the current masks"
    with pytest.raises(_lib.GcreOutOfRange):  # beyond the limit; the setting stays as it was
        ex.setPermutationStrata(np.arange(n) % (STRATA_LIMIT + 1))
    ex.generatePermutedMasks(7, 5)
    assert np.array_equal(ex.getPermutedMasks(), synth.make_perm_masks_philox(nc, nt, 33, 7, first_perm=5, strata=np.arange(n) % 3))
    with pytest.raises(_lib.GcreAssertion):
        ex.setPermutationStrata(np.zeros(n - 1, np.int32))
    with pytest.raises(_lib.GcreOutOfRange):
        ex.getPermutedMasks(34)
    relabelled = (np.arange(n) % 3) * -11 + 4
    ex.setPermutationStrata(relabelled)
    ex.generatePermutedMasks(7, 5)
    assert np.array_equal(ex.getPermutedMasks(), synth.make_perm_masks_philox(nc, nt, 33, 7, first_perm=5, strata=np.arange(n) % 3))
    ex.setPermutationStrata(None)
    ex.generatePermutedMasks(7, 5)
    assert np.array_equal(ex.getPermutedMasks(), synth.make_perm_masks_philox(nc, nt, 33, 7, first_perm=5))
    assert np.array_equal(ex.getPermutedMasks(3), synth.make_perm_masks_philox(nc, nt, 3, 7, first_perm=5))
    zero = engine.JoinExec("method1", nc, nt, 0)
    zero.generatePermutedMasks(7)  # nothing to do
    assert zero.getPermutedMasks().shape == (0, synth.words_for(n))


def test_int_matrix_masks_are_inspectable(engine):
    w = synth.make_workload(40, 57, 30, 60, 70, seed=3, max_path_length=3)
    bits = np.unpackbits(w.perm_masks.view(np.uint8), axis=1, bitorder="little")[:, :97].astype(bool)
    is_case = np.arange(97) < 40
    ex = engine.JoinExec("method1", 40, 57, 70)
    ex.setPermutedCases((bits == is_case[None, :]).astype(np.int32))
    assert np.array_equal(ex.getPermutedMasks(), w.perm_masks)


def _workload(shape, seed, strata=None, first=0):
    nc, nt, g, e, perms, top_k = shape
    w = synth.make_workload(nc, nt, g, e, perms, seed=seed, max_path_length=5, real_table=(nc % 2 == 0), max_freq=0.12, zero_frac=0.3)
    w.perm_masks = synth.make_perm_masks_philox(nc, nt, perms, SEED, first_perm=first, strata=strata)
    return w, top_k


def _engine_exec(engine, kernel):
    class Exec(engine.JoinExec):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.kernel = kernel

    return Exec


@pytest.mark.parametrize("kernel", FORMS)
@pytest.mark.parametrize("method", ["method1", "method2"])
@pytest.mark.parametrize("shape,strata", [(SHAPES[1], None), (SHAPES[4], 5)])
def test_schedule_on_generated_masks(engine, oracles, method, shape, strata, kernel, monkeypatch):
    _form_env(kernel, monkeypatch)
    n = shape[0] + shape[1]
    labels = labels_for(n, strata)
    first = 2**32 - 100
    w, top_k = _workload(shape, seed=2000 + n, strata=labels, first=first)
    want, kept_want, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 5, top_k)
    host, _, _ = helpers.run_schedule(_engine_exec(engine, kernel), engine.UidRelSet, w, method, 5, top_k)
    ex = _engine_exec(engine, kernel)(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    if labels is not None:
        ex.setPermutationStrata(labels)
    ex.generatePermutedMasks(SEED, first)
    assert np.array_equal(ex.getPermutedMasks(), w.perm_masks)
    got, kept = schedule.replay_levels(ex, engine.UidRelSet, w, 5)
    for k in kept_want:
        assert np.array_equal(kept[k].to_numpy(), kept_want[k]), f"kept {k} differs"
    for lvl in want:
        helpers.assert_same_results(got[lvl], want[lvl], what=f"{method} L{lvl} vs oracle")
        helpers.assert_same_results(got[lvl], host[lvl], what=f"{method} L{lvl} vs host masks")
        assert got[lvl].info["kernel"] == kernel
    if isinstance(kernel, _Tail):
        assert got["4"].info["tail_form"]


@pytest.mark.parametrize("form", ["precount", "tail"])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_regenerated_masks_drop_kept_counts(engine, oracles, method, form, monkeypatch):
    """Levels 1a-3 hand count tables to level 4 (pre-counted form, or the tail form's gene-row counts); regenerating the masks
    in between must make level 4 count against the new masks."""
    monkeypatch.setenv("GCRE_TEST_NO_SPLIT", "1")
    monkeypatch.setenv("GCRE_THR", "0")
    monkeypatch.setenv("GCRE_SC_PTS", "0")
    monkeypatch.setenv("GCRE_TEST_PRECOUNT", "1" if form == "precount" else "0")
    if form == "tail":
        monkeypatch.setenv("GCRE_TEST_TAIL", "1")
    shape = SHAPES[4]
    w, top_k = _workload(shape, seed=4300, first=0)
    w_new = synth.Workload(w.n_cases, w.n_ctrls, w.n_perms, w.gene_bits, w.gene_bits2,
                           synth.make_perm_masks_philox(w.n_cases, w.n_ctrls, w.n_perms, SEED, first_perm=2**40), w.value_table, w.net)
    want_old, _, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, method, 4, top_k)
    want_new, _, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w_new, method, 4, top_k)
    ex = _engine_exec(engine, _lib.KERNEL_SPARSE)(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    ex.generatePermutedMasks(SEED, 0)

    def regenerate(name, _):
        if name == "3":
            ex.generatePermutedMasks(SEED, 2**40)

    got, _ = schedule.replay_levels(ex, engine.UidRelSet, w, 4, on_level=regenerate)
    for lvl in ("1a", "1b", "2", "3"):
        helpers.assert_same_results(got[lvl], want_old[lvl], what=f"{method} L{lvl}")
    helpers.assert_same_results(got["4"], want_new["4"], what=f"{method} L4 after regeneration")
    assert got["4"].info["precounted" if form == "precount" else "tail_form"]
    assert not (np.asarray(got["4"].permuted_scores) == np.asarray(want_old["4"].permuted_scores)).all()


@pytest.mark.parametrize("per", [100, 257])
@pytest.mark.parametrize("method", ["method1", "method2"])
def test_replay_permutation_batches_equals_one_exec(engine, method, per):
    shape = SHAPES[3]
    nc, nt = shape[0], shape[1]
    w, top_k = _workload(shape, seed=4400)
    total, first = 3 * per - 7, 2**32 - per
    ex = engine.JoinExec(method, nc, nt, per)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    got = schedule.replay_permutation_batches(ex, engine.UidRelSet, w, 5, total, SEED, first_perm=first)
    one = engine.JoinExec(method, nc, nt, total)
    one.top_k = top_k
    one.setValueTable(w.value_table)
    one.generatePermutedMasks(SEED, first)
    want, _ = schedule.replay_levels(one, engine.UidRelSet, w, 5)
    assert set(got) == set(want)
    for lvl in want:
        helpers.assert_same_results(got[lvl], want[lvl], what=f"{method} L{lvl} batches of {per}")


def test_generation_on_caller_stream(engine, oracles):
    """Generated on a caller's stream that is still busy, then joined with no host synchronisation in between."""
    import torch

    shape = SHAPES[4]
    w, top_k = _workload(shape, seed=4500, first=77)
    want, _, _ = helpers.run_schedule(oracles.OracleExec, oracles.UidRelSet, w, "method2", 4, top_k)
    stream = torch.cuda.Stream()
    ex = engine.JoinExec("method2", w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.set_stream(stream.cuda_stream)
    ex.setValueTable(w.value_table)
    with torch.cuda.stream(stream):
        torch.cuda._sleep(20_000_000)  # the stream is busy for ~10 ms when the generation is queued behind it
    ex.generatePermutedMasks(SEED, 77)
    got, _ = schedule.replay_levels(ex, engine.UidRelSet, w, 4)
    for lvl in want:
        helpers.assert_same_results(got[lvl], want[lvl], what=f"L{lvl}")
    ex.set_stream(None)


def _build_kat(tmp_path):
    exe = str(tmp_path / "perm_gen_kat")
    lib_dir = os.path.join(ROOT, "geneticscre_b200")
    subprocess.check_call(["g++", "-std=c++11", "-O1", "-pthread", "-I", os.path.join(ROOT, "include", "gcre"),
                           os.path.join(ROOT, "tests", "cpp", "perm_gen_kat.cpp"), "-L", lib_dir, "-lgcre_b200",
                           f"-Wl,-rpath,{lib_dir}", "-o", exe])
    return exe


def _run_kat(exe, gpus):
    env = {k: v for k, v in os.environ.items() if k not in ("GCRE_DEVICES", "GCRE_DEVICE")}
    env["GCRE_GPUS"] = str(gpus)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "perm gen: OK" in out.stdout
    return [line for line in out.stdout.splitlines() if line.startswith("join:")]


def test_cpp_known_answers(tmp_path, engine):
    lines = _run_kat(_build_kat(tmp_path), 1)
    assert len(lines) == 2


def test_cpp_two_gpus_match_one(tmp_path, engine):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    exe = _build_kat(tmp_path)
    assert _run_kat(exe, 2) == _run_kat(exe, 1)
