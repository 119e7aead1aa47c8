"""CPU tests of bench.py --dump-outputs: the dumped maxima are the real permutations of every batch and rank, never the
kernels' padded slots, and an oversized dump keeps the same seeded sample of every block."""
import numpy as np

import bench
from geneticscre_b200.api import Score, joined_res

WORLD, N_BATCHES, IP, BATCH, N_PERMS = 2, 2, 640, 600, 1000  # batch 1 holds 400 real permutations; ip pads to the 128-wide tile


def fake_perm_all():
    """[rank][batch][ip] with value rank * 10,000 + permutation index in real slots and -1 in padded ones."""
    v = np.full((WORLD, N_BATCHES, IP), -1.0, dtype=np.float32)
    for r in range(WORLD):
        for b in range(N_BATCHES):
            nb = min(BATCH, N_PERMS - b * BATCH)
            v[r, b, :nb] = r * 10000 + b * BATCH + np.arange(nb)
    return v.reshape(-1)


def fake_step():
    """run_batches' return for one method: per level, each batch's maxima (already cut to its real permutations)."""
    top = [Score(float("-inf"), -1, -1, 0, 0), Score(2.5, 3, 4, 5, 6)]
    res = {k: joined_res(top, np.zeros(BATCH)) for k in ("1b", "2", "3", "4")}
    parts = {k: [np.arange(BATCH, dtype=np.float64), BATCH + np.arange(N_PERMS - BATCH, dtype=np.float64)] for k in res}
    return ({}, res, res, parts)


def test_device_perm_max_drops_padding():
    got = bench.device_perm_max(fake_perm_all(), WORLD, N_BATCHES, IP, BATCH, N_PERMS)
    want = np.concatenate([r * 10000 + np.arange(N_PERMS) for r in range(WORLD)]).astype(np.float64)
    assert got.dtype == np.float64 and np.array_equal(got, want)


def test_dump_outputs_writes_real_permutations(tmp_path):
    last_out = {"method1": fake_step(), "method2": fake_step()}
    last_perm = {"method1": bench.device_perm_max(fake_perm_all(), WORLD, N_BATCHES, IP, BATCH, N_PERMS)}
    bench.dump_outputs(str(tmp_path), last_out, ["1a", "1b", "2", "3", "4"], last_perm, N_PERMS)
    names = sorted(p.name for p in tmp_path.iterdir())
    assert names == sorted(f"{m}_level{k}_{kind}.npy" for m in ("method1", "method2") for k in ("1b", "2", "3", "4") for kind in ("perm_max", "topk"))
    assert np.array_equal(np.load(tmp_path / "method1_level4_perm_max.npy"), last_perm["method1"])
    for m, k in (("method1", "3"), ("method2", "4")):
        assert np.array_equal(np.load(tmp_path / f"{m}_level{k}_perm_max.npy"), np.arange(N_PERMS, dtype=np.float64))
    top = np.load(tmp_path / "method2_level2_topk.npy")
    assert top.dtype == np.float64 and top.shape == (2, 5) and top[0, 0] == -np.inf and list(top[1]) == [2.5, 3, 4, 5, 6]


def test_oversized_dump_keeps_one_sample_of_every_block(tmp_path):
    last_out = {"method1": fake_step()}
    last_perm = {"method1": bench.device_perm_max(fake_perm_all(), WORLD, N_BATCHES, IP, BATCH, N_PERMS)}
    limit = 2 * 8 * 5 * N_PERMS // 4  # maxima of 5 blocks (1b, 2, 3 and the two ranks of 4) -> a quarter of them kept
    bench.dump_outputs(str(tmp_path), last_out, ["1b", "2", "3", "4"], last_perm, N_PERMS, limit=limit)
    keep = np.load(tmp_path / "perm_sample_index.npy").astype(np.int64)
    assert keep.size == N_PERMS // 4 and np.all(np.diff(keep) > 0) and keep.max() < N_PERMS
    assert np.array_equal(np.load(tmp_path / "method1_level2_perm_max.npy"), keep.astype(np.float64))
    last = np.load(tmp_path / "method1_level4_perm_max.npy")
    assert np.array_equal(last, np.concatenate([r * 10000 + keep for r in range(WORLD)]).astype(np.float64))
    bench.dump_outputs(str(tmp_path / "again"), last_out, ["1b", "2", "3", "4"], last_perm, N_PERMS, limit=limit)
    assert np.array_equal(np.load(tmp_path / "again" / "perm_sample_index.npy"), keep.astype(np.float64))
