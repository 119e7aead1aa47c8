"""Cost of decorated p-values for whole top-K lists on the device (gcre_exec_decorated_paths, csrc/decorated.cuh) against the host
implementation (decorated.decorated_pvalues_for_path) on the same splits.  Writes one JSON.

    python tools/decorated_timing.py --out profiles/r8_decorated.json

* cohort: config 3 (5,000 cases + 5,000 controls, 15,000 genes, 150,000 edges), value table from generateValueTable, seed of
  bench.py.  Levels 2-4 are replayed with top_k = 1,000 per method: 1,000 paths of each length, 12,000 splits per method.
* device: the whole list in one call, gene rows resident (a path set loaded once, as data1 is during a run), no strata and 16
  random strata (setPermutationStrata).  CUDA events on the exec's stream around `reps` calls after one warm-up call; the call
  ends in a host wait, so the events span everything it does (split forming, count pass, read-back of the sizes, joint kernels).
* host: decorated_pvalues_for_path per path on a seeded sample of the same paths (exact mode, with and without the same strata);
  the time per split is scaled to the 12,000 splits.  The sample's device values are compared with the host's (max relative
  difference of the p-values; scores and counts must be equal).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LEVELS = ("2", "3", "4")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:  # informational only
        return None


def time_device(ex, gs, genes, signs, lengths, stratified, reps, stream):
    """ms per call of gcre_exec_decorated_paths over the whole list (CUDA events, mean of `reps` calls after a warm-up)."""
    import torch

    from geneticscre_b200 import _lib

    k = lengths.shape[0]
    out = (_lib.DecoratedC * (8 * k))()
    i32 = C.POINTER(C.c_int32)
    args = (ex._h, gs._h, genes.ctypes.data_as(i32), signs.ctypes.data_as(i32), lengths.ctypes.data_as(i32), k, int(stratified), out)
    _lib.check(ex._lib.gcre_exec_decorated_paths(*args))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t = time.perf_counter()
    e0.record(stream)
    for _ in range(reps):
        _lib.check(ex._lib.gcre_exec_decorated_paths(*args))
    e1.record(stream)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t) * 1e3 / reps
    return e0.elapsed_time(e1) / reps, wall


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--top-k", type=int, default=1000)
    ap.add_argument("--host-paths", type=int, default=60, help="paths per method whose splits the host computes")
    ap.add_argument("--strata", type=int, default=16)
    a = ap.parse_args()
    import torch

    from bench import WORKLOAD as W
    from geneticscre_b200 import api, build, decorated, schedule, synth

    build.build()
    gpu = gpu_info()
    w = synth.make_workload(W["n_cases"], W["n_ctrls"], W["n_genes"], W["n_edges"], 100, W["seed"], max_path_length=4, host_table=False)
    n = w.n_patients
    rows = synth.unpack_bits(w.gene_bits, n).astype(bool)
    labels = np.random.default_rng(W["seed"]).integers(0, a.strata, n).astype(np.int32)
    stream = torch.cuda.Stream()  # not the default stream: its handle is 0, which set_stream reads as "the exec's own stream"
    result = {"gpu": gpu, "cohort": {"n_cases": W["n_cases"], "n_ctrls": W["n_ctrls"], "n_genes": W["n_genes"], "n_edges": W["n_edges"],
                                     "seed": W["seed"], "value_table": "generateValueTable"},
              "top_k": a.top_k, "levels": list(LEVELS), "strata": a.strata, "reps": a.reps, "methods": {}}
    for method in (1, 2):
        ex = api.JoinExec("method1" if method == 1 else "method2", w.n_cases, w.n_ctrls, w.n_perms)
        ex.set_stream(stream.cuda_stream)
        ex.top_k = a.top_k
        ex.generateValueTable()
        ex.setPermutedMasks(w.perm_masks)
        res, _ = schedule.replay_levels(ex, api.UidRelSet, w, 4)
        parts = []
        for lv in LEVELS:
            sc = [s for s in res[lv].scores if s.src >= 0]
            parts.append(synth.path_genes(w.net, lv, [s.src for s in sc], [s.trg for s in sc]))
        genes = np.ascontiguousarray(np.concatenate([p[0] for p in parts]))
        signs = np.ascontiguousarray(np.concatenate([p[1] for p in parts]))
        lengths = np.ascontiguousarray(np.concatenate([p[2] for p in parts]))
        n_splits = int((2 * (lengths - 1)).sum())
        gs = ex.createPathSet(w.gene_bits.shape[0])
        gs.load_bits(w.gene_bits)
        vt = ex.getValueTable()
        row = {"paths": int(lengths.shape[0]), "splits": n_splits}
        sample = np.random.default_rng(1).choice(lengths.shape[0], size=min(a.host_paths, lengths.shape[0]), replace=False)
        for stratified in (False, True):
            ex.setPermutationStrata(labels if stratified else None)
            ev_ms, wall_ms = time_device(ex, gs, genes, signs, lengths, stratified, a.reps, stream)
            dev = decorated.decorated_pvalues_device(ex, gs, genes[sample], signs[sample], lengths[sample], stratified=stratified)
            t = time.perf_counter()
            host = [decorated.decorated_pvalues_for_path(rows[genes[i, :lengths[i]]], signs[i, :lengths[i]], w.n_cases, w.n_ctrls, method, vt,
                                                         strata=labels if stratified else None) for i in sample]
            host_s = time.perf_counter() - t
            host_splits = sum(len(h) for h in host)
            worst, same = 0.0, True
            for d, h in zip(dev, host):
                for x, y in zip(d, h):
                    same &= (x["score"], x["cases1"], x["controls1"], x["cases2"], x["controls2"]) == (y["score"], y["cases1"], y["controls1"], y["cases2"], y["controls2"])
                    worst = max(worst, abs(x["decorated_pvalue"] - y["decorated_pvalue"]) / max(y["decorated_pvalue"], 1e-300))
            host_ms_per_split = host_s * 1e3 / max(host_splits, 1)
            key = f"strata_{a.strata}" if stratified else "no_strata"
            row[key] = {"device_ms": round(ev_ms, 3), "device_wall_ms": round(wall_ms, 3), "device_us_per_split": round(ev_ms * 1e3 / n_splits, 3),
                        "host_splits_timed": host_splits, "host_ms_per_split": round(host_ms_per_split, 4),
                        "host_ms_all_splits_scaled": round(host_ms_per_split * n_splits, 1),
                        "host_over_device": round(host_ms_per_split * n_splits / ev_ms, 1),
                        "sample_scores_and_counts_equal": bool(same), "sample_max_rel_diff_pvalue": worst}
            print(json.dumps({"method": method, key: row[key]}), flush=True)
        ex.setPermutationStrata(None)
        result["methods"][f"method{method}"] = row
        ex.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
