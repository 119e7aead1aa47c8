"""Cost of the seeded permutation-mask generator (gcre_exec_generate_permuted_masks, csrc/perm_gen.cuh) against building the
same number of masks on the host (synth.make_perm_masks), and a byte-identity check on bench.py's workload.  Writes one JSON.

    python tools/perm_gen_timing.py --out profiles/r4_perm_gen.json

* device: CUDA events around `reps` generator calls on one stream (the call includes the rebuild of the word-major mask layout,
  masks_to_word_major_kernel); the generator kernel alone and the layout rebuild alone from torch.profiler over the same calls.
  The masks are written, never read back, and at most 26 MB: they stay in L2 between calls, as they do between batches of a job.
* host: synth.make_perm_masks (one rng.permutation per mask).  Shapes that would take minutes are sampled: `host_perms_timed`
  masks are timed and the time is scaled to the shape (`host_scaled`: true).
* bench workload (bench.py's WORKLOAD: config 3, methods 1 + 2): replays of the level schedule (schedule.replay_levels, inputs
  uploaded inside the step) after generatePermutedMasks(seed) and after setPermutedMasks(make_perm_masks_philox(seed)); top-K
  and maxima must be identical byte for byte.  The replay's time is mostly uploads and host work, so it varies with the load of
  the host by tens of ms.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED = 20261021


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:  # informational only
        return None


def kernel_us(prof, name):
    for e in prof.key_averages():
        if name in e.key:
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = getattr(e, "cuda_time_total", 0.0)
            return t / max(e.count, 1)
    return None


def time_device(api, n, perms, strata, reps):
    import torch

    nc = n // 2
    ex = api.JoinExec("method1", nc, n - nc, perms)
    stream = torch.cuda.Stream()  # not the default stream: its handle is 0, which set_stream reads as "the exec's own stream"
    ex.set_stream(stream.cuda_stream)
    if strata:
        ex.setPermutationStrata(np.random.default_rng(1).integers(0, strata, n).astype(np.int32))
    for r in range(3):
        ex.generatePermutedMasks(SEED, r * perms)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for r in range(reps):
        ex.generatePermutedMasks(SEED, r * perms)
    e1.record(stream)
    torch.cuda.synchronize()
    total_ms = e0.elapsed_time(e1) / reps
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for r in range(reps):
            ex.generatePermutedMasks(SEED, r * perms)
        torch.cuda.synchronize()
    gen_us, layout_us = kernel_us(prof, "perm_gen_kernel"), kernel_us(prof, "masks_to_word_major_kernel")
    ex.close()
    return {"ms_per_call_with_layout": round(total_ms, 4), "kernel_ms": None if gen_us is None else round(gen_us / 1e3, 4),
            "layout_rebuild_kernel_ms": None if layout_us is None else round(layout_us / 1e3, 4)}


def time_host(n, perms, budget_s):
    from geneticscre_b200 import synth

    nc = n // 2
    t = time.perf_counter()
    synth.make_perm_masks(nc, n - nc, 4, SEED)
    per = (time.perf_counter() - t) / 4
    k = int(min(perms, max(4, budget_s / max(per, 1e-9))))
    t = time.perf_counter()
    synth.make_perm_masks(nc, n - nc, k, SEED)
    dt = time.perf_counter() - t
    return {"host_ms": round(dt * perms / k * 1e3, 2), "host_perms_timed": k, "host_scaled": k < perms}


def bench_check(api, schedule, synth):
    import torch

    from bench import WORKLOAD as W

    w = synth.make_workload(W["n_cases"], W["n_ctrls"], W["n_genes"], W["n_edges"], W["n_perms"], W["seed"], max_path_length=W["path_length"],
                            real_table=True)
    masks = synth.make_perm_masks_philox(w.n_cases, w.n_ctrls, w.n_perms, W["seed"])
    out = {"workload": W, "generator_seed": W["seed"], "methods": {}}
    for method in ("method1", "method2"):
        res, ms = {}, {}
        for how in ("generated", "host_philox"):
            ex = api.JoinExec(method, w.n_cases, w.n_ctrls, w.n_perms)
            ex.top_k = W["top_k"]
            ex.setValueTable(w.value_table)
            times = []
            for _ in range(3):  # first is warm-up
                torch.cuda.synchronize()
                t = time.perf_counter()
                if how == "generated":
                    ex.generatePermutedMasks(W["seed"])
                else:
                    ex.setPermutedMasks(masks)
                r, _ = schedule.replay_levels(ex, api.UidRelSet, w, W["path_length"])
                torch.cuda.synchronize()
                times.append((time.perf_counter() - t) * 1e3)
            assert np.array_equal(ex.getPermutedMasks(), masks)
            res[how] = r
            ms[how] = [round(x, 2) for x in times[1:]]
            ex.close()
        same = True
        for lvl in res["generated"]:
            a, b = res["generated"][lvl], res["host_philox"][lvl]
            same &= [(s.score, s.src, s.trg, s.cases, s.ctrls) for s in a.scores] == [(s.score, s.src, s.trg, s.cases, s.ctrls) for s in b.scores]
            same &= np.asarray(a.permuted_scores).tobytes() == np.asarray(b.permuted_scores).tobytes()
        out["methods"][method] = {"byte_identical": bool(same), "step_ms_generated": ms["generated"], "step_ms_host_masks": ms["host_philox"],
                                  "levels": sorted(res["generated"])}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-budget-s", type=float, default=3.0, help="host seconds per shape before the host time is sampled and scaled")
    a = ap.parse_args()
    from geneticscre_b200 import api, build, schedule, synth

    build.build()
    rows = []
    for n in (10_000, 50_000):
        for perms in (100, 1000, 4096):
            host = time_host(n, perms, a.host_budget_s)
            for strata in (None, 16):
                d = time_device(api, n, perms, strata, a.reps)
                row = {"patients": n, "perms": perms, "strata": strata or 1, **d, **host}
                row["host_over_device"] = round(host["host_ms"] / d["ms_per_call_with_layout"], 1)
                rows.append(row)
                print(json.dumps(row), flush=True)
    result = {"gpu": gpu_info(), "seed": SEED, "reps": a.reps, "shapes": rows, "bench_workload": bench_check(api, schedule, synth)}
    print(json.dumps(result["bench_workload"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
