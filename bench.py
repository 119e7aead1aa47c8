#!/usr/bin/env python
"""Benchmark of the path-join + permutation-scoring hot path (BASELINE.json metric: path-pair*perm scores / s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE config 3 - synthetic cohort of 10,000 patients (5,000 cases), 15,000 genes, path
length 4, 1,000 permutations, methods 1 + 2 - on a seeded heavy-tailed signed network (the reference's Rels.dat is not
in the checkout; sizes generated are reported in `config`).  One step = the whole level schedule 1a,1b,2,3,4 of
`ProcessPaths` (src/wrapper.cpp:225-269) for method 1 and then method 2.

  value      device-timed throughput with all inputs resident in HBM (packed gene rows, permutation masks, value table)
  e2e        the same schedule through the reference-facing calls with HOST buffers in the R-facing formats
             (IntegerMatrix data, CaseORControl int matrix, value table), uploads and result read-back inside the timing
  roofline   the level-4 join kernels against the roof that binds them: warp-instruction issue for the sparse kernels (ncu
             instruction counts / live CUDA-event time vs the issue rate measured with tools/int_peak.cu), the measured POPC rate
             for the dense kernel; the SURVEY 8d algorithmic bytes / word-ops are kept as `algorithmic` (speed-ups, not fractions)
  cpu_baseline  the reference's own join (oracle/_ref, built from the unmodified reference sources with
             g++ -O3 -march=<host level> -mpopcnt) on all host cores over a bounded sample of the same level-4 join

--steps K sets the timed steps of every timed leg (resident, e2e, strong).  --dump-outputs DIR writes what the last timed
resident step returned to its caller (see dump_outputs); the inputs depend only on the workload arguments and the seed, so
two builds run with the same arguments can be compared output for output.

Multi-GPU (N > 1), one process per GPU:
  --shard perms (default)  every GPU scores ALL pairs against its own block of n_perms permutations (the decomposition of
             BASELINE config 4/5: more permutations, same cohort); the per-permutation maxima are merged with ONE NCCL
             allreduce(max) over the N x n_perms vector (each rank fills its block), top-K is identical on every rank.  Per-GPU work is fixed => "scaling": "weak"; value counts
             N x n_perms permutations.
  --shard rows             the last level's upstream rows are split by pair count, levels 1-3 are computed redundantly,
             permutation maxima are merged with ONE NCCL allreduce(max) per join, top-K lists with an all-gather +
             merge.  Fixed total work => "scaling": "strong".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(n_cases=5000, n_ctrls=5000, n_genes=15000, n_edges=150000, n_perms=1000, path_length=4, top_k=10, seed=20261021)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of every timed leg; the e2e leg needs about 30 for a stable figure (host contention comes in bursts)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "dense", "sparse"])
    ap.add_argument("--shard", default="perms", choices=["perms", "rows"],
                    help="N > 1: 'perms' = every GPU scores all pairs against its own block of n_perms permutations (weak scaling, "
                         "results concatenated); 'rows' = the last level's upstream rows are split, maxima merged with one NCCL allreduce(max)")
    ap.add_argument("--table", default="auto", choices=["auto", "host", "device"],
                    help="value table: numpy on the host and uploaded (what R does), or generated on the device (needed for n >= 50k)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the fixed-work (row-sharded) measurement reported as `strong`")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-threads", type=int, default=2, choices=[1, 2],
                    help="e2e leg: 2 = submit the two methods from two host threads (uploads of one overlap joins of the other); 1 = sequential")
    ap.add_argument("--perm-batch", type=int, default=4096,
                    help="permutations scored per pass over the level schedule; more are processed as sequential batches of this size with the "
                         "masks resident on the device (permutations are independent: maxima concatenate, the top-K is the same in every batch). "
                         "Keeps the per-row count tables the joins hand from level to level (2 KB per row, half and 1,024 permutations) inside HBM")
    ap.add_argument("--cpu-edges", type=int, default=0,
                    help="CPU leg on a SUB-SHAPE: the same cohort size (identical W) and value table, but a network of this many edges (default: "
                         "the benchmarked network up to 20,000 patients, n_edges / 20 above - the reference replays levels 1-3 on the host first "
                         "and keeps an (n+1)^2 table per method-2 thread, SURVEY App. D)")
    ap.add_argument("--cpu-perms", type=int, default=1000, help="permutations the CPU baseline / parity leg scores (the reference's cost per pair*perm does not depend on the count)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed end-to-end steps (default: --steps)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU work per method for the baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last timed step (per method and level: permutation maxima and top-K) "
                         "as DIR/<name>.npy")
    for k, v in WORKLOAD.items():
        ap.add_argument("--" + k.replace("_", "-"), type=type(v), default=v)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results: not with --impl reference")
    return a


def make_workload(a):
    from geneticscre_b200 import synth

    t = time.time()
    host_table = a.table == "host" or (a.table == "auto" and a.n_cases + a.n_ctrls <= 20000)
    w = synth.make_workload(a.n_cases, a.n_ctrls, a.n_genes, a.n_edges, a.n_perms, a.seed, max_path_length=a.path_length, real_table=True,
                            host_table=host_table)
    return w, time.time() - t


def workload_config(a, w):
    lv = w.net.levels
    return {
        "workload": ("BASELINE config 3" if (w.n_patients, a.n_genes, a.path_length, a.n_perms) == (10000, 15000, 4, 1000) else "custom") +
                    ": synthetic cohort, methods 1+2, full level schedule 1a,1b,2,3,4" + (",5" if a.path_length >= 5 else "") + " per method",
        "value_table": "host numpy, uploaded" if w.value_table is not None else "generated on the device",
        "arithmetic": "u64 bitsets / u16 carrier lists, u32+u16 integer counts, f64 score table (f32 copy for method-1 permutation look-ups)",
        "patients": w.n_patients, "cases": w.n_cases, "genes_in_network": w.net.n_genes, "genes_requested": a.n_genes,
        "edges": int(w.net.edges_src.shape[0]), "path_length": a.path_length, "permutations": a.n_perms, "top_k": a.top_k,
        "pairs_per_level": {k: lv[k].n_pairs for k in lv}, "words_per_row_m1": (w.n_patients + 63) // 64,
        "l2_policy": "inputs larger than L2: path sets + tables per method exceed the 126 MB L2",
        "seed": a.seed,
    }


def full_config(a, w, world):
    """config of the JSON line - the same object in both arms (the reference arm describes its own run in cpu_baseline)."""
    shard_perms = world > 1 and a.shard == "perms"
    last = ["1a", "1b", "2", "3", "4", "5"][a.path_length]
    cfg = workload_config(a, w)
    cfg["permutations_total"] = w.n_perms * (world if shard_perms else 1)
    if w.n_perms > a.perm_batch:
        cfg["permutation_batches"] = f"{(w.n_perms + a.perm_batch - 1) // a.perm_batch} sequential batches of <= {a.perm_batch} permutations per GPU (masks resident)"
    cfg["parallelism"] = ("1 GPU" if world == 1 else
                          f"{world} GPUs, one block of {w.n_perms} permutations per GPU over all pairs; maxima merged with one NCCL allreduce(max)" if shard_perms else
                          f"{world} GPUs, level-{last} upstream rows sharded by pair count; one NCCL allreduce(max) per join + top-K gather")
    return cfg


def pairs_per_step(w, path_length):
    names = ["1a", "1b", "2", "3", "4", "5"][: path_length + 1]
    return sum(w.net.levels[k].n_pairs for k in names) * 2  # methods 1 + 2


# ----------------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled through NVML INSIDE the timed region (one sample after every timed step).

    NVML is initialised before the warm-up steps.  (An `nvidia-smi -lms 100` child process, and also a background NVML
    polling thread, were measured to stretch this process's CUDA API calls by 2-10x on the shared hosts - the step is
    made of many short launches - so the samples are taken inline, ~0.1 ms each.)"""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, device):
        self.device, self.sm, self.reasons, self.smax, self.err, self.nv = device, [], set(), None, None, None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.device)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def sample(self):
        nv = self.nv
        if nv is None:
            return
        try:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            try:
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:  # noqa: BLE001
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for name, bit in self.REASONS.items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml unavailable: {self.err}"]}
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.smax, "samples": len(self.sm),
                "reasons": sorted(self.reasons), "how": "NVML, one sample after every timed step (inside the timed region)"}


# ----------------------------------------------------------------------------------------------------------------------
# CPU reference arm
# ----------------------------------------------------------------------------------------------------------------------
# The reference's JoinMethod has no virtual destructor (src/gcre.h:92-99) and its workers are held through
# unique_ptr<JoinMethod>, so every method-2 worker's private (n+1)^2 clone of the value table (src/methods.h:128: 800 MB at
# n = 10,000) is never freed: nthreads x 800 MB leak per method-2 join.  The unmodified reference therefore runs in WORKER
# SUBPROCESSES that are replaced after a bounded number of joins (round 1's in-process arm was OOM-killed on the 1-GPU box).
# The workers load only oracle/_ref/*.so; the process that owns the GPU never maps the reference, and the reference arm never
# maps the CUDA engine.
REF_JOINS_PER_WORKER = {"method1": 64, "method2": 6}  # method 2: upper limit, lowered to what the RAM allows


def mem_available_bytes():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 64 << 30


def workload_file(w, a):
    """The workload as an uncompressed .npz in shared memory (workers map it instead of regenerating it).  The CPU leg scores
    the first min(n_perms, --cpu-perms) permutations."""
    import tempfile

    cpu_perms = cpu_perm_count(w, a)

    net = w.net
    need = w.value_table.nbytes + w.gene_bits.nbytes + w.gene_bits2.nbytes + (64 << 20)
    d = tempfile.gettempdir()
    try:
        st = os.statvfs("/dev/shm")
        if os.access("/dev/shm", os.W_OK) and st.f_bavail * st.f_frsize > need:
            d = "/dev/shm"
    except OSError:
        pass
    path = os.path.join(d, f"gcre_bench_workload_{os.getpid()}.npz")
    np.savez(path, n_cases=w.n_cases, n_ctrls=w.n_ctrls, n_perms=cpu_perms, gene_bits=w.gene_bits, gene_bits2=w.gene_bits2,
             perm_masks=w.perm_masks[:cpu_perms], value_table=w.value_table, n_genes=net.n_genes, edges_src=net.edges_src, edges_trg=net.edges_trg,
             edges_sign=net.edges_sign, ents2=net.ents2, path_length=a.path_length)
    return path


def cpu_perm_count(w, a):
    return int(max(1, min(w.n_perms, getattr(a, "cpu_perms", 1000), getattr(a, "perm_batch", 4096))))


def load_workload_file(path):
    from geneticscre_b200 import synth

    z = np.load(path, allow_pickle=False)
    net = synth.network_from_edges(int(z["n_genes"]), z["edges_src"], z["edges_trg"], z["edges_sign"], ents2=z["ents2"],
                                   max_path_length=max(int(z["path_length"]), 4))
    return synth.Workload(int(z["n_cases"]), int(z["n_ctrls"]), int(z["n_perms"]), z["gene_bits"], z["gene_bits2"], z["perm_masks"],
                          z["value_table"], net)


def ref_worker_main(path, method, kind, threads, top_k):
    """Worker process: the reference's own JoinExec (kind "reference") or the scalar restatement (kind "port") with levels
    1-3 replayed once; then one level-4 join over the first x upstream rows per request line on stdin."""
    from geneticscre_b200 import schedule
    from oracle import pyoracle as po

    real_out = os.dup(1)
    os.dup2(2, 1)  # the reference printf()s progress lines on every join

    def reply(obj):
        os.write(real_out, (json.dumps(obj) + "\n").encode())

    t0 = time.time()
    w = load_workload_file(path)
    if kind == "reference":
        ex = po.RefExec(method, w.n_cases, w.n_ctrls, w.n_perms)
        ex.nthreads = threads
    else:
        ex = po.OracleExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    _, kept = schedule.replay_levels(ex, po.UidRelSet, w, 3, only=())
    p0, p1 = kept["paths3"], kept["paths2"]
    lv = w.net.levels["4"]
    csum = np.cumsum(lv.count.astype(np.int64))
    reply({"ready": True, "setup_s": time.time() - t0})
    for line in sys.stdin:
        req = json.loads(line)
        if req.get("quit"):
            break
        x = int(min(max(req["x"], 1), lv.n_uids))
        uids = po.UidRelSet(4, lv.src[:x], lv.trg[:x], lv.count[:x], lv.location[:x], lv.signs[:x])
        sub = p0 if x == lv.n_uids else p0.select(np.arange(x, dtype=np.int32))
        t = time.time()
        r = ex.join(uids, sub, p1, ex.createPathSet(0))
        dt = time.time() - t
        out = {"seconds": dt, "pairs": int(csum[x - 1]), "x": x}
        if req.get("results"):
            out["scores"] = [[s.score if np.isfinite(s.score) else repr(s.score), s.src, s.trg, s.cases, s.ctrls] for s in r.scores]
            out["perm"] = np.asarray(r.permuted_scores, dtype=np.float64).tolist()  # repr round-trips doubles exactly
        reply(out)


class RefWorker:
    def __init__(self, path, method, kind, threads, top_k):
        env = dict(os.environ)
        env.pop("GCRE_B200_LIB", None)
        self.proc = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--ref-worker", path, method, kind, str(threads), str(top_k)],
                                     stdin=subprocess.PIPE, stdout=subprocess.PIPE, env=env, cwd=ROOT)
        self.joins = 0
        self.setup_s = self._read()["setup_s"]

    def _read(self):
        line = self.proc.stdout.readline()
        if not line:
            raise RuntimeError(f"reference worker died (exit code {self.proc.poll()})")
        return json.loads(line)

    def join(self, x, results=False):
        self.proc.stdin.write((json.dumps({"x": int(x), "results": bool(results)}) + "\n").encode())
        self.proc.stdin.flush()
        self.joins += 1
        return self._read()

    def close(self):
        if self.proc.poll() is None:
            try:
                self.proc.stdin.write(b'{"quit": true}\n')
                self.proc.stdin.flush()
                self.proc.stdin.close()
                self.proc.wait(timeout=60)
            except Exception:  # noqa: BLE001
                self.proc.kill()
                self.proc.wait()


class ReferenceArm:
    """The reference's own JoinExec::join (oracle/_ref: unmodified reference sources, g++ -O3 -march=<host level> -mpopcnt)
    on all host cores, in worker subprocesses.  Each worker replays levels 1-3 once (untimed, like our arm's resident
    inputs); sample() times the last-level join - the whole join when it fits the time budget, else a bounded prefix of
    upstream rows - and can return that join's results for the parity check against the GPU."""

    def __init__(self, w, a, methods=("method1", "method2")):
        if a.path_length < 4:
            raise RuntimeError("the CPU baseline times the level-4 join: needs path_length >= 4")
        if w.value_table is None:
            raise RuntimeError("the CPU baseline needs the value table on the host")
        sys.path.insert(0, ROOT)
        from oracle import pyoracle as po  # (availability / ISA level only; the joins run in the workers)

        self.w, self.a, self.methods = w, a, methods
        self.n_perms = cpu_perm_count(w, a)
        self.kind = "reference" if po.ref_available() else "port"
        self.variant = po.ref_variant()
        self.cores = (os.cpu_count() or 1) if self.kind == "reference" else 1
        # method 2 of the reference needs (and leaks) one (n+1)^2 f64 table per worker thread and join: bound both by the RAM
        table_bytes = (w.n_patients + 1) ** 2 * 8
        # (a worker's set-up replays levels 1a, 2 and 3 through the reference: three more joins that leave their copies behind)
        budget = 0.5 * mem_available_bytes() - 2.5 * table_bytes
        self.threads = {"method1": self.cores, "method2": int(max(1, min(self.cores, budget // (4 * table_bytes))))}
        self.joins_per_worker = {"method1": REF_JOINS_PER_WORKER["method1"],
                                 "method2": int(max(1, min(REF_JOINS_PER_WORKER["method2"], budget // (self.threads["method2"] * table_bytes) - 3)))}
        self.lv = w.net.levels["4"]
        self.csum = np.cumsum(self.lv.count.astype(np.int64))
        self.path = workload_file(w, a)
        self.workers, self.plan, self.setup_s = {}, {}, {}

    def close(self):
        for wk in self.workers.values():
            wk.close()
        self.workers = {}
        try:
            os.unlink(self.path)
        except OSError:
            pass

    def _worker(self, method, need=1):
        wk = self.workers.get(method)
        if wk is not None and wk.joins + need > max(self.joins_per_worker[method], need):
            wk.close()
            wk = None
        if wk is None:
            wk = self.workers[method] = RefWorker(self.path, method, self.kind, self.threads[method], self.a.top_k)
            self.setup_s[method] = wk.setup_s
        return wk

    def calibrate(self, method, target_s):
        """two-point calibration: a join call has a fixed cost (per-thread state; for method 2 a per-thread clone of the
        (n+1)^2 table, src/methods.h:128) plus a per-pair cost"""
        lv = self.lv
        x1 = max(64, lv.n_uids // 400)
        r1 = self._worker(method).join(x1)
        r2 = self._worker(method).join(min(lv.n_uids, 4 * x1))
        rate = max(r2["pairs"] - r1["pairs"], 1) / max(r2["seconds"] - r1["seconds"], 1e-6)
        t_fixed = max(r1["seconds"] - r1["pairs"] / rate, 0.0)
        if t_fixed + lv.n_pairs / rate <= 3.0 * target_s:
            x = lv.n_uids
        else:
            x = int(np.searchsorted(self.csum, max(target_s - t_fixed, 0.25 * target_s) * rate)) + 1
        self.plan[method] = (min(x, lv.n_uids), t_fixed)

    def sample(self, target_s, results=False):
        """One bounded sample per method; returns the cpu_baseline object (and, with `results`, each join's output)."""
        lv, w = self.lv, self.w
        total_pp, total_t, detail, outputs = 0.0, 0.0, {}, {}
        for method in self.methods:
            if method not in self.plan:
                self.calibrate(method, target_s)
            x, t_fixed = self.plan[method]
            r = self._worker(method).join(x, results=results)
            # a join's fixed cost (thread start-up; method 2: every thread's private copy of the (n+1)^2 table) is paid once per
            # join whatever its size: a prefix sample is charged its share of it, so the figure estimates the WHOLE join's rate
            share = r["pairs"] / max(lv.n_pairs, 1)
            fixed = min(t_fixed, 0.9 * r["seconds"])
            t_eff = r["seconds"] - fixed * (1.0 - share)
            total_pp += r["pairs"] * self.n_perms
            total_t += t_eff
            detail[method] = {"pairs": r["pairs"], "of_level4_pairs": lv.n_pairs, "upstream_rows": r["x"], "seconds_measured": round(r["seconds"], 3),
                              "seconds_charged": round(t_eff, 3), "pair_perm_per_s": r["pairs"] * self.n_perms / t_eff,
                              "fixed_s_per_join": round(t_fixed, 3), "threads": self.threads[method],
                              "setup_levels_1_3_s": round(self.setup_s[method], 2)}
            if results:
                outputs[method] = r
        compiler = ""
        try:
            compiler = open(os.path.join(ROOT, "oracle", "_ref", "COMPILER.txt")).read().strip()
        except OSError:
            pass
        how = (f"reference built with {compiler} -O3 -march={self.variant} -mpopcnt" if self.kind == "reference"
               else "scalar C restatement (oracle/gcre_oracle.c), the reference build is absent")
        out = {"value": total_pp / total_t, "unit": "pair*perm/s", "cores": self.cores, "kind": self.kind,
               "sample": f"level-4 join (paths3 x paths2) per method ({'+'.join(self.methods)}): the whole join when it fits ~{3 * target_s:.0f} s, "
                         f"else the first upstream rows sized for ~{target_s:.0f} s; {self.n_perms} perms, W64={(w.n_patients + 63) // 64}; {how}; "
                         f"nthreads={self.threads['method1']} (method 2: {self.threads['method2']}); a prefix sample is charged its pro-rata share of the "
                         f"join's fixed cost (method 2 copies the (n+1)^2 table once per thread and join); run in worker subprocesses replaced every "
                         f"{self.joins_per_worker['method2']} method-2 joins (the reference never frees those copies)",
               "seconds": round(total_t, 3), "detail": detail}
        return (out, outputs) if results else out


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.time()
    w, _ = make_workload(a)
    arm = ReferenceArm(w, a)
    try:
        # K + W bounded samples inside ~3 minutes for the driver's --steps 20 --warmup 5: ~1.2 s of join time per method and sample,
        # on top of method 2's ~1 s fixed cost per join and ~6 s of worker set-up (value table, masks, levels 1-3) every few joins
        per_method_s = max(0.5, min(a.cpu_seconds, 60.0 / max(a.steps + a.warmup, 1) / 2))
        vals = []
        for i in range(a.warmup + a.steps):
            r = arm.sample(per_method_s)
            if i >= a.warmup:
                vals.append(r)
            sys.stderr.write(f"[bench] reference step {i}: {r['value']:.4g} pair*perm/s in {r['seconds']:.2f} s\n")
    finally:
        arm.close()
    value = float(np.mean([v["value"] for v in vals])) if vals else 0.0
    last = vals[-1] if vals else {"cores": arm.cores, "kind": arm.kind, "sample": ""}
    ms = 1e3 * float(np.mean([v["seconds"] for v in vals])) if vals else None
    cfg = full_config(a, w, max(a.gpus, 1))
    line = {"metric": "path-pair*perm scores/s", "value": value, "unit": "pair*perm/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "impl": "reference", "config": cfg,
            "cpu_baseline": {"value": value, "unit": "pair*perm/s", "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
            "e2e": {"value": value, "unit": "pair*perm/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": round(time.time() - t0, 1)}
    emit_line(line)


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  NCCL ("NCCL version ..."), the reference's printf progress lines and any
    library chatter also write to file descriptor 1, so fd 1 is pointed at stderr for the whole run and the JSON line is
    written to the saved original descriptor at the end."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_line(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def check_parity(ref_out, last_out, state, lv4, w, api, cpu_perms, reset_masks):
    """GPU level-4 results against the reference's on the same inputs -> the `parity` object of the line (raises on mismatch).

    The CPU leg scored the first `cpu_perms` permutations (they belong to the first permutation batch).  When the reference ran
    the whole join, the result of the last TIMED step (first batch) is compared; when it ran a prefix of the upstream rows
    (bounded sample), the GPU re-runs exactly that prefix (uid_range) on its resident operands."""
    from oracle import pyoracle as po  # the checker

    out = {"checked": True, "rule": "SURVEY App. A.7: f32 permutation maxima bit-exact, top-K score multiset bit-exact, entries above the K-th score identical",
           "against": "the reference's own join (oracle/_ref) in the cpu_baseline leg of this run", "permutations_compared": int(cpu_perms),
           "level4_pairs": 0, "mismatches": 0, "methods": {}}
    for method, r in ref_out.items():
        want = po.JoinedRes([po.Score(float(s[0]), int(s[1]), int(s[2]), int(s[3]), int(s[4])) for s in r["scores"]], np.asarray(r["perm"], dtype=np.float64))
        x = int(r["x"])
        if x == lv4.n_uids and "4" in last_out[method][2]:
            got, how = last_out[method][2]["4"], "whole join, result of the last timed step"
        else:
            reset_masks(state[method])
            got, how = rerun_level4_prefix(state[method], lv4, w, x, api), f"first {x} upstream rows, re-run on the GPU with uid_range"
        got = po.JoinedRes(got.scores, np.asarray(got.permuted_scores, dtype=np.float64)[:cpu_perms])
        try:
            po.compare_results(got, want, what=f"bench parity {method}")
            bad = 0
        except AssertionError as e:
            sys.stderr.write(f"[bench] PARITY MISMATCH {method}: {e}\n")
            bad = 1
        out["methods"][method] = {"pairs": int(r["pairs"]), "compared": how, "perm_maxima": int(want.permuted_scores.shape[0]), "top_k": len(want.scores), "mismatch": bad}
        out["level4_pairs"] += int(r["pairs"])
        out["mismatches"] += bad
    if out["mismatches"]:
        raise AssertionError(f"GPU results differ from the reference's on the benchmarked workload: {out}")
    return out


DUMP_LIMIT_BYTES = 64 << 20


def device_perm_max(perm_all, world, n_batches, ip, batch_perms, n_perms):
    """The device vector of last-level maxima, laid out [rank][batch][ip], -> float64 [world * n_perms]: the real permutations of
    every block, in order.  ip is the batch padded to the kernels' tile, and the slots of a short last batch past its real
    permutations are scored on copies of real ones: neither is part of the result."""
    v = np.asarray(perm_all, dtype=np.float64).reshape(world, n_batches, ip)
    return np.concatenate([v[r, b, : min(batch_perms, n_perms - b * batch_perms)] for r in range(world) for b in range(n_batches)])


def dump_outputs(d, last_out, names, last_perm, n_perms, limit=DUMP_LIMIT_BYTES):
    """What one step returns to its caller, for each method and each level whose result the step keeps (1b and up):
    <method>_level<k>_perm_max.npy (float64 [n_perms]: the f32 permutation maxima of all batches, widened as the API returns
    them) and <method>_level<k>_topk.npy (float64 [rows, 5]: score, src, trg, cases, ctrls in the API's ascending order, -inf
    sentinel row included).  `last_perm[method]` replaces the last level's maxima with the merged [world * n_perms] vector
    of a perm-sharded run.  Should the maxima exceed half of `limit`, the same fixed, seeded sample of permutation indices is
    kept from every block of n_perms and the indices are written as perm_sample_index.npy."""
    os.makedirs(d, exist_ok=True)
    out, perms = {}, {}
    for method, step in last_out.items():
        res, parts = step[1], step[3]
        for k in [k for k in names if k in res]:
            v = last_perm[method] if k == names[-1] and method in last_perm else np.concatenate(parts[k])
            perms[f"{method}_level{k}_perm_max"] = np.asarray(v, dtype=np.float64).reshape(-1, n_perms)
            out[f"{method}_level{k}_topk"] = np.array([[s.score, s.src, s.trg, s.cases, s.ctrls] for s in res[k].scores], dtype=np.float64).reshape(-1, 5)
    total = sum(v.nbytes for v in perms.values())
    if total > limit // 2:
        keep = np.sort(np.random.default_rng(0).choice(n_perms, size=max(1, int(n_perms * (limit // 2) // total)), replace=False))
        perms = {k: v[:, keep] for k, v in perms.items()}
        out["perm_sample_index"] = keep.astype(np.float64)
    out.update({k: v.reshape(-1) for k, v in perms.items()})
    for k, v in out.items():
        np.save(os.path.join(d, k + ".npy"), v)


def rerun_level4_prefix(st, lv4, w, x, api):
    """Levels 1-3 again (resident inputs) and the level-4 join over the first x upstream rows."""
    ex, d1, d2 = st["ex"], st["d1"], st["d2"]
    lv = w.net.levels
    p1 = ex.createPathSet(lv["1a"].n_pairs)
    ex.join(st["uid"]["1a"], ex.createPathSet(lv["1a"].n_uids), d1.select(w.net.data_idx["1a"]), p1)
    p2 = ex.createPathSet(lv["2"].n_pairs)
    ex.join(st["uid"]["2"], p1, d1.select(w.net.data_idx["2"]), p2)
    p3 = ex.createPathSet(lv["3"].n_pairs)
    ex.join(st["uid"]["3"], p2, d1.select(w.net.data_idx["3"]), p3)
    return ex.join(st["uid"]["4"], p3, p2, ex.createPathSet(0), uid_range=(0, x))


def load_json(*parts):
    try:
        return json.load(open(os.path.join(ROOT, *parts)))
    except (OSError, ValueError):
        return None


def roofline_of(last_out, last, w, a, n, ms_step, world):
    """The `roofline` object of the line for the dominant kernel (the last-level join of methods 1 + 2).

    The sparse (carrier-list) kernels do not move the algorithmic bytes of SURVEY 8d nor execute its word-ops - that is their
    point - so neither HBM nor the POPC pipe can be their roof: they are bound by warp-instruction ISSUE (ALU-pipe LOP3s, the
    filter pass and the mask gathers).  achieved = warp instructions of the launches (ncu smsp__inst_executed.sum of the same
    command, profiles/r2_counts.json) / the kernel time measured live with CUDA events; peak = the issue rate measured on this
    pool's B200 with tools/int_peak.cu (profiles/r2_int_peak.json).  The dense (AND + POPC) kernel does the 8d word-ops: its roof
    is the measured POPC rate.  The 8d algorithmic figures are kept as `algorithmic` and are SPEED-UPS of the sparse formulation
    over a kernel that would do that work, not utilisations."""
    W64 = (n + 63) // 64
    ker_ms, alg_bytes, word_ops, kname = 0.0, 0.0, 0.0, None
    for method, m in (("method1", 1), ("method2", 2)):
        inf = last_out[method][0][last]
        ker_ms += inf["kernel_ms"]
        pairs = inf["pairs"]
        alg_bytes += pairs * 2 * W64 * m * 8 + W64 * w.n_perms * 8 + 4 * w.n_perms
        word_ops += pairs * w.n_perms * W64 * m
        kname = {1: "dense", 2: "sparse"}.get(inf["kernel"], "?")
        if inf.get("split_carrier"):
            kname = "sparse_sc"  # <= 512 permutations (join_sparse_sc.cuh)
    ker_s = max(ker_ms, 1e-9) * 1e-3
    peaks = load_json("MEASURED_PEAKS.json") or {}
    ip = (load_json("profiles", "r2_int_peak.json") or {}).get("summary", {})
    issue_peak = float(ip.get("issue_peak_warp_inst_per_s", 148 * 4 * 1.965e9))
    word_peak = float(ip.get("word_ops_per_s (1 word-op = 2 POPC32, SURVEY 8d)", 148 * 16 * 1.965e9 / 2))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    counts, batches = None, max(1, (w.n_perms + a.perm_batch - 1) // a.perm_batch)
    for x in (load_json("profiles", "r2_counts.json") or {}).get("workloads", []):
        c = x["config"]
        if (c["patients"], c["edges"], c["permutations"], c["path_length"]) == (n, a.n_edges, min(w.n_perms, a.perm_batch), a.path_length) and world == 1:
            counts = x
    algorithmic = {"bytes": alg_bytes, "GB_per_s": alg_bytes / ker_s / 1e9, "x_measured_hbm_peak": alg_bytes / ker_s / 1e9 / hbm_peak,
                   "word_ops_per_s": word_ops / ker_s, "x_measured_popc_peak": word_ops / ker_s / word_peak,
                   "note": "SURVEY 8d figures (read both operand rows of every pair; one AND+POPC per word and permutation). For the sparse kernels these "
                           "ratios are the SPEED-UP over a kernel that does that work at the measured HBM / POPC peak, not a utilisation"}
    base = {"kernel": f"join_{kname}_kernel, level-{last} joins of methods 1+2 (this rank's shard)", "kernel_ms_per_step": ker_ms,
            "kernel_share_of_step": ker_ms / ms_step, "algorithmic": algorithmic}
    if kname == "dense":
        ach = word_ops / ker_s
        return dict(base, bound="xu_popc", achieved=ach, peak=word_peak, unit="word-ops/s", frac=ach / word_peak, traffic=None,
                    peak_source="measured POPC rate (tools/int_peak.cu, profiles/r2_int_peak.json)")
    if counts is None:
        return dict(base, bound="issue", achieved=None, peak=issue_peak, unit="warp-inst/s", frac=None, traffic=None,
                    peak_source="measured issue rate (tools/int_peak.cu, profiles/r2_int_peak.json)",
                    note="no ncu instruction count is committed for this workload (profiles/r2_counts.json): the issue-slot fraction needs one")
    inst = sum(v["warp_instructions"] for v in counts["launches"].values()) * batches
    traffic = sum(v["dram_bytes"] for v in counts["launches"].values()) * batches
    ach = inst / ker_s
    return dict(base, bound="issue", achieved=ach, peak=issue_peak, unit="warp-inst/s", frac=ach / issue_peak, traffic=traffic,
                peak_source="measured issue rate (tools/int_peak.cu, profiles/r2_int_peak.json: 3.97 warp instructions / clk / SM)",
                warp_instructions_per_step=inst, dram_GB_per_s=traffic / ker_s / 1e9, hbm_frac=traffic / ker_s / 1e9 / hbm_peak,
                ncu={k: {kk: v[kk] for kk in ("kernel", "ncu_ms", "issue_active_pct", "alu_pipe_pct")} for k, v in counts["launches"].items()},
                counts_source=f"profiles/r2_counts.json ({counts.get('source', '')}): smsp__inst_executed.sum and dram bytes of the same launches under ncu; time live",
                note="issue-bound: the ALU pipe (LOP3 carry-save adds, compares, address arithmetic; measured peak 2 warp instructions / clk / SM) is the busiest unit; "
                     "DRAM traffic is a few per cent of the HBM peak because the working set (masks, look-up rows) lives in L1/L2")


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--ref-worker":
        return ref_worker_main(sys.argv[2], sys.argv[3], sys.argv[4], int(sys.argv[5]), int(sys.argv[6]))
    a = parse_args()
    claim_stdout()
    if a.impl == "reference":
        return run_reference_arm(a)

    import torch
    import torch.distributed as dist

    from geneticscre_b200 import _lib, api, build, synth
    from geneticscre_b200 import dist as gdist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    build.build()
    lib = _lib.load()
    kernel = {"auto": _lib.KERNEL_AUTO, "dense": _lib.KERNEL_DENSE, "sparse": _lib.KERNEL_SPARSE}[a.kernel]

    w, gen_s = make_workload(a)
    shard_perms = world > 1 and a.shard == "perms"
    if shard_perms and rank > 0:
        # this rank's own block of permutations (same cohort, network and table on every rank)
        w.perm_masks = synth.make_perm_masks(w.n_cases, w.n_ctrls, w.n_perms, a.seed + 3 + 1000 * rank)
    # host cores are shared by the ranks of one box: the engine packs int matrices on the host only with >= 8 threads
    # (gcre_pathset_load_i32), so with several ranks per host it falls back to packing on the device
    os.environ.setdefault("GCRE_HOST_PACK_THREADS", str(min(16, (os.cpu_count() or 1) // max(world, 1))))
    lv = w.net.levels
    n = w.n_patients
    names = ["1a", "1b", "2", "3", "4", "5"][: a.path_length + 1]
    last = names[-1]
    shards = gdist.shard_bounds(lv[last].count, world)
    my_shard = shards[rank]
    # Fixed-work decomposition at path length 4: the level-4 shard of a rank is a contiguous range of paths3 rows, so the rank
    # builds ONLY those rows at level 3 (a contiguous range of level-3 upstream rows, cut where a level-3 row's results end);
    # ranges are balanced by level-4 pairs plus the level-3 pairs they cost (a KEEP pair ~ 4 score-only pairs).
    l3_shard = l4_rows = None
    if a.path_length == 4 and world > 1:
        c3 = lv["3"].count.astype(np.int64)
        pidx3 = np.concatenate([[0], np.cumsum(c3)])
        cs4 = np.concatenate([[0], np.cumsum(lv["4"].count.astype(np.int64))])
        weight = cs4[pidx3[1:]] - cs4[pidx3[:-1]] + 4 * c3
        l3_shard = gdist.shard_bounds(weight, world)[rank]
        l4_rows = (int(pidx3[l3_shard[0]]), int(pidx3[l3_shard[1]]))
    default_mode = "perms" if shard_perms else ("rows" if world > 1 else "single")
    stream = torch.cuda.current_stream()

    def launches():
        import ctypes

        c = ctypes.c_uint64(0)
        lib.gcre_kernel_launch_count(ctypes.byref(c))
        return c.value

    # ---- resident state: one exec per method with table + masks + packed gene rows in HBM ----
    # permutations beyond --perm-batch are scored as sequential batches through the same exec (masks of every batch resident)
    batch_perms = int(min(w.n_perms, max(a.perm_batch, 1)))
    n_batches = (w.n_perms + batch_perms - 1) // batch_perms
    if a.dump_outputs and world > 1 and not shard_perms and n_batches > 1:
        # each batch's row shards are merged on their own and only the last batch's merged maxima reach the host
        raise SystemExit("bench.py: --dump-outputs with --shard rows needs n_perms <= --perm-batch")
    W1m = (n + 63) // 64
    masks_dev = torch.from_numpy(np.ascontiguousarray(w.perm_masks).view(np.int64)).cuda() if n_batches > 1 else None
    state = {}
    for method in ("method1", "method2"):
        ex = api.JoinExec(method, w.n_cases, w.n_ctrls, batch_perms, device=local_rank)
        ex.set_stream(stream.cuda_stream)
        ex.kernel = kernel
        ex.top_k = a.top_k
        if w.value_table is None:
            ex.generateValueTable()
        else:
            ex.setValueTable(w.value_table)
        ex.setPermutedMasks(w.perm_masks[:batch_perms])
        d1 = ex.createPathSet(w.gene_bits.shape[0])
        d1.load_bits(w.gene_bits)
        d2 = ex.createPathSet(w.gene_bits2.shape[0])
        d2.load_bits(w.gene_bits2)
        # the join indices are inputs like the gene rows: resident on the device for the `value` measurement
        uid = {k: api.UidRelSet(lv[k].path_length, lv[k].src, lv[k].trg, lv[k].count, lv[k].location, lv[k].signs).make_resident(ex) for k in names}
        state[method] = dict(ex=ex, d1=d1, d2=d2, uid=uid, perm_t=torch.zeros(ex.iterations, dtype=torch.float32, device="cuda"),
                             perm_all=torch.zeros(world * n_batches * ex.iterations, dtype=torch.float32, device="cuda"))

    def export_block(st, b):
        """This rank's maxima of batch b into its slot of the [rank][batch][Ip] result vector (device to device, on the exec's stream)."""
        ex = st["ex"]
        with torch.cuda.stream(st.get("stream", stream)):
            if b == 0 and shard_perms:
                st["perm_all"].zero_()
            off = (rank * n_batches + b) * ex.iterations
            _lib.check(lib.gcre_exec_export_perm_max(ex._h, st["perm_all"].data_ptr() + 4 * off, ex.iterations))

    def merge_last_level(st, results=None):
        """The one data-path collective of a perm-sharded job: every rank has dropped its maxima into its slots of a zeroed
        [N][batches][Ip] vector and ONE NCCL allreduce(max) over NVLink merges them (maxima are >= +0, so max against the zeros
        is concatenation)."""
        if not shard_perms:
            return
        with torch.cuda.stream(st.get("stream", stream)):  # the stream the exec launches on
            dist.all_reduce(st["perm_all"], op=dist.ReduceOp.MAX)

    def schedule_resident(st, results, collective=True, single=False, mode=None):
        """Levels 1a,1b,2,3,(4,5) with device-resident inputs; the last level is sharded across ranks
        (`single`: this rank alone does the whole job - the cross-check of the multi-GPU result).
        mode: "perms" (own permutation block, all pairs), "rows" (fixed work: upstream rows sharded), "single"."""
        mode = "single" if single else (mode or default_mode)
        ex, d1, d2, uid = st["ex"], st["d1"], st["d2"], st["uid"]
        zero = ex.createPathSet(0)
        info = {}
        p1 = ex.createPathSet(lv["1a"].n_pairs)
        r = ex.join(uid["1a"], ex.createPathSet(lv["1a"].n_uids), d1.select(w.net.data_idx["1a"]), p1); info["1a"] = r.info
        r = ex.join(uid["1b"], ex.createPathSet(lv["1b"].n_uids), d2.select(w.net.data_idx["1b"]), zero); info["1b"] = r.info; results["1b"] = r
        prev = p1
        for k in names[2:]:
            keep = lv[k].keep and k != last
            if k in ("2", "3"):
                operand = d1.select(w.net.data_idx[k])
            elif k == "4":
                operand = results["_p2"]
            else:
                operand = results["_p3"]
            res_set = ex.createPathSet(lv[k].n_pairs) if (keep or (k in ("2", "3") and a.path_length > int(k))) else zero
            if k == last and mode == "perms":
                r = ex.join(uid[k], prev, operand, res_set, skip_host_perm=n_batches > 1)
                export_block(st, st.get("batch", 0))
                if collective and st.get("batch", 0) == n_batches - 1:
                    merge_last_level(st, results)
            elif k == "3" and mode == "rows" and l3_shard is not None:
                # this rank's slice of level 3: exactly the paths3 rows its level-4 shard reads
                r = ex.join(uid[k], prev, operand, res_set, uid_range=l3_shard)
            elif k == last and mode == "rows":
                r = ex.join(uid[k], prev, operand, zero, uid_range=(l4_rows if l4_rows is not None else my_shard), skip_host_perm=True)
                _lib.check(lib.gcre_exec_export_perm_max(ex._h, st["perm_t"].data_ptr(), ex.iterations))
                # ONE data-path collective per join: NCCL allreduce(max) of the f32 maxima (+ a K-entry gather)
                gdist.merge_shard_result(r, a.top_k, api.merge_topk, api.Score, dist, device_perm=st["perm_t"], n_perms=w.n_perms)
            else:
                r = ex.join(uid[k], prev, operand, res_set)
            info[k] = r.info
            results[k] = r
            if k == "2":
                results["_p2"] = res_set
            if k == "3":
                results["_p3"] = res_set
            if k in ("2", "3"):
                prev = res_set
        return info

    def run_batches(st, collective=True, single=False):
        """All permutation batches of one method; returns (per-level info with kernel times summed over the batches, results of the
        last batch, results of batch 0, per level the list of every batch's permutation maxima)."""
        info_sum, res_last, res_first, perms = None, None, None, {}
        for b in range(n_batches):
            ex = st["ex"]
            st["batch"] = b
            nb = min(batch_perms, w.n_perms - b * batch_perms)
            if n_batches > 1:
                ex.setPermutedMasksDevice(masks_dev.data_ptr() + 8 * b * batch_perms * W1m, nb)
            res = {}
            info = schedule_resident(st, res, collective=collective, single=single)
            if n_batches > 1 and not shard_perms:
                export_block(st, b)
            for k in [k for k in res if k.startswith("_")]:
                del res[k]  # kept path sets go back to the block cache now, not when the next step overwrites `last_out`
            for k, r in res.items():
                perms.setdefault(k, []).append(r.permuted_scores[:nb])  # a short last batch is padded with copies of real permutations
            if info_sum is None:
                info_sum, res_first = info, res
            else:
                for k in info:
                    info_sum[k]["kernel_ms"] += info[k]["kernel_ms"]
                    info_sum[k]["exact_pairs"] += info[k].get("exact_pairs", 0)
            res_last = res
        st["batch"] = 0
        return info_sum, res_last, res_first, perms

    def step_resident():
        out = {}
        for method in ("method1", "method2"):
            out[method] = run_batches(state[method])
        return out

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- warm-up + timed region (CUDA events on the stream the engine launches on) ----
    dbg = bool(os.environ.get("GCRE_BENCH_DEBUG"))
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for i in range(a.warmup):
        t_dbg = time.perf_counter()
        step_resident()
        sampler.sample()  # NVML's first queries are slow and perturb the following step: take them during warm-up
        if dbg:
            torch.cuda.synchronize()
            sys.stderr.write(f"[bench] warmup step {i}: {(time.perf_counter() - t_dbg) * 1e3:.1f} ms\n")
    sync_all()
    import gc

    gc.collect()
    gc.freeze()   # keep the interpreter's cyclic GC (hundreds of ms with torch imported) out of the timed region
    gc.disable()
    l0 = launches()
    sampler.sm.clear()
    sampler.reasons.clear()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    last_out = None
    for i in range(a.steps):
        t_dbg = time.perf_counter()
        last_out = step_resident()
        sampler.sample()
        if dbg:
            sys.stderr.write(f"[bench] timed step {i}: {(time.perf_counter() - t_dbg) * 1e3:.1f} ms (host clock, no sync)\n")
    ev1.record(stream)
    sync_all()
    ms_total = ev0.elapsed_time(ev1)
    if a.dump_outputs and rank == 0:
        # perm-sharded, the last level's merged maxima of every rank are only in perm_all (which later legs overwrite)
        last_perm = {m: device_perm_max(state[m]["perm_all"].cpu().numpy(), world, n_batches, state[m]["ex"].iterations, batch_perms, w.n_perms)
                     for m in state} if shard_perms else {}
        dump_outputs(a.dump_outputs, last_out, names, last_perm, w.n_perms)
    n_launch = launches() - l0
    clocks = sampler.stop() if rank == 0 else None
    gc.enable()
    t_ms = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_step = float(t_ms.item()) / a.steps
    pp_step = pairs_per_step(w, a.path_length) * w.n_perms * (world if shard_perms else 1)  # whole job, all ranks
    value = pp_step / (ms_step * 1e-3)

    # ---- N > 1: the merged result against a single-rank recomputation (after the timed region) ----
    multi_parity = None
    if world > 1 and last_out is not None:
        bad = 0
        for method in ("method1", "method2"):
            st = state[method]
            ex = st["ex"]
            merged = last_out[method][1][last]
            if shard_perms:
                # rank r recomputes, alone, the block of permutations rank (r + 1) % N scored, and compares it bit for bit with
                # that block of the all-reduced N x I vector; the top-K (permutation independent) must be the same on every rank
                # (with several permutation batches: the neighbour's first batch)
                blk = (rank + 1) % world
                all_red = st["perm_all"].cpu().numpy().astype(np.float64)
                ex.setPermutedMasks(synth.make_perm_masks(w.n_cases, w.n_ctrls, w.n_perms, a.seed + 3 + 1000 * blk)[:batch_perms])
                res = {}
                st["batch"] = 0
                schedule_resident(st, res, collective=False, single=True)
                mine = res[last]
                o0 = blk * n_batches * ex.iterations
                bad += int(not np.array_equal(mine.permuted_scores.view(np.uint64), all_red[o0: o0 + batch_perms].view(np.uint64)))
                bad += int([(s_.score, s_.src, s_.trg, s_.cases, s_.ctrls) for s_ in mine.scores] != [(s_.score, s_.src, s_.trg, s_.cases, s_.ctrls) for s_ in merged.scores])
                ex.setPermutedMasks(w.perm_masks[:batch_perms])
                del res
            else:
                # every rank recomputes the whole last-level join and compares it with the merged shards
                res = {}
                schedule_resident(st, res, single=True)
                mine = res[last]
                bad += int(not np.array_equal(mine.permuted_scores.view(np.uint64), np.asarray(merged.permuted_scores, dtype=np.float64).view(np.uint64)))
                bad += int([(s_.score, s_.src, s_.trg, s_.cases, s_.ctrls) for s_ in mine.scores] != [(s_.score, s_.src, s_.trg, s_.cases, s_.ctrls) for s_ in merged.scores])
                del res
            tops = [None] * world
            dist.all_gather_object(tops, [(s_.score, s_.src, s_.trg, s_.cases, s_.ctrls) for s_ in merged.scores])
            bad += int(any(t_ != tops[0] for t_ in tops))
        t_bad = torch.tensor([bad], dtype=torch.int64, device="cuda")
        dist.all_reduce(t_bad, op=dist.ReduceOp.SUM)
        multi_parity = {"checked": True, "mismatches": int(t_bad.item()),
                        "what": ("every rank recomputed, alone, the permutation block of its neighbour and compared it bit for bit with that block of the "
                                 "all-reduced maxima; top-K identical on all ranks" if shard_perms else
                                 "every rank recomputed the whole last-level join alone and compared maxima (bit for bit) and top-K with the merged shards")}
        if multi_parity["mismatches"]:
            raise AssertionError(f"multi-GPU result differs from the single-rank recomputation: {multi_parity}")

    # ---- N > 1: the same FIXED job (rank 0's permutations, first batch) row-sharded over the N GPUs vs done by one GPU alone ----
    strong = None
    if world > 1 and not a.no_strong and last_out is not None:
        block0 = synth.make_perm_masks(w.n_cases, w.n_ctrls, w.n_perms, a.seed + 3)[:batch_perms] if rank > 0 else w.perm_masks[:batch_perms]
        for st in state.values():
            st["ex"].setPermutedMasks(block0)
            st["batch"] = 0

        def timed(mode, steps):
            def one():
                for method in ("method1", "method2"):
                    res = {}
                    schedule_resident(state[method], res, mode=mode)
                    del res
            for _ in range(2):
                one()
            sync_all()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                one()
            e1.record(stream)
            sync_all()
            t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        k_steps = a.steps
        ms_one = timed("single", k_steps)
        ms_rows = timed("rows", k_steps)
        strong = {"job": f"the N=1 job ({batch_perms} permutations, all pairs, methods 1+2) done once by the {world} GPUs together",
                  "decomposition": ("level-4 upstream rows sharded by pair count; each rank builds only its own paths3 rows at level 3; levels 1a/1b/2 replicated; "
                                    "one NCCL allreduce(max) + top-K gather per method" if l3_shard is not None else
                                    "last level's upstream rows sharded by pair count, earlier levels replicated; one NCCL allreduce(max) + top-K gather per method"),
                  "ms_per_step_one_gpu": ms_one, "ms_per_step": ms_rows, "speedup": ms_one / ms_rows, "efficiency": ms_one / ms_rows / world, "steps": k_steps,
                  "timing": "CUDA events on the launching stream, max over ranks"}
        for st in state.values():
            st["ex"].setPermutedMasks(w.perm_masks[:batch_perms])

    # ---- roofline of the dominant kernel: the last-level join of each method, timed live by CUDA events inside join ----
    roof = None
    if last_out is not None:
        roof = roofline_of(last_out, last, w, a, n, ms_step, world)

    # ---- SURVEY 8d: the metric per level as well as in aggregate (kernel time of each join, CUDA events inside gcre_join) ----
    per_level = None
    if last_out is not None:
        per_level = {}
        for method in ("method1", "method2"):
            per_level[method] = {}
            for k in names:
                inf = last_out[method][0][k]
                kms = float(inf["kernel_ms"])
                per_level[method][k] = {"pairs": int(inf["pairs"]), "kernel_ms": kms, "kernel": {1: "dense", 2: "sparse"}.get(inf["kernel"], "none") + ("+precount" if inf.get("precounted") else "") + ("+split-carrier" if inf.get("split_carrier") else "") + ("+thresholded" if inf.get("thresholded") else ""),
                                        "exact_lookup_fraction": (inf["exact_pairs"] / max(1, inf["pairs"] * ((batch_perms + 1023) // 1024) * n_batches)) if inf.get("thresholded") else None,
                                        "pair_perm_per_s": (inf["pairs"] * w.n_perms / (kms * 1e-3)) if kms > 0 else None}

    # ---- end-to-end through the reference-facing calls with HOST buffers (R-facing int matrices), N GPUs ----
    e2e = None
    if not a.no_e2e and w.value_table is None:
        sys.stderr.write("[bench] e2e skipped: no host value table at this size (generated on the device)\n")
    if not a.no_e2e and w.value_table is not None and n_batches > 1:
        sys.stderr.write("[bench] e2e skipped: several permutation batches (the int permutation matrix would not fit the host)\n")
    if not a.no_e2e and w.value_table is not None and n_batches == 1:
        data1_i = torch.from_numpy(synth.unpack_bits(w.gene_bits, n)).pin_memory().numpy()
        data2_i = torch.from_numpy(synth.unpack_bits(w.gene_bits2, n)).pin_memory().numpy()
        bits = np.unpackbits(w.perm_masks.view(np.uint8), axis=1, bitorder="little")[:, :n].astype(bool)
        is_case = np.zeros(n, dtype=bool)
        is_case[: w.n_cases] = True
        perm_i = torch.from_numpy((bits == is_case[None, :]).astype(np.int32)).pin_memory().numpy()
        table = torch.from_numpy(np.ascontiguousarray(w.value_table)).pin_memory().numpy()
        d2h_holder = [0]

        uid_host = {k: api.UidRelSet(lv[k].path_length, lv[k].src, lv[k].trg, lv[k].count, lv[k].location, lv[k].signs) for k in names}

        def pinned(arr):  # the join indices are host inputs like the matrices: page-locked, so their copies run at PCIe rate
            t = torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).reshape(-1)).pin_memory()
            return t.numpy().view(arr.dtype).reshape(arr.shape)

        for u in uid_host.values():
            u._packed, u.signs = pinned(u._packed), pinned(u.signs)
        idx_bytes = sum(u._packed.nbytes + u.signs.nbytes for u in uid_host.values())
        W1 = (n + 63) // 64
        bits_bytes = (data1_i.shape[0] + data2_i.shape[0]) * W1 * 8
        pack_threads = int(os.environ["GCRE_HOST_PACK_THREADS"])
        host_packed = pack_threads >= 8 and min(data1_i.nbytes, data2_i.nbytes) >= (32 << 20)  # gcre_pathset_load_i32's own rule
        # Multi-GPU, permutation blocks: cohort matrices and value table are the same on every rank, so rank 0 alone reads them
        # (host-packed), uploads them once per step and NCCL broadcasts the 47 MB of bits + the table over NVLink; every rank
        # uploads only its own block of permutations.  Without this eight ranks pull 8 x 2.9 GB per step through one host.
        fanout = world > 1 and shard_perms
        if fanout:
            h2d = (bits_bytes + table.nbytes if rank == 0 else 0) + 2 * (perm_i.nbytes + idx_bytes)
            bits1_h = torch.zeros((data1_i.shape[0], W1), dtype=torch.int64).pin_memory()
            bits2_h = torch.zeros((data2_i.shape[0], W1), dtype=torch.int64).pin_memory()
            table_h = torch.from_numpy(table)
        else:
            h2d = 2 * ((bits_bytes if host_packed else data1_i.nbytes + data2_i.nbytes) + perm_i.nbytes + table.nbytes + idx_bytes)  # per method
        host_input_bytes = 2 * (data1_i.nbytes + data2_i.nbytes + perm_i.nbytes + table.nbytes + idx_bytes)
        # The two methods are independent jobs (two GWASPA() calls upstream).  Run from two host threads on two streams the
        # second method's uploads hide under the first method's joins; the collectives stay on the main thread, in order.
        overlap = a.e2e_threads > 1 and (world == 1 or shard_perms)
        e2e_streams = {m: (torch.cuda.Stream() if overlap else stream) for m in ("method1", "method2")}
        shared = {}

        def fan_out():
            """rank 0: pack + upload once; everyone: receive over NVLink (main thread, default process group)."""
            with torch.cuda.stream(stream):
                tab_d = torch.empty(table.shape, dtype=torch.float64, device="cuda")
                b1_d = torch.empty(bits1_h.shape, dtype=torch.int64, device="cuda")
                b2_d = torch.empty(bits2_h.shape, dtype=torch.int64, device="cuda")
                if rank == 0:
                    tab_d.copy_(table_h, non_blocking=True)
                    api.host_pack(data1_i, threads=min(16, os.cpu_count() or 1), out=bits1_h.numpy().view(np.uint64))
                    b1_d.copy_(bits1_h, non_blocking=True)
                    api.host_pack(data2_i, threads=min(16, os.cpu_count() or 1), out=bits2_h.numpy().view(np.uint64))
                    b2_d.copy_(bits2_h, non_blocking=True)
                for t in (tab_d, b1_d, b2_d):
                    dist.broadcast(t, src=0)
            stream.synchronize()  # the method threads launch on their own streams
            shared.update(table=tab_d, bits1=b1_d, bits2=b2_d)

        def e2e_method(method, results, gate_in, gate_out):
            t_in = time.perf_counter()
            try:
                torch.cuda.set_device(local_rank)
                if gate_in is not None:
                    gate_in.wait()
                t_go = time.perf_counter()
                ex = api.JoinExec(method, w.n_cases, w.n_ctrls, w.n_perms, device=local_rank)
                ex.set_stream(e2e_streams[method].cuda_stream)
                ex.kernel = kernel
                ex.top_k = a.top_k
                if fanout:
                    ex.setValueTableDevice(shared["table"].data_ptr(), table.shape[0], table.shape[1])
                    ex.setPermutedCases(perm_i)
                    d1 = ex.createPathSet(data1_i.shape[0]); d1.load_bits_device(shared["bits1"].data_ptr(), data1_i.shape[0], W1)
                    d2 = ex.createPathSet(data2_i.shape[0]); d2.load_bits_device(shared["bits2"].data_ptr(), data2_i.shape[0], W1)
                else:
                    ex.setValueTable(table)
                    ex.setPermutedCases(perm_i)
                    d1 = ex.createPathSet(data1_i.shape[0]); d1.load(data1_i)
                    d2 = ex.createPathSet(data2_i.shape[0]); d2.load(data2_i)
            finally:
                if gate_out is not None:
                    gate_out.set()
            t_up = time.perf_counter()
            st = dict(ex=ex, d1=d1, d2=d2, uid=uid_host, stream=e2e_streams[method], perm_t=state[method]["perm_t"], perm_all=state[method]["perm_all"])
            res = {}
            schedule_resident(st, res, collective=not overlap)
            results[method] = (st, res)
            if dbg:
                sys.stderr.write(f"[bench] e2e {method}: waited {(t_go - t_in) * 1e3:.1f} ms, uploads {(t_up - t_go) * 1e3:.1f} ms, "
                                 f"joins {(time.perf_counter() - t_up) * 1e3:.1f} ms\n")

        def step_e2e():
            import threading

            d2h = 0
            results = {}
            if fanout:
                t_f = time.perf_counter()
                fan_out()
                if dbg:
                    sys.stderr.write(f"[bench] rank {rank} e2e fan-out: {(time.perf_counter() - t_f) * 1e3:.1f} ms\n")
            if overlap:
                gate = threading.Event()
                errs = []

                def guarded(*args):
                    try:
                        e2e_method(*args)
                    except BaseException as e:  # re-raised on the main thread
                        errs.append(e)

                # method 1 first: its shorter joins are done by the time method 2's uploads finish (65.9 vs 68.2 ms the other way round)
                first, second = ("method2", "method1") if os.environ.get("GCRE_BENCH_E2E_ORDER") == "21" else ("method1", "method2")
                th = [threading.Thread(target=guarded, args=(first, results, None, gate)),
                      threading.Thread(target=guarded, args=(second, results, gate, None))]
                for t in th:
                    t.start()
                for t in th:
                    t.join()
                if errs:
                    raise errs[0]
                for method in ("method1", "method2"):
                    merge_last_level(*results[method])
            else:
                for method in ("method1", "method2"):
                    e2e_method(method, results, None, None)
            for method in ("method1", "method2"):
                st, res = results.pop(method)
                for k, r in res.items():
                    if not k.startswith("_"):
                        d2h += r.permuted_scores.nbytes // 2 + len(r.scores) * 24
                ex = st["ex"]
                del res, st
                ex.close()
            d2h_holder[0] = d2h

        for _ in range(2):  # untimed: block cache, page-locked staging and the copy streams reach their steady state
            step_e2e()
        # A freshly started host stretches single steps 2-6x for its first seconds (profiles/README.md: the first 2-GPU run of
        # round 2).  Keep warming up, untimed, until three consecutive steps agree within 15 % - at most 20 more steps (~1.2 s);
        # every rank sees the same (max over ranks) times, so all ranks stop together.
        e2e_warmup, recent = 2, []
        for _ in range(20):
            sync_all()
            t_w = time.perf_counter()
            step_e2e()
            torch.cuda.synchronize()
            t_w = torch.tensor([time.perf_counter() - t_w], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t_w, op=dist.ReduceOp.MAX)
            e2e_warmup += 1
            recent = (recent + [float(t_w.item())])[-3:]
            if len(recent) == 3 and max(recent) <= 1.15 * min(recent):
                break
        sync_all()
        gc.collect()
        gc.freeze()
        gc.disable()  # as in the resident region: a cyclic GC pass costs 100+ ms with torch imported
        e2e_steps = a.steps if a.e2e_steps <= 0 else a.e2e_steps  # host contention comes in ~0.5 s bursts: a stable e2e figure needs ~30 steps
        per_step = []
        for i in range(e2e_steps):
            sync_all()  # every rank starts the step together; the step's own time is host wall clock, result read-back included
            t_dbg = time.perf_counter()
            step_e2e()
            torch.cuda.synchronize()
            per_step.append(time.perf_counter() - t_dbg)
        gc.enable()
        t_steps = torch.tensor(per_step, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t_steps, op=dist.ReduceOp.MAX)  # per step: the slowest rank
        per_step = t_steps.cpu().numpy()
        if rank == 0:
            sys.stderr.write("[bench] e2e ms per step (max over ranks): " + " ".join(f"{1e3 * t:.1f}" for t in per_step) + "\n")
        # E = work per step / MEDIAN step time: the step is ~60 ms of host packing, PCIe copies and joins on a shared host, and
        # single steps are stretched by tens of ms when the host is busy (mean, min and max are in the object too)
        dt = torch.tensor([float(np.median(per_step))], dtype=torch.float64)
        e2e = {"value": pp_step / float(dt.item()), "unit": "pair*perm/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h_holder[0]),
               "ms_per_step": float(dt.item()) * 1e3, "steps": e2e_steps, "warmup_steps": e2e_warmup, "ms_per_step_mean": float(per_step.mean()) * 1e3,
               "ms_per_step_max": float(per_step.max()) * 1e3, "ms_per_step_min": float(per_step.min()) * 1e3,
               "value_from_mean": pp_step / float(per_step.mean()),
               "timing": "host wall clock per step incl. uploads and result read-back, max over ranks per step; value = pair*perm per step / MEDIAN step time", "host_input_bytes_per_step": int(host_input_bytes),
               "input_path": ("rank 0 packs the int matrices on host threads and uploads bits + table once per step, NCCL broadcast to the other ranks; "
                              "every rank uploads its own permutation block" if fanout else
                              "int matrices packed to bits by host threads inside gcre_pathset_load_i32, bits uploaded" if host_packed else
                              "int matrices uploaded, packed on the device"),
               "host_threads": 2 if overlap else 1,
               "note": "host IntegerMatrix data + CaseORControl int matrix + f64 value table + join indices uploaded every step (pinned), per method; "
                       "the two methods are submitted from two host threads on two streams, so one method's uploads overlap the other's joins"
                       if overlap else
                       "host IntegerMatrix data + CaseORControl int matrix + f64 value table + join indices uploaded every step (pinned), per method"}

    # ---- CPU baseline + parity of what was benchmarked: the reference's own level-4 join on the bench inputs, compared with
    #      the GPU's level-4 result of the last timed step (SURVEY App. A.7 rule: f32 maxima bit for bit, the multiset of top-K
    #      scores, every entry above the K-th score; entries tied with the K-th score only need to carry that score) ----
    cpu, parity = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline and w.value_table is None and (w.n_cases + 1) * (w.n_ctrls + 1) * 8 <= (8 << 30):
        # the table was generated on the device (no host generator finishes at this size): the CPU leg gets a copy of it
        w.value_table = state["method1"]["ex"].getValueTable()
    if rank == 0 and world == 1 and not a.no_cpu_baseline and w.value_table is not None and a.path_length >= 4:
        arm = None
        cpu_edges = a.cpu_edges or (a.n_edges if w.n_patients <= 20000 else max(2000, a.n_edges // 20))
        try:
            if cpu_edges >= a.n_edges:
                arm = ReferenceArm(w, a)
                cpu, ref_out = arm.sample(a.cpu_seconds, results=True)
                parity = check_parity(ref_out, last_out, state, lv["4"], w, api, cpu_perm_count(w, a),
                                      lambda st: st["ex"].setPermutedMasks(w.perm_masks[:batch_perms]))
            else:
                # SURVEY 8d: where the reference cannot run the shape, time the largest runnable sub-shape with identical W - the same
                # cohort size, permutations and value table over a smaller network (its cost per pair*perm depends on W and I only)
                a_sub = argparse.Namespace(**vars(a))
                a_sub.n_edges, a_sub.n_genes = cpu_edges, max(200, int(a.n_genes * cpu_edges / a.n_edges))
                w_sub = synth.make_workload(a.n_cases, a.n_ctrls, a_sub.n_genes, a_sub.n_edges, cpu_perm_count(w, a), a.seed, max_path_length=a.path_length,
                                            real_table=True, host_table=False)
                w_sub.value_table = w.value_table
                # method 1 only: at this cohort size every method-2 thread needs its own (n+1)^2 f64 table (20 GB at 50,000 patients),
                # copied again for every join and never freed - one thread would be all this host can hold
                arm = ReferenceArm(w_sub, a_sub, methods=("method1",))
                cpu = arm.sample(a.cpu_seconds)
                cpu["sample"] = (f"SUB-SHAPE with the benchmark's W64 and value table: {w_sub.n_patients} patients, {w_sub.net.n_genes} genes, {a_sub.n_edges} edges "
                                 f"({w_sub.net.levels['4'].n_pairs} level-4 pairs); ") + cpu["sample"]
                parity = {"checked": False, "why": "the CPU leg ran a sub-shape (smaller network); parity of this cohort size is covered by tests/test_fullsize_gpu.py "
                                                   "and the 32-bit-carrier tests"}
        except AssertionError:
            raise
        except Exception as e:  # the GPU numbers stand on their own
            cpu = {"value": None, "unit": "pair*perm/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e!r}"}
        finally:
            if arm is not None:
                arm.close()

    if rank == 0:
        cfg = full_config(a, w, world)
        line = {"metric": "path-pair*perm scores/s", "value": value, "unit": "pair*perm/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak" if (shard_perms or world == 1) else "strong", "vs_baseline": None,
                "dtype": "u64", "data": "synthetic", "config": cfg, "clocks": clocks,
                "e2e": e2e, "gpu_launches": int(n_launch), "roofline": roof, "cpu_baseline": cpu, "parity": parity, "multi_gpu_parity": multi_parity, "strong": strong, "per_level": per_level,
                "pair_perm_per_step": pp_step, "workload_gen_s": round(gen_s, 1)}
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
