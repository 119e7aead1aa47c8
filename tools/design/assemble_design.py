"""DESIGN.md = tools/design/DESIGN.template.md with its tables (NUMBERS_TABLE, CONFIGS_TABLE, PERM_GEN_TABLE) filled from the JSON files under profiles/.

    python tools/design/assemble_design.py
"""
import json
import os
ROOT=os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
P=os.path.join(ROOT,"profiles")+"/"
L=lambda f: json.load(open(P+f))
def ms(d,m,l): return d["per_level"][m][l]["kernel_ms"]
n1=L("r2_bench_n1.json"); ref=L("r2_bench_reference_arm.json")
r3=L("r3_bench_n1.json")
e2=n1["e2e"]
numbers=f"""| what | result | file (`profiles/`) |
|---|---|---|
| whole level schedule, inputs resident (`value`) | **{n1['value']:.3g} pair·perm/s, {n1['ms_per_step']:.1f} ms per step** (round 1: 5.9e11, 45.6 ms) | `r2_bench_n1.json` |
| round 3, tail form of the level-4 join (§4.2) | **{r3['value']:.3g} pair·perm/s, {r3['ms_per_step']:.1f} ms per step**; level 4 {ms(r3,'method1','4'):.1f} / {ms(r3,'method2','4'):.1f} ms; `e2e` {r3['e2e']['value']:.3g}, {r3['e2e']['ms_per_step']:.0f} ms per step. A/B against the round-2 build in one call, three runs each: 7.22-7.29e+11 → 8.42-8.68e+11 (+15 to +20 % per pairing), outputs identical byte for byte; set-up it adds per method and step: provenance recording 0.3-0.4 ms, the eligibility pass 0.4 ms, `P` of data1 0.03 ms (`r3_level_schedule_kernels.json`). Config 5 at 1,000 permutations 2.69e+11 → 4.29e+11 (100 → 63 ms per step), path length 5 +2 %, 100 permutations (no tail form) within 0.3 ms per step. NVIDIA B200 at 1,000 W | `r3_bench_n1.json`, `r3_tail_form_ab.txt`, `r3_regressions.txt` |
| round 2 build: level-4 join (12.0 M pairs), method 1 / method 2 | {ms(n1,'method1','4'):.1f} / {ms(n1,'method2','4'):.1f} ms = {11988861*1000/ms(n1,'method1','4')*1e3:.3g} / {11988861*1000/ms(n1,'method2','4')*1e3:.3g} pair·perm/s (round 1: 11.2 / 19.4 ms) | same, `per_level` |
| … level 3 (1.35 M pairs, rows + counts kept) | {ms(n1,'method1','3'):.1f} / {ms(n1,'method2','3'):.1f} ms; levels 1a + 1b + 2: {ms(n1,'method1','1a')+ms(n1,'method1','1b')+ms(n1,'method1','2'):.1f} / {ms(n1,'method2','1a')+ms(n1,'method2','1b')+ms(n1,'method2','2'):.1f} ms; carrier-list construction and row selection ≈ 4 % of the step's kernel time | `r2_step_launches.txt` |
| roofline of the level-4 launches | `bound: issue`: {n1['roofline']['achieved']:.3g} warp instructions/s = **{n1['roofline']['frac']:.2f}** of the measured issue rate; ncu: issue slots 70 % / 67 % active, ALU pipe 65 % / 61 %; DRAM traffic {n1['roofline']['traffic']/1e9:.1f} GB per step = {n1['roofline']['hbm_frac']:.2f} of the HBM peak; algorithmic (SURVEY 8d): {n1['roofline']['algorithmic']['x_measured_popc_peak']:.0f}× the measured POPC roof, {n1['roofline']['algorithmic']['x_measured_hbm_peak']:.2f}× the HBM peak | `r2_bench_n1.json`, `r2_counts.json`, `r2_final_full.txt` |
| from host R-format int matrices (`e2e`, median of ≥ 20 steps) | **{e2['value']:.3g}, {e2['ms_per_step']:.0f} ms per step** (mean {e2['ms_per_step_mean']:.0f}, min {e2['ms_per_step_min']:.0f}, max {e2['ms_per_step_max']:.0f}: the host is shared and single steps are stretched by tens of ms); uploads ≈ 17 ms per method (two 600 MB int matrices packed to bits on 16 host threads - AVX-512 compare-to-mask, 160 GB/s, 4 ms each - and uploaded, value table 4 ms, permutation matrix 1 ms; every setter returns only when the caller's buffer is free again), joins 20 / 25 ms, the second method's uploads overlap the first's joins (`r2_e2e_debug.err`); round 1: 3.9e11, 68.6 ms | `r2_bench_n1.json`, `r2_e2e_debug.err` |
| reference `join_base.cpp`, g++ -O3 AVX-512, 16 host cores of the same box | whole level-4 joins: {n1['cpu_baseline']['value']:.3g} (method 1 {n1['cpu_baseline']['detail']['method1']['pair_perm_per_s']:.3g} in {n1['cpu_baseline']['detail']['method1']['seconds_measured']:.1f} s, method 2 {n1['cpu_baseline']['detail']['method2']['pair_perm_per_s']:.3g} in {n1['cpu_baseline']['detail']['method2']['seconds_measured']:.1f} s); `--impl reference --steps 20 --warmup 5`: {ref['value']:.3g}, {ref['wall_s']:.0f} s wall | `r2_bench_n1.json`, `r2_bench_reference_arm.json` |
| parity of the benchmarked workload | 23,977,722 level-4 pairs × 1,000 permutations, both methods, against the reference's join in the same run: 0 mismatches | `r2_bench_n1.json` `parity` |"""
rows=[]
def strong(n):
    d=L(f"r2_bench_n{n}.json"); s=d["strong"]
    return d, f"{s['ms_per_step_one_gpu']:.1f} → {s['ms_per_step']:.1f} ms = {s['speedup']:.2f}× ({s['efficiency']:.2f})"
n2,s2=strong(2); n4,s4=strong(4); n8,s8=strong(8)
c4={n:L(f"r2_config4_n{n}.json") for n in (2,4,8)}
c5={p:L(f"r2_config5_n1_p{p}.json") for p in (100,1000,10000,100000)}
c58a=L("r2_config5_n8_p8000total.json"); c58b=L("r2_config5_n8_p100000total.json")
p100=L("r2_bench_config3_p100.json"); len5=L("r2_bench_config3_len5.json")
cpu5=c5[1000]["cpu_baseline"]
configs=f"""| Config | How it is covered | Result |
|---|---|---|
| 1 vignette m1 len2 p100, 2 vignette m2 len3 p1000 | golden fixtures from the reference itself on the bundled `random.phenotype.data` (`tests/golden/vignette_*.npz`), CPU + GPU, every kernel form | bit-exact; a whole run (new JoinExec, table, masks, all joins) takes 1.2 ms and 1.9 ms against 1.9 ms and 29 ms for the reference on one host core - launch-latency bound |
| 3 synthetic 10k patients, 15k genes, len 4, 1,000 perms, m1+m2 | `bench.py` default; parity inside the run and in `tests/test_bench_workload_gpu.py` | 1 GPU {n1['value']:.3g} ({n1['ms_per_step']:.1f} ms/step); one block of 1,000 permutations per GPU (weak): 2 / 4 / 8 GPUs {n2['value']:.3g} / {n4['value']:.3g} / {n8['value']:.3g} ({n2['ms_per_step']:.1f} / {n4['ms_per_step']:.1f} / {n8['ms_per_step']:.1f} ms per step; `e2e` {n2['e2e']['value']:.3g} / {n4['e2e']['value']:.3g} / {n8['e2e']['value']:.3g}); the same fixed job row-sharded (`strong`): 2 GPUs {s2}, 4 GPUs {s4}, 8 GPUs {s8} - limited by the replicated levels 1a/1b/2 (3.2 ms of kernels), the per-join set-up kernels and host work (≈ 4 ms on one GPU, not sharded) and the merge (allreduce + top-K gather through the host), not by the collective: 38.6 ms (the build these multi-GPU runs used: one kernel change, 3.6 %, behind the final one) = ≈ 7 (not sharded) + 31.5 (levels 3 + 4), so 4 GPUs cannot do better than ≈ 15 ms (efficiency 0.64) and reach {n4['strong']['ms_per_step']:.1f} ms; the ≥ 0.7 target at 4 GPUs is not met |
| 3 at GWASPA's default of 100 permutations | `bench.py --n-perms 100` (split-carrier kernels, masks in shared memory at level 4) | {p100['value']:.3g} ({p100['ms_per_step']:.1f} ms/step, round 1 and the start of round 2: 30.2; level 4 {ms(p100,'method1','4'):.1f} / {ms(p100,'method2','4'):.1f} ms, level 3 {ms(p100,'method1','3'):.1f} / {ms(p100,'method2','3'):.1f}; issue-slot roofline {p100['roofline']['frac']:.2f}); 256 / 500 permutations: 24.6 / 32.9 ms per step (33 / 41 in round 1). VERDICT's ≤ 20 ms is not met: the kernels take 17.0 ms, ten joins' host work and set-up kernels the rest |
| 3 at path length 5 (108 M level-5 pairs) | `bench.py --path-length 5` | {len5['value']:.3g} ({len5['ms_per_step']:.0f} ms per step; level 5 {ms(len5,'method1','5'):.0f} / {ms(len5,'method2','5'):.0f} ms; round 1: 6.0e11, 406 ms) |
| 4 100k patients, len 5, 10,000 perms over 2/4/8 GPUs | `bench.py --n-cases 50000 --n-ctrls 50000 --path-length 5 --n-perms 10000/N` under torchrun; 32-bit carrier indices, value table generated on the device, 2 permutation batches at N = 2 (the reference cannot run this shape: App. D) | 2 / 4 / 8 GPUs: {c4[2]['value']:.3g} / {c4[4]['value']:.3g} / {c4[8]['value']:.3g} pair·perm/s = {c4[2]['ms_per_step']/1e3:.2f} / {c4[4]['ms_per_step']/1e3:.2f} / {c4[8]['ms_per_step']/1e3:.2f} s per 2.4e12-pair·perm step (level 5 of method 2: {ms(c4[2],'method2','5')/1e3:.1f} / {ms(c4[4],'method2','5')/1e3:.1f} / {ms(c4[8],'method2','5')/1e3:.1f} s); merged maxima checked against a single-rank recomputation (`multi_gpu_parity`: 0 mismatches). Not linear in N because a 1,024-permutation block is the unit of work: 5,000 / 2,500 / 1,250 permutations per GPU are 5 / 3 / 2 blocks. Limiter at 8 GPUs: the level-5 kernels themselves (90 % of the step), neither the replicated levels nor the collective (one 40 KB allreduce per method) |
| 5 perm sweep at 50k patients, len 4 | `--n-cases 25000 --n-ctrls 25000 --n-perms P`; more than 4,096 permutations run as sequential batches with the masks resident (`--perm-batch`) | 1 GPU, 100 / 1,000 / 10,000 / 100,000 permutations: {c5[100]['value']:.3g} / {c5[1000]['value']:.3g} / {c5[10000]['value']:.3g} / {c5[100000]['value']:.3g} ({c5[100]['ms_per_step']:.0f} ms / {c5[1000]['ms_per_step']:.0f} ms / {c5[10000]['ms_per_step']/1e3:.2f} s / {c5[100000]['ms_per_step']/1e3:.2f} s per step); issue-slot roofline {c5[100]['roofline']['frac']:.2f} (100, split-carrier kernels) and {c5[1000]['roofline']['frac']:.2f} (1,000); 8 GPUs, 8,000 / 100,000 permutations in total (the second one measured with the build before the last two kernel changes): {c58a['value']:.3g} / {c58b['value']:.3g} ({c58a['ms_per_step']:.0f} ms / {c58b['ms_per_step']/1e3:.2f} s per step). CPU beside it (`r2_config5_n1_p1000.json`): the reference on the largest sub-shape it can run with the same W64 = 782 and value table (50,000 patients, 7,500 edges, 849 k level-4 pairs, method 1, 16 threads): {cpu5['value']:.3g} pair·perm/s - method 2 needs a private 20 GB table per thread and join and never frees it (one thread is all a 196 GB host can hold) |"""
pg=L("r4_perm_gen.json")
perm_gen="| patients | permutations | strata | generator call (incl. layout rebuild) | generator kernel | layout rebuild | host `make_perm_masks` | host / device |\n|---|---|---|---|---|---|---|---|\n"
for r in pg["shapes"]:
    host=f"{r['host_ms']:,.0f} ms"+(f" (scaled from {r['host_perms_timed']:,} masks)" if r["host_scaled"] else "")
    perm_gen+=f"| {r['patients']:,} | {r['perms']:,} | {r['strata']} | {r['ms_per_call_with_layout']:.3f} ms | {r['kernel_ms']:.3f} ms | {r['layout_rebuild_kernel_ms']:.3f} ms | {host} | {r['host_over_device']:,.0f}× |\n"
bw=pg["bench_workload"]["methods"]
perm_gen+=(f"\n{pg['gpu']}; CUDA events over {pg['reps']} calls, kernel times from torch.profiler (`profiles/r4_perm_gen.json`, "
           f"`tools/perm_gen_timing.py`). Bench workload (config 3): a level-schedule replay after `generatePermutedMasks` gives outputs "
           f"byte-identical to one after `setPermutedMasks(make_perm_masks_philox(...))`: method 1 {'yes' if bw['method1']['byte_identical'] else 'NO'}, method 2 "
           f"{'yes' if bw['method2']['byte_identical'] else 'NO'}. Replay steps (methods 1 / 2, two timed each): {' / '.join(', '.join(f'{x:.0f}' for x in bw[m]['step_ms_generated']) for m in ('method1', 'method2'))} ms "
           f"after `generatePermutedMasks`, {' / '.join(', '.join(f'{x:.0f}' for x in bw[m]['step_ms_host_masks']) for m in ('method1', 'method2'))} ms with the host masks uploaded; "
           f"a replay uploads its inputs inside the step, so these are host-bound and vary by tens of ms with the load of the shared host. "
           f"The gap between the two method-1 columns cannot come from the generator, which takes 0.06 ms at this shape (table above).")
s=open(os.path.join(ROOT,"tools","design","DESIGN.template.md")).read()
s=s.replace("NUMBERS_TABLE",numbers).replace("CONFIGS_TABLE",configs).replace("PERM_GEN_TABLE",perm_gen)
s=s.replace("SC_P100_MS","%.1f"%p100['ms_per_step']).replace("SC_P100_L4","%.1f / %.1f"%(ms(p100,'method1','4'),ms(p100,'method2','4')))
open(os.path.join(ROOT,"DESIGN.md"),"w").write(s)
print("DESIGN.md written", len(s))
