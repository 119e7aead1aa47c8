# kernel times and launch counts of one level schedule (bench workload) per method under torch.profiler, every kernel: carrier-list
# builds (half_popcount / build_lists), P build of data1, eligibility pass, provenance recording, level-3 and level-4 joins.
# Run from the root of the tree whose build is measured.
import json, os, sys
sys.path.insert(0, os.getcwd())
import torch
from torch.profiler import profile, ProfilerActivity
from geneticscre_b200 import api, synth, schedule, build
build.build()
w = synth.make_workload(5000, 5000, 15000, 150000, 1000, 20261021, max_path_length=4, real_table=True)
out = {}
for method in ("method1", "method2"):
    ex = api.JoinExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = 10
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    schedule.replay_levels(ex, api.UidRelSet, w, 4)  # warm-up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res, _ = schedule.replay_levels(ex, api.UidRelSet, w, 4)
        torch.cuda.synchronize()
    agg = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            k = e.name.split("(")[0][:90]
            a = agg.setdefault(k, [0, 0.0])
            a[0] += 1
            a[1] += e.device_time_total / 1000.0 if hasattr(e, "device_time_total") else e.cuda_time_total / 1000.0
    out[method] = {"level3_info": res["3"].info, "level4_info": res["4"].info,
                   "kernels_ms": {k: v for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])}}
    ex.close()
print(json.dumps(out, indent=1))
