"""Where the time of fs_create_cohort_bn goes on 1 000 trios (tools/bench_cohort_bn.py, workload a): torch.profiler's
CUDA time per kernel over 10 device-resident FP64 calls, beside fs_create_cohort (ES) on the same file.
Usage: python profiles/cohort_bn_profile.py > out.txt"""
import os
import sys

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import famseq_b200 as fs  # noqa: E402
from bench_families import gpu_name_and_power, time_engine  # noqa: E402
from famseq_b200 import synth  # noqa: E402

ped, _ = synth.forest([synth.trio()] * 1000)
S, V = ped.n, 5479
print(gpu_name_and_power())
for method, kind in ((fs.BN, dict(cohort_bn=True)), (fs.ES, dict(cohort=True))):
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=0, **kind) as e:
        time_engine(e, V, S, False, steps=3, method=method)  # warm-up
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            time_engine(e, V, S, False, steps=10, warmup=0, method=method)
    print(list(kind)[0])
    print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=8, max_name_column_width=70))
