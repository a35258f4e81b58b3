"""Device-resident Bayesian network on cohort ped files (fs_create_cohort_bn): prints one JSON line.

FP64 and compact (PL) input, post + single + gt + status written, samples/s; inputs sized past the 126 MB L2
(tools/bench_families.py: time_engine).  Workloads:
  (a) 1 000 trios through fs_create_cohort_bn, beside fs_create_cohort (ES) on the same file;
  (b) 1 000 trios plus 100 each of sibship(4), half_sibs and cousins_loop (a looped family) through fs_create_cohort_bn;
  (c) a forest of 5 trios through fs_create BN (3^15 configurations per variant: compute-bound, so 4 096 variants) and
      through fs_create_cohort_bn (27 configurations per family), whose outputs agree to 1e-9 (checked).
Usage: python tools/bench_cohort_bn.py [--out DIR]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import famseq_b200 as fs  # noqa: E402
from bench_families import bytes_per_sample, gpu_name_and_power, time_engine  # noqa: E402
from famseq_b200 import synth  # noqa: E402


def measure(workload, path, ped, compact, method, V=None, **kind):
    S = len(ped.sequenced_cols())
    V = V or max(4096, int(1.2e9 // (S * bytes_per_sample(compact))))  # ~1.2 GB moved per call: far past the L2
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=0, **kind) as e:
        ms = time_engine(e, V, S, compact, steps=10 if V == 4096 else 20, method=method)
        launches = e.info()["kernel_launches"]
    return dict(workload=workload, path=path, S=S, compact=compact, V=V, ms=ms, samples_per_s=V * S / ms * 1e3, launches=launches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rows, checks = [], {}
    a, _ = synth.forest([synth.trio()] * 1000)
    b, _ = synth.forest([synth.trio()] * 1000 + [synth.sibship(4), synth.half_sibs(), synth.cousins_loop()] * 100)
    c, _ = synth.forest([synth.trio()] * 5)
    for compact in (False, True):
        rows.append(measure("a", "cohort_bn", a, compact, fs.BN, cohort_bn=True))
        rows.append(measure("a", "cohort_es", a, compact, fs.ES, cohort=True))
        rows.append(measure("b", "cohort_bn", b, compact, fs.BN, cohort_bn=True))
        rows.append(measure("c", "fs_create_bn", c, compact, fs.BN, V=4096))
        rows.append(measure("c", "cohort_bn", c, compact, fs.BN, cohort_bn=True))
    lk, fl = synth.synth_likelihoods(c, 2048, seed=4, x_fraction=0.2)
    args_c = (c.ids, c.mids, c.fids, c.genders, c.sequenced_cols())
    with fs.Engine(*args_c, device=0) as x, fs.Engine(*args_c, device=0, cohort_bn=True) as y:
        p, q = x.run(fs.BN, lk, fl), y.run(fs.BN, lk, fl)
    checks["c_outputs_agree_1e-9"] = bool(np.array_equal(p.status, q.status) and np.array_equal(p.gt, q.gt)
                                         and np.allclose(p.post, q.post, rtol=1e-9, atol=0))
    res = dict(gpu=gpu_name_and_power(), checks=checks, rows=rows)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "cohort_bn_bench.json"), "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
