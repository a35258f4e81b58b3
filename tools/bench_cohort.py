"""Device-resident Elston-Stewart on cohort ped files with extended families (fs_create_cohort): prints one JSON line.

FP64 and compact (PL) input, post + single + gt + status written, samples/s; inputs sized past the 126 MB L2
(tools/bench_families.py: time_engine).  Workloads:
  (a) 1 000 trios and 100 three-generation families (three_generations(3)) through fs_create_cohort;
  (b) the same 1 000 trios alone, through fs_create_families and fs_create_cohort (no program family: the same kernel,
      so the same bytes -- checked -- and the same speed);
  (c) a forest of 128 members mixing ped14, half_sibs, three_wives, sibship(8) and 28 trios, through fs_create (the
      whole-forest interpreter, FAMSEQ_ES_JIT=0) and through fs_create_cohort (one vector file per family).
Usage: python tools/bench_cohort.py [--out DIR]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
os.environ["FAMSEQ_ES_JIT"] = "0"  # fs_create's pedigree runs in the interpreter: the generated kernel is another path
import famseq_b200 as fs  # noqa: E402
from bench_families import bytes_per_sample, gpu_name_and_power, time_engine  # noqa: E402
from famseq_b200 import synth  # noqa: E402


def outputs(eng, S, V=2048, seed=3):
    """post, single, gt, status of one run_pl_device call on seeded PLs."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    pl = torch.randint(0, 60, (V, S, 3), device="cuda", dtype=torch.int16, generator=g)
    pl[..., 0] = 0
    flags = torch.randint(0, 4, (V,), device="cuda", dtype=torch.uint8, generator=g)
    post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
    single = torch.empty_like(post)
    gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
    status = torch.empty(V, dtype=torch.uint8, device="cuda")
    eng.run_pl_device(fs.ES, V, pl.data_ptr(), flags.data_ptr(), post.data_ptr(), single.data_ptr(), gt.data_ptr(), status.data_ptr(),
                      stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in (post, single, gt, status)]


def measure(workload, path, ped, S, compact, **kind):
    V = max(4096, int(1.2e9 // (S * bytes_per_sample(compact))))  # ~1.2 GB moved per call: far past the L2
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=0, **kind) as e:
        ms = time_engine(e, V, S, compact)
    return dict(workload=workload, path=path, S=S, compact=compact, V=V, ms=ms, samples_per_s=V * S / ms * 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rows, checks = [], {}
    trios, _ = synth.forest([synth.trio()] * 1000)
    a, _ = synth.forest([synth.trio()] * 1000 + [synth.three_generations(3)] * 100)
    c, _ = synth.forest([synth.ped14(), synth.half_sibs(), synth.three_wives(), synth.sibship(8)] + [synth.trio()] * 28, shuffle_seed=1)
    assert c.n == 128
    for compact in (False, True):
        rows.append(measure("a", "cohort", a, a.n, compact, cohort=True))
        rows.append(measure("b", "families", trios, trios.n, compact, families=True))
        rows.append(measure("b", "cohort", trios, trios.n, compact, cohort=True))
        rows.append(measure("c", "interpreter", c, c.n, compact))
        rows.append(measure("c", "cohort", c, c.n, compact, cohort=True))
    args_b = (trios.ids, trios.mids, trios.fids, trios.genders, trios.sequenced_cols())
    with fs.Engine(*args_b, device=0, families=True) as x, fs.Engine(*args_b, device=0, cohort=True) as y:
        checks["b_outputs_equal"] = all(np.array_equal(p, q) for p, q in zip(outputs(x, trios.n), outputs(y, trios.n)))
    args_c = (c.ids, c.mids, c.fids, c.genders, c.sequenced_cols())
    with fs.Engine(*args_c, device=0) as x, fs.Engine(*args_c, device=0, cohort=True) as y:
        checks["c_outputs_equal"] = all(np.array_equal(p, q) for p, q in zip(outputs(x, c.n), outputs(y, c.n)))
    res = dict(gpu=gpu_name_and_power(), checks=checks, rows=rows)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "cohort_bench.json"), "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
