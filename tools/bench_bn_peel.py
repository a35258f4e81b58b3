"""Device-resident exact posteriors by conditioned peeling (method 4, BN_PEEL): prints one JSON line.

Variants/s of run_device with post + single + gt + status written, FP64 gene-dropped likelihoods (synth), -LRC 5 so that
every variant goes through the pedigree, CUDA events around `steps` calls after `warmup` calls.  Workloads:
  ped40         BN_PEEL (3 loop breakers, 27 peels) against the Gibbs sampler at 1 000 + 10 000 sweeps (its generated kernel,
                FAMSEQ_MCMC_JIT=1), the only other method that runs on it (BN enumeration refuses 40 members, ES refuses loops);
  cousins_loop  BN_PEEL (1 breaker, 3 peels) against BN enumeration (3^9 configurations);
  ped14         BN_PEEL (no breaker, one peel) against the ES interpreter (FAMSEQ_ES_JIT=0): the cost of the accumulators.
Usage: python tools/bench_bn_peel.py [--out DIR]"""
import argparse
import json
import os
import sys

os.environ["FAMSEQ_ES_JIT"] = "0"  # read at fs_create: the ES baseline is the interpreter
os.environ["FAMSEQ_MCMC_JIT"] = "1"  # the Gibbs baseline is the generated kernel, compiled during the warm-up calls

import numpy as np  # noqa: E402
import torch  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import famseq_b200 as fs  # noqa: E402
from bench_families import gpu_name_and_power  # noqa: E402
from famseq_b200 import synth  # noqa: E402


def time_method(e, method, lk, fl, steps, warmup=2, burn=0, rep=1):
    V, S = lk.shape[:2]
    x, flags = torch.from_numpy(lk).cuda(), torch.from_numpy(fl).cuda()
    post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
    single = torch.empty_like(post)
    gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
    status = torch.empty(V, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def call():
        e.run_device(method, V, x.data_ptr(), flags.data_ptr(), post.data_ptr(), single.data_ptr(), gt.data_ptr(),
                     status.data_ptr(), burn=burn, rep=rep, seed=1, stream=stream)
    for _ in range(warmup):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return ms, fs.Result(post.cpu().numpy(), single.cpu().numpy(), gt.cpu().numpy(), status.cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    prm = fs.Params.default()
    prm.lrc = 5.0
    rows, checks = [], {}
    cases = [("ped40", synth.ped40(), [("bn_peel", fs.BN_PEEL, 1 << 18, 0, 1), ("mcmc_1000_10000", fs.MCMC, 1 << 16, 1000, 10000)]),
             ("cousins_loop", synth.cousins_loop(), [("bn_peel", fs.BN_PEEL, 1 << 21, 0, 1), ("bn", fs.BN, 1 << 18, 0, 1)]),
             ("ped14", synth.ped14(), [("bn_peel", fs.BN_PEEL, 1 << 21, 0, 1), ("es_interpreter", fs.ES, 1 << 21, 0, 1)])]
    for name, ped, paths in cases:
        cols = ped.sequenced_cols()
        V_max = max(p[2] for p in paths)
        lk, fl = synth.synth_likelihoods(ped, V_max, seed=7, x_fraction=0.1)
        res = {}
        with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=prm, device=0) as e:
            breakers = len(e.bn_peel_program()[2])
            for path, method, V, burn, rep in paths:
                ms, res[path] = time_method(e, method, lk[:V], fl[:V], steps=3 if method == fs.MCMC else 10, burn=burn, rep=rep)
                rows.append(dict(pedigree=name, n=ped.n, path=path, breakers=breakers if method == fs.BN_PEEL else None, V=V,
                                 ms=ms, variants_per_s=V / ms * 1e3))
        other = [p[0] for p in paths if p[0] != "bn_peel"][0]
        a, b = res["bn_peel"], res[other]
        n = len(b.status)
        if other == "es_interpreter":
            checks[f"{name}_bytes_equal_es"] = bool(np.array_equal(a.post[:n], b.post) and np.array_equal(a.gt[:n], b.gt)
                                                   and np.array_equal(a.status[:n], b.status))
        elif other == "bn":
            checks[f"{name}_within_1e-9_of_bn"] = bool(np.array_equal(a.status[:n], b.status)
                                                      and np.allclose(a.post[:n], b.post, rtol=1e-9, atol=0))
        else:
            ok = (a.status[:n] == 0) & (b.status == 0)
            checks[f"{name}_max_abs_diff_vs_mcmc"] = float(np.abs(a.post[:n][ok] - b.post[ok]).max())
    line = json.dumps(dict(gpu=gpu_name_and_power(), lrc=5.0, checks=checks, rows=rows))
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bn_peel_bench.json"), "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
