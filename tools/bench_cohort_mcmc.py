"""Device-resident Gibbs sampler on cohort ped files (fs_create_cohort_mcmc): prints one JSON line.

FP64 and compact (PL) input, post + single + gt + status written, 1 000 burn-in + 10 000 sampling sweeps.  V is chosen from a
probe so that each timed call takes about a second ((c): one full wave of fs_create's kernel).  Workloads:
  (a) 1 000 trios;
  (b) 1 000 trios plus 10 x ped40 (double first cousins, 40 members: a looped family past the BN limit);
  (c) the 126-member forest of 42 trios, beside fs_create on the same file with its table-driven sampler
      (FAMSEQ_MCMC_JIT=0) and with the generated one (=1); the cohort engine's outputs equal the table-driven ones (checked).
For every row: variants/s, samples/s and Gibbs steps/s (V * (burn + rep) * members / time).  For (c), a torch.profiler
run splits one cohort call into head / class / finish kernel time.
Usage: python tools/bench_cohort_mcmc.py [--out DIR]"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import famseq_b200 as fs  # noqa: E402
from bench_families import gpu_name_and_power  # noqa: E402
from famseq_b200 import synth  # noqa: E402

BURN, REP = 1000, 10000


class Batch:
    """Device-resident random PL rows (and their FP64 decoding), flags and outputs for V variants of S columns."""

    def __init__(self, V, S, compact, seed=1):
        g = torch.Generator(device="cuda").manual_seed(seed)
        pl = torch.randint(0, 60, (V, S, 3), device="cuda", dtype=torch.int16, generator=g)
        pl[..., 0] = 0
        self.V, self.compact = V, compact
        self.x = pl if compact else torch.from_numpy(synth.pl_table()).cuda()[pl.long()]
        self.flags = torch.randint(0, 4, (V,), device="cuda", dtype=torch.uint8, generator=g)
        self.post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
        self.single = torch.empty_like(self.post)
        self.gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
        self.status = torch.empty(V, dtype=torch.uint8, device="cuda")

    def call(self, e):
        f = e.run_pl_device if self.compact else e.run_device
        f(fs.MCMC, self.V, self.x.data_ptr(), self.flags.data_ptr(), self.post.data_ptr(), self.single.data_ptr(), self.gt.data_ptr(),
          self.status.data_ptr(), burn=BURN, rep=REP, seed=7, v_offset=0, stream=torch.cuda.current_stream().cuda_stream)


def timed(e, b, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        b.call(e)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def engine(ped, jit=None, **kind):
    if jit is not None:
        os.environ["FAMSEQ_MCMC_JIT"] = jit
    try:
        return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=0, **kind)
    finally:
        os.environ.pop("FAMSEQ_MCMC_JIT", None)


def pick_v(ped, S, make):
    """V for a call of about a second: doubled (or more) from 256 until a call takes 0.7 s; the first calls also warm up
    modules and run-time compiles."""
    V = 256
    with make() as e:
        while True:
            b = Batch(V, S, False)
            b.call(e)
            torch.cuda.synchronize()
            ms = timed(e, b, 1)
            if ms >= 700 or V >= 1 << 20:
                return V
            V = int(min(1 << 20, V * max(2.0, min(16.0, 1000.0 / ms)))) // 256 * 256


def measure(workload, path, ped, make, V):
    S = len(ped.sequenced_cols())
    rows = []
    for compact in (False, True):
        b = Batch(V, S, compact)
        with make() as e:
            b.call(e)  # warm-up
            torch.cuda.synchronize()
            ms = timed(e, b, 2)
            info = e.info()
        rows.append(dict(workload=workload, path=path, members=ped.n, S=S, compact=compact, V=V, burn=BURN, rep=REP, ms=ms,
                         variants_per_s=V / ms * 1e3, samples_per_s=V * S / ms * 1e3,
                         gibbs_steps_per_s=V * (BURN + REP) * ped.n / ms * 1e3, gibbs_generator=info["gibbs_generator"]))
    return rows


def profile_split(ped, V):
    """Kernel time of one cohort call (FP64 input) by kernel: the head, each launch class, the finish."""
    S = len(ped.sequenced_cols())
    b = Batch(V, S, False)
    with engine(ped, cohort_mcmc=True) as e:
        b.call(e)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            b.call(e)
            torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        name = ev.key
        kind = ("head" if "es_cohort_head_kernel" in name else "finish" if "es_cohort_finish_kernel" in name
                else "mcmc_cohort_kernel" if "mcmc_cohort_kernel" in name else None)
        if kind:
            t = getattr(ev, "device_time_total", None)
            t = ev.cuda_time_total if t is None else t
            split[kind] = split.get(kind, 0.0) + t / 1e3
    return dict(V=V, ms=split)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    t0 = time.time()
    rows, checks = [], {}
    a, _ = synth.forest([synth.trio()] * 1000)
    b, _ = synth.forest([synth.trio()] * 1000 + [synth.ped40()] * 10)
    c, _ = synth.forest([synth.trio()] * 42)
    for name, ped in (("a", a), ("b", b)):
        make = lambda ped=ped: engine(ped, cohort_mcmc=True)  # noqa: E731
        rows += measure(name, "cohort_mcmc", ped, make, pick_v(ped, len(ped.sequenced_cols()), make))
    makes = {"cohort_mcmc": lambda: engine(c, cohort_mcmc=True), "fs_create_table": lambda: engine(c, jit="0"),
             "fs_create_generated": lambda: engine(c, jit="1")}
    # fs_create's table-driven kernel keeps 3 blocks of 256 chains resident per SM and a block's chains run for the whole
    # call, so any V up to one full wave takes the same time: time it (and the others) at one full wave
    Vc = torch.cuda.get_device_properties(0).multi_processor_count * 3 * 256
    for path, make in makes.items():
        rows += measure("c", path, c, make, Vc)
    split = profile_split(c, Vc)
    lk, fl = synth.synth_likelihoods(c, 512, seed=4, x_fraction=0.2)
    with makes["fs_create_table"]() as x, makes["cohort_mcmc"]() as y:
        p, q = x.run(fs.MCMC, lk, fl, burn=50, rep=200, seed=3), y.run(fs.MCMC, lk, fl, burn=50, rep=200, seed=3)
    checks["c_outputs_equal_table_driven"] = bool(all(np.array_equal(getattr(p, k), getattr(q, k)) for k in ("post", "single", "gt", "status")))
    res = dict(gpu=gpu_name_and_power(), checks=checks, rows=rows, c_profile_split=split, wall_s=time.time() - t0)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "cohort_mcmc_bench.json"), "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
