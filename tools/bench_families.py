"""Device-resident Elston-Stewart on cohort ped files (fs_create_families, es_families_kernel): prints one JSON line.

For cohorts of 42 and 1000 trios, FP64 and compact (PL) input, post + single + gt + status written: variants/s, samples/s
and the bytes the kernel must move per sample over the HBM bandwidth they imply.  Inputs are sized past the 126 MB L2.
Beside them, at the same number of samples per call:
  (a) the message-program interpreter on the 42-trio forest through fs_create (the path cohorts of <= 128 members take);
  (b) the nuclear trio kernel on V x T trio variants, the ceiling: the same arithmetic with no cross-family reduction.
Usage: python tools/bench_families.py [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import famseq_b200 as fs  # noqa: E402
from famseq_b200 import synth  # noqa: E402


def gpu_name_and_power():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name(0)


def time_engine(eng, V, S, compact, steps=20, warmup=3, seed=1, method=fs.ES):
    """ms per call of run_device / run_pl_device on V variants of S columns (random PLs, device-resident)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    pl = torch.randint(0, 60, (V, S, 3), device="cuda", dtype=torch.int16, generator=g)
    pl[..., 0] = 0
    x = pl if compact else torch.from_numpy(synth.pl_table()).cuda()[pl.long()]
    flags = torch.randint(0, 4, (V,), device="cuda", dtype=torch.uint8, generator=g)
    post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
    single = torch.empty_like(post)
    gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
    status = torch.empty(V, dtype=torch.uint8, device="cuda")
    f = eng.run_pl_device if compact else eng.run_device
    stream = torch.cuda.current_stream().cuda_stream

    def call():
        f(method, V, x.data_ptr(), flags.data_ptr(), post.data_ptr(), single.data_ptr(), gt.data_ptr(), status.data_ptr(), stream=stream)
    for _ in range(warmup):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        call()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def bytes_per_sample(compact):
    # in (24 or 6) + post 24 + single 24 + gt 1; flags and status are per variant and negligible at these widths
    return (6 if compact else 24) + 49


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    hbm = 7.7e12
    rows = []
    for trios in (42, 1000):
        ped, _ = synth.forest([synth.trio()] * trios)
        S = ped.n
        for compact in (False, True):
            V = max(4096, int(1.2e9 // (S * bytes_per_sample(compact))))  # ~1.2 GB moved per call: far past the L2
            with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=0, families=True) as e:
                ms = time_engine(e, V, S, compact)
            row = dict(path="cohort", trios=trios, S=S, compact=compact, V=V, ms=ms, variants_per_s=V / ms * 1e3,
                       samples_per_s=V * S / ms * 1e3)
            row["hbm_fraction"] = row["samples_per_s"] * bytes_per_sample(compact) / hbm
            rows.append(row)
            if trios == 42:  # (a) the interpreter through fs_create on the same forest
                with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=0) as e:
                    ms = time_engine(e, V, S, compact)
                rows.append(dict(path="interpreter", trios=trios, S=S, compact=compact, V=V, ms=ms, variants_per_s=V / ms * 1e3,
                                 samples_per_s=V * S / ms * 1e3, hbm_fraction=V * S / ms * 1e3 * bytes_per_sample(compact) / hbm))
            # (b) the nuclear trio kernel on V x T trio variants
            t = synth.trio()
            with fs.Engine(t.ids, t.mids, t.fids, t.genders, [0, 1, 2], device=0) as e:
                ms = time_engine(e, V * trios, 3, compact)
            rows.append(dict(path="nuclear_trio", trios=trios, S=3, compact=compact, V=V * trios, ms=ms, variants_per_s=V * trios / ms * 1e3,
                             samples_per_s=V * S / ms * 1e3, hbm_fraction=V * S / ms * 1e3 * bytes_per_sample(compact) / hbm))
    res = dict(gpu=gpu_name_and_power(), hbm_bytes_per_s=hbm, rows=rows)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_families.json"), "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
