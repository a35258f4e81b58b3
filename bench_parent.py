#!/usr/bin/env python
"""bench.py -- variants/second of the B200-native FamSeq posterior engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Headline workload (BASELINE.json configs[2], the one quoted at 1/2/4/8 GPUs): synthetic trio pedigree,
Elston-Stewart peeling, 10 M variants PER GPU (weak scaling: every rank owns its own contiguous slice of
sites, no data-path collective).  A "step" is one pass of the kernel over the rank's resident batch.
  value    : whole-job variants/s, inputs and outputs resident in HBM, CUDA events, max over ranks
  e2e      : the same batch through the C ABI on HOST (pinned) buffers, H2D + D2H inside: fs_run_pl() -- uint16 PL
             fields up, post + gt + status down (single = NULL); `e2e_fp64_full` is fs_run() with FP64 likelihoods up
             and post + single down; both carry the plain-memcpy ceiling of the same byte mix measured in this run
  roofline : HBM, algorithmic bytes = 73*S+2 per variant (221 B for a trio), peak from MEASURED_PEAKS.json;
             `layouts` has the compact-input kernels (167 B and 95 B per variant) with their own rooflines
  methods  : ES on ped14, BN (3^14 exhaustive enumeration, ped14) and MCMC (ped40 with loops, 1 000 + 10 000
             sweeps) timed the same way; also as flat top-level scalars (bn_ped14_variants_per_s, ...)
  cpu_baseline : the reference's own CPU engine (oracle/_ref/ref_harness, built from the unmodified
             reference sources) on all host cores, one pass over the whole 10 M-variant configuration
  cli_e2e  : file -> file through this repo's FamSeq command line; ref_cuda_bn: the reference's own CUDA build
`--impl reference` times that CPU engine as the reference arm (same metric string, same sample definition).
For N > 1 the line also carries `e2e_single_process`: ONE fs_create_multi engine over all N GPUs writing one ordered buffer.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 20261018
METHOD_ID = {"bn": 1, "es": 2, "mcmc": 3}
# ONE metric string for both arms (the driver divides the two lines only when they name the same metric)
METRIC = "variants/sec (ES peeling, trio)"
UNIT = "variants/s"


def algorithmic_bytes(S: int, compact_in: bool = False, single: bool = True) -> int:
    """SURVEY 8(d): lk 24S (compact input: 6S) + 1 flag byte in; post (+ single) 24S each, gt S, status 1 out.
    Canonical layout 73 S + 2 (221 B for a trio); compact input 55 S + 2 (167 B); compact input without the
    individual-only posteriors 31 S + 2 (95 B)."""
    return (6 if compact_in else 24) * S + 1 + (48 if single else 24) * S + S + 1


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


# ----------------------------------------------------------------------------------------------------
# clocks during the timed region
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.nvml = None
        self.samples = []  # (sm_mhz, max_mhz, reasons bitmask) polled through NVML every ~1 ms
        self._stop = False
        self._max = None
        self.error = None

    def sample_now(self):
        """One synchronous NVML sample (called by the timing loop while the kernels are in flight)."""
        if self.nvml is None:
            return
        import pynvml as nv

        h = self.nvml
        try:
            if self._max is None:
                self._max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception as ex:  # noqa: BLE001
            self.error = repr(ex)
            return
        try:
            reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:  # noqa: BLE001
            try:
                reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            except Exception as ex:  # noqa: BLE001
                self.error = repr(ex)
                reasons = 0
        self.samples.append((sm, self._max, reasons))

    def _poll(self):
        while not self._stop:
            self.sample_now()
            time.sleep(0.001)

    def __enter__(self):
        try:  # NVML polling catches regions of a few milliseconds that an nvidia-smi loop would miss
            import pynvml as nv

            nv.nvmlInit()
            self.nvml = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.nvml is not None:
            self._stop = True
            self.t.join(timeout=2)
            return
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        if self.nvml is not None and self.samples:
            import pynvml as nv

            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            seen = 0
            for s in self.samples:
                seen |= s[2]
            return {"sm_mhz": int(statistics.median(s[0] for s in self.samples)), "sm_max_mhz": int(self.samples[0][1]),
                    "reasons": sorted(k for k, b in bits.items() if seen & b), "samples": len(self.samples), "source": "nvml"}
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6 or not f[0].isdigit():
                continue
            sm.append(int(f[0])); mx.append(int(f[1]))
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "error": self.error}
        return {"sm_mhz": int(statistics.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# CPU reference arm
# ----------------------------------------------------------------------------------------------------
class CpuSample:
    """The reference CPU engine on every host core: one single-threaded process per core on disjoint slices of ONE
    prepared sample of the workload (BASELINE.md section 4).  The inputs are generated and written once; every run()
    is one pass of all processes over the whole sample and returns variants/s (engine only: set_LK + calPostProb* +
    accessors, timed inside the harness; no file I/O).  The same object -- the same sample definition -- serves the
    `cpu_baseline` of our arm and every step of `--impl reference`."""

    def __init__(self, ped, method: str, variants: int, burn: int = 0, rep: int = 0):
        from famseq_b200 import synth
        from oracle import oracle as O

        self.O, self.ped, self.method, self.variants, self.burn, self.rep = O, ped, method, variants, burn, rep
        self.cores = os.cpu_count() or 1
        self.per_core = max(1, variants // self.cores)
        self.variants = self.per_core * self.cores
        self.td = tempfile.TemporaryDirectory()
        self.kind = "reference" if O.have_ref() else "port"
        self.ped_path = os.path.join(self.td.name, "p.ped")
        ped.write(self.ped_path)
        self.inputs = []
        for c in range(self.cores):
            lk, fl = synth.synth_likelihoods(ped, self.per_core, SEED + 1, v0=c * self.per_core)
            if self.kind == "reference":
                fin = os.path.join(self.td.name, f"in{c}.bin")
                with open(fin, "wb") as fh:
                    fh.write(np.array([lk.shape[0], lk.shape[1]], np.int32).tobytes())
                    fh.write(fl.tobytes())
                    fh.write(np.ascontiguousarray(lk).tobytes())
                self.inputs.append(fin)
            else:
                self.inputs.append((lk, fl))
        self.sample = (f"{self.variants} variants of the same synthetic workload = {self.cores} single-threaded processes x "
                       f"{self.per_core} variants, one pass per step (engine only: set_LK + calPostProb + accessors, no file I/O)")

    def run(self) -> float:
        O, mid, cols = self.O, METHOD_ID[self.method], self.ped.sequenced_cols()
        if self.kind == "reference":
            cmds = [[O.REF_HARNESS, f"ped={self.ped_path}", f"method={mid}", f"burn={self.burn}", f"rep={self.rep}", "seed=1",
                     "cols=" + ",".join(str(x) for x in cols), "repeat=1", f"in={fin}"] for fin in self.inputs]
            running = [subprocess.Popen(a, stdout=subprocess.PIPE, text=True) for a in cmds]
            outs = [json.loads(p.communicate()[0].strip().splitlines()[-1]) for p in running]
            return self.variants / max(o["elapsed_s"] for o in outs)
        import multiprocessing as mp

        with mp.Pool(self.cores) as pool:  # the C restatement, one process per core
            res = pool.starmap(_port_worker, [(self.ped, mid, lk, fl, self.burn, self.rep) for lk, fl in self.inputs])
        return self.variants / max(res)

    def baseline(self, runs: int = 3) -> dict:
        self.run()  # page cache, CPU clocks
        v = float(statistics.mean(self.run() for _ in range(runs)))
        return {"value": v, "unit": UNIT, "cores": self.cores, "kind": self.kind, "sample": self.sample + f"; mean of {runs} passes"}

    def close(self):
        self.td.cleanup()


def _port_worker(ped, mid, lk, fl, burn, rep):
    from oracle import oracle as O

    t0 = time.perf_counter()
    O.run(ped, ped.sequenced_cols(), lk, fl, method=mid, burn=burn, rep=rep, rng=O.RNG_LIBC, seed=1)
    return time.perf_counter() - t0


# variants of the bounded CPU samples (ES: the whole 10 M-variant configuration, ~0.7 s per pass on 16 cores)
CPU_SAMPLE = {"bn": 64, "mcmc": 2048}


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, name, ped, method, variants, burn=0, rep=0):
        self.name, self.ped, self.method, self.variants, self.burn, self.rep = name, ped, method, variants, burn, rep


def time_device_path(torch, dist, fs, eng, wl: Workload, rank, world, steps, warmup, device_index, compact=False, single=True, data=None):
    """Kernel-only timing: inputs/outputs resident in HBM, CUDA events on the launch stream, max over ranks."""
    from famseq_b200 import synth

    V, S = wl.variants, len(wl.ped.sequenced_cols())
    if data is None:
        pl, fl = synth.synth_pl(wl.ped, V, SEED + METHOD_ID[wl.method], v0=rank * V)
        data = dict(h_pl=torch.from_numpy(pl.astype(np.uint16).view(np.int16)).pin_memory(), h_fl=torch.from_numpy(fl).pin_memory())
        data["h_lk"] = torch.from_numpy(synth.pl_to_likelihood(pl)).pin_memory()
        del pl
    d_in = (data["h_pl"] if compact else data["h_lk"]).cuda(non_blocking=True)
    d_fl = data["h_fl"].cuda(non_blocking=True)
    d_post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
    d_single = torch.empty_like(d_post) if single else None
    d_gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
    d_st = torch.empty(V, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()
    mid = METHOD_ID[wl.method]
    call = eng.run_pl_device if compact else eng.run_device

    def step():
        call(mid, V, d_in.data_ptr(), d_fl.data_ptr(), d_post.data_ptr(), d_single.data_ptr() if single else None, d_gt.data_ptr(),
             d_st.data_ptr(), burn=wl.burn, rep=wl.rep, seed=SEED, v_offset=rank * V, stream=stream.cuda_stream)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches0 = eng.info()["kernel_launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(device_index) as clk:
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(steps):
            step()
        e1.record(stream)
        clk.sample_now()  # the launches above are asynchronous: this sample is taken while they run
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.info()["kernel_launches"] - launches0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    failed = int(d_st.sum().item())
    keep = dict(data, d_post=d_post, d_gt=d_gt, d_st=d_st)
    return ms / steps, launches, clk.summary(), failed, keep


def time_e2e_path(torch, dist, eng, wl: Workload, rank, world, steps, warmup, keep, compact=True, single=False, phred=False):
    """The reference-facing call on pinned HOST buffers, H2D and D2H inside the timed region: fs_run_pl() (compact input,
    post + gt + status out), fs_run() (FP64 likelihoods in, single as well out) or fs_run_pl_phred() (compact input,
    posteriors as the six Phred digits the reference prints, 4 bytes per value)."""
    V, S = wl.variants, len(wl.ped.sequenced_cols())
    h_in, h_fl = (keep["h_pl"] if compact else keep["h_lk"]), keep["h_fl"]
    h_post = (torch.empty((V, S, 3), dtype=torch.int32) if phred else torch.empty((V, S, 3), dtype=torch.float64)).pin_memory()
    fixes = np.zeros(1 << 16, dtype=[("index", np.int64), ("p", np.float64)])
    n_fixes = [0]
    h_single = torch.empty((V, S, 3), dtype=torch.float64).pin_memory() if single else None
    h_gt = torch.empty((V, S), dtype=torch.uint8).pin_memory()
    h_st = torch.empty(V, dtype=torch.uint8).pin_memory()
    mid = METHOD_ID[wl.method]
    call = eng.run_pl_raw if compact else eng.run_raw

    def step():
        if phred:
            n_fixes[0] = eng.run_pl_phred_raw(mid, V, h_in.data_ptr(), h_fl.data_ptr(), h_post.data_ptr(), None, h_gt.data_ptr(), h_st.data_ptr(),
                                              fixes, len(fixes), burn=wl.burn, rep=wl.rep, seed=SEED, v_offset=rank * V)
            return
        call(mid, V, h_in.data_ptr(), h_fl.data_ptr(), h_post.data_ptr(), h_single.data_ptr() if single else None, h_gt.data_ptr(),
             h_st.data_ptr(), burn=wl.burn, rep=wl.rep, seed=SEED, v_offset=rank * V)

    for _ in range(max(1, min(warmup, 2))):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([sec], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    # the device-resident and the host path must have produced the same bytes
    same = bool(torch.equal(keep["d_gt"].cpu(), h_gt) and torch.equal(keep["d_st"].cpu(), h_st))
    if phred:  # every code must print what the reference prints for the device path's double (checked on the first 20 000 variants)
        import famseq_b200 as fs
        from oracle import oracle as O

        n = min(V, 20000) * S * 3
        codes = h_post.numpy().view(np.uint32).reshape(-1)[:n]
        exact = keep["d_post"][:min(V, 20000)].cpu().numpy().reshape(-1)
        decided = (codes >> 30) != 3
        same = same and n_fixes[0] <= len(fixes) and all(fs.phred_text(int(c)) == O.phred_text(float(x)) for c, x in zip(codes[decided], exact[decided]))
    else:
        same = same and bool(torch.equal(keep["d_post"].cpu(), h_post))
    h2d = h_in.numel() * h_in.element_size() + h_fl.numel()
    d2h = h_post.numel() * h_post.element_size() + (h_single.numel() * 8 if single else 0) + h_gt.numel() + h_st.numel() + (8 + 16 * min(n_fixes[0], len(fixes)) if phred else 0)
    return sec / steps, h2d, d2h, same


def host_copy_ceiling(torch, dist, world, h2d_bytes, d2h_bytes, reps=4):
    """What the host side can move at all: plain pinned cudaMemcpyAsync of the e2e step's byte mix -- `h2d_bytes` up and
    `d2h_bytes` down per rank, both directions concurrently on two streams, in 48 MB pieces like the engine's pipeline,
    all ranks at once -- no kernel.  Returns aggregate GB/s (both directions summed, max-over-ranks time)."""
    piece = 48 << 20
    up_h = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    dn_h = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    up_d = torch.empty(h2d_bytes, dtype=torch.uint8, device="cuda")
    dn_d = torch.empty(d2h_bytes, dtype=torch.uint8, device="cuda")
    s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()

    def once():
        with torch.cuda.stream(s_up):
            for o in range(0, h2d_bytes, piece):
                up_d[o:o + piece].copy_(up_h[o:o + piece], non_blocking=True)
        with torch.cuda.stream(s_dn):
            for o in range(0, d2h_bytes, piece):
                dn_h[o:o + piece].copy_(dn_d[o:o + piece], non_blocking=True)

    once()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([sec], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    return world * (h2d_bytes + d2h_bytes) * reps / sec / 1e9


def pin_rank_to_cores(local_rank: int, local_world: int):
    """Each rank gets its own contiguous share of the host cores (set before any pinned allocation, so that first-touch
    places the staging buffers near the threads that feed them)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        share = max(1, len(cores) // max(1, local_world))
        mine = cores[local_rank * share:(local_rank + 1) * share] or cores
        os.sched_setaffinity(0, mine)
        return mine
    except (AttributeError, OSError):
        return None


def profile_json(name):
    p = os.path.join(ROOT, "profiles", name)
    return json.load(open(p)) if os.path.exists(p) else {}


def cli_file_to_file(variants: int):
    """File -> file through the command line (SURVEY 8(d)): this repo's FamSeq on a synthetic trio VCF, wall clock of the
    whole process (CUDA context creation included) and the pipeline rate its own timers report."""
    from famseq_b200 import synth

    exe = os.path.join(ROOT, "famseq_b200", "bin", "FamSeq")
    if not os.path.exists(exe):
        return {"unavailable": "famseq_b200/bin/FamSeq is not built"}
    ped = synth.trio()
    with tempfile.TemporaryDirectory() as td:
        pp, vcf, out = os.path.join(td, "trio.ped"), os.path.join(td, "in.vcf"), os.path.join(td, "out.vcf")
        ped.write(pp)
        pl, fl = synth.synth_pl(ped, variants, seed=99)
        synth.write_vcf(vcf, ped, pl, fl)
        env = dict(os.environ, FAMSEQ_STATS="1")
        best = None
        for _ in range(3):  # first run warms the page cache
            t0 = time.perf_counter()
            r = subprocess.run([exe, "vcf", "-vcfFile", vcf, "-pedFile", pp, "-output", out, "-method", "2"], capture_output=True, text=True, env=env)
            wall = time.perf_counter() - t0
            if r.returncode != 0:
                return {"unavailable": f"FamSeq exited {r.returncode}: {r.stdout[-200:]}"}
            st = json.loads(r.stderr.strip().splitlines()[-1]) if r.stderr.strip() else {}
            if best is None or wall < best[0]:
                best = (wall, st)
        wall, st = best
        res = {"workload": f"{variants}-record synthetic trio VCF ({os.path.getsize(vcf)} bytes), -method 2, file -> file", "wall_s": wall,
               "variants_per_s_wall": variants / wall, "stats": st, "out_bytes": os.path.getsize(out)}
        if st.get("total_s"):
            res["variants_per_s_pipeline"] = variants / max(1e-9, st["total_s"] - st.get("start_wait_s", 0.0))
        ref = os.path.join(ROOT, "oracle", "_ref", "FamSeq")
        if os.path.exists(ref):  # the reference binary on a bounded head of the same file, and the byte comparison
            n = min(variants, 100_000)
            small, r_out, o_out = os.path.join(td, "small.vcf"), os.path.join(td, "r.vcf"), os.path.join(td, "o.vcf")
            synth.write_vcf(small, ped, pl[:n], fl[:n])
            t0 = time.perf_counter()
            subprocess.run([ref, "vcf", "-vcfFile", small, "-pedFile", pp, "-output", r_out, "-method", "2"], capture_output=True)
            res["reference_cli"] = {"variants": n, "variants_per_s_wall": n / (time.perf_counter() - t0), "cores": 1}
            subprocess.run([exe, "vcf", "-vcfFile", small, "-pedFile", pp, "-output", o_out, "-method", "2"], capture_output=True)
            res["identical_output"] = open(o_out, "rb").read() == open(r_out, "rb").read()
        return res


def reference_cuda_bn():
    """The reference's own CUDA build (family.cu compiled unmodified for sm_100a, BN only) on this GPU: the kernel to beat."""
    tool = os.path.join(ROOT, "tools", "bench_ref_gpu.py")
    try:
        r = subprocess.run([sys.executable, tool, "--large", "72", "--ours-large", "100000"], capture_output=True, text=True, timeout=300)
        d = json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as ex:  # noqa: BLE001
        return {"unavailable": repr(ex)[:200]}
    if "unavailable" in d:
        return d
    return {"workload": "ped14 BN through the command lines, file -> file", "reference_cuda_variants_per_s": d["reference_cuda"]["variants_per_s"],
            "ours_cli_variants_per_s": d["ours"]["variants_per_s"], "outputs_agree": d["outputs_agree"], "speedup": d["speedup"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variants", type=int, default=10_000_000, help="ES trio variants per GPU")
    ap.add_argument("--bn-variants", type=int, default=1_000_000)
    ap.add_argument("--mcmc-variants", type=int, default=1_000_000)
    ap.add_argument("--es14-variants", type=int, default=4_000_000)
    ap.add_argument("--cli-variants", type=int, default=2_000_000)
    ap.add_argument("--methods", default="es,es14,bn,mcmc,cli,refgpu", help="which lines to time (es is the headline)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--single-process", action="store_true", help="(default for N > 1; kept for compatibility)")
    ap.add_argument("--no-single-process", action="store_true",
                    help="N > 1: skip the e2e of ONE fs_create_multi engine over all N GPUs writing one ordered host buffer (rank 0 drives all GPUs)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    from famseq_b200 import synth

    trio, ped14, ped40 = synth.trio(), synth.ped14(), synth.ped40()
    config = {"workload": "synthetic trio pedigree, ES peeling (-method 2), 10 M variants per GPU (BASELINE.json configs[2])",
              "variants_per_gpu": args.variants, "pedigree_members": 3, "sequenced": 3,
              "layout": "lk[V][S][3] f64 + flags[V] u8 -> post,single[V][S][3] f64, gt[V][S] u8, status[V] u8",
              "l2_note": "per-step inputs+outputs (>= 0.95 GB) exceed the 126 MB L2, no flush needed",
              "parallelism": f"variant-sharded x{world}, no collective"}

    # ------------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        cpu = CpuSample(trio, "es", args.variants)
        rates = []
        for k in range(args.warmup + args.steps):
            v = cpu.run()
            if k >= args.warmup:
                rates.append(v)
        value = cpu.variants / float(statistics.mean(cpu.variants / r for r in rates))  # variants / mean step time
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * cpu.variants / value,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cpu.cores, "kind": cpu.kind, "sample": cpu.sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        cpu.close()
        return

    # ------------------------------------------------------------------------------------------------
    cores = pin_rank_to_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    import torch
    import torch.distributed as dist

    import famseq_b200 as fs

    if not torch.cuda.is_available() or fs.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; this engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    hbm_peak, peak_src, _ = measured_peaks()
    fp64_peak = fs.engine.measure_fp64_tflops(local_rank)
    methods = [m.strip() for m in args.methods.split(",") if m.strip()]

    def engine(ped, device=local_rank):
        return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=device)

    out = {}
    # ---- headline: ES trio ---------------------------------------------------------------------------
    wl = Workload("es", trio, "es", args.variants)
    e2e_steps = max(2, min(args.steps, 5))
    layouts = {}
    with engine(trio) as eng:
        # canonical layout (SURVEY 8(d)): FP64 likelihoods in, post + single out -- the headline `value`
        ms_step, launches, clocks, failed, keep = time_device_path(torch, dist, fs, eng, wl, rank, world, args.steps, args.warmup, local_rank)
        e2e64_s, h2d64, d2h64, same64 = time_e2e_path(torch, dist, eng, wl, rank, world, e2e_steps, args.warmup, keep, compact=False, single=True)
        data = {k: keep[k] for k in ("h_pl", "h_fl", "h_lk")}
        want_post, want_gt = keep["d_post"].clone(), keep["d_gt"].clone()
        del keep
        # compact input (fs_run_pl: uint16 PL decoded on the device), with and without the individual-only posteriors
        for tag, single in (("compact_in", True), ("compact_in_no_single", False)):
            ms_c, l_c, _, f_c, keep = time_device_path(torch, dist, fs, eng, wl, rank, world, args.steps, args.warmup, local_rank,
                                                        compact=True, single=single, data=data)
            ab = algorithmic_bytes(3, True, single)
            ach = ab * args.variants / (ms_c * 1e-3) / 1e9
            traffic = profile_json("es_trio_traffic.json").get(tag, {}).get("dram_bytes_per_variant")
            layouts[tag] = {"kernel": "es_nuclear_stream_kernel<1,%s,true> (uint16 PL tiles in, 4 per block, each prefetched by TMA under the one before; decode-table gather, identity column map)" % ("true" if single else "false"),
                            "value": world * args.variants / (ms_c * 1e-3), "unit": UNIT, "ms_per_step": ms_c, "gpu_launches": l_c,
                            "failed_variants": f_c, "same_bytes_as_canonical": bool(torch.equal(keep["d_post"], want_post) and torch.equal(keep["d_gt"], want_gt)),
                            "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                                         "traffic": traffic * args.variants if traffic else None, "algorithmic_bytes_per_variant": ab,
                                         "note": "these two layouts are bound by instruction issue / the FP64 pipe (~740 / ~650 instructions per variant, 325 of "
                                                 "them FP64; issue slots 72-74 % busy, FP64 pipe 58 %, profiles/r2x_r2x_es_l3.txt, _l5.txt), not by HBM"}}
        # headline e2e: the compact entry on pinned host buffers (2 B per likelihood up, post + gt + status down)
        e2e_s, h2d, d2h, same = time_e2e_path(torch, dist, eng, wl, rank, world, e2e_steps, args.warmup, keep, compact=True, single=False)
        # ... and with the posteriors as the reference prints them (Phred, six digits), 4 bytes per value
        e2ep_s, h2dp, d2hp, samep = time_e2e_path(torch, dist, eng, wl, rank, world, e2e_steps, args.warmup, keep, compact=True, single=False, phred=True)
        del keep, want_post, want_gt
    torch.cuda.empty_cache()
    ceiling = host_copy_ceiling(torch, dist, world, h2d, d2h)
    ceiling64 = host_copy_ceiling(torch, dist, world, h2d64, d2h64)
    ceilingp = host_copy_ceiling(torch, dist, world, h2dp, d2hp)
    value = world * args.variants / (ms_step * 1e-3)
    achieved = algorithmic_bytes(3) * args.variants / (ms_step * 1e-3) / 1e9
    tr = profile_json("es_trio_traffic.json").get("canonical", {})
    out.update({
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                     "traffic": tr.get("dram_bytes_per_variant", 0.0) * args.variants or None, "traffic_source": tr.get("source"),
                     "peak_source": peak_src, "algorithmic_bytes_per_variant": algorithmic_bytes(3),
                     "kernel": "es_nuclear_kernel<1,32,false,true,false> (one warp per block, TMA bulk load/store of a 32-variant tile, register-resident peeling: fast pass + complete pass)"},
        "e2e": {"value": world * args.variants / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_s * 1e3, "api": "fs_run_pl() on pinned host buffers: uint16 PL + flags up, post + gt + status down (single = NULL)",
                "matches_device_path": same, "mode": "one process per GPU",
                "host_copy_ceiling_gbs": ceiling, "achieved_gbs": world * (h2d + d2h) / e2e_s / 1e9,
                "frac_of_host_copy_ceiling": world * (h2d + d2h) / e2e_s / 1e9 / ceiling,
                "ceiling_note": "plain pinned cudaMemcpyAsync of the same byte mix, both directions at once, all ranks at once, no kernel"},
        "e2e_fp64_full": {"value": world * args.variants / e2e64_s, "unit": UNIT, "h2d_bytes_per_step": h2d64, "d2h_bytes_per_step": d2h64,
                          "ms_per_step": e2e64_s * 1e3, "api": "fs_run() on pinned host buffers: FP64 likelihoods up, post + single + gt + status down",
                          "matches_device_path": same64, "host_copy_ceiling_gbs": ceiling64,
                          "frac_of_host_copy_ceiling": world * (h2d64 + d2h64) / e2e64_s / 1e9 / ceiling64},
        "e2e_phred": {"value": world * args.variants / e2ep_s, "unit": UNIT, "h2d_bytes_per_step": h2dp, "d2h_bytes_per_step": d2hp,
                      "ms_per_step": e2ep_s * 1e3, "api": "fs_run_pl_phred() on pinned host buffers: uint16 PL + flags up; FPP as the six Phred digits the "
                      "reference prints (uint32 codes, device-encoded, exact: values next to a rounding boundary come back as doubles), gt, status down",
                      "codes_print_what_the_reference_prints": samep, "host_copy_ceiling_gbs": ceilingp,
                      "frac_of_host_copy_ceiling": world * (h2dp + d2hp) / e2ep_s / 1e9 / ceilingp},
        "layouts": layouts,
        "gpu_launches": launches, "clocks": clocks, "failed_variants": failed,
        "fp64_peak_tflops_measured": fp64_peak, "host_cores_of_rank0": len(cores) if cores else None,
        "notes": "compute-sanitizer is closed on this GPU pool (SURVEY section 5): memory safety rests on the bit-exact parity tests",
    })

    # ---- N GPUs behind ONE engine, one ordered host buffer (rank 0 drives every GPU) ---------------------------
    if world > 1 and not args.no_single_process:
        dist.barrier()
        if rank == 0:
            VV = world * args.variants
            pl, fl = synth.synth_pl(trio, args.variants, SEED + 2)
            h_pl = torch.from_numpy(np.tile(pl.astype(np.uint16).view(np.int16), (world, 1, 1))).pin_memory()
            h_fl = torch.from_numpy(np.tile(fl, world)).pin_memory()
            h_post = torch.empty((VV, 3, 3), dtype=torch.float64).pin_memory()
            h_gt = torch.empty((VV, 3), dtype=torch.uint8).pin_memory()
            h_st = torch.empty(VV, dtype=torch.uint8).pin_memory()
            with engine(trio, device=list(range(world))) as eng:
                for _ in range(2):
                    eng.run_pl_raw(2, VV, h_pl.data_ptr(), h_fl.data_ptr(), h_post.data_ptr(), None, h_gt.data_ptr(), h_st.data_ptr())
                t0 = time.perf_counter()
                for _ in range(e2e_steps):
                    eng.run_pl_raw(2, VV, h_pl.data_ptr(), h_fl.data_ptr(), h_post.data_ptr(), None, h_gt.data_ptr(), h_st.data_ptr())
                sec = (time.perf_counter() - t0) / e2e_steps
            slices_equal = bool(torch.equal(h_post[:args.variants], h_post[-args.variants:]) and torch.equal(h_gt[:args.variants], h_gt[-args.variants:]))
            out["e2e_single_process"] = {"value": VV / sec, "unit": UNIT, "ms_per_step": sec * 1e3, "mode": "fs_create_multi: one process, one engine, "
                                         f"{world} GPUs, one ordered pinned buffer of {VV} variants", "every_gpu_slice_has_the_same_bytes": slices_equal}
            del h_pl, h_fl, h_post, h_gt, h_st
        dist.barrier()

    # ---- the other methods -----------------------------------------------------------------------------------
    sub = {}
    if "es14" in methods:  # ES on a pedigree that is not a nuclear family (any loop-free pedigree), HBM roofline
        wl = Workload("es14", ped14, "es", args.es14_variants)
        # the message program as generated straight-line code (csrc/cuda/es_jit.cu); compiled in the warm-up step here,
        # on a worker thread after 2e10 variants otherwise (FAMSEQ_ES_JIT=0: the interpreter of es_kernel.cu)
        os.environ.setdefault("FAMSEQ_ES_JIT", "1")
        with engine(ped14) as eng:
            ms_e, l_e, clk_e, failed_e, keep = time_device_path(torch, dist, fs, eng, wl, rank, world, 5, 2, local_rank)
            jit_e = eng.info()["jit_launches"]
        del keep
        torch.cuda.empty_cache()
        ach = algorithmic_bytes(14) * args.es14_variants / (ms_e * 1e-3) / 1e9
        sub["ES_ped14"] = {"workload": "synthetic 14-member 3-generation pedigree, ES peeling (compiled message program)",
                           "kernel": "famseq_es (generated for the pedigree, NVRTC)" if jit_e else "es_kernel (message-program interpreter)",
                           "variants_per_gpu": args.es14_variants, "value": world * args.es14_variants / (ms_e * 1e-3),
                           "unit": UNIT, "ms_per_step": ms_e, "steps": 5, "warmup": 2, "gpu_launches": l_e, "clocks": clk_e,
                           "failed_variants": failed_e,
                           "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                                        "algorithmic_bytes_per_variant": algorithmic_bytes(14)}}
    if "bn" in methods:
        N = 14
        wl = Workload("bn", ped14, "bn", args.bn_variants)
        with engine(ped14) as eng:
            ms_b, l_b, clk_b, failed_b, keep = time_device_path(torch, dist, fs, eng, wl, rank, world, 2, 1, local_rank)
        del keep
        torch.cuda.empty_cache()
        # roofline: FP64 instructions the kernel EXECUTES per configuration (ncu: smsp__inst_executed_pipe_fp64 of one
        # launch / (variants x 3^N), profiles/bn_fp64_instr.json) against the FP64 issue peak = measured DFMA peak / 2
        prof = profile_json("bn_fp64_instr.json")
        ipc = float(prof.get("fp64_instr_per_configuration", 2.39))
        instr_rate = ipc * 3 ** N * args.bn_variants / (ms_b * 1e-3)  # FP64 thread-instructions per second
        ach = 2.0 * instr_rate / 1e12                                    # each counted like the DFMA the peak is measured with
        flops = 2.0 * N * 3 ** N
        sub["BN"] = {"workload": "synthetic 14-member 3-generation pedigree, exhaustive 3^14 enumeration (-method 1)",
                     "variants_per_gpu": args.bn_variants, "value": world * args.bn_variants / (ms_b * 1e-3), "unit": UNIT,
                     "ms_per_step": ms_b, "steps": 2, "warmup": 1, "gpu_launches": l_b, "clocks": clk_b, "failed_variants": failed_b,
                     "roofline": {"bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach / fp64_peak,
                                  "fp64_instr_per_configuration": ipc, "fp64_instr_source": prof.get("source", "profiles/r1q_bn_r1q.txt (FP64 pipe 71.8 % -> 2.39 instr/config)"),
                                  "algorithmic_note": f"SURVEY 8(d) counts 2 N 3^N = {flops:.4g} flop per variant for the reference's algorithm (N multiplies + N adds "
                                                      f"per configuration); by that count this run does {flops * args.bn_variants / (ms_b * 1e-3) / 1e12:.1f} TFLOP/s. The kernel "
                                                      "shares prefix products, so it executes far fewer: frac is executed FP64 instructions / issue peak"}}
        # Not the contract number: the same kernel with the opt-in closed-form sum over the innermost block of childless
        # members (FAMSEQ_BN_FACTOR=1, bn_kernel.cu: bn_block_factored) -- 3^9 instead of 3^14 configurations visited.
        os.environ["FAMSEQ_BN_FACTOR"] = "1"
        try:
            with engine(ped14) as eng:
                ms_f, l_f, _, failed_f, keep = time_device_path(torch, dist, fs, eng, wl, rank, world, 2, 1, local_rank)
        finally:
            del os.environ["FAMSEQ_BN_FACTOR"]
        del keep
        torch.cuda.empty_cache()
        sub["BN_leaves_summed_analytically"] = {
            "workload": "same as BN; opt-in FAMSEQ_BN_FACTOR=1: the 3^5 configurations of the five innermost (childless) members "
                        "are summed in closed form, 3^9 configurations are enumerated; same marginals to 1e-9",
            "variants_per_gpu": args.bn_variants, "value": world * args.bn_variants / (ms_f * 1e-3), "unit": UNIT,
            "ms_per_step": ms_f, "steps": 2, "warmup": 1, "gpu_launches": l_f, "failed_variants": failed_f}
    if "mcmc" in methods:
        N, founders, burn, rep = 40, 9, 1000, 10000
        wl = Workload("mcmc", ped40, "mcmc", args.mcmc_variants, burn, rep)
        # The Gibbs kernel of a large batch is generated for the pedigree and compiled at run time (csrc/cuda/gibbs_jit.cu).
        # By default that happens on a worker thread while the table-driven kernel carries on; here the compile is made
        # synchronous so that it falls into the warm-up step and every timed step runs the same kernel.
        os.environ.setdefault("FAMSEQ_MCMC_JIT", "1")
        with engine(ped40) as eng:
            ms_m, l_m, clk_m, failed_m, keep = time_device_path(torch, dist, fs, eng, wl, rank, world, 2, 1, local_rank)
            info_m = eng.info()
        del keep
        torch.cuda.empty_cache()
        flops = (burn + rep) * (14.0 * N + 3.0 * 2 * (N - founders))
        ach = flops * args.mcmc_variants / (ms_m * 1e-3) / 1e12
        sub["MCMC"] = {"workload": "synthetic 40-member pedigree with loops, Gibbs 1000 burn-in + 10000 sweeps (-method 3)",
                       "variants_per_gpu": args.mcmc_variants, "value": world * args.mcmc_variants / (ms_m * 1e-3), "unit": UNIT,
                       "ms_per_step": ms_m, "steps": 2, "warmup": 1, "gpu_launches": l_m, "clocks": clk_m, "failed_variants": failed_m,
                       "kernel": "famseq_gibbs (generated for the pedigree, NVRTC)" if info_m["jit_launches"] else "mcmc_kernel (table-driven)",
                       "chains_redone_by_the_table_driven_kernel": info_m["mcmc_fixups"],
                       "roofline": {"bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach / fp64_peak,
                                    "algorithmic_flops_per_variant": flops,
                                    "note": "SURVEY 8(d) flop count of the reference's sweep against the measured DFMA peak; a Gibbs step has "
                                            "no FMAs, so the DFMA peak counts every FP64 instruction twice"}}
    out["methods"] = sub
    # the other configurations also as flat scalars (C4 = BN ped14, C5 = MCMC ped40), for records that keep top-level keys only
    for key, name in (("ES_ped14", "es_ped14"), ("BN", "bn_ped14"), ("MCMC", "mcmc_ped40"), ("BN_leaves_summed_analytically", "bn_ped14_leaves_summed")):
        if key in sub:
            out[f"{name}_variants_per_s"] = sub[key]["value"]
            if "roofline" in sub[key]:
                out[f"{name}_roofline_frac"] = sub[key]["roofline"]["frac"]
    out["e2e_phred_variants_per_s"] = out["e2e_phred"]["value"]
    out["e2e_fp64_full_variants_per_s"] = out["e2e_fp64_full"]["value"]
    for tag, L in layouts.items():
        out[f"es_trio_{tag}_variants_per_s"] = L["value"]
        out[f"es_trio_{tag}_roofline_frac"] = L["roofline"]["frac"]

    # ---- CPU baseline beside it, file -> file, the reference's CUDA build (rank 0, N = 1 only) ----------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = CpuSample(trio, "es", args.variants)
        out["cpu_baseline"] = cpu.baseline()
        cpu.close()
        if "bn" in methods:
            cpu = CpuSample(ped14, "bn", CPU_SAMPLE["bn"])
            out["methods"]["BN"]["cpu_baseline"] = cpu.baseline(1)
            out["bn_ped14_cpu_variants_per_s"] = out["methods"]["BN"]["cpu_baseline"]["value"]
            cpu.close()
        if "mcmc" in methods:
            cpu = CpuSample(ped40, "mcmc", CPU_SAMPLE["mcmc"], 1000, 10000)
            out["methods"]["MCMC"]["cpu_baseline"] = cpu.baseline(1)
            out["mcmc_ped40_cpu_variants_per_s"] = out["methods"]["MCMC"]["cpu_baseline"]["value"]
            cpu.close()
    if rank == 0 and world == 1:
        if "cli" in methods:
            out["cli_e2e"] = cli_file_to_file(args.cli_variants)
            out["cli_e2e_variants_per_s_wall"] = out["cli_e2e"].get("variants_per_s_wall")
            out["cli_e2e_variants_per_s_pipeline"] = out["cli_e2e"].get("variants_per_s_pipeline")
        if "refgpu" in methods:
            out["ref_cuda_bn"] = reference_cuda_bn()
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
