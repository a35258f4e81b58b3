"""ctypes binding of libfamseq_b200.so (C ABI: include/famseq_b200.h).

This is host-side plumbing for tests and bench.py; the product is the shared library and the
`FamSeq` command line built from famseq_b200/csrc.  There is no Python or CPU implementation of the
posterior engine here: if the library is missing the import of this module fails, and if no sm_100
GPU is usable `Engine(...)` raises.

Names follow the reference's `class family` (src/family.h:262-389): `calPostProbBN`,
`calPostProbPeeling`, `calPostProbMCMC`, but each call takes a whole batch of variants.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfamseq_b200.so")

BN, ES, MCMC, BN_PEEL = 1, 2, 3, 4  # BN_PEEL: BN's answer by conditioned peeling (-method 1 -peelLoops)
FLAG_KNOWN, FLAG_CHRX = 1, 2

FS_ERRORS = {
    -1: "FS_E_ARG", -2: "FS_E_HALF_PARENTS", -3: "FS_E_GENDER", -4: "FS_E_LOOP", -5: "FS_E_TOO_LARGE",
    -6: "FS_E_CUDA", -7: "FS_E_NOMEM",
}


class FamSeqError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{FS_ERRORS.get(code, code)}: {message}")
        self.code = code


class _Pedigree(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int32), ("id", ctypes.c_void_p), ("mother_id", ctypes.c_void_p),
                ("father_id", ctypes.c_void_p), ("gender", ctypes.c_void_p), ("s", ctypes.c_int32),
                ("cols", ctypes.c_void_p)]


class Params(ctypes.Structure):
    """fs_params: -mRate, -LRC and the four prior vectors (reference defaults via `Params.default()`)."""
    _fields_ = [("mrate", ctypes.c_double), ("lrc", ctypes.c_double), ("geno_prob_n", ctypes.c_double * 3),
                ("geno_prob_k", ctypes.c_double * 3), ("geno_prob_xn", ctypes.c_double * 3),
                ("geno_prob_xk", ctypes.c_double * 3)]

    @staticmethod
    def default() -> "Params":
        p = Params()
        lib().fs_default_params(ctypes.byref(p))
        return p

    def priors(self) -> np.ndarray:
        return np.array([list(self.geno_prob_n), list(self.geno_prob_k), list(self.geno_prob_xn),
                         list(self.geno_prob_xk)], dtype=np.float64)


class _Info(ctypes.Structure):
    _fields_ = [(k, ctypes.c_int32) for k in ("n", "s", "n_founders", "has_loop", "es_ops", "es_slots", "bn_levels",
                                               "bn_group", "mcmc_links", "device")] + [("kernel_launches", ctypes.c_int64),
                                                                                      ("jit_launches", ctypes.c_int64),
                                                                                      ("mcmc_fixups", ctypes.c_int64),
                                                                                      ("n_devices", ctypes.c_int32),
                                                                                      ("gibbs_generator", ctypes.c_int32)]


_lib = None


def lib() -> ctypes.CDLL:
    """Loads the shared library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(make -C famseq_b200/csrc). There is no CPU or PyTorch fallback.")
        L = ctypes.CDLL(LIB_PATH)
        P, I32, I64, U64, D = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double
        L.fs_default_params.restype = None
        L.fs_default_params.argtypes = [P]
        L.fs_device_count.restype = ctypes.c_int
        L.fs_create.restype = ctypes.c_int
        L.fs_create.argtypes = [P, P, ctypes.c_int, P]
        L.fs_create_multi.restype = ctypes.c_int
        L.fs_create_multi.argtypes = [P, P, P, ctypes.c_int, P]
        L.fs_create_families.restype = ctypes.c_int
        L.fs_create_families.argtypes = [P, P, P, ctypes.c_int, P]
        L.fs_get_families.restype = ctypes.c_int
        L.fs_get_families.argtypes = [P, P, P, P]
        L.fs_create_cohort.restype = ctypes.c_int
        L.fs_create_cohort.argtypes = [P, P, P, ctypes.c_int, P]
        L.fs_create_cohort_bn.restype = ctypes.c_int
        L.fs_create_cohort_bn.argtypes = [P, P, P, ctypes.c_int, P]
        L.fs_create_cohort_mcmc.restype = ctypes.c_int
        L.fs_create_cohort_mcmc.argtypes = [P, P, P, ctypes.c_int, P]
        L.fs_get_family_program.restype = ctypes.c_int
        L.fs_get_family_program.argtypes = [P, I32, P, I32, P, P, P, P, P]
        L.fs_run_pl.restype = ctypes.c_int
        L.fs_run_pl.argtypes = [P, ctypes.c_int, I64, P, P, I32, I32, U64, I64, P, P, P, P]
        L.fs_run_pl_device.restype = ctypes.c_int
        L.fs_run_pl_device.argtypes = [P, ctypes.c_int, I64, P, P, I32, I32, U64, I64, P, P, P, P, P]
        L.fs_get_pl_table.restype = ctypes.c_int
        L.fs_get_pl_table.argtypes = [P, P]
        L.fs_run_pl_phred.restype = ctypes.c_int
        L.fs_run_pl_phred.argtypes = [P, ctypes.c_int, I64, P, P, I32, I32, U64, I64, P, P, P, P, P, I64, P]
        L.fs_phred_encode.restype = ctypes.c_int
        L.fs_phred_encode.argtypes = [P, I64, P, P, P, I64, P]
        L.fs_phred_text.restype = ctypes.c_int
        L.fs_phred_text.argtypes = [ctypes.c_uint32, ctypes.c_char_p]
        L.fs_phred_text_exact.restype = ctypes.c_int
        L.fs_phred_text_exact.argtypes = [D, ctypes.c_char_p]
        L.fs_destroy.restype = None
        L.fs_destroy.argtypes = [P]
        L.fs_last_error.restype = ctypes.c_char_p
        L.fs_run.restype = ctypes.c_int
        L.fs_run.argtypes = [P, ctypes.c_int, I64, P, P, I32, I32, U64, I64, P, P, P, P]
        L.fs_run_device.restype = ctypes.c_int
        L.fs_run_device.argtypes = [P, ctypes.c_int, I64, P, P, I32, I32, U64, I64, P, P, P, P, P]
        L.fs_get_info.restype = ctypes.c_int
        L.fs_get_info.argtypes = [P, P]
        L.fs_get_tables.restype = ctypes.c_int
        L.fs_get_tables.argtypes = [P, P, P, P, P, P]
        L.fs_alloc_pinned.restype = P
        L.fs_alloc_pinned.argtypes = [ctypes.c_size_t]
        L.fs_free_pinned.restype = None
        L.fs_free_pinned.argtypes = [P]
        L.fs_last_kernel_ms.restype = D
        L.fs_last_kernel_ms.argtypes = [P]
        L.fs_get_es_program.restype = ctypes.c_int
        L.fs_get_es_program.argtypes = [P, P, I32, P, P]
        L.fs_get_bn_peel_program.restype = ctypes.c_int
        L.fs_get_bn_peel_program.argtypes = [P, P, I32, P, P, P, I32, P, P]
        L.fs_bench_fp64_tflops.restype = ctypes.c_int
        L.fs_bench_fp64_tflops.argtypes = [ctypes.c_int, P]
        _lib = L
    return _lib


EXPORTED_SYMBOLS = ["fs_default_params", "fs_device_count", "fs_create", "fs_destroy", "fs_last_error", "fs_run",
                    "fs_run_device", "fs_get_info", "fs_get_tables", "fs_alloc_pinned", "fs_free_pinned",
                    "fs_last_kernel_ms", "fs_bench_fp64_tflops", "fs_get_es_program", "fs_get_gibbs_kernel", "fs_get_es_kernel", "fs_warmup",
                    "fs_create_multi", "fs_run_pl", "fs_run_pl_device", "fs_get_pl_table",
                    "fs_run_pl_phred", "fs_phred_encode", "fs_phred_text", "fs_phred_text_exact",
                    "fs_create_families", "fs_get_families", "fs_create_cohort", "fs_get_family_program", "fs_create_cohort_bn",
                    "fs_create_cohort_mcmc", "fs_get_bn_peel_program"]


def _check(rc: int) -> None:
    if rc != 0:
        raise FamSeqError(rc, lib().fs_last_error().decode("utf-8", "replace"))


def _i32(x):
    return np.ascontiguousarray(x, dtype=np.int32)


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(ctypes.c_void_p)
    return ctypes.c_void_p(int(a))  # raw address (e.g. torch.Tensor.data_ptr())


PHRED_FIX_DTYPE = np.dtype([("index", np.int64), ("p", np.float64)])  # fs_phred_fix
PHRED_KIND_FIX = 3
PHRED_FIX_SINGLE = 1 << 62


def phred_text(code: int) -> str | None:
    """Text of one packed Phred code (fs_phred_text); None for an exception code (kind FS_PHRED_FIX)."""
    buf = ctypes.create_string_buffer(16)
    n = lib().fs_phred_text(int(code), buf)
    return None if n < 0 else buf.raw[:n].decode()


def phred_text_exact(p: float) -> str:
    """The reference's text of one probability (fs_phred_text_exact: libm log10 + "%g")."""
    buf = ctypes.create_string_buffer(40)
    n = lib().fs_phred_text_exact(float(p), buf)
    return buf.raw[:n].decode()


@dataclass
class PhredResult:
    post: np.ndarray            # [V][S][3] uint32 packed Phred codes of the pedigree-aware posterior
    single: np.ndarray | None   # the same for the individual-only posterior, or None
    gt: np.ndarray
    status: np.ndarray
    fixes: np.ndarray           # PHRED_FIX_DTYPE records: values the host formats itself (exact doubles)
    n_fixes: int                # how many there were (may exceed len(fixes) = the capacity given)


@dataclass
class Result:
    post: np.ndarray    # [V][S][3] pedigree-aware posterior (FPP)
    single: np.ndarray  # [V][S][3] individual-only posterior (GPP)
    gt: np.ndarray      # [V][S] uint8 called genotype (FGT): 0 RR, 1 RA, 2 AA, 255 = the reference's -1
    status: np.ndarray  # [V] uint8, 1 = "this variant hasn't been calculated" (the reference returned false)


class Engine:
    """One pedigree compiled for one GPU (fs_create) or, with `device` a list of GPUs, for several (fs_create_multi:
    every batch call is cut into one contiguous slice of variants per GPU).  families=True takes a cohort ped file of
    nuclear families and lone individuals of any size (fs_create_families, Elston-Stewart only; `device` an int or a
    list, -1 = host side only); cohort=True takes one whose families may also have any other loop-free shape
    (fs_create_cohort, same rules).  cohort_bn=True runs the Bayesian network on a cohort ped file of any size, each family
    (looped ones included, at most 31 members each) enumerated on its own (fs_create_cohort_bn, BN only; `device` as for
    cohort=True).  cohort_mcmc=True runs the Gibbs sampler on a cohort ped file of any size, each family (looped ones
    included, at most 128 members each) on its own chain, which is the whole file's chain restricted to that family
    (fs_create_cohort_mcmc, MCMC only; `device` as for cohort=True)."""

    def __init__(self, ids, mother_ids, father_ids, genders, cols, params: Params | None = None, device=0, families: bool = False,
                 cohort: bool = False, cohort_bn: bool = False, cohort_mcmc: bool = False):
        self._h = ctypes.c_void_p()
        self._keep = [_i32(ids), _i32(mother_ids), _i32(father_ids), _i32(genders), _i32(cols)]
        ped = _Pedigree(len(self._keep[0]), _ptr(self._keep[0]), _ptr(self._keep[1]), _ptr(self._keep[2]),
                        _ptr(self._keep[3]), len(self._keep[4]), _ptr(self._keep[4]))
        self.params = params if params is not None else Params.default()
        self.device = device
        if families or cohort or cohort_bn or cohort_mcmc:
            devs = _i32(list(device) if isinstance(device, (list, tuple)) else [device])
            create = (lib().fs_create_cohort_mcmc if cohort_mcmc else lib().fs_create_cohort_bn if cohort_bn
                      else lib().fs_create_cohort if cohort else lib().fs_create_families)
            _check(create(ctypes.byref(ped), ctypes.byref(self.params), _ptr(devs), len(devs), ctypes.byref(self._h)))
        elif isinstance(device, (list, tuple)):
            devs = _i32(list(device))
            _check(lib().fs_create_multi(ctypes.byref(ped), ctypes.byref(self.params), _ptr(devs), len(devs), ctypes.byref(self._h)))
        else:
            _check(lib().fs_create(ctypes.byref(ped), ctypes.byref(self.params), device, ctypes.byref(self._h)))
        self.n, self.s = ped.n, ped.s

    def close(self) -> None:
        if self._h:
            lib().fs_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- introspection ------------------------------------------------------------------------------
    def info(self) -> dict:
        i = _Info()
        _check(lib().fs_get_info(self._h, ctypes.byref(i)))
        return {k: getattr(i, k) for k, _ in _Info._fields_}

    def tables(self):
        a, xf, xm = np.zeros(27), np.zeros(27), np.zeros(27)
        mo, fa = np.zeros(self.n, np.int32), np.zeros(self.n, np.int32)
        _check(lib().fs_get_tables(self._h, _ptr(a), _ptr(xf), _ptr(xm), _ptr(mo), _ptr(fa)))
        return a, xf, xm, mo, fa

    def families(self):
        """(family[n], n_children[F]) of an engine made with families=True or a cohort constructor: the family index of
        each ped row (families numbered by their first row) and each family's number of children (0 = a lone individual;
        the non-founder members of a family peeled by a message program or run by cohort_bn / cohort_mcmc)."""
        nf = ctypes.c_int32(0)
        _check(lib().fs_get_families(self._h, None, ctypes.byref(nf), None))
        fam, kids = np.zeros(self.n, np.int32), np.zeros(nf.value, np.int32)
        _check(lib().fs_get_families(self._h, _ptr(fam), None, _ptr(kids)))
        return fam, kids

    def family_program(self, f: int):
        """(words, n_slots, cols, program) of family f of a cohort=True engine: the message program it runs, the global input
        column of each of its local columns, and the program's index (-1 and empty arrays: the nuclear kernel peels it)."""
        n_words, n_slots, n_cols, prog = ctypes.c_int32(0), ctypes.c_int32(0), ctypes.c_int32(0), ctypes.c_int32(0)
        _check(lib().fs_get_family_program(self._h, f, None, 0, ctypes.byref(n_words), ctypes.byref(n_slots), None,
                                           ctypes.byref(n_cols), ctypes.byref(prog)))
        words, cols = np.zeros(n_words.value, np.uint32), np.zeros(n_cols.value, np.int32)
        _check(lib().fs_get_family_program(self._h, f, _ptr(words), n_words.value, None, None, _ptr(cols), None, None))
        return words, int(n_slots.value), cols, int(prog.value)

    def es_program(self):
        """(words, n_slots) of the compiled Elston-Stewart message program (introspection, see es_program.hpp)."""
        n_words, n_slots = ctypes.c_int32(0), ctypes.c_int32(0)
        _check(lib().fs_get_es_program(self._h, None, 0, ctypes.byref(n_words), ctypes.byref(n_slots)))
        words = np.zeros(n_words.value, np.uint32)
        _check(lib().fs_get_es_program(self._h, _ptr(words), n_words.value, None, None))
        return words, int(n_slots.value)

    def bn_peel_program(self):
        """(words, n_slots, breaker_rows, clamp_slots) of the conditioned program of BN_PEEL (fs_get_bn_peel_program):
        clamp_slots[j] = (vector of breaker j's clamped likelihood, vector of its indicator)."""
        n_words, n_slots, k = ctypes.c_int32(0), ctypes.c_int32(0), ctypes.c_int32(0)
        _check(lib().fs_get_bn_peel_program(self._h, None, 0, ctypes.byref(n_words), ctypes.byref(n_slots), None, 0,
                                            ctypes.byref(k), None))
        words, rows, clamps = np.zeros(n_words.value, np.uint32), np.zeros(k.value, np.int32), np.zeros((k.value, 2), np.int32)
        _check(lib().fs_get_bn_peel_program(self._h, _ptr(words), n_words.value, None, None, _ptr(rows), k.value, None,
                                            _ptr(clamps)))
        return words, int(n_slots.value), rows, clamps

    def es_kernel(self, compile: bool = False):
        """(text, cubin_bytes): the CUDA C++ generated for this pedigree's Elston-Stewart peeling, or the compile log."""
        return self._generated("fs_get_es_kernel", compile)

    def _generated(self, symbol: str, compile: bool):
        n, cb = ctypes.c_size_t(0), ctypes.c_size_t(0)
        f = getattr(lib(), symbol)
        f.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t),
                      ctypes.POINTER(ctypes.c_size_t)]
        f.restype = ctypes.c_int
        buf = ctypes.create_string_buffer(16 << 20)
        _check(f(self._h, 1 if compile else 0, buf, len(buf), ctypes.byref(n), ctypes.byref(cb)))
        return buf.value.decode("utf-8", "replace"), int(cb.value)

    def gibbs_kernel(self, compile: bool = False):
        """(text, cubin_bytes): the CUDA C++ the engine generates for this pedigree's Gibbs sampler, or, with
        compile=True, the NVRTC/ptxas log of compiling it for sm_100a (no device needed) and the cubin size."""
        n, cb = ctypes.c_size_t(0), ctypes.c_size_t(0)
        f = lib().fs_get_gibbs_kernel
        f.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t),
                      ctypes.POINTER(ctypes.c_size_t)]
        f.restype = ctypes.c_int
        buf = ctypes.create_string_buffer(4 << 20)
        _check(f(self._h, 1 if compile else 0, buf, len(buf), ctypes.byref(n), ctypes.byref(cb)))
        return buf.value.decode("utf-8", "replace"), int(cb.value)

    def pl_table(self) -> np.ndarray:
        """The 65 536-entry PL decode table of fs_run_pl (built on the host with libm's pow)."""
        out = np.empty(65536, np.float64)
        _check(lib().fs_get_pl_table(self._h, _ptr(out)))
        return out

    def last_kernel_ms(self) -> float:
        return float(lib().fs_last_kernel_ms(self._h))

    # -- batch calls on host buffers ------------------------------------------------------------------
    def run(self, method: int, lk, flags=None, burn: int = 1000, rep: int = 100000, seed: int = 0,
            v_offset: int = 0, out: Result | None = None, want_single: bool = True) -> Result:
        """fs_run on numpy arrays.  want_single=False passes single = NULL (Result.single is then None)."""
        return self._run_host("fs_run", np.float64, method, lk, flags, burn, rep, seed, v_offset, out, want_single)

    def run_pl(self, method: int, pl, flags=None, burn: int = 1000, rep: int = 100000, seed: int = 0,
               v_offset: int = 0, out: Result | None = None, want_single: bool = True) -> Result:
        """fs_run_pl: compact input, pl[V][S][3] uint16 Phred-scaled likelihoods (lk = 10^(-pl/10), file.cpp:588-590)."""
        return self._run_host("fs_run_pl", np.uint16, method, pl, flags, burn, rep, seed, v_offset, out, want_single)

    def _run_host(self, symbol, dtype, method, x, flags, burn, rep, seed, v_offset, out, want_single) -> Result:
        x = np.ascontiguousarray(x, dtype=dtype)
        if x.ndim != 3 or x.shape[1] != self.s or x.shape[2] != 3:
            raise ValueError(f"input must be [V][{self.s}][3]")
        V = x.shape[0]
        if flags is not None:
            flags = np.ascontiguousarray(flags, dtype=np.uint8)
            if flags.shape != (V,):
                raise ValueError("flags must be [V]")
        if out is None:
            out = Result(np.empty((V, self.s, 3)), np.empty((V, self.s, 3)) if want_single else None,
                         np.empty((V, self.s), np.uint8), np.empty(V, np.uint8))
        _check(getattr(lib(), symbol)(self._h, method, V, _ptr(x), _ptr(flags), burn, rep, seed, v_offset, _ptr(out.post),
                                      _ptr(out.single), _ptr(out.gt), _ptr(out.status)))
        return out

    def run_raw(self, method: int, V: int, lk_ptr, flags_ptr, post_ptr, single_ptr, gt_ptr, status_ptr, burn=1000,
                rep=100000, seed=0, v_offset=0) -> None:
        """fs_run on raw HOST addresses (e.g. pinned torch tensors)."""
        _check(lib().fs_run(self._h, method, V, _ptr(lk_ptr), _ptr(flags_ptr), burn, rep, seed, v_offset, _ptr(post_ptr),
                            _ptr(single_ptr), _ptr(gt_ptr), _ptr(status_ptr)))

    def run_pl_phred(self, method: int, pl, flags=None, burn: int = 1000, rep: int = 100000, seed: int = 0, v_offset: int = 0,
                     want_single: bool = True, fix_capacity: int = 4096) -> PhredResult:
        """fs_run_pl_phred: compact input AND compact output (Phred codes, 4 bytes per value)."""
        pl = np.ascontiguousarray(pl, dtype=np.uint16)
        if pl.ndim != 3 or pl.shape[1] != self.s or pl.shape[2] != 3:
            raise ValueError(f"input must be [V][{self.s}][3]")
        V = pl.shape[0]
        if flags is not None:
            flags = np.ascontiguousarray(flags, dtype=np.uint8)
        out = PhredResult(np.empty((V, self.s, 3), np.uint32), np.empty((V, self.s, 3), np.uint32) if want_single else None,
                          np.empty((V, self.s), np.uint8), np.empty(V, np.uint8), np.zeros(fix_capacity, PHRED_FIX_DTYPE), 0)
        n = ctypes.c_int64(0)
        _check(lib().fs_run_pl_phred(self._h, method, V, _ptr(pl), _ptr(flags), burn, rep, seed, v_offset, _ptr(out.post), _ptr(out.single),
                                     _ptr(out.gt), _ptr(out.status), _ptr(out.fixes), fix_capacity, ctypes.byref(n)))
        out.n_fixes = int(n.value)
        out.fixes = out.fixes[:min(out.n_fixes, fix_capacity)]
        return out

    def run_pl_phred_raw(self, method: int, V: int, pl_ptr, flags_ptr, post32_ptr, single32_ptr, gt_ptr, status_ptr, fixes_ptr, fix_capacity,
                         burn=1000, rep=100000, seed=0, v_offset=0) -> int:
        """fs_run_pl_phred on raw HOST addresses; returns the number of exceptions."""
        n = ctypes.c_int64(0)
        _check(lib().fs_run_pl_phred(self._h, method, V, _ptr(pl_ptr), _ptr(flags_ptr), burn, rep, seed, v_offset, _ptr(post32_ptr),
                                     _ptr(single32_ptr), _ptr(gt_ptr), _ptr(status_ptr), _ptr(fixes_ptr), fix_capacity, ctypes.byref(n)))
        return int(n.value)

    def phred_encode(self, p, fix_capacity: int = 4096):
        """fs_phred_encode: (codes uint32 like p, fixes, n_fixes) for an array of probabilities."""
        p = np.ascontiguousarray(p, dtype=np.float64)
        out = np.empty(p.shape, np.uint32)
        fixes = np.zeros(fix_capacity, PHRED_FIX_DTYPE)
        n = ctypes.c_int64(0)
        _check(lib().fs_phred_encode(self._h, p.size, _ptr(p), _ptr(out), _ptr(fixes), fix_capacity, ctypes.byref(n)))
        return out, fixes[:min(int(n.value), fix_capacity)], int(n.value)

    def run_pl_raw(self, method: int, V: int, pl_ptr, flags_ptr, post_ptr, single_ptr, gt_ptr, status_ptr, burn=1000,
                   rep=100000, seed=0, v_offset=0) -> None:
        """fs_run_pl on raw HOST addresses; single_ptr may be None."""
        _check(lib().fs_run_pl(self._h, method, V, _ptr(pl_ptr), _ptr(flags_ptr), burn, rep, seed, v_offset, _ptr(post_ptr),
                               _ptr(single_ptr), _ptr(gt_ptr), _ptr(status_ptr)))

    def run_pl_device(self, method: int, V: int, pl_ptr, flags_ptr, post_ptr, single_ptr, gt_ptr, status_ptr, burn=1000,
                      rep=100000, seed=0, v_offset=0, stream=0) -> None:
        """fs_run_pl_device on raw DEVICE addresses; asynchronous on `stream`; single_ptr may be None."""
        _check(lib().fs_run_pl_device(self._h, method, V, _ptr(pl_ptr), _ptr(flags_ptr), burn, rep, seed, v_offset,
                                      _ptr(post_ptr), _ptr(single_ptr), _ptr(gt_ptr), _ptr(status_ptr),
                                      ctypes.c_void_p(int(stream))))

    def run_device(self, method: int, V: int, lk_ptr, flags_ptr, post_ptr, single_ptr, gt_ptr, status_ptr, burn=1000,
                   rep=100000, seed=0, v_offset=0, stream=0) -> None:
        """fs_run_device on raw DEVICE addresses; asynchronous on `stream` (a cudaStream_t handle)."""
        _check(lib().fs_run_device(self._h, method, V, _ptr(lk_ptr), _ptr(flags_ptr), burn, rep, seed, v_offset,
                                   _ptr(post_ptr), _ptr(single_ptr), _ptr(gt_ptr), _ptr(status_ptr),
                                   ctypes.c_void_p(int(stream))))

    # -- the reference's method names -------------------------------------------------------------------
    def calPostProbBN(self, lk, flags=None) -> Result:
        return self.run(BN, lk, flags)

    def calPostProbPeeling(self, lk, flags=None) -> Result:
        return self.run(ES, lk, flags)

    def calPostProbMCMC(self, lk, numBurnIn: int, numRep: int, flags=None, seed: int = 0, v_offset: int = 0) -> Result:
        return self.run(MCMC, lk, flags, burn=numBurnIn, rep=numRep, seed=seed, v_offset=v_offset)


def device_count() -> int:
    return int(lib().fs_device_count())


def measure_fp64_tflops(device: int = 0) -> float:
    """Plain FP64 (DFMA) throughput of the device, measured by fs_bench_fp64_tflops."""
    out = ctypes.c_double(0.0)
    _check(lib().fs_bench_fp64_tflops(device, ctypes.byref(out)))
    return float(out.value)
