"""famseq_b200 -- B200-native FamSeq posterior-genotype engine (BN / ES / MCMC).

The product is `libfamseq_b200.so` (C ABI, include/famseq_b200.h) and the `FamSeq` command line, both
built from famseq_b200/csrc for sm_100a.  This package only binds the library for tests and bench.py
and generates synthetic inputs; it contains no CPU implementation of the engine.
"""
from . import synth  # noqa: F401
from .engine import (BN, BN_PEEL, ES, MCMC, FLAG_CHRX, FLAG_KNOWN, Engine, FamSeqError, Params, PhredResult, Result,  # noqa: F401
                     device_count, lib, phred_text, phred_text_exact)
