"""bamsignals_b200 — B200-native (sm_100a) counting path of bamsignals behind the reference's own interface.

Only what the hot path needs lives here: csrc/ (CUDA kernels, host fetch pipeline, C ABI -> libbamsignals_cuda.so)
and api.py (the Python mirror of the R functions bamCount / bamProfile / bamCoverage and of CountSignals).
"""
from .api import (BamsignalsError, BsgOpts, CountSignals, CoverageRuns, GRanges, ProfileRuns, Stage, debug_plan,  # noqa: F401
                  bamCount, bamCoverage, bamProfile, core_args, coverage_core, coverage_runs_core, default_opts, flagMask,
                  lib, pileup_core, profile_runs_core, timings, writeSamAsBamAndIndex)

__version__ = "0.1.0"
