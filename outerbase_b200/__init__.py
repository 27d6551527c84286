"""outerbase_b200 -- B200-native implementation of outerbase's hot path.

`lib()` returns the binding over the CUDA library (built in-tree by `build()` /
`__graft_entry__.build()`); creating it needs a B200: there is no CPU fallback and
no code path in this package touches the oracle under /oracle.
"""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

from .binding import (Library, getpara, gethyp, header_symbols, loglik_gauss, loglik_gda, logpr_gauss, lpdf, lpdfvec,  # noqa: F401
                      outerbase, outermod, predictor, setcovfs, setknot, sobol, sobol_pairs,
                      sobol_shapley)

ROOT = Path(__file__).resolve().parent
REPO = ROOT.parent
CSRC = ROOT / "csrc"
LIBDIR = ROOT / "_lib"
LIBPATH = LIBDIR / "libouterbase_b200.so"
HEADER = REPO / "include" / "outerbase_b200.h"
MULTI_HEADER = REPO / "include" / "outerbase_b200_multi.h"  # the multi-response extension
PERCOL_HEADER = REPO / "include" / "outerbase_b200_multi_percol.h"  # its per-column para variants
MULTI_GDA_HEADER = REPO / "include" / "outerbase_b200_multi_gda.h"  # multi-response loglik_gda (two-stage fits)
DRAWS_HEADER = REPO / "include" / "outerbase_b200_draws.h"  # posterior draws of a fitted model
SOBOL_HEADER = REPO / "include" / "outerbase_b200_sobol.h"  # Sobol sensitivity indices of a fitted model
SOBOL_PAIRS_HEADER = REPO / "include" / "outerbase_b200_sobol_pairs.h"  # their second-order (input-pair) forms
SOBOL_SHAPLEY_HEADER = REPO / "include" / "outerbase_b200_sobol_shapley.h"  # Shapley effects of a fitted model

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _sources():
    return [CSRC / "ob_kernels.cu", CSRC / "ob_spec_rt.cu", CSRC / "ob_capi.cu"]


def _stale() -> bool:
    if not LIBPATH.exists():
        return True
    t = LIBPATH.stat().st_mtime
    deps = list(CSRC.glob("*")) + [HEADER, MULTI_HEADER, PERCOL_HEADER, MULTI_GDA_HEADER, DRAWS_HEADER, SOBOL_HEADER,
                                   SOBOL_PAIRS_HEADER, SOBOL_SHAPLEY_HEADER]
    return any(p.stat().st_mtime > t for p in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every CUDA source of the package for sm_100a into _lib/ (in-tree)."""
    if not force and not _stale():
        return LIBPATH
    LIBDIR.mkdir(exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, *NVCC_FLAGS, "-o", str(LIBPATH), *map(str, _sources()), "-ldl"]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    subprocess.run(cmd, check=True, cwd=str(CSRC))
    return LIBPATH


_LIB = None


def lib(device: int | None = None) -> Library:
    """The process-wide binding (one context on `device`, default LOCAL_RANK or 0)."""
    global _LIB
    if _LIB is None:
        if not LIBPATH.exists():
            raise RuntimeError(f"{LIBPATH} is missing: run outerbase_b200.build() (needs nvcc); no CPU fallback exists")
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        _LIB = Library(LIBPATH, "ob_", device=device)
    return _LIB


def load_symbols_only() -> Library:
    """Load the shared library without creating a GPU context (CPU-side ABI checks)."""
    return Library(LIBPATH, "ob_", create_ctx=False)
