"""The deterministic backward executes no floating-point atomic: in the compiled library (cuobjdump -sass), only the
default backward's kernels contain a floating-point RED / ATOM add.  Together with the kernel-list check of
tests/test_gpu_deterministic.py (none of those kernels launches under the flag) a deterministic step runs no float
atomic.  Runs without a GPU."""
import os
import re
import shutil
import subprocess

import pytest

# The default (atomic) backward path; every other kernel must be free of floating-point atomics.
ALLOWED = {"k_edge_bwd", "k_lin_dw_tc", "k_split_colsum", "k_lin_dx_simt", "k_lin_dw_simt", "k_update_bwd",
           "k_fold_bwd_w", "k_fold_bwd_rel"}

FLOAT_ATOMIC = re.compile(r"\b(?:RED|REDG|REDAS|ATOM|ATOMG|ATOMS)\.[A-Z0-9_.]*?(?:ADD|CAS)[A-Z0-9_.]*?\.(?:F16|BF16|F32|F64)")
SHARED_CAS = re.compile(r"\bATOMS\.CAST?\.SPIN")          # emulated floating-point add on shared memory


def _cuobjdump():
    for cand in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump"),
                 shutil.which("cuobjdump")):
        if cand and os.path.exists(cand):
            return cand
    pytest.skip("cuobjdump not found")


def _kernel_name(mangled):
    hit = re.search(r"\d(k_[a-z0-9_]+?)(?:I|E|$)", mangled)
    return hit.group(1) if hit else mangled


def _float_atomic_kernels():
    import __graft_entry__ as ge
    lib = ge.build()
    sass = subprocess.run([_cuobjdump(), "-sass", lib], capture_output=True, text=True, check=True).stdout
    found, fn = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = m.group(1)
            continue
        if fn and (FLOAT_ATOMIC.search(line) or SHARED_CAS.search(line)):
            found.setdefault(_kernel_name(fn), set()).add(fn)
    return found


def test_only_the_default_backward_kernels_contain_float_atomics():
    found = _float_atomic_kernels()
    assert set(found) - ALLOWED == set(), sorted(set(found) - ALLOWED)
    # the pattern does see the default path's reductions (guards against a SASS spelling the regex misses)
    assert {"k_edge_bwd", "k_lin_dw_tc", "k_lin_dw_simt"} <= set(found), sorted(found)
