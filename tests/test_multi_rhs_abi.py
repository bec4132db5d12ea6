"""CPU: argument checks of the many-sources entry points (batched DDHTransfer action, lockstep FP32 GMRES) return an error status
before any CUDA call, the C++ overloads compile, and the new kernels compile without spills."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import pytest

from cuddhelmholtz_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def _ptrs(k):
    # non-null stand-ins: the checks under test reject the call before any pointer is dereferenced
    return (C.c_void_p * max(k, 1))(*([0x1000 * (j + 1) for j in range(max(k, 1))]))


def _err(lib):
    return (lib.cuddh_b200_last_error() or b"").decode()


@pytest.mark.parametrize("k", [0, 33])
def test_transfer_action_batch_rejects_k_out_of_range(k):
    lib = capi.load()
    assert lib.cuddh_b200_ddh_transfer_action_batch(None, k, _ptrs(k), _ptrs(k), None) != 0
    assert "k must be in [1, 32]" in _err(lib)


def test_transfer_action_batch_rejects_null_arrays():
    lib = capi.load()
    assert lib.cuddh_b200_ddh_transfer_action_batch(None, 2, None, _ptrs(2), None) != 0
    assert "null pointer array" in _err(lib)
    assert lib.cuddh_b200_ddh_transfer_action_batch(None, 2, _ptrs(2), None, None) != 0
    assert "null pointer array" in _err(lib)
    assert lib.cuddh_b200_ddh_transfer_as_apply_batch(None, 2, _ptrs(2), None, None) != 0


def _gmres_batch(lib, k, x, b, m=20, A=True):
    fn = C.cast(lib.cuddh_b200_ddh_transfer_as_apply_batch, C.c_void_p) if A else None
    so = (capi.SolverOut * max(k, 1))()
    return lib.cuddh_b200_gmres_f_batch(64, k, x, fn, None, b, m, 10, 1e-4, 60.0, so, None, None, 0, None)


@pytest.mark.parametrize("k", [0, 33])
def test_gmres_batch_rejects_k_out_of_range(k):
    lib = capi.load()
    assert _gmres_batch(lib, k, _ptrs(k), _ptrs(k)) != 0
    assert "k must be in [1, 32]" in _err(lib)


def test_gmres_batch_rejects_null_arrays_and_callback():
    lib = capi.load()
    assert _gmres_batch(lib, 3, None, _ptrs(3)) != 0
    assert "null pointer array" in _err(lib)
    assert _gmres_batch(lib, 3, _ptrs(3), None) != 0
    assert "null pointer array" in _err(lib)
    assert _gmres_batch(lib, 3, _ptrs(3), _ptrs(3), A=False) != 0
    assert "null operator callback" in _err(lib)


@pytest.mark.parametrize("m", [0, -1])
def test_gmres_batch_rejects_m_below_one(m):
    lib = capi.load()
    assert _gmres_batch(lib, 3, _ptrs(3), _ptrs(3), m=m) != 0
    assert "m must be >= 1" in _err(lib)


SNIPPET = r"""
#include "DDH.hpp"
#include <vector>
std::vector<cuddh::solver_out> solve_many(const cuddh::DDHTransfer & T, int n, int k, float * const * x, const float * const * b,
                                          const float * const * v, float * const * w)
{
    T.action(k, v, w);
    cuddh_ddh_transfer_t raw = T.handle();
    (void)raw;
    return cuddh::gmres(n, k, x, T, b, 20, 100, 1e-4f);
}
"""


def _syntax_check(src, tmp):
    path = os.path.join(tmp, "many_sources.cpp")
    with open(path, "w") as f:
        f.write(src)
    cx = os.path.join(ROOT, "cuddhelmholtz_b200", "cxx")
    # the headers launch kernels (<<< >>>), so g++ sees them through nvcc's front end; -fsyntax-only stops g++ at the parse
    cmd = [NVCC, "-x", "cu", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "g++", "-Xcompiler", "-fsyntax-only",
           "-I", cx, "-I", os.path.join(cx, "include"), "-I", os.path.join(ROOT, "include"), "-c", path, "-o", os.path.join(tmp, "x.o")]
    return subprocess.run(cmd, capture_output=True, text=True)


def test_cxx_batched_overloads_compile():
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not found")
    with tempfile.TemporaryDirectory() as tmp:
        r = _syntax_check(SNIPPET, tmp)
        assert r.returncode == 0, r.stderr[-3000:]
        # and the check has teeth: a wrong argument list fails
        r = _syntax_check(SNIPPET.replace("cuddh::gmres(n, k, x, T, b,", "cuddh::gmres(n, k, x, &T, b,"), tmp)
        assert r.returncode != 0


def test_new_kernels_compile_for_sm100a_without_spills():
    obj = os.path.join(ROOT, "cuddhelmholtz_b200", "lib", "obj")
    found = {}
    for name in ("ddh_transfer", "linalg"):
        log = open(os.path.join(obj, name + ".ptxas.log")).read()
        for m in re.finditer(r"Compiling entry function '(\w+)' for 'sm_100a'\n.*?Function properties.*?\n(.*?)\n(.*?)\n", log):
            if "_batch_kernel" in m.group(1):
                found[m.group(1)] = m.group(2) + " " + m.group(3)
    # 4 transfer instances (TF 96 / 112 / 192 / 224) + 5 GMRES kernels
    assert len(found) == 9, sorted(found)
    for fn, info in found.items():
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in info, (fn, info)
    regs = [int(re.search(r"Used (\d+) registers", i).group(1)) for f, i in found.items() if "ddh_transfer" in f]
    assert len(regs) == 4 and max(regs) <= 128, regs  # two 256-thread CTAs per SM
