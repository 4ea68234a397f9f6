"""The C-ABI library loads, exports every symbol include/mpc_b200.h declares, and fails loudly without a GPU
(no compute calls are made here)."""
import ctypes
import os
import re

import pytest
import torch

import __graft_entry__ as g
from python_mpc_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "mpc_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mpcb_[a-z0-9_]+)\s*\(", src)))


def test_header_binding_and_library_agree():
    names = declared_symbols()
    assert len(names) >= 25
    assert sorted(_lib.EXPORTED_SYMBOLS) == names
    lib = ctypes.CDLL(g.build_cuda())
    for n in names:
        assert hasattr(lib, n), "libmpc_b200.so does not export %s" % n
    lib.mpcb_version.restype = ctypes.c_int
    assert lib.mpcb_version() >= 100


def test_library_is_compiled_for_sm_100a():
    import subprocess
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")        # the toolkit build_cuda() compiles with
    out = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-lelf", g.build_cuda()], capture_output=True,
                         text=True).stdout
    assert "sm_100a" in out


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour of a GPU-less host")
def test_product_fails_loudly_without_a_gpu():
    with pytest.raises(_lib.MpcError, match="no CPU fallback"):
        _lib.cuda_backend()
    # and the library itself reports the CUDA error instead of computing anything
    be = _lib.Backend(ctypes.CDLL(g.build_cuda()), "cpu")
    p = _lib.Problem(); p.horizon, p.nx, p.nu, p.dtype = 20, 4, 1, _lib.MPCB_F64
    for i in range(4):
        p.xmin[i], p.xmax[i] = -1.0, 1.0
    p.umin[0], p.umax[0] = -1.0, 1.0
    h = ctypes.c_void_p()
    rc = be.lib.mpcb_create(ctypes.byref(p), None, 32, ctypes.byref(h))
    assert rc == -2 and b"cuda" in be.lib.mpcb_last_error().lower()


def test_argument_validation_in_the_abi(emu_backend):
    lib = emu_backend.lib
    p = _lib.Problem(); p.horizon, p.nx, p.nu, p.dtype = 20, 4, 1, _lib.MPCB_F64
    h = ctypes.c_void_p()
    assert lib.mpcb_create(None, None, 1, ctypes.byref(h)) == -1
    assert lib.mpcb_create(ctypes.byref(p), None, 0, ctypes.byref(h)) == -1
    p.nx = 9
    assert lib.mpcb_create(ctypes.byref(p), None, 4, ctypes.byref(h)) == -1
    assert b"unsupported" in lib.mpcb_last_error()
    p.nx = 4; p.xmin[0] = 1.0; p.xmax[0] = -1.0
    assert lib.mpcb_create(ctypes.byref(p), None, 4, ctypes.byref(h)) == -1
    assert b"lower bound must be lower than or equal to upper bound" in lib.mpcb_last_error()
    p.xmin[0] = -1.0; p.xmax[0] = 1.0
    assert lib.mpcb_create(ctypes.byref(p), None, 4, ctypes.byref(h)) == 0
    assert lib.mpcb_num_variables(h) == 21 * 4 + 20 and lib.mpcb_num_constraints(h) == 2 * 21 * 4 + 20
    assert lib.mpcb_solve(h, None) == -3                     # solve before setup
    assert lib.mpcb_setup(h, 8, 32, None, None, None, None, None, None) == -1
    lib.mpcb_destroy(h)
