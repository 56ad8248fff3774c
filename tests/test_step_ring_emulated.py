"""The staged form of the step kernels (csrc/qp.cu: qs_step_ring_kernel) reads the operands of qs_step from a per-warp ring of chunks
(csrc/qp_split.cuh: qs_sp) instead of global memory.  tests/step_ring_host.cpp runs the same chunk table through a memcpy ring on the
host that checks every read against the chunks held at that moment, and compares what qs_step stores with the global-memory form bit
for bit: every mode, both iterate buffers, every stage flag combination the controllers produce, both storage flavours."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest

from tests.common import make_problem

HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {}


def _lib(f32):
    if f32 not in _LIBS:
        d = tempfile.mkdtemp(prefix='step_ring_')
        so = os.path.join(d, 'step_ring_host.so')
        flav = ['-DQS_REAL=float', '-DQS_FLAVOUR=f32'] if f32 else []
        subprocess.run(['g++', '-O2', '-std=c++17', '-fPIC', '-shared'] + flav + ['-o', so, os.path.join(HERE, 'step_ring_host.cpp')], check=True)
        lib = C.CDLL(so)
        lib.step_ring_check.restype = C.c_int
        _LIBS[f32] = lib
    return _LIBS[f32]


@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('controller', ['st', 'htwa', 'naive', 'receding', 'real_receding', 'constraint_everywhere'])
def test_ring_operands_match_global_reads(controller, f32):
    lib = _lib(f32)
    prob, params, md = make_problem(controller, N=12)
    errors = C.c_int(-1)
    bad = lib.step_ring_check(C.byref(prob), C.c_int(3), C.c_uint64(7), C.byref(errors))
    assert errors.value == 0, f'{errors.value} reads or copies outside the ring protocol'
    assert bad == 0, f'{bad} of 6 (iteration parity, mode) runs store different bits'
