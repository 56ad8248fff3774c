"""The schedule of a QP solve captured into a CUDA graph (csrc/qp_split.cuh: qs_graph_drive -- no compaction, fixed kernel forms, step<2> /
red(true) in every iteration, the iteration index in device memory and the loop body repeated while qs_loop_step says so) against the
host-driven loop the eager path runs (qs_drive at depth 0).  tests/graph_loop_host.cpp runs both on the host build of the kernel source;
the results must agree bit for bit, in both storage flavours, including solves that the iteration limit ends."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle.oracle import Oracle
from safe_mpc_b200 import abi
from tests.common import make_problem, start_states, rollout_guess

HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {}


def _lib(f32):
    if f32 not in _LIBS:
        d = tempfile.mkdtemp(prefix='graph_loop_')
        so = os.path.join(d, 'graph_loop_host.so')
        flav = ['-DQS_REAL=float', '-DQS_FLAVOUR=f32'] if f32 else []
        subprocess.run(['g++', '-O2', '-std=c++17', '-fPIC', '-shared'] + flav + ['-o', so, os.path.join(HERE, 'graph_loop_host.cpp')], check=True)
        lib = C.CDLL(so)
        lib.graph_loop_solve.restype = C.c_int
        _LIBS[f32] = lib
    return _LIBS[f32]


def _p(a):
    return C.c_void_p(a.ctypes.data)


def _solve(lib, prob, lin, x0, r, act, graph):
    B, N = lin.shape[0], prob.N
    xt = np.full((B, N + 1, 10), np.nan); ut = np.full((B, N, 5), np.nan)
    status = np.full(B, -1, dtype=np.int32); it = np.full(B, -1, dtype=np.int32); qst = np.full(B, -1, dtype=np.int32)
    res = np.zeros((B, 5))
    n = lib.graph_loop_solve(C.byref(prob), C.c_int(B), _p(lin), _p(x0), _p(r), _p(act), C.c_int(graph),
                             _p(xt), _p(ut), _p(status), _p(it), _p(qst), _p(res))
    return n, dict(xt=xt, ut=ut, status=status, iter=it, qp_status=qst, res=res)


def _case(controller, iter_max=None, f32=False):
    N, B = 12, 70                      # three tiles, the last one padded
    prob64, params, md = make_problem(controller, N=N)
    prob, _, _ = make_problem(controller, N=N, precision='f32' if f32 else 'f64')
    if iter_max is not None:
        prob.qp_iter_max = iter_max
    o = Oracle(prob64, B, 2)
    x0 = start_states(B, seed=41, vel=0.6)
    x0[::3, 5:] *= 4.0                 # every third problem starts fast: spread iteration counts, some infeasible
    xg, ug = rollout_guess(x0, N, params.dt, seed=42)
    o.set_guess(xg, ug)
    r = np.full(B, 5 if controller in ('receding', 'real_receding') else N, dtype=np.int32)
    o.set_state(abi.STATE_R, r)
    o.rti_solve(x0)
    lin = np.ascontiguousarray(o.get_lin())
    act = np.ones(B, dtype=np.uint8); act[7::11] = 0
    return prob, lin, np.ascontiguousarray(x0), r, act


def _assert_same(e, g, act):
    for key in ('status', 'iter', 'qp_status', 'res'):
        assert np.array_equal(e[key], g[key]), key
    on = act == 1
    assert np.array_equal(e['xt'][on], g['xt'][on]) and np.array_equal(e['ut'][on], g['ut'][on])
    assert np.isnan(g['xt'][~on]).all() and (g['status'][~on] == -1).all()     # masked problems stay untouched


@pytest.mark.parametrize('f32', [False, True])
@pytest.mark.parametrize('controller', ['st', 'htwa', 'naive', 'receding', 'real_receding', 'constraint_everywhere'])
def test_graph_schedule_matches_host_loop(controller, f32):
    lib = _lib(f32)
    prob, lin, x0, r, act = _case(controller, f32=f32)
    n_host, e = _solve(lib, prob, lin, x0, r, act, graph=0)
    n_body, g = _solve(lib, prob, lin, x0, r, act, graph=1)
    assert len(set(e['iter'][act == 1].tolist())) >= 2, 'the case should spread the iteration counts'
    _assert_same(e, g, act)
    # the body runs once per iteration of the host loop, plus the one in which the last problem finished
    assert n_body == n_host + 1


@pytest.mark.parametrize('f32', [False, True])
def test_graph_schedule_iteration_limit_ends_the_loop(f32):
    lib = _lib(f32)
    prob, lin, x0, r, act = _case('st', iter_max=5, f32=f32)
    n_host, e = _solve(lib, prob, lin, x0, r, act, graph=0)
    n_body, g = _solve(lib, prob, lin, x0, r, act, graph=1)
    _assert_same(e, g, act)
    assert (e['qp_status'][act == 1] == 1).any(), 'some solve should end at the iteration limit'
    assert n_body == 6                 # iterations 0 .. 5: the loop step stops at kk = qp_iter_max
