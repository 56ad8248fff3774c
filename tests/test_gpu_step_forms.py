"""The step kernels run in two forms (csrc/qp.cu): the staged form reads the operands of qs_step from a per-warp ring of bulk copies in
shared memory, the thread form (SMPC_QP_STEP=thread) straight from global memory.  Every lane runs the same instructions on the same
values in both, so whole solves and closed loops must agree bit for bit, in both storage flavours."""
import os
from contextlib import contextmanager

import numpy as np
import pytest

from safe_mpc_b200 import abi
from tests.common import make_problem, start_states, rollout_guess, cfg0_initial_states, cfg0_plants, sqp_warm_start, run_closed_loop

pytestmark = pytest.mark.gpu


@contextmanager
def _env(env):
    env = {'SMPC_QP_SOLO': '0', **env}     # small batches would otherwise be served by the solo kernel, which has no staged form
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)


def _solve(controller, precision, env):
    from safe_mpc_b200.engine import Engine
    Bc, Nc = 1280, 16
    with _env(env):
        prob, params, md = make_problem(controller, N=Nc, precision=precision)
        eng = Engine(prob, Bc, 0)
    x0 = start_states(Bc, seed=41, vel=0.5)
    x0[::3, 5:] *= 4.0                     # fast starts: more iterations, centering fallbacks, infeasible problems
    xg, ug = rollout_guess(x0, Nc, params.dt, seed=42, scale=1.0)
    act = np.ones(Bc, dtype=np.uint8); act[3::19] = 0
    eng.set_guess(xg, ug)
    st = eng.rti_solve(x0, act)
    xt, ut = eng.get_temp()
    it = eng.get_state(abi.STATE_QP_ITER)
    eng.close()
    return st, xt, ut, it


@pytest.mark.parametrize('precision', ['f64', 'f32'])
@pytest.mark.parametrize('controller', ['st', 'htwa', 'receding', 'constraint_everywhere'])
def test_step_forms_agree_bitwise(controller, precision):
    thread = _solve(controller, precision, {'SMPC_QP_STEP': 'thread'})
    staged = _solve(controller, precision, {})
    for i in range(4):
        assert np.array_equal(thread[i], staged[i], equal_nan=True), i


@pytest.mark.parametrize('precision', ['f64', 'f32'])
@pytest.mark.parametrize('controller', ['st', 'htwa', 'receding', 'constraint_everywhere'])
def test_step_forms_closed_loop_agree_bitwise(controller, precision):
    from safe_mpc_b200.engine import Engine, Sim
    B, N, steps = 100, 30, 40
    prob, params, md = make_problem(controller, N=N, precision=precision)
    bprob, _, _ = make_problem('backup', cost='zero', N=params.back_hor, precision=precision)
    eng = Engine(prob, B, 0)
    x0 = cfg0_initial_states(eng, md, params, B, 'halton')
    pin, tn = cfg0_plants(md, params, B, 0.0, 0.0)
    xg, ug = sqp_warm_start(eng, x0, N, 10)
    eng.close()
    runs = []
    for env in ({'SMPC_QP_STEP': 'thread'}, {}):
        with _env(env):
            runs.append(run_closed_loop(Engine, Sim, prob, bprob, x0, xg, ug, pin, tn, steps))
    a, b = runs
    assert np.array_equal(a['outcome'], b['outcome'])
    assert np.array_equal(a['x'], b['x'], equal_nan=True) and np.array_equal(a['u'], b['u'], equal_nan=True)
    assert a['counters'] == b['counters']
