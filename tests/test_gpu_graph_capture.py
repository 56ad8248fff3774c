"""Controller and plant steps captured into a CUDA graph (torch.cuda.graph on the handle's stream, INTEGRATION.md) and replayed: the QP
solve runs its interior-point loop from a conditional WHILE node on the device (csrc/qp.cu, qp_split.cuh: qs_graph_drive), or as the one
launch of the solo kernel for small batches.  A twin handle runs the same steps eagerly; every replay must agree with it bit for bit."""
import os

import numpy as np
import pytest

from safe_mpc_b200 import abi
from tests.common import make_problem, cfg0_initial_states, cfg0_plants, sqp_warm_start

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_CUDA, ERR_UNSUPPORTED = -1, -2, -3


def _engine_with_env(prob, B, env):
    from safe_mpc_b200.engine import Engine
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return Engine(prob, B, 0)               # (the switches are read when the handle is created)
    finally:
        for k, v in old.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)


def _setup(controller, precision, B, N=30, nn_precision=None, **kw):
    from safe_mpc_b200.engine import Engine
    prob, params, md = make_problem(controller, N=N, precision=precision, nn_precision=nn_precision)
    for k, v in kw.items():
        setattr(prob, k, v)
    eng = Engine(prob, B, 0)
    x0 = cfg0_initial_states(eng, md, params, B, 'halton')
    pin, tn = cfg0_plants(md, params, B, 0.1, 2.0)
    xg, ug = sqp_warm_start(eng, x0, N, 3)
    eng.close()
    pair = []
    for _ in range(2):
        e = Engine(prob, B, 0)
        e.set_guess(xg, ug); e.reset_controller()
        e.set_plant_inertial(pin); e.set_torque_noise(tn)
        pair.append(e)
    return pair, x0


def _snapshot(eng, x, u, ab):
    import torch
    xg, ug = eng.get_guess(like=x)
    out = dict(x=x, u=u, abort=ab, xg=xg, ug=ug)
    for name, f in (('status', abi.STATE_STATUS), ('qp_iter', abi.STATE_QP_ITER), ('fails', abi.STATE_FAILS), ('r', abi.STATE_R)):
        out[name] = eng.get_state(f, like=x)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


@pytest.mark.parametrize('B', [256, 4096])
@pytest.mark.parametrize('precision', ['f64', 'f32'])
@pytest.mark.parametrize('controller', ['naive', 'st', 'htwa', 'receding', 'constraint_everywhere'])
def test_captured_closed_loop_matches_eager(controller, precision, B):
    _closed_loop(controller, precision, B)


def test_captured_closed_loop_tf32x3():
    _closed_loop('htwa', 'f64', 4096, nn_precision='tf32x3')


def _closed_loop(controller, precision, B, nn_precision=None, steps=40):
    import torch
    (eg, ee), x0 = _setup(controller, precision, B, nn_precision=nn_precision)
    s = torch.cuda.Stream()
    eg.set_stream(s)
    x_g = torch.tensor(x0, device='cuda')
    x_e = x_g.clone()
    s.wait_stream(torch.cuda.current_stream())
    # warm-up: one eager step on both handles (the same step, so the twins stay in lock-step)
    with torch.cuda.stream(s):
        u, ab = eg.controller_step(x_g)
        xn, _ = eg.plant_step(x_g, u)
        x_g.copy_(xn)
    u_e, ab_e = ee.controller_step(x_e)
    x_e, _ = ee.plant_step(x_e, u_e)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        u_s, ab_s = eg.controller_step(x_g)
        xn_s, _ = eg.plant_step(x_g, u_s)
        x_g.copy_(xn_s)
    n_iters = set()
    for j in range(steps):
        g.replay()
        u_e, ab_e = ee.controller_step(x_e)
        x_e, _ = ee.plant_step(x_e, u_e)
        a = _snapshot(eg, x_g, u_s, ab_s)
        b = _snapshot(ee, x_e, u_e, ab_e)
        for k in a:
            assert np.array_equal(a[k], b[k], equal_nan=True), (j, k)
        n_iters.add(int(b['qp_iter'].max()))
    assert max(n_iters) > 0
    eg.close(); ee.close()


def test_captured_solve_ends_at_the_iteration_limit():
    import torch
    B = 4096
    (eg, ee), x0 = _setup('st', 'f64', B, qp_iter_max=5)
    s = torch.cuda.Stream()
    eg.set_stream(s)
    x = torch.tensor(x0, device='cuda')
    x[::3, 5:] = 0.8                  # moving starts: solves that need more than five iterations
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eg.rti_solve(x)               # warm-up
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        st_g = eg.rti_solve(x)
    g.replay()
    st_e = ee.rti_solve(x)
    torch.cuda.synchronize()
    assert torch.equal(st_g, st_e)
    for f in (abi.STATE_QP_ITER, abi.STATE_QP_STATUS):
        a, b = eg.get_state(f, like=x), ee.get_state(f, like=x)
        torch.cuda.synchronize()
        assert torch.equal(a, b), f
    qst = ee.get_state(abi.STATE_QP_STATUS)
    assert (qst == 1).any() and ee.get_state(abi.STATE_QP_ITER).max() == 5
    eg.close(); ee.close()


def _refused(eng, fn, code):
    import torch
    s = torch.cuda.Stream()
    eng.set_stream(s)
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):         # (the capture must still end cleanly after the refusal)
        with pytest.raises(RuntimeError, match=rf'failed \({code}\)'):
            fn()
    torch.cuda.synchronize()


def test_capture_refusals():
    import torch
    from safe_mpc_b200.engine import Engine
    B = 64
    (eng, _), x0 = _setup('htwa', 'f64', B)
    x = torch.tensor(x0, device='cuda')
    _refused(eng, lambda: eng.controller_step(x0), ERR_ARG)                  # host arrays
    _refused(eng, lambda: eng.rti_solve(x0), ERR_ARG)
    _refused(eng, lambda: eng.plant_step(x0, np.zeros((B, abi.NU))), ERR_ARG)
    eng.set_profiling(True)
    _refused(eng, lambda: eng.controller_step(x), ERR_UNSUPPORTED)          # profiling reads the timeline on the host
    eng.set_profiling(False)
    u, ab = eng.controller_step(x)                                         # the handle still works eagerly
    torch.cuda.synchronize()
    assert torch.isfinite(u).all()
    eng.close()
    prob, params, md = make_problem('parallel', N=20)
    par = Engine(prob, B, 0)
    _refused(par, lambda: par.controller_step(x), ERR_UNSUPPORTED)          # early stop reads a counter on the host
    par.close()


def test_capture_refusals_trace_groups_and_invalidated_capture():
    import torch
    prob, params, md = make_problem('st', N=20)
    x = torch.zeros((8192, abi.NX), dtype=torch.float64, device='cuda')
    tr = _engine_with_env(prob, 64, {'SMPC_QP_TRACE': '1'})
    _refused(tr, lambda: tr.controller_step(x[:64]), ERR_UNSUPPORTED)      # the trace reads the kernel timeline on the host
    tr.close()
    gr = _engine_with_env(prob, 8192, {'SMPC_QP_GROUPS': '2'})
    _refused(gr, lambda: gr.rti_solve(x), ERR_UNSUPPORTED)                 # several tile groups
    gr.close()
    from safe_mpc_b200.engine import Engine
    eng = Engine(prob, 64, 0)
    s = torch.cuda.Stream()
    eng.set_stream(s)
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError):
        with torch.cuda.graph(g, stream=s, capture_error_mode='relaxed'):
            try:
                s.query()                       # not allowed while capturing: invalidates the capture
            except RuntimeError:
                pass
            with pytest.raises(RuntimeError, match=rf'failed \({ERR_CUDA}\)'):
                eng.controller_step(x[:64])
    torch.cuda.synchronize()
    eng.close()


def _sim_pair(B, steps):
    """the stress case of tools/long_run_check.py: receding controller, N = 20, 5 % model noise, three-fold initial velocities (aborts and
    backup solves in the first steps, none once the problems have settled or ended)"""
    import bench
    from safe_mpc_b200.engine import Engine, Sim
    N = 20
    params, md, x0, pin = bench.workload('receding', N, 5.0, 3, 0, B)
    x0[:, 5:] *= 3.0
    out = []
    for _ in range(2):
        main, bk, prob = bench.make_handles(Engine, params, md, 'receding', B, 0)
        main.set_plant_inertial(pin)
        bench.warm_guess(main, x0, N, 3)
        sim = Sim(main, bk, steps)
        sim.reset(x0)
        out.append((sim, main, bk))
    return out


def test_captured_sim_step_matches_eager_sim_run():
    """smpc_sim_step captured once (after one eager step) and replayed: the backup solve sits in a conditional IF node (with the WHILE node
    of its QP inside); outcome codes, logs and counters equal those of an eager smpc_sim_run of the same closed loop, and the loop has steps
    with and without backup solves."""
    import torch
    B, steps = 256, 200
    (sg, mg, bg), (se, me, be) = _sim_pair(B, steps)
    se.run(steps)
    s = torch.cuda.Stream()
    mg.set_stream(s)
    sg.step()                                   # warm-up: one eager step
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        sg.step()
    with_backup = without_backup = 0
    seen = sg.counters()['backup_solves']
    for j in range(steps - 1):
        g.replay()
        torch.cuda.synchronize()
        n = sg.counters()['backup_solves']
        with_backup += n > seen
        without_backup += n == seen
        seen = n
    a_x, a_u = sg.log(); b_x, b_u = se.log()
    assert np.array_equal(np.asarray(sg.outcome()), np.asarray(se.outcome()))
    assert np.array_equal(a_x, b_x, equal_nan=True) and np.array_equal(a_u, b_u, equal_nan=True)
    assert sg.counters() == se.counters()
    assert with_backup > 0 and without_backup > 0, (with_backup, without_backup)
    for sim, m, b in ((sg, mg, bg), (se, me, be)):
        sim.close() if hasattr(sim, 'close') else None
        m.close(); b.close()
