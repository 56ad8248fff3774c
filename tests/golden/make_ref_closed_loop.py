"""Golden of the REFERENCE's own closed-loop script (reference scripts/mpc.py:87-287: per-test loop, safe-abort handling, PD following and
hold, break conditions, outcome sets -- row a12 of SURVEY.md section 8) driving the REFERENCE's own controller classes (controller.py,
rows a8 / a9), run in the build container.

mpc.py is a flat script that builds acados solvers at its top; the statements of its simulation part (from ``conv_idx, ... = [], [], []`` to
``unconv_idx = ...``) are taken out of the file with ``ast`` and executed UNMODIFIED in a namespace that holds what they reference:
  * ``controller``     an instance of the reference's controller class (class body extracted from controller.py, no ``__init__``) whose
                       ``solve`` returns a scripted outcome per (test, step);
  * ``safe_ocp``       the backup OCP: ``solve`` returns a scripted outcome per (test, step);
  * ``model``          predicates, plant step and end-effector position evaluated by the oracle (bounds / collision checks, plant_step with
                       the nominal plant, kinematics), so that the scripted trajectories mean the same to both sides;
  * the remaining names (params, args, counters, ...) as plain values.
Recorded: the x / u logs (NaN padded), conv / collisions / viable / unconv index sets, the initial states.  The scripted outcomes are
not stored: ``scripted_inputs`` draws them again from their seeds, and ``input_digest`` (stored) pins them bit for bit.

    python tests/golden/make_ref_closed_loop.py   ->  tests/golden/ref_closed_loop.npz
"""
import ast
import hashlib
import os
import sys
import types
from copy import deepcopy
from functools import reduce

import numpy as np
import scipy.linalg as lin

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
MPC = '/root/reference/scripts/mpc.py'
CTRL = '/root/reference/src/safe_mpc/controller.py'
CLASSES = {'naive': 'NaiveController', 'htwa': 'HTWAController', 'receding': 'RecedingController'}
N, NB, B, STEPS = 8, 6, 10, 40


def reference_classes():
    ns = {'np': np, 'lin': lin, 'deepcopy': deepcopy}
    exec(compile(ast.Module(body=[n for n in ast.parse(open(CTRL).read()).body if isinstance(n, ast.ClassDef)], type_ignores=[]), CTRL, 'exec'), ns)
    return ns


def simulation_statements():
    """module-level statements of mpc.py from the initialisation of the index lists to the computation of unconv_idx"""
    tree = ast.parse(open(MPC).read())
    first = next(i for i, n in enumerate(tree.body) if isinstance(n, ast.Assign) and isinstance(n.targets[0], ast.Tuple)
                 and [getattr(e, 'id', None) for e in n.targets[0].elts] == ['conv_idx', 'collisions_idx', 'viable_idx'])
    last = next(i for i, n in enumerate(tree.body) if isinstance(n, ast.Assign) and getattr(n.targets[0], 'id', None) == 'unconv_idx')
    return compile(ast.Module(body=tree.body[first:last + 1], type_ignores=[]), MPC, 'exec')


def scripted_inputs(name, x_init):
    """the scripted outcomes of the main and backup solves per (test, step) of one controller's run, drawn from its seed"""
    rng = np.random.default_rng({'naive': 11, 'htwa': 12, 'receding': 13}[name])
    status = rng.choice([0, 0, 0, 0, 4], size=(B, STEPS)).astype(np.int32)
    status[:4, 5:16] = 4                                           # a long run of failures for the first tests -> abort
    if name == 'receding':
        status[4:6, :] = 0
    xt = x_init[:, None, None, :] + 0.02 * rng.standard_normal((B, STEPS, N + 1, 10))
    xt[:, :, :, 5:] *= rng.choice([0.05, 1.0, 4.0], size=(B, STEPS, 1, 1))
    ut = 2.0 * rng.standard_normal((B, STEPS, N, 5))
    bk_status = rng.choice([0, 0, 0, 4], size=(B, STEPS)).astype(np.int32)
    bk_xt = x_init[:, None, None, :] + 0.02 * rng.standard_normal((B, STEPS, NB + 1, 10))
    bk_xt[:, :, :, 5:] *= 0.1
    bk_xt[1, :, -1, 5:] = 0.5                                      # test 1: the abort trajectory does not end at rest -> PD hold (mpc.py:143-144)
    bk_ut = 0.5 * rng.standard_normal((B, STEPS, NB, 5))
    return {'status': status, 'xt': xt, 'ut': ut, 'bk_status': bk_status, 'bk_xt': bk_xt, 'bk_ut': bk_ut}


def input_digest(inputs):
    """sha256 of the arrays of scripted_inputs, in key order"""
    h = hashlib.sha256()
    for k in sorted(inputs):
        h.update(np.ascontiguousarray(inputs[k]).tobytes())
    return h.hexdigest()


class _Solver:
    def cost_set(self, *a): pass
    def set(self, *a): pass
    def constraints_set(self, *a): pass
    def get_stats(self, *a): return 0


def main():
    from tests.common import make_problem, start_states
    from oracle.oracle import Oracle
    cls = reference_classes()
    code = simulation_statements()
    out = {'N': N, 'NB': NB, 'B': B, 'STEPS': STEPS}
    for name, cls_name in CLASSES.items():
        prob, params, md = make_problem(name, N=N)
        orc = Oracle(prob, 1, 1)
        tol = params.tol_safe_set
        x_init = start_states(B, seed=17, vel=0.4)
        xg0 = np.repeat(x_init[:, None, :], N + 1, axis=1)
        ug0 = np.zeros((B, N, 5))
        script = scripted_inputs(name, x_init)
        status, xt, ut, bk_status, bk_xt, bk_ut = (script[k] for k in ('status', 'xt', 'ut', 'bk_status', 'bk_xt', 'bk_ut'))

        def state_in_bounds(x):
            return bool(np.all((x >= md.x_min - params.tol_x) & (x <= md.x_max + params.tol_x)))

        def collision_free(x):
            if not np.all(np.isfinite(x)):
                return False
            _, dist = orc.kinematics(np.asarray(x)[None])
            return bool(np.all((np.array(prob.pair_lo_chk) <= dist[0]) & (dist[0] <= prob.pair_hi + params.tol_obs)))

        def check_state_constraints(traj):                             # env_model.py:170-173 with the early return of :236-243
            return bool(np.all((traj >= md.x_min - params.tol_x) & (traj <= md.x_max + params.tol_x)) and collision_free(traj[0]))

        def check_safe(x):
            c = orc.nn_constraint(np.asarray(x)[None], grad=False)[0]
            return bool((0.0 - tol <= c) and (c <= 1e6 + tol))

        def integrate(x, u):
            xn, a = orc.plant_step(np.asarray(x)[None], np.asarray(u)[None])
            return xn[0], a[0]

        def joint_to_ee(x):
            if not np.all(np.isfinite(x)):
                return np.full((3, 1), np.nan)
            ee, _ = orc.kinematics(np.asarray(x)[None])
            return ee[0].reshape(3, 1)

        mparams = types.SimpleNamespace(dt=params.dt, alpha=params.alpha, ws_t=params.ws_t, ws_r=params.ws_r, abort_flag=bool(params.abort_flag), N=N,
                                        use_net=True)
        cmodel = types.SimpleNamespace(nx=10, nu=5, ee_ref=np.array(params.ee_ref), x_min=md.x_min, x_max=md.x_max, params=mparams,
                                       checkStateConstraints=check_state_constraints, checkCollision=collision_free,
                                       update_randomized_dynamics=lambda **k: None,
                                       integrate_naively=lambda x, u, dt=params.dt: np.hstack([x[:5] + dt * x[5:] + 0.5 * dt * dt * u, x[5:] + dt * u]))
        controller = cls[cls_name].__new__(cls[cls_name])
        controller.model = cmodel; controller.N = N; controller.fails = 0; controller.current_step = 0; controller.r = N
        controller.abort_flag = mparams.abort_flag; controller.x_guess = xg0[0].copy(); controller.u_guess = ug0[0].copy()
        controller.x_temp = np.zeros((N + 1, 10)); controller.u_temp = np.zeros((N, 5)); controller.x_viable = xg0[0][-1].copy()
        controller.ocp_solver = _Solver(); controller.zl = np.zeros(0); controller.zl_e = np.zeros(1); controller.last_status = 4
        controller.checkSafeConstraints = check_safe
        controller.getTime = lambda: np.zeros(7)
        controller.time_fields = ['t'] * 7
        ns = {'np': np, 'reduce': reduce, 'CALLBACK': False, 'nq': 5, 'cont_name': name, 'args': {'noise': 0.0, 'controller': name},
              'params': types.SimpleNamespace(test_num=B, n_steps=STEPS, alpha=params.alpha, tol_x=params.tol_x, tol_tau=params.tol_tau,
                                              tol_conv=params.tol_conv, urdf_name='z1'),
              'x_guess': xg0, 'u_guess': ug0, 'x_init': x_init, 'controller': controller}

        def solve(x):
            i, j = ns['i'], ns['j']
            controller.x_temp = xt[i, j].copy(); controller.u_temp = ut[i, j].copy(); controller.last_status = int(status[i, j])
            return int(status[i, j])
        controller.solve = solve
        safe = types.SimpleNamespace(N=NB, model=types.SimpleNamespace(update_randomized_dynamics=lambda **k: None), x_temp=None, u_temp=None)
        safe.setGuess = lambda xg, ug: None

        def bk_solve(x):
            i, j = ns['i'], ns['j']
            safe.x_temp = bk_xt[i, j].copy(); safe.u_temp = bk_ut[i, j].copy()
            return int(bk_status[i, j])
        safe.solve = bk_solve
        ns['safe_ocp'] = safe
        ns['model'] = types.SimpleNamespace(nx=10, nu=5, ee_ref=np.array(params.ee_ref), x_min=md.x_min, x_max=md.x_max, reset_seed=lambda i: None,
                                            tau_fun=lambda x, u: np.zeros((5, 1)), checkStateConstraints=check_state_constraints,
                                            checkTorqueBounds=lambda tau: True, integrate=integrate, checkStateBounds=state_in_bounds,
                                            jointToEE=joint_to_ee)
        ns['model_backup'] = types.SimpleNamespace(reset_seed=lambda i: None)
        exec(code, ns)
        xv_first = np.full((B, 10), np.nan)
        # x_viable is appended once per abort, in test order: recover the first abort of every test from the logs of the loop
        out[f'{name}_x'] = np.asarray(ns['x_sim_list']); out[f'{name}_u'] = np.asarray(ns['u_list'])
        out[f'{name}_conv'] = np.array(sorted(ns['conv_idx']), dtype=np.int64); out[f'{name}_coll'] = np.array(sorted(set(ns['collisions_idx'])), dtype=np.int64)
        out[f'{name}_viable'] = np.array(sorted(ns['viable_idx']), dtype=np.int64); out[f'{name}_unconv'] = np.array(sorted(ns['unconv_idx']), dtype=np.int64)
        out[f'{name}_n_aborts'] = len(ns['x_viable'])
        out[f'{name}_x_init'] = x_init
        out[f'{name}_input_digest'] = input_digest(script)
        print(name, 'conv', ns['conv_idx'], 'collisions', sorted(set(ns['collisions_idx'])), 'viable', sorted(ns['viable_idx']), 'unconv', ns['unconv_idx'],
              'aborts', len(ns['x_viable']))
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'ref_closed_loop.npz')
    np.savez_compressed(path, **out)
    print('wrote', path)


if __name__ == '__main__':
    main()
