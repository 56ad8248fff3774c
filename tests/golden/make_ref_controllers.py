"""Golden of the REFERENCE's own controller state machines (reference src/safe_mpc/controller.py: NaiveController.step :274-284,
STWAController.step :375-388, RecedingController.step :448-498, RealReceding.step :524-565, ControllerSafeSetEverywhere.step :651-660,
provideControl :169-184, guessCorrection :226-231 -- rows a8 / a9 of SURVEY.md section 8), run in the build container.

controller.py cannot be imported (acados, casadi), so the class definitions are taken out of the file with ``ast`` and executed
UNMODIFIED; instances are made without ``__init__`` (which builds the acados OCP) and given the attributes the step methods use.  The
three things a step calls outside the class are stand-ins:
  * ``solve(x)``                 returns a scripted status and stores scripted x_temp / u_temp (the solve itself is row a7, pinned elsewhere);
  * ``model.checkStateConstraints``  is the reference's own method (env_model.py:170-177,236-243, bodies extracted unmodified: bounds on
                                 every row, collision check that returns after the first row) over the oracle's capsule distances;
  * ``checkSafeConstraints``     the oracle's viability value >= -tol (the network is pinned separately);
  * ``model.integrate_naively``  the double integrator of env_model.py:63-71.
What is recorded is everything the reference logic decides: control returned, abort flag, fails, receding index, viable state, next guess.
The scripted inputs are not stored: ``scripted_inputs`` draws them again from their seed, given the few values they depend on (stored:
the start states, the upper bound of joint 0, a colliding configuration per controller), and ``input_digest`` (stored) pins them bit for bit.

    python tests/golden/make_ref_controllers.py   ->  tests/golden/ref_controllers.npz
"""
import ast
import hashlib
import os
import sys
import types
from copy import deepcopy

import numpy as np
import scipy.linalg as lin

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
SRC = '/root/reference/src/safe_mpc/controller.py'
CLASSES = {'naive': 'NaiveController', 'zerovel': 'TerminalZeroVelocity', 'st': 'STController', 'stwa': 'STWAController', 'htwa': 'HTWAController',
           'receding': 'RecedingController', 'real_receding': 'RealReceding', 'constraint_everywhere': 'ControllerSafeSetEverywhere'}
N, B, STEPS = 8, 12, 14


def reference_classes():
    tree = ast.parse(open(SRC).read())
    ns = {'np': np, 'lin': lin, 'deepcopy': deepcopy}
    body = [n for n in tree.body if isinstance(n, ast.ClassDef)]
    exec(compile(ast.Module(body=body, type_ignores=[]), SRC, 'exec'), ns)
    return ns


def reference_checks():
    ENV = '/root/reference/src/safe_mpc/env_model.py'
    cls = next(n for n in ast.parse(open(ENV).read()).body if isinstance(n, ast.ClassDef) and n.name == 'AdamModel')
    keep = [n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name in ('checkStateConstraints', 'checkStateBounds', 'checkCollision')]
    assert len(keep) == 3
    mod = ast.Module(body=[ast.ClassDef(name='RefChecks', bases=[], keywords=[], body=keep, decorator_list=[])], type_ignores=[])
    ast.fix_missing_locations(mod)
    ns = {'np': np, 'deepcopy': deepcopy}
    exec(compile(mod, ENV, 'exec'), ns)
    return ns['RefChecks']()


def scripted_inputs(x0, x_max0, colliding):
    """the scripted guesses, states and solve outcomes of every controller, drawn in CLASSES order from one seeded stream:
    {name: {xg0, ug0, x, status, xt, ut}}, the last four per step.  x0: start states [B, 10]; x_max0: upper bound of joint 0;
    colliding[name]: a colliding configuration [10] or None."""
    rng = np.random.default_rng(123)
    out = {}
    for name in CLASSES:
        xg0 = np.repeat(x0[:, None, :], N + 1, axis=1) + 0.01 * rng.standard_normal((B, N + 1, 10))
        ug0 = 0.5 * rng.standard_normal((B, N, 5))
        rec = {k: [] for k in ('x', 'status', 'xt', 'ut')}
        for step in range(STEPS):
            x = x0 + 0.02 * step * rng.standard_normal((B, 10))
            # scripted solve outcomes: mostly successes inside the bounds, some failures, some trajectories out of bounds / unsafe
            status = rng.choice([0, 0, 0, 4, 2, 1], size=B).astype(np.int32)
            if step in (3, 4, 5, 6, 7, 8, 9, 10):
                status[:4] = 4                                          # a run of failures: exercises fails == N - 1 -> abort (N = 8)
            xt = np.repeat(x[:, None, :], N + 1, axis=1) + 0.05 * rng.standard_normal((B, N + 1, 10))
            xt[:, :, 5:] *= rng.choice([0.2, 1.0, 3.0], size=(B, 1, 1))   # slow / fast trajectories: safe / unsafe under the viability row
            viol = rng.random(B) < 0.15
            xt[viol, 3, 0] = x_max0 + 0.5                               # state-bound violation on a later row
            if colliding[name] is not None:
                late = rng.random(B) < 0.2
                xt[late, 4, :5] = colliding[name][:5]                   # a collision on a LATER row: not seen by the reference's checkCollision
                first = (rng.random(B) < 0.1) & ~late
                xt[first, 0, :5] = colliding[name][:5]                  # a collision on row 0: seen
            ut = rng.standard_normal((B, N, 5))
            for k, v in zip(('x', 'status', 'xt', 'ut'), (x, status, xt, ut)):
                rec[k].append(v)
        out[name] = {'xg0': xg0, 'ug0': ug0, **{k: np.array(v) for k, v in rec.items()}}
    return out


def input_digest(inputs):
    """sha256 of the arrays of scripted_inputs, controller by controller in CLASSES order, keys in sorted order"""
    h = hashlib.sha256()
    for name in CLASSES:
        for k in sorted(inputs[name]):
            h.update(np.ascontiguousarray(inputs[name][k]).tobytes())
    return h.hexdigest()


class _Solver:                                   # ocp_solver: the step methods only program flags / bounds on it
    def cost_set(self, *a): pass
    def set(self, *a): pass
    def constraints_set(self, *a): pass


def main():
    from tests.common import make_problem, random_states, start_states
    from oracle.oracle import Oracle
    ns = reference_classes()
    out = {'N': N, 'B': B, 'STEPS': STEPS}
    x0 = start_states(B, seed=7, vel=0.5)
    colliding = {}
    for name in CLASSES:
        prob, params, md = make_problem(name, N=N)
        cand = random_states(md, 4000, seed=3, vel_scale=0.0)
        dd = Oracle(prob, 1, 1).kinematics(cand)[1]
        bad = np.flatnonzero((dd < np.array(prob.pair_lo_chk)).any(axis=1) & ((cand >= md.x_min) & (cand <= md.x_max)).all(axis=1))
        colliding[name] = cand[bad[0]] if len(bad) else None
    x_max0 = float(md.x_max[0])
    inputs = scripted_inputs(x0, x_max0, colliding)
    out['x0'] = x0; out['x_max0'] = x_max0; out['input_digest'] = input_digest(inputs)
    for name, cls_name in CLASSES.items():
        prob, params, md = make_problem(name, N=N)
        orc = Oracle(prob, 1, 1)
        tol = params.tol_safe_set
        assert float(md.x_max[0]) == x_max0
        out[f'{name}_colliding'] = np.full(10, np.nan) if colliding[name] is None else colliding[name]

        # the reference's own predicates (env_model.py:170-177,236-243: checkStateConstraints -> bounds on every row and checkCollision,
        # which returns after the FIRST row of a trajectory), method bodies extracted unmodified; the capsule distance functions they
        # call are the oracle's
        checks = reference_checks()
        checks.x_min, checks.x_max, checks.params = md.x_min, md.x_max, types.SimpleNamespace(tol_x=params.tol_x)
        checks.collisions_constr_fun = [[(lambda x, p=p, orc=orc: float(orc.kinematics(np.asarray(x)[None])[1][0, p])), prob.pair_lo_chk[p],
                                         prob.pair_hi + params.tol_obs] for p in range(6)]
        check_state = checks.checkStateConstraints

        def check_safe(x, orc=orc):                                      # safe_set.py:61-68
            c = orc.nn_constraint(np.asarray(x)[None], grad=False)[0]
            return bool((0.0 - tol <= c) and (c <= 1e6 + tol))

        model = types.SimpleNamespace(nx=10, nu=5, ee_ref=np.array(params.ee_ref), x_min=md.x_min, x_max=md.x_max,
                                      params=types.SimpleNamespace(dt=params.dt, alpha=params.alpha, ws_t=params.ws_t, ws_r=params.ws_r,
                                                                   abort_flag=bool(params.abort_flag), N=N, use_net=True),
                                      checkStateConstraints=check_state,
                                      integrate_naively=lambda x, u, dt=params.dt: np.hstack([x[:5] + dt * x[5:] + 0.5 * dt * dt * u, x[5:] + dt * u]))
        rec = {k: [] for k in ('u', 'abort', 'fails', 'r', 'xv', 'xg', 'ug')}
        objs = []
        xg0, ug0 = inputs[name]['xg0'], inputs[name]['ug0']
        for b in range(B):
            o = ns[cls_name].__new__(ns[cls_name])
            o.model = model; o.N = N; o.fails = 0; o.current_step = 0; o.r = N; o.abort_flag = model.params.abort_flag
            o.x_guess = xg0[b].copy(); o.u_guess = ug0[b].copy(); o.x_temp = np.zeros((N + 1, 10)); o.u_temp = np.zeros((N, 5))
            o.x_viable = np.copy(o.x_guess[-1]); o.ocp_solver = _Solver(); o.zl = np.zeros(0); o.zl_e = np.zeros(1)
            o.checkSafeConstraints = check_safe
            objs.append(o)
        for step in range(STEPS):
            x, status, xt, ut = (inputs[name][k][step] for k in ('x', 'status', 'xt', 'ut'))
            us, abs_, fl, rr, xv, xgn, ugn = [], [], [], [], [], [], []
            for b, o in enumerate(objs):
                def solve(xx, o=o, b=b):
                    o.x_temp = xt[b].copy(); o.u_temp = ut[b].copy(); o.last_status = int(status[b])
                    return int(status[b])
                o.solve = solve
                u, ab = o.step(x[b])
                us.append(np.array(u, dtype=float)); abs_.append(bool(ab)); fl.append(o.fails); rr.append(getattr(o, 'r', N))
                xv.append(np.array(o.x_viable, dtype=float)); xgn.append(o.x_guess.copy()); ugn.append(o.u_guess.copy())
            for k, v in zip(('u', 'abort', 'fails', 'r', 'xv', 'xg', 'ug'), (us, abs_, fl, rr, xv, xgn, ugn)):
                rec[k].append(np.array(v))
        for k, v in rec.items():
            out[f'{name}_{k}'] = np.array(v)
        print(name, 'aborts', int(out[f'{name}_abort'].sum()), 'max fails', int(out[f'{name}_fails'].max()), 'r values', sorted(set(out[f'{name}_r'].ravel().tolist())))
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'ref_controllers.npz')
    np.savez_compressed(path, **out)
    print('wrote', path)


if __name__ == '__main__':
    main()
