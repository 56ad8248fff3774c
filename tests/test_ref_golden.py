"""Golden vectors computed with the REFERENCE's own ``NeuralNetwork`` class (tests/golden/make_ref_golden.py, run in the build container
where /root/reference is mounted): the one piece of the hot path that executes without casadi / acados / adam / l4casadi.
They pin row a5 of SURVEY.md section 8 -- architecture, layer order, GELU(tanh), psi(x), c(x) and dc/dx -- on reference code instead of on
a restatement: the oracle must reproduce the fp64 evaluation of the reference class to rounding, and the reference's fp32 evaluation
(what its L4CasADi call computes) to fp32 accuracy; the CUDA kernels are held to the same vectors."""
import functools
import os

import numpy as np
import pytest

from tests.common import make_problem

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_network.npz'))


def test_oracle_matches_the_reference_network_class():
    from oracle.oracle import Oracle
    prob, params, md = make_problem('st', N=10, alpha=float(G['alpha']))
    orc = Oracle(prob, 4, 0)
    c, g = orc.nn_constraint(G['x'])
    assert np.abs(c - G['c']).max() <= 1e-9 * max(1.0, np.abs(G['c']).max())          # fp32 weights, fp64 accumulation on both sides
    assert np.abs(g - G['grad']).max() <= 1e-9 * max(1.0, np.abs(G['grad']).max())
    # what the reference itself computes (fp32 inside libtorch) differs from both by fp32 rounding only
    s = (100.0 - float(G['alpha'])) / 100.0
    assert np.abs((G['y32'] - G['y64']) * s).max() <= 2e-6


@pytest.mark.gpu
@pytest.mark.parametrize('precision,kernel,tol', [('strict', 'single', 1e-9), ('tf32x3', 'single', 2e-5), ('tf32x3', 'pair', 2e-5)])
def test_engine_matches_the_reference_network_class(precision, kernel, tol):
    from safe_mpc_b200.engine import Engine
    prob, params, md = make_problem('st', N=10, alpha=float(G['alpha']), nn_precision=precision)
    old = os.environ.get('SMPC_MLP_TC')
    os.environ['SMPC_MLP_TC'] = kernel
    try:
        eng = Engine(prob, 4, 0)
    finally:
        if old is None:
            os.environ.pop('SMPC_MLP_TC', None)
        else:
            os.environ['SMPC_MLP_TC'] = old
    c, g = eng.nn_constraint(G['x'])
    assert np.abs(c - G['c']).max() <= tol * max(1.0, np.abs(G['c']).max())
    assert np.abs(g - G['grad']).max() <= tol * max(1.0, np.abs(G['grad']).max())


# ---------------------------------------------------------------------------------------------------------------------------
# reference parser.py (Parameters, parse_args) evaluated on the reference's own config.yaml  ->  tests/golden/ref_parameters.json
# ---------------------------------------------------------------------------------------------------------------------------
import json

P = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_parameters.json')))
ARGV = {'default': [],
        'margins': ['--joint_bounds_margin', '5', '--collision_margin', '0.02', '--noise', '10', '-c', 'receding', '--horizon', '35', '--alpha', '20']}


# placeholders of the moving capsules that env_model.py:131-151 later fills with CasADi functions (the engine has no such objects)
CASADI_SLOTS = {'end_points_T_fun', 'end_points_fk', 'end_points_fk_fun'}


def _same(a, b, path=''):
    """recursive comparison of a value of this repo's Parameters with the reference's (lists / arrays / dicts / scalars)"""
    if isinstance(b, dict):
        keys = set(b) - CASADI_SLOTS
        assert isinstance(a, dict) and keys <= set(a), f'{path}: keys {sorted(keys - set(a))} missing'
        for k in keys:
            _same(a[k], b[k], f'{path}.{k}')
    elif isinstance(b, list):
        a = a.tolist() if isinstance(a, np.ndarray) else list(a)
        assert len(a) == len(b), f'{path}: length {len(a)} != {len(b)}'
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, f'{path}[{i}]')
    elif isinstance(b, float):
        assert abs(float(a) - b) <= 1e-15 * max(1.0, abs(b)), f'{path}: {a} != {b}'
    elif b is None:
        assert a is None, f'{path}: {a} is not None'
    else:
        a = a.item() if isinstance(a, (np.integer, np.floating, np.bool_)) else a
        assert a == b, f'{path}: {a!r} != {b!r}'


@pytest.mark.parametrize('tag', ['default', 'margins'])
def test_parameters_match_the_reference_parser(tag):
    from safe_mpc_b200.parser import Parameters, parse_args
    args = parse_args(ARGV[tag])
    for k, v in P[tag]['args'].items():                    # the reference's CLI: same keys, same defaults (parser.py:9-34)
        assert args[k] == v, f'args[{k}]'
    p = Parameters(args, 'z1', rti=True)
    ref = P[tag]['params']
    assert len(ref) >= 50
    for k, v in ref.items():
        assert hasattr(p, k), f'Parameters.{k} missing'
        _same(getattr(p, k), v, k)


# ---------------------------------------------------------------------------------------------------------------------------
# reference utils.py: randomize_model (a13) and rot_mat_x/y/z, executed unmodified (tests/golden/make_ref_randomize.py)
# ---------------------------------------------------------------------------------------------------------------------------
R = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_randomize.npz'))


@pytest.mark.parametrize('seed', [1, 2])
def test_randomized_inertials_match_the_reference_function(seed):
    """the draw order and the perturbation of the reference's randomize_model (mass, 6 inertia entries, CoM, link by link) -- the
    per-problem plant parameters of the model-noise ensemble (BASELINE.json configs[3])"""
    from safe_mpc_b200 import urdf as U
    from safe_mpc_b200.robot_model import nominal_link_inertials, randomized_link_inertials
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    nominal = nominal_link_inertials(U.URDF.from_xml_file(os.path.join(root, 'robots', 'z1_description', 'urdf', 'z1.urdf')))
    pct = float(R[f'pct_{seed}'])
    count = R[f'mass_{seed}'].shape[0]
    ours = randomized_link_inertials(nominal, pct, pct, pct, count, seed=seed)
    # the reference writes the numbers through str() into the URDF text and reads them back: exact round trip for doubles
    np.testing.assert_allclose(ours['mass'], R[f'mass_{seed}'], rtol=1e-15, atol=0)
    np.testing.assert_allclose(ours['inertia6'], R[f'inertia6_{seed}'], rtol=1e-15, atol=0)
    np.testing.assert_allclose(ours['com'], R[f'com_{seed}'], rtol=1e-15, atol=0)


def test_rotation_helpers_match_the_reference_functions():
    from safe_mpc_b200.robot_model import rot_mat_x, rot_mat_y, rot_mat_z
    for i, t in enumerate(R['theta']):
        np.testing.assert_array_equal(rot_mat_x(t), R['rot_x'][i])
        np.testing.assert_array_equal(rot_mat_y(t), R['rot_y'][i])
        np.testing.assert_array_equal(rot_mat_z(t), R['rot_z'][i])


def test_capsule_distances_match_the_reference_function():
    """row a4: squared segment-segment distances with the clamped parameters and the R^2 + 1e-5 regulariser of the reference's
    casadi_segment_dist, evaluated by the reference function itself on the capsule end points of 64 random configurations"""
    from oracle.oracle import Oracle
    prob, params, md = make_problem('naive', N=10)
    orc = Oracle(prob, 4, 0)
    ee, dist = orc.kinematics(R['dist_x'])
    np.testing.assert_allclose(dist, R['dist'], rtol=1e-11, atol=1e-13)


# ---------------------------------------------------------------------------------------------------------------------------
# reference controller.py: the step state machines, provideControl and guessCorrection (rows a8 / a9), driven with scripted solve
# outcomes (tests/golden/make_ref_controllers.py); the oracle is driven with the same sequences
# ---------------------------------------------------------------------------------------------------------------------------
CG = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_controllers.npz'))


@functools.lru_cache(maxsize=None)
def controller_script():
    """the scripted inputs the golden outputs were recorded with, drawn again from their seed (only the outputs are stored)"""
    from tests.golden.make_ref_controllers import CLASSES, input_digest, scripted_inputs
    colliding = {n: None if np.isnan(CG[f'{n}_colliding']).all() else CG[f'{n}_colliding'] for n in CLASSES}
    script = scripted_inputs(CG['x0'], float(CG['x_max0']), colliding)
    assert input_digest(script) == str(CG['input_digest']), 'the seeded stream no longer reproduces the recorded scripted inputs'
    return script


@pytest.mark.parametrize('name', ['naive', 'zerovel', 'st', 'stwa', 'htwa', 'receding', 'real_receding', 'constraint_everywhere'])
def test_controller_state_machines_match_the_reference_classes(name):
    from oracle.oracle import Oracle
    from safe_mpc_b200 import abi
    N, B, steps = int(CG['N']), int(CG['B']), int(CG['STEPS'])
    CI = controller_script()[name]
    prob, params, md = make_problem(name, N=N)
    orc = Oracle(prob, B, 1)
    orc.set_guess(CI['xg0'], CI['ug0'])
    orc.reset_controller()
    for s in range(steps):
        u, ab = orc.controller_step_scripted(CI['x'][s], CI['status'][s], CI['xt'][s], CI['ut'][s])
        where = f'{name}, step {s}'
        np.testing.assert_array_equal(ab, CG[f'{name}_abort'][s], err_msg=f'abort flag, {where}')
        np.testing.assert_array_equal(orc.get_state(abi.STATE_FAILS), CG[f'{name}_fails'][s], err_msg=f'fails, {where}')
        if name in ('receding', 'real_receding'):
            np.testing.assert_array_equal(orc.get_state(abi.STATE_R), CG[f'{name}_r'][s], err_msg=f'receding index, {where}')
        np.testing.assert_allclose(u, CG[f'{name}_u'][s], rtol=0, atol=1e-14, err_msg=f'control, {where}')
        xg, ug = orc.get_guess()
        np.testing.assert_allclose(xg, CG[f'{name}_xg'][s], rtol=0, atol=1e-13, err_msg=f'x_guess, {where}')
        np.testing.assert_allclose(ug, CG[f'{name}_ug'][s], rtol=0, atol=1e-14, err_msg=f'u_guess, {where}')
        if name in ('stwa', 'htwa', 'receding', 'real_receding'):
            aborted = CG[f'{name}_abort'][:s + 1].any(axis=0) | (CG[f'{name}_fails'][:s + 1] > 0).any(axis=0)
            np.testing.assert_allclose(orc.get_x_viable()[aborted], CG[f'{name}_xv'][s][aborted], rtol=0, atol=1e-13, err_msg=f'x_viable, {where}')


# ---------------------------------------------------------------------------------------------------------------------------
# reference scripts/mpc.py: the closed-loop simulation statements (row a12), executed unmodified around the reference's own controller
# classes with scripted solve outcomes (tests/golden/make_ref_closed_loop.py); the oracle's closed loop is driven with the same script
# ---------------------------------------------------------------------------------------------------------------------------
LG = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_closed_loop.npz'))


@pytest.mark.parametrize('name', ['naive', 'htwa', 'receding'])
def test_closed_loop_matches_the_reference_script(name):
    from oracle.oracle import Oracle, OracleSim
    from safe_mpc_b200 import abi
    N, NB, B, steps = int(LG['N']), int(LG['NB']), int(LG['B']), int(LG['STEPS'])
    from tests.golden.make_ref_closed_loop import input_digest, scripted_inputs
    prob, params, md = make_problem(name, N=N)
    bprob, _, _ = make_problem('backup', cost='zero', N=NB)
    main, bk = Oracle(prob, B, 1), Oracle(bprob, B, 1)
    x_init = LG[f'{name}_x_init']
    SI = scripted_inputs(name, x_init)                    # drawn again from its seed: only the outputs are stored
    assert input_digest(SI) == str(LG[f'{name}_input_digest']), 'the seeded stream no longer reproduces the recorded scripted inputs'
    main.set_guess(np.repeat(x_init[:, None, :], N + 1, axis=1).copy(), np.zeros((B, N, abi.NU)))
    main.reset_controller()
    sim = OracleSim(main, bk, steps)
    sim.reset(x_init)
    for j in range(steps):
        sim.set_script(SI['status'][:, j], SI['xt'][:, j], SI['ut'][:, j], SI['bk_status'][:, j], SI['bk_xt'][:, j], SI['bk_ut'][:, j])
        sim.step()
    x, u = sim.log()
    gx, gu = LG[f'{name}_x'], LG[f'{name}_u']
    np.testing.assert_array_equal(np.isnan(x), np.isnan(gx), err_msg='termination pattern of the state log')
    np.testing.assert_array_equal(np.isnan(u), np.isnan(gu), err_msg='termination pattern of the control log')
    np.testing.assert_allclose(np.nan_to_num(x), np.nan_to_num(gx), rtol=0, atol=1e-10)
    np.testing.assert_allclose(np.nan_to_num(u), np.nan_to_num(gu), rtol=0, atol=1e-9)
    out = sim.outcome()
    conv = np.flatnonzero(out & abi.OUT_CONVERGED)
    coll = np.flatnonzero(out & abi.OUT_COLLIDED)
    viable = np.flatnonzero((out & abi.OUT_ABORTED) != 0) if hasattr(abi, 'OUT_ABORTED') else None
    viable = np.array([i for i in viable if i not in conv and i not in coll], dtype=np.int64)      # mpc.py:273-285
    unconv = np.setdiff1d(np.arange(B), np.concatenate([conv, coll, viable]))
    np.testing.assert_array_equal(conv, LG[f'{name}_conv']); np.testing.assert_array_equal(coll, LG[f'{name}_coll'])
    np.testing.assert_array_equal(viable, LG[f'{name}_viable']); np.testing.assert_array_equal(unconv, LG[f'{name}_unconv'])


# ---------------------------------------------------------------------------------------------------------------------------
# reference env_model.py: AdamModel.integrate (row a11), method body executed unmodified (tests/golden/make_ref_plant.py)
# ---------------------------------------------------------------------------------------------------------------------------
PG = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_plant.npz'))


def test_plant_step_matches_the_reference_method():
    from oracle.oracle import Oracle
    B = PG['x'].shape[0]
    prob, params, md = make_problem('naive', N=10)
    orc = Oracle(prob, B, 1)
    orc.set_plant_inertial(PG['pin'])
    xn, a = orc.plant_step(PG['x'], PG['u'])
    assert PG['sat'].sum() >= 5 and (~PG['sat']).sum() >= 5          # both branches of the saturation are exercised
    np.testing.assert_allclose(a, PG['acc'], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(xn, PG['xn'], rtol=1e-11, atol=1e-11)


@pytest.mark.gpu
def test_engine_plant_step_matches_the_reference_method():
    from safe_mpc_b200.engine import Engine
    B = PG['x'].shape[0]
    prob, params, md = make_problem('naive', N=10)
    eng = Engine(prob, B, 0)
    eng.set_plant_inertial(PG['pin'])
    xn, a = eng.plant_step(PG['x'], PG['u'])
    np.testing.assert_allclose(a, PG['acc'], rtol=1e-8, atol=1e-8)
    np.testing.assert_allclose(xn, PG['xn'], rtol=1e-10, atol=1e-10)
