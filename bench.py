#!/usr/bin/env python
"""Headline benchmark: RTI iterations/s of the batched closed-loop MPC (BASELINE.json metric).

A step = one closed-loop control step of every problem of the batch (controller.step = RTI solve, backup solve
on abort, plant step; scripts/mpc.py:125-264).  Workload at 1 GPU = BASELINE.json configs[1]: Z1(-like) ST
controller with the viability-network terminal constraint, N=45, dt=5 ms, batch 10 000 per GPU (weak scaling).

  python bench.py [--gpus N --steps K --warmup W]          this engine (one process per GPU under torchrun)
  python bench.py --impl reference ...                      the CPU path (oracle port of the acados RTI path,
                                                            all host threads, bounded sample of the same workload)
  python bench.py --config cfg0|cfg1|cfg2|cfg3|cfg4 ...     the other BASELINE.json configurations (see PRESETS); the default and
                                                            the N = 1 headline stay cfg1
  python bench.py ... --dump-outputs DIR                    also write what the last timed step computed as DIR/<name>.npy (see
                                                            dump_outputs), so that two builds can be compared output for output
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

from safe_mpc_b200 import abi, distributed as D  # noqa: E402
from safe_mpc_b200.parser import Parameters, default_args  # noqa: E402
from safe_mpc_b200.problem import ModelData, build_problem  # noqa: E402

METRIC = 'rti_iterations_per_sec'
UNIT = 'RTI iterations/s'
Q0 = np.array([-0.3, 0.8, -1.65, 0.658, 0.0])


NN_PRECISION = 'strict'      # set from --nn-precision

# BASELINE.json configs -> bench arguments (explicit flags win).  cfg2 names three controllers: pick with --controller.
PRESETS = {
    'cfg0': dict(controller='naive', horizon=45, batch=100, noise=0.0,
                 what="configs[0]: naive RTI MPC, N=45, dt=5 ms, 100 initial states (the reference's own test_num)"),
    'cfg1': dict(controller='st', horizon=45, batch=10000, noise=0.0,
                 what='configs[1]: ST controller with the viability-network terminal constraint, batch 10k on 1 GPU'),
    'cfg2': dict(controller='receding', horizon=45, batch=12500, noise=0.0, nn_precision='tf32x3',
                 what='configs[2]: HTWA / receding / constraint_everywhere (--controller), 12.5k problems per GPU = 100k on 8 GPUs; '
                      'viability network on the tensor cores (fp32 class, the precision of the reference libtorch call)'),
    'cfg3': dict(controller='st', horizon=45, batch=50000, noise=5.0,
                 what='configs[3]: model-noise ensemble, per-problem perturbed inertial parameters (5 %), batch 50k'),
    'cfg4': dict(controller='st', horizon=45, batch=10000, noise=0.0,
                 what='configs[4]: horizon / alpha sweep point (--horizon in {20,35,45,60,80}, --alpha in {10,..,50})'),
}


ALPHA = None                 # set from --alpha (default: config.yaml)
PRECISION = 'f64'            # set from --precision


def workload(controller, N, noise, seed, lo, hi):
    """Synthetic inputs of problems [lo, hi): initial states around the shipped IC, perturbed plants, torque noise."""
    args = default_args(controller=controller, horizon=N, noise=noise, nn_precision=NN_PRECISION, precision=PRECISION)
    params = Parameters(args, 'z1', rti=True)
    params.N = N
    if ALPHA is not None:
        params.alpha = float(ALPHA)
    md = ModelData(params)
    B = hi - lo
    x0 = np.zeros((B, abi.NX)); pin = np.zeros((B, abi.NQ, 10))
    for i, gi in enumerate(range(lo, hi)):          # per-problem streams -> independent of the sharding
        rng = np.random.default_rng([seed, gi])
        x0[i, :abi.NQ] = Q0 + 0.15 * rng.uniform(-1, 1, abi.NQ)
        x0[i, abi.NQ:] = 0.2 * rng.uniform(-1, 1, abi.NQ)
        pin[i] = md.inertial * (1 + noise / 100 * rng.uniform(-1, 1, (abi.NQ, 10)))
    return params, md, x0, pin


def make_handles(E, params, md, controller, B, arg):
    prob, keep = build_problem(params, controller, cost='ext', model=md)
    bprob, bkeep = build_problem(params, 'backup', cost='zero', N=params.back_hor, model=md)
    main, bk = E(prob, B, arg), E(bprob, B, arg)
    main._keepalive = (prob, keep); bk._keepalive = (bprob, bkeep)
    return main, bk, prob


def warm_guess(main, x0, N, iters):
    """Warm start: a few full-step SQP iterations from the constant guess (x0 repeated, u = 0), untimed."""
    xg = np.repeat(x0[:, None, :], N + 1, axis=1).copy()
    ug = np.zeros((x0.shape[0], N, abi.NU))
    main.set_guess(xg, ug)
    for _ in range(iters):
        main.rti_solve(x0)
        xt, ut = main.get_temp()
        main.set_guess(xt, ut)
    main.reset_controller()


DUMP_LIMIT = 64_000_000     # bytes --dump-outputs may write


def dump_outputs(path, sim, main, step):
    """What the closed loop hands its caller after `step` steps, as float64 .npy files under `path`: the plant state x [B, NX] after the
    step and the control u [B, NU] applied in it, terminated [B] (1 for a problem whose simulation has ended, mpc.py's break: its log
    rows are NaN, written here as zeros so that every output is finite), the main controller's warm start x_guess [B, N+1, NX] /
    u_guess [B, N, NU] and its solve status [B].
    When the batch would exceed DUMP_LIMIT, the same arrays for a fixed seeded sample of the problems; problem_index says which."""
    x, u = sim.log()
    x, u = x[:, step], u[:, step - 1]
    terminated = np.isnan(x).any(axis=1) | np.isnan(u).any(axis=1)
    xg, ug = main.get_guess()
    out = {'x': np.where(terminated[:, None], 0.0, x), 'u': np.where(terminated[:, None], 0.0, u), 'terminated': terminated.astype(np.float64),
           'x_guess': xg, 'u_guess': ug, 'status': main.get_state(abi.STATE_STATUS).astype(np.float64)}
    B = main.B
    per_problem = 8 * (1 + sum(v[0].size for v in out.values()))
    idx = np.arange(B)
    if B * per_problem > DUMP_LIMIT:
        idx = np.sort(np.random.default_rng(0).choice(B, DUMP_LIMIT // per_problem, replace=False))
    out = {k: np.ascontiguousarray(v[idx], dtype=np.float64) for k, v in out.items()}
    out['problem_index'] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + '.npy'), v)


class ClockSampler:
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={gpu_index}', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill(); out, _ = self.proc.communicate()
        sm, smax, reasons = [], [], set()
        for line in out.splitlines():
            f = [s.strip() for s in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def time_oracle(controller, N, noise, seed, n_problems, steps, warmup, sqp_iters, dump=None):
    """The CPU path (oracle port of the reference's acados RTI path) on a bounded sample of the workload; `dump`: dump_outputs directory."""
    from oracle.oracle import Oracle, OracleSim
    params, md, x0, pin = workload(controller, N, noise, seed, 0, n_problems)
    main, bk, prob = make_handles(Oracle, params, md, controller, n_problems, 0)
    main.set_plant_inertial(pin)
    warm_guess(main, x0, N, sqp_iters)
    sim = OracleSim(main, bk, warmup + steps)
    sim.reset(x0)
    sim.run(warmup)
    c0 = sim.counters()
    t0 = time.perf_counter()
    sim.run(steps)
    dt = time.perf_counter() - t0
    c1 = sim.counters()
    if dump:
        dump_outputs(dump, sim, main, warmup + steps)
    solves = (c1['rti_solves'] - c0['rti_solves']) + (c1['backup_solves'] - c0['backup_solves'])
    return {'value': solves / dt, 'seconds': dt, 'solves': solves, 'cores': main.num_threads(),
            'ipm_per_solve': (c1['ipm_iterations'] - c0['ipm_iterations']) / max(1, solves),
            'sample': f'{n_problems} problems x {steps} closed-loop steps of the same workload ({controller}, N={N})',
            'outcome': D.outcome_counts(sim.outcome())}


def run_reference(a):
    rank, _, world = D.env_world()
    if rank != 0:
        return
    n = a.ref_problems
    r = time_oracle(a.controller, a.horizon, a.noise, a.seed, n, a.steps, a.warmup, a.sqp_iters, dump=a.dump_outputs)
    line = {'metric': METRIC, 'value': r['value'], 'unit': UNIT, 'impl': 'reference', 'n_gpus': a.gpus, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': 1e3 * r['seconds'] / a.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
            'data': 'synthetic',
            'config': {'workload': f'{a.config}: closed-loop RTI MPC, controller={a.controller}, N={a.horizon}, dt=5ms, '
                                   f'synthetic Z1-like 5-DOF chain + random-init viability MLP 10-256-256-256-1',
                       'preset': PRESETS[a.config]['what'], 'batch': n, 'noise_percent': a.noise, 'note': 'CPU path: oracle port of the acados SQP_RTI/HPIPM path (acados, CasADi, adam, l4casadi are not installable offline)'},
            'cpu_baseline': {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port', 'sample': r['sample']},
            'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'ipm_iterations_per_solve': r['ipm_per_solve'], 'outcome': r['outcome']}
    print(json.dumps(line), flush=True)


def run_engine(a):
    import torch
    from safe_mpc_b200.engine import Engine, Sim
    rank, local_rank, world = D.init('nccl')
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; this engine has no CPU fallback (use --impl reference for the CPU path)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    B = a.batch                                   # per GPU (weak scaling)
    lo, hi = rank * B, (rank + 1) * B
    params, md, x0, pin = workload(a.controller, a.horizon, a.noise, a.seed, lo, hi)
    N = a.horizon
    main, bk, prob = make_handles(Engine, params, md, a.controller, B, local_rank)
    main.set_plant_inertial(pin)
    warm_guess(main, x0, N, a.sqp_iters)
    guess0 = [np.array(v, copy=True) for v in main.get_guess()]     # the e2e arm replays the same closed loop from the same warm start
    total_steps = a.warmup + a.steps + 2 * a.probe_steps        # (the roofline probe continues the same closed loop)
    sim = Sim(main, bk, total_steps)
    sim.reset(x0)
    stream = torch.cuda.ExternalStream(main.stream(), device=dev)
    sim.run(a.warmup)
    main.sync()
    c0 = sim.counters(); l0 = main.launch_count() + bk.launch_count()
    D.barrier(); torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    try:                                          # the sampler's nvidia-smi must not outlive a failed run
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
        evs[0].record(stream)
        for i in range(a.steps):
            sim.step()
            evs[i + 1].record(stream)
        main.sync(); torch.cuda.synchronize()
        D.barrier()
    finally:
        clocks = sampler.stop() if sampler else None
    if a.dump_outputs:
        dump_outputs(a.dump_outputs if world == 1 else os.path.join(a.dump_outputs, f'rank{rank}'), sim, main, a.warmup + a.steps)
    ms = evs[0].elapsed_time(evs[-1])
    lat = np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(a.steps)])
    c1 = sim.counters(); l1 = main.launch_count() + bk.launch_count()
    solves = (c1['rti_solves'] - c0['rti_solves']) + (c1['backup_solves'] - c0['backup_solves'])
    ipm = c1['ipm_iterations'] - c0['ipm_iterations']

    # ---- per-kernel times of the QP solves of further closed-loop steps (roofline) ----
    # The same closed loop simply continues after the timed region: first a few steps that only read the acados-style time fields of
    # the step (time_qp, time_lin), then a few steps with one CUDA-event pair around every kernel on the stream it is launched on
    # (smpc_set_profiling; the solver runs a single tile group, so no two kernels of a solve overlap while they are timed).  The
    # event pairs cost launch gaps, so these steps are outside the timed region; what is summed is kernel durations only.
    xs = torch.tensor(x0, device=dev)
    tq = []
    for _ in range(a.probe_steps):
        sim.step(); main.sync()
        tq.append(main.times())
    kern = {}
    span_ms, it_max = 0.0, 0
    cp0 = sim.counters()
    main.set_profiling(True)
    tq_prof = []
    for _ in range(a.probe_steps):
        sim.step(); main.sync()
        k1, sp1, itm1 = main.profile()
        for k, (ms_k, n_k) in k1.items():
            o = kern.get(k, (0.0, 0))
            kern[k] = (o[0] + ms_k, o[1] + n_k)
        span_ms += sp1; it_max = max(it_max, itm1)
        tq_prof.append(main.times())
    main.set_profiling(False)
    cp1 = sim.counters()
    probe_solves = cp1['rti_solves'] - cp0['rti_solves']
    probe_ipm = cp1['ipm_iterations'] - cp0['ipm_iterations']
    # a problem takes part in the launches kk = 0 .. iter of its solve
    probe_visits = float(probe_ipm + probe_solves) * (N + 1)
    qp_ms = float(np.median([t['time_qp'] for t in tq]) * 1e3)
    qp_ms_1group = float(np.median([t['time_qp'] for t in tq_prof]) * 1e3)
    lin_ms = float(np.median([t['time_lin'] for t in tq]) * 1e3)
    it_qp = probe_ipm / max(1, probe_solves)
    it_sum = float(probe_ipm) / a.probe_steps                                     # IPM iterations of one batched solve
    kern = {k: (v[0] / a.probe_steps, v[1] / a.probe_steps) for k, v in kern.items()}   # -> per solve
    kern_total = sum(v[0] for v in kern.values())

    # ---- the linearisation kernel alone: a handle without viability rows (time_lin = linearize_kernel only), same B and N ----
    lin_probe = None
    if rank == 0:
        nprob, nkeep = build_problem(params, 'naive', cost='ext', model=md)
        neng = Engine(nprob, B, local_rank); neng._keepalive = (nprob, nkeep)
        neng.set_guess(*main.get_guess())
        neng.rti_solve(xs); neng.sync()
        tl = []
        for _ in range(3):
            neng.rti_solve(xs); neng.sync()
            tl.append(neng.times()['time_lin'] * 1e3)
        lin_probe = float(np.median(tl))
        neng.close()

    # ---- measured FP64 / FP32 FMA peaks (MEASURED_PEAKS.json has none) ----
    fp64_peak = fp32_peak = None
    if rank == 0:
        fp64_peak, fp32_peak = Engine.measure_peaks(local_rank)

    # ---- end to end through the C ABI with host buffers (H2D / D2H inside the timed region) ----
    e2e = None
    if not a.no_e2e:
        # the same W + K closed-loop steps from the same warm start, every step through the C ABI with HOST buffers:
        # x (H2D) -> smpc_controller_step -> u, abort (D2H);  x, u (H2D) -> smpc_plant_step -> x_next, a (D2H)
        main.set_guess(*guess0)
        main.reset_controller()
        xh = torch.tensor(x0).pin_memory().numpy()
        x_cur = xh.copy()
        for _ in range(a.warmup):
            u, ab = main.controller_step(x_cur); x_cur, _ = main.plant_step(x_cur, u)
        main.sync()
        D.barrier()
        t0 = time.perf_counter()
        n_e2e = a.steps
        for _ in range(n_e2e):
            u, ab = main.controller_step(x_cur)
            x_cur, _ = main.plant_step(x_cur, u)
        main.sync()
        e2e_s = time.perf_counter() - t0
        e2e = {'steps': n_e2e, 'seconds': e2e_s, 'solves': n_e2e * B,
               'h2d': B * (abi.NX * 8) + B * (abi.NX + abi.NU) * 8, 'd2h': B * (abi.NU * 8 + 1) + B * (abi.NX + abi.NU) * 8}

    # ---- the viability network kernels timed alone on the row count of configs[2] (a row per problem and stage) ----
    mlp = None
    rk4 = None
    if rank == 0 and not a.no_mlp:
        mlp = time_mlp(params, md, B * N, local_rank, dev)
        rk4 = time_rk4(params, md, B * (N + 1), local_rank, dev)

    # ---- aggregate over ranks ----
    vec = [ms, solves, ipm, l1 - l0, (e2e['seconds'] if e2e else 0.0), (e2e['solves'] if e2e else 0.0)]
    allv = D.all_gather_vector(vec, device=dev)
    ms_max = max(v[0] for v in allv)
    solves_all = sum(v[1] for v in allv)
    outcome = D.gather_outcomes(sim.outcome(), device=dev)
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s (B200_PROFILING.md)'
    fp64_src = 'measured in this run (smpc_measure_peaks: 16 independent DFMA chains per thread, CUDA events)'
    if not fp64_peak:
        fp64_peak, fp64_src = 37.0, 'nominal 37 TFLOP/s (SURVEY.md section 8d placeholder; smpc_measure_peaks failed)'
    # Per-kernel roofline of one QP solve.  A "visit" = one (problem, stage) handled by one launch; a problem takes part in the launches
    # kk = 0 .. iter_b of a solve.  Two bases per kernel (DESIGN.md section 3.2):
    #   bytes  what the kernel has to stream per visit in THIS design (solver state resident in HBM), doubles read + written
    #   flop   SURVEY.md section 8(d) / BASELINE.md section 4 dense counts per stage and IPM iteration: factorisation 4 875, one
    #          solve 1 250, inequality condensation 2 475
    sb = 8 if a.precision == 'f64' else 4             # bytes of a value of the storage type (records, directions, factors); the iterate is fp64
    UNITS = {                       # kernel family -> (fp64 values, storage-type values, flop) per visit
        'qs_prep': (250, 451, 2475.0),                # update + residuals + condensation: 436 read + 265 written
        'qs_ric1': (0, 145 + 155 + 100 + 15, 4875.0 + 1250.0),   # factorisation + affine solve (backward + forward)
        'qs_step0': (122, 228, 0.0),                  # affine (dlam, dt), products, corrector terms (row products: not in the 8(d) count)
        'qs_ric2': (0, 155 + 30 + 180 + 50, 2 * 1250.0), # corrector and centering solves in one pass
        'qs_step1': (122, 292, 0.0),
        'qs_step2_centering': (122, 301, 0.0),
    }
    # the solo kernel (one CTA per problem, whole IPM iterations in one launch: small batches) runs every phase above on the same arrays
    UNITS['qs_solo'] = tuple(sum(u[i] for k, u in UNITS.items() if k != 'qs_step2_centering') for i in range(3))
    UNITS = {k: ((d * 8 + v * sb) / 8.0, fl) for k, (d, v, fl) in UNITS.items()}    # -> (fp64-equivalents per visit, flop)
    visits = probe_visits / a.probe_steps                                       # (problem, stage) visits of one batched solve
    table = {}
    for k, (dbl, flop) in UNITS.items():
        ms_k, n_k = kern[k]
        if n_k == 0 or ms_k <= 0:
            continue
        v = visits if k != 'qs_step2_centering' else None     # (only the problems that switch direction: not tracked per launch)
        if k == 'qs_prep' and kern.get('qs_solo', (0, 0))[1] > 0 and kern.get('qs_ric1', (0, 0))[1] == 0:
            v = float(probe_solves) / a.probe_steps * (N + 1)   # solo path: only the cold-start prep is a launch of its own
        row = {'ms_per_solve': round(ms_k, 3), 'launches': n_k, 'share_of_qp_solve': ms_k / max(kern_total, 1e-9)}
        if v is not None:
            row.update({'hbm_gbs': v * dbl * 8 / (ms_k * 1e-3) / 1e9, 'hbm_frac': v * dbl * 8 / (ms_k * 1e-3) / 1e9 / hbm_peak,
                        'fp64_tflops': v * flop / (ms_k * 1e-3) / 1e12, 'fp64_frac': v * flop / (ms_k * 1e-3) / 1e12 / fp64_peak,
                        'bytes_per_visit': int(dbl * 8), 'flop_per_visit': flop})
        table[k] = row
    dom = max((k for k in table if 'hbm_gbs' in table[k]), key=lambda k: table[k]['ms_per_solve'])
    dname = {'qs_prep': 'qs_prep_coop_kernel / qs_prep_kernel', 'qs_ric1': 'qs_ric1x_kernel / qs_ric1t_kernel', 'qs_ric2': 'qs_ric2_kernel / qs_ric2t_kernel',
             'qs_step0': 'qs_step_kernel<0>', 'qs_step1': 'qs_step_kernel<1>', 'qs_solo': 'qs_solo_kernel'}[dom]
    d = table[dom]
    # ncu --set full captures of the round-2 kernels, one all-active launch each (dram__bytes_read.sum + dram__bytes_write.sum)
    ncu_traffic = {'qs_prep': (1.549120e9 + 0.930624e9, 'profiles/r02_prep_coop_rolled_raw.csv'),
                   'qs_ric1': (0.876355e9 + 0.582946e9, 'profiles/r02_ric1x_raw.csv'),
                   'qs_ric2': (1.219103e9 + 0.277923e9, 'profiles/r02_ric2_raw.csv')}
    traffic, traffic_file = ncu_traffic.get(dom, (None, None)) if (B, N) == (10000, 45) else (None, None)
    # bytes the whole solve moves per problem against what is algorithmically necessary (SURVEY 8d: ~11 KB per problem and RTI iteration)
    moved = sum(table[k]['bytes_per_visit'] for k in table if 'bytes_per_visit' in table[k] and not (k == 'qs_prep' and 'qs_solo' in table)) * visits / B
    necessary = ((N + 1) * abi.NX + N * abi.NU) * 8 * 2 + 200
    flops_solve = 0.48e6 * (N + 1) / 46.0 * it_sum                              # SURVEY section 8(d): 0.48 MFLOP per IPM iteration at N = 45
    value = solves_all / (ms_max * 1e-3)
    roofline = {'kernel': dname, 'bound': 'hbm', 'achieved': d['hbm_gbs'], 'peak': hbm_peak, 'unit': 'GB/s', 'frac': d['hbm_frac'],
                'traffic': traffic, 'traffic_source': 'ncu dram__bytes_read+write of one all-active launch (313 tiles x %d stages), %s (B=10000, N=45 only)' % (N + 1, traffic_file),
                'traffic_algorithmic_all_active': d['bytes_per_visit'] * 313 * 32 * (N + 1) if traffic else None,
                'peak_source': peak_src, 'selection': 'the QP kernel family with the largest summed duration in one solve (kernel_ms below)',
                'algorithmic_bytes_per_launch': d['bytes_per_visit'] * visits / max(1, d['launches']), 'launch_ms': d['ms_per_solve'] / max(1, d['launches']),
                'launches_per_solve': d['launches'], 'share_of_qp_solve': d['share_of_qp_solve'],
                'bytes_basis': 'design traffic: solver state resident in HBM, %d doubles per (problem, stage) visit' % (d['bytes_per_visit'] // 8),
                'fp64': {'achieved': d['fp64_tflops'], 'peak': fp64_peak, 'unit': 'TFLOP/s', 'frac': d['fp64_frac'], 'flop_per_visit': d['flop_per_visit'],
                         'peak_source': fp64_src, 'basis': 'SURVEY.md section 8(d) dense flop count of this phase'},
                'solve_traffic': {'bytes_moved_per_problem': moved, 'necessary_bytes_per_problem': necessary, 'ratio': moved / necessary,
                                  'note': 'HBM bytes one RTI solve streams per problem (sum over the kernels of bytes_per_visit x visits) against the '
                                          'warm start in / out + x0 + status that SURVEY 8(d) calls algorithmically necessary: the solver state '
                                          '(~340 KB per problem) does not fit on chip for the ~1 500 problems the sequential Riccati recursion needs in flight, '
                                          'so every IPM iteration re-streams it (DESIGN.md section 3.2)'},
                'note': 'bytes and time are summed over every launch of the family in the solves of the probe steps; a launch only touches the problems still iterating'
                        + ('; the solo kernel serves a batch smaller than the machine out of L2 (working set below the L2 size): it is bound by the latency of one '
                           'problem\'s dependent chain, the HBM basis is reported for completeness only' if dom == 'qs_solo' else '')}
    # linearisation kernel against the FP64 pipe (BASELINE.md section 4: flop per stage from the executed-instruction tally)
    roof_dyn = None
    if lin_probe:
        fl = LINEARIZE_FLOP_PER_STAGE * B * (N + 1)
        roof_dyn = {'kernel': 'linearize_kernel', 'bound': 'fp64', 'achieved': fl / (lin_probe * 1e-3) / 1e12, 'peak': fp64_peak, 'unit': 'TFLOP/s',
                    'frac': fl / (lin_probe * 1e-3) / 1e12 / fp64_peak, 'launch_ms': lin_probe, 'flop_per_stage': LINEARIZE_FLOP_PER_STAGE,
                    'flop_source': LINEARIZE_FLOP_SOURCE, 'peak_source': fp64_src,
                    'hbm_gbs_written': B * (N + 1) * abi.REC * 8 / (lin_probe * 1e-3) / 1e9}
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
        'ms_per_step': ms_max / a.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64' if a.precision == 'f64' else 'f32-storage/f64-accumulate',
        'data': 'synthetic',
        'config': {'workload': f'{a.config}: closed-loop RTI MPC, controller={a.controller}, N={N}, dt=5ms, '
                               f'synthetic Z1-like 5-DOF chain + random-init viability MLP 10-256-256-256-1',
                   'preset': PRESETS[a.config]['what'],
                   'batch_per_gpu': B, 'global_batch': B * world, 'parallelism': f'dp{world} (problem sharding, no hot-path collective)',
                   'l2': f'working set {B * (main_qp_bytes(N)) / 1e9:.2f} GB per GPU > 126 MB L2 (no flush needed)' if B * main_qp_bytes(N) > 2.5e8
                         else f'working set {B * (main_qp_bytes(N)) / 1e6:.0f} MB per GPU: L2-resident (small-batch latency case, not a bandwidth measurement)',
                   'noise_percent': a.noise, 'alpha': float(params.alpha), 'sqp_warm_start_iters': a.sqp_iters, 'nn_precision': a.nn_precision,
                   'precision': a.precision},
        'p50_step_ms': float(np.percentile(lat, 50)), 'p99_step_ms': float(np.percentile(lat, 99)),
        'ipm_iterations_per_solve': ipm / max(1, solves),
        'gpu_launches': int(sum(v[3] for v in allv)),
        'clocks': clocks,
        'roofline': roofline,
        'roofline_kernels': table,
        'roofline_dynamics': roof_dyn,
        'peaks': {'hbm_gbs': hbm_peak, 'fp64_tflops': fp64_peak, 'fp32_tflops': fp32_peak, 'fp64_source': fp64_src},
        'qp_solve': {'ms': qp_ms, 'ms_single_tile_group': qp_ms_1group, 'linearize_ms': lin_ms, 'ipm_iterations_mean': it_qp, 'ipm_iterations_max': it_max,
                     'algorithmic_fp64_tflops': flops_solve / (qp_ms * 1e-3) / 1e12, 'algorithmic_fp64_frac': flops_solve / (qp_ms * 1e-3) / 1e12 / fp64_peak,
                     'kernel_ms': {k: round(v[0], 3) for k, v in kern.items()}, 'kernel_launches': {k: round(v[1], 1) for k, v in kern.items()},
                     'kernel_ms_note': f'per-kernel sums per solve, averaged over the solves of {a.probe_steps} further closed-loop steps timed with one '
                                       'CUDA-event pair per kernel (single tile group: no overlap between kernels)'},
        'outcome': D.outcome_counts(outcome),
    }
    if mlp:
        tpeak = mlp.pop('tf32_peak_measured', None)
        if tpeak:
            mlp['tensor_peak_source'] = 'measured in this run: torch.matmul fp32 8192^3 with allow_tf32 (cuBLAS TF32 tensor-core GEMM), best of 5, CUDA events'
        else:
            tpeak = float(peaks.get('bf16_tflops', peaks.get('bf16_dense_tflops', 1590.0))) / 2
            mlp['tensor_peak_source'] = 'half of the dense bf16 peak of MEASURED_PEAKS.json (the TF32 GEMM measurement failed)'
        mlp['tensor_peak_tf32_tflops'] = tpeak
        mlp['tf32x3']['frac_of_tensor_peak'] = mlp['tf32x3']['executed_tf32_tflops'] / tpeak
        line['viability_network'] = mlp
    if rk4:
        rk4['fp64_frac'] = rk4['fp64_tflops'] / fp64_peak
        line['torque_input_rk4'] = rk4
    if e2e:
        e2e_s = max(v[4] for v in allv)
        line['e2e'] = {'value': sum(v[5] for v in allv) / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': e2e['h2d'], 'd2h_bytes_per_step': e2e['d2h'],
                       'api': 'smpc_controller_step + smpc_plant_step with host buffers', 'steps': e2e['steps'],
                       'note': 'same warm start and the same W + K closed-loop steps as the device-resident arm (no abort occurs in this workload)'}
    if world == 1 and not a.no_cpu:
        r = time_oracle(a.controller, N, a.noise, a.seed, a.cpu_problems, a.cpu_steps, 1, a.sqp_iters)
        line['cpu_baseline'] = {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port', 'sample': r['sample'],
                                'ipm_iterations_per_solve': r['ipm_per_solve']}
    print(json.dumps(line), flush=True)


def time_rk4(params, md, n_rows, device_index, dev):
    """Extension kernel of SURVEY 8(f)4, not on the closed-loop path: one torque-input RK4 step with sensitivities (smpc_rk4_sens) for a
    row per (problem, stage), buffers resident in HBM."""
    import torch
    from safe_mpc_b200.engine import Engine
    rng = np.random.default_rng(9)
    mid, half = 0.5 * (md.x_min + md.x_max), 0.5 * (md.x_max - md.x_min)
    x = mid + 0.8 * half * rng.uniform(-1, 1, (n_rows, abi.NX))
    x[:, abi.NQ:] *= 0.6
    xd = torch.tensor(x, device=dev); td = torch.tensor(rng.uniform(-8, 8, (n_rows, abi.NU)), device=dev)
    prob, keep = build_problem(params, 'naive', cost='ext', model=md)
    eng = Engine(prob, 64, device_index)
    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    out = {'kernel': 'rk4_sens_kernel', 'rows': n_rows, 'flop_per_row': 81657,
           'flop_source': 'executed FP64 instructions under ncu (2 DFMA + DADD + DMUL per row): profiles/r02_rk4_sens.md',
           'note': 'extension beyond the reference formulation (SURVEY 8(f)4), not part of the timed closed loop'}
    for sens in (True, False):
        eng.rk4_sens(xd, td, params.dt, sens=sens); eng.sync()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        ev[0].record(stream)
        for i in range(5):
            eng.rk4_sens(xd, td, params.dt, sens=sens)
            ev[i + 1].record(stream)
        eng.sync(); torch.cuda.synchronize()
        ms = float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(5)]))
        if sens:
            out.update({'ms': ms, 'rows_per_s': n_rows / (ms * 1e-3), 'fp64_tflops': n_rows * 81657 / (ms * 1e-3) / 1e12})
        else:
            out['ms_value_only'] = ms
    eng.close()
    return out


def time_mlp(params, md, n_rows, device_index, dev):
    """c(x) and dc/dx of n_rows states resident in HBM through smpc_nn_constraint: strict kernel vs tensor-core kernel."""
    import torch
    from safe_mpc_b200.engine import Engine
    rng = np.random.default_rng(7)
    mid, half = 0.5 * (md.x_min + md.x_max), 0.5 * (md.x_max - md.x_min)
    x = mid + 0.8 * half * rng.uniform(-1, 1, (n_rows, abi.NX))
    xd = torch.tensor(x, device=dev)
    out = {'rows': n_rows, 'algorithmic_flop_per_row': 535040}
    try:                                           # TF32 tensor-core peak of this GPU (library GEMM, measurement only)
        torch.backends.cuda.matmul.allow_tf32 = True
        a_ = torch.randn(8192, 8192, device=dev); b_ = torch.randn(8192, 8192, device=dev)
        torch.matmul(a_, b_); torch.cuda.synchronize()
        best = 0.0
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a_, b_); e1.record(); torch.cuda.synchronize()
            best = max(best, 2 * 8192 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        out['tf32_peak_measured'] = best
        del a_, b_
        torch.backends.cuda.matmul.allow_tf32 = False
    except Exception:
        pass
    for name in ('strict', 'tf32x3'):
        prob, keep = build_problem(params, 'st', cost='ext', model=md, nn_precision=name)
        eng = Engine(prob, 64, device_index)
        stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
        eng.nn_constraint(xd); eng.sync()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        ev[0].record(stream)
        for i in range(5):
            eng.nn_constraint(xd)
            ev[i + 1].record(stream)
        eng.sync(); torch.cuda.synchronize()
        ms = float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(5)]))
        out[name] = {'ms': ms, 'algorithmic_tflops': n_rows * 535040 / (ms * 1e-3) / 1e12}
        if name == 'tf32x3':
            # the four 256 x 256 contractions (491 520 of the 535 040 flop) run as three tf32 products each
            out[name]['executed_tf32_tflops'] = n_rows * 3 * 4 * 2 * 256 * 256 / (ms * 1e-3) / 1e12
        eng.close()
    return out


# linearize_kernel: FP64 flop per (problem, stage) = 2 x DFMA + DADD + DMUL thread instructions executed / (B (N+1)), from ncu
# (smsp__sass_thread_inst_executed_op_d{fma,add,mul}_pred_on.sum; profiles/r02_linearize_flops.md).  Frozen in BASELINE.md section 4.
LINEARIZE_FLOP_PER_STAGE = 16274.0
LINEARIZE_FLOP_SOURCE = 'executed FP64 instructions of linearize_kernel under ncu, 2 DFMA + DADD + DMUL per (problem, stage): profiles/r02_linearize_flops.md'


def main_qp_bytes(N):
    sb = 8 if PRECISION == 'f64' else 4
    return (N + 1) * ((2 * 120 + 8 + 4) * 8 + (abi.REC + 120 + 25 + 345 + 46) * sb)     # per problem: iterate x2, partials (fp64); records, step, solver block, products (storage type)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='engine', choices=['engine', 'reference'])
    ap.add_argument('--config', default='cfg1', choices=sorted(PRESETS), help='BASELINE.json configuration (default cfg1 = the headline)')
    ap.add_argument('--controller', default=None)
    ap.add_argument('--horizon', type=int, default=None)
    ap.add_argument('--batch', type=int, default=None, help='problems per GPU')
    ap.add_argument('--noise', type=float, default=None)
    ap.add_argument('--alpha', type=float, default=None, help='safety margin in percent (config.yaml alpha)')
    ap.add_argument('--precision', default='f64', choices=['f64', 'f32'], help='storage precision of the QP solver state')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--sqp-iters', type=int, default=5, dest='sqp_iters')
    ap.add_argument('--ref-problems', type=int, default=256, dest='ref_problems')
    ap.add_argument('--cpu-problems', type=int, default=256, dest='cpu_problems')
    ap.add_argument('--cpu-steps', type=int, default=8, dest='cpu_steps')
    ap.add_argument('--probe-steps', type=int, default=5, dest='probe_steps', help='closed-loop steps after the timed region that are timed kernel by kernel')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-mlp', action='store_true', dest='no_mlp')
    ap.add_argument('--nn-precision', default=None, choices=['strict', 'tf32x3'], dest='nn_precision',
                    help='viability network arithmetic of the timed closed loop (the tensor-core kernel is always timed alone as well)')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR', dest='dump_outputs',
                    help='after the timed steps, write what the last of them computed as DIR/<name>.npy (float64, at most 64 MB; '
                         'with several GPUs DIR/rank<r>/)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    pre = PRESETS[a.config]
    for key in ('controller', 'horizon', 'batch', 'noise'):
        if getattr(a, key) is None:
            setattr(a, key, pre[key])
    if a.nn_precision is None:
        a.nn_precision = pre.get('nn_precision', 'strict')
    global NN_PRECISION, ALPHA, PRECISION
    NN_PRECISION = a.nn_precision
    ALPHA = a.alpha
    PRECISION = a.precision
    if a.warmup < 3 and a.impl == 'engine':
        a.warmup = 3
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_engine(a)
        D.finalize()


if __name__ == '__main__':
    main()
