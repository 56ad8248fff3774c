"""dev: the two forms of the QP step kernels on the cfg[1] closed loop, alternated in one process.

    python tools/step_forms_ab.py [--rounds 3] [--steps 20] [--warmup 3] [--batch 10000] [--precision f64]

Each run builds fresh handles (the form is read when a handle is created: SMPC_QP_STEP=thread -> thread form, unset -> staged form),
replays the same seeded warm start and closed loop as bench.py, times `--steps` steps with CUDA events after `--warmup` untimed ones,
then profiles two more steps kernel by kernel (smpc_set_profiling; CUDA events around every launch).  Prints one line per run and the
mean / spread per form, with the card's name and power limit."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

import numpy as np
import torch

import bench

FAMILIES = ('qs_prep_kernel', 'qs_ric1_kernel', 'qs_step_kernel<0>', 'qs_ric2_kernel', 'qs_step_kernel<1>', 'qs_step_kernel<2>', 'qs_compact')


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = 'unknown'
    return out or torch.cuda.get_device_name(0)


def run(form, a):
    from safe_mpc_b200.engine import Engine, Sim
    if form == 'thread':
        os.environ['SMPC_QP_STEP'] = 'thread'
    else:
        os.environ.pop('SMPC_QP_STEP', None)
    params, md, x0, pin = bench.workload('st', 45, 0.0, 0, 0, a.batch)
    main, bk, prob = bench.make_handles(Engine, params, md, 'st', a.batch, 0)
    main.set_plant_inertial(pin)
    bench.warm_guess(main, x0, 45, 5)
    sim = Sim(main, bk, a.warmup + a.steps + 2)
    sim.reset(x0)
    stream = torch.cuda.ExternalStream(main.stream(), device=torch.device('cuda', 0))
    sim.run(a.warmup)
    main.sync(); torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
    evs[0].record(stream)
    for i in range(a.steps):
        sim.step()
        evs[i + 1].record(stream)
    main.sync(); torch.cuda.synchronize()
    lat = np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(a.steps)])
    kern = {}
    main.set_profiling(True)
    for _ in range(2):
        sim.step(); main.sync()
        for k, (ms, n) in main.profile()[0].items():
            o = kern.get(k, (0.0, 0))
            kern[k] = (o[0] + ms, o[1] + n)
    main.set_profiling(False)
    x, u = sim.log()
    sim.close() if hasattr(sim, 'close') else None
    main.close(); bk.close()
    return lat, {k: kern.get(k, (0.0, 0))[0] / 2 for k in FAMILIES}, np.nan_to_num(x[:, a.warmup + a.steps])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=10000)
    ap.add_argument('--precision', default='f64', choices=['f64', 'f32'])
    a = ap.parse_args()
    bench.PRECISION = a.precision
    print(f'card: {card()}   cfg[1] ST N=45 B={a.batch} {a.precision}, {a.steps} timed steps per run')
    res = {'thread': [], 'staged': []}
    xs = {}
    for r in range(a.rounds):
        for form in ('thread', 'staged') if r % 2 == 0 else ('staged', 'thread'):
            lat, kern, x = run(form, a)
            res[form].append(lat.mean())
            if form in xs and not np.array_equal(xs[form], x):
                print(f'  {form}: the closed loop is not reproducible from run to run')
            xs[form] = x
            fam = '  '.join(f'{k.replace("qs_", "").replace("_kernel", "")}={v:.2f}' for k, v in kern.items())
            print(f'round {r} {form:6s}  ms/step p50 {np.median(lat):6.2f} mean {lat.mean():6.2f}   per step (ms): {fam}')
    print('same final states in both forms:', np.array_equal(xs['thread'], xs['staged']))
    for form, v in res.items():
        v = np.array(v)
        print(f'{form:6s}  mean ms/step {v.mean():.2f}  spread (max - min) {v.max() - v.min():.2f}  runs {np.round(v, 2).tolist()}')
    t, s = np.mean(res['thread']), np.mean(res['staged'])
    print(f'staged / thread: {s / t:.4f}  ({100 * (t - s) / t:+.1f} % of a step)')


if __name__ == '__main__':
    main()
