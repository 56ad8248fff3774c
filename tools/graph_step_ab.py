"""dev: one controller step + plant step of the cfg[0] (naive, B = 100) and cfg[1] (ST, B = 10 000) closed loops, run eagerly and as a
replay of a captured CUDA graph (INTEGRATION.md), alternated in one process.

    python tools/graph_step_ab.py [--rounds 3] [--steps 40] [--warmup 3] [--precision f64]

Per configuration: two handles with the same seeded workload and warm start as bench.py; one runs the steps eagerly on its own stream,
the other captures `controller_step` + `plant_step` once (after an eager warm-up step) and replays the graph.  Each round times `--steps`
steps of each arm with CUDA events (the arms alternate between rounds and run the same number of steps).  Prints ms per step (mean, p50,
p99) per arm, the number of nodes of the captured graph, the number of problems whose states differ between the arms at the end (NaN equal
to NaN), and the card's name and power limit."""
import argparse
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

import numpy as np
import torch

import bench


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = 'unknown'
    return out or torch.cuda.get_device_name(0)


def graph_nodes(g):
    """node count of the top level of a captured torch graph (conditional nodes count once; their bodies are not expanded)"""
    rt = None
    try:
        raw = g.raw_cuda_graph()
    except (AttributeError, RuntimeError):
        return -1
    for name in ('libcudart.so.12', 'libcudart.so'):
        try:
            rt = C.CDLL(name)
            break
        except OSError:
            continue
    if rt is None:
        return -1
    n = C.c_size_t(0)
    rc = rt.cudaGraphGetNodes(C.c_void_p(raw), None, C.byref(n))
    return int(n.value) if rc == 0 else -1


def arm(controller, B):
    from safe_mpc_b200.engine import Engine
    params, md, x0, pin = bench.workload(controller, 45, 0.0, 0, 0, B)
    main, bk, prob = bench.make_handles(Engine, params, md, controller, B, 0)
    bk.close()
    main.set_plant_inertial(pin)
    bench.warm_guess(main, x0, 45, 5)
    return main, x0


def timed(fn, stream, steps):
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record(stream)
    for i in range(steps):
        fn()
        evs[i + 1].record(stream)
    torch.cuda.synchronize()
    return np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(steps)])


def run_config(name, controller, B, a):
    eng_e, x0 = arm(controller, B)
    eng_g, _ = arm(controller, B)
    s = torch.cuda.Stream()
    eng_g.set_stream(s)
    x_e = torch.tensor(x0, device='cuda')
    x_g = x_e.clone()
    s.wait_stream(torch.cuda.current_stream())
    cur = torch.cuda.current_stream()

    def eager():
        nonlocal x_e
        u, _ = eng_e.controller_step(x_e)
        x_e, _ = eng_e.plant_step(x_e, u)

    with torch.cuda.stream(s):
        for _ in range(a.warmup):
            u, _ = eng_g.controller_step(x_g)
            xn, _ = eng_g.plant_step(x_g, u)
            x_g.copy_(xn)
    for _ in range(a.warmup):
        eager()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        u_s, _ = eng_g.controller_step(x_g)
        xn_s, _ = eng_g.plant_step(x_g, u_s)
        x_g.copy_(xn_s)
    torch.cuda.synchronize()
    nodes = graph_nodes(g)
    res = {'eager': [], 'graph': []}
    for r in range(a.rounds):
        for which in ('eager', 'graph') if r % 2 == 0 else ('graph', 'eager'):
            lat = timed(eager if which == 'eager' else g.replay, cur, a.steps)
            res[which].append(lat)
    differ = int((~((x_e == x_g) | (torch.isnan(x_e) & torch.isnan(x_g)))).any(dim=1).sum())
    print(f'{name}: {controller} N=45 B={B} {a.precision}, {a.rounds} rounds x {a.steps} steps per arm; graph nodes (top level) {nodes}; '
          f'problems whose states differ after the last step: {differ}')
    for which, v in res.items():
        lat = np.concatenate(v)
        per_round = ' '.join(f'{x.mean():.3f}' for x in v)
        print(f'  {which:5s}  ms/step mean {lat.mean():7.3f}  p50 {np.percentile(lat, 50):7.3f}  p99 {np.percentile(lat, 99):7.3f}   rounds {per_round}')
    e, gr = np.concatenate(res['eager']).mean(), np.concatenate(res['graph']).mean()
    print(f'  graph / eager: {gr / e:.4f}  ({100 * (e - gr) / e:+.1f} % of a step)')
    eng_e.close(); eng_g.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--precision', default='f64', choices=['f64', 'f32'])
    a = ap.parse_args()
    bench.PRECISION = a.precision
    print(f'card: {card()}')
    run_config('cfg[0]', 'naive', 100, a)
    run_config('cfg[1]', 'st', 10000, a)


if __name__ == '__main__':
    main()
