"""Exact posterior draws (RaoTehChains.draw_posterior) against Rao-Teh sweeps at the C4 configuration
(synth.config_c4: 4-state HKY, 64-leaf tree; 4096 chains x 1e4 sites = 4.1e7 trajectories), in one
process: after warm-up, one draw and `--sweeps` sweeps are timed in turn with CUDA events, `--reps`
times, both with statistics.  Prints one JSON line: the card and its power limit, draws/s and
sweeps/s (trajectories x draws or sweeps per second, medians over the repetitions), and the time to
an unbiased estimate on the C4-shape test's schedule: 1 draw + 200 sweeps against initialize() +
1000 burn-in + 200 sweeps.

    python tools/time_posterior_draw.py [--chains 4096] [--sites 10000] [--reps 5] [--sweeps 10]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--chains', type=int, default=4096)
    ap.add_argument('--sites', type=int, default=10_000)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--sweeps', type=int, default=10)
    ap.add_argument('--cap', type=int, default=112)
    ap.add_argument('--time-dtype', default='float32', choices=['float32', 'float64'])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    from raoteh_b200 import engine, synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains
    cfg = synth.config_c4(n_sites=a.sites)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    ch = RaoTehChains(sched, cfg['Q'], obs, n_chains=a.chains, root_distn=cfg['pi'], seed=20260204,
                      cap=a.cap, time_dtype=a.time_dtype)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    # initialize(): the start the sweeps otherwise use (timed once, after a warm-up call)
    ch.initialize()
    e0, e1 = ev(), ev()
    e0.record()
    ch.initialize()
    e1.record()
    torch.cuda.synchronize()
    ms_init = e0.elapsed_time(e1)
    # warm-up of both timed calls (module loads, the draw's P and partials, workspaces)
    ch.draw_posterior()
    ch.sweep(2)
    torch.cuda.synchronize()
    ms_draw, ms_sweep = [], []
    for _ in range(a.reps):
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        ch.draw_posterior()
        e1.record()
        ch.sweep(a.sweeps)
        e2.record()
        torch.cuda.synchronize()
        ms_draw.append(e0.elapsed_time(e1))
        ms_sweep.append(e1.elapsed_time(e2) / a.sweeps)
    n = ch.n_traj
    d, s = float(np.median(ms_draw)), float(np.median(ms_sweep))
    name, power = card()
    print(json.dumps(dict(
        workload='C4: 4-state HKY, 64-leaf tree, %d chains x %d sites = %d trajectories, %s event times'
                 % (a.chains, a.sites, n, a.time_dtype),
        gpu=name, power_limit=power,
        draw_ms=d, sweep_ms=s, draw_ms_all=ms_draw, sweep_ms_all=ms_sweep, initialize_ms=ms_init,
        draws_per_s=n / (d * 1e-3), sweeps_per_s=n / (s * 1e-3), draw_over_sweep=d / s,
        mean_real_jumps_per_trajectory=float(ch.ev_total.double().mean()),
        unbiased_c4_schedule_ms=dict(draw_then_200_sweeps=d + 200 * s,
                                     initialize_1000_burn_in_200_sweeps=ms_init + 1200 * s))))


if __name__ == '__main__':
    main()
