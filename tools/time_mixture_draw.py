"""Exact posterior draws under site-class mixtures (SiteMixtureMJP.history_draws) against the
single-class draw (RaoTehChains.draw_posterior) at the C4 configuration (synth.config_c4: 4-state
HKY, 64-leaf tree; 4096 chains x 1e4 sites = 4.1e7 trajectories), in one process: after warm-up,
one draw of every trajectory under HKY+G4 (alpha = 0.5), under HKY+G4+I and under the single-class
model is timed in turn with CUDA events, `--reps` times, all with statistics.  Prints one JSON line:
the card and its power limit, the median times and the ratios to the single-class draw.

    python tools/time_mixture_draw.py [--chains 4096] [--sites 10000] [--reps 3]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from time_posterior_draw import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--chains', type=int, default=4096)
    ap.add_argument('--sites', type=int, default=10_000)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--cap', type=int, default=112)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    from raoteh_b200 import engine, synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.mixture import SiteMixtureMJP, discrete_gamma_rates
    from raoteh_b200.raoteh import RaoTehChains
    cfg = synth.config_c4(n_sites=a.sites)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    Q, pi = cfg['Q'], cfg['pi']
    g4 = discrete_gamma_rates(0.5, 4)
    runs = {
        'single': RaoTehChains(sched, Q, obs, n_chains=a.chains, root_distn=pi, seed=1, cap=a.cap),
        'g4': SiteMixtureMJP(sched, Q, root_distn=pi, rates=g4).history_draws(
            obs, n_chains=a.chains, seed=1, cap=a.cap),
        'g4_i': SiteMixtureMJP(sched, Q, root_distn=pi, rates=np.concatenate([[0.0], g4]),
                               weights=[0.2, 0.2, 0.2, 0.2, 0.2]).history_draws(
            obs, n_chains=a.chains, seed=1, cap=a.cap),
    }
    step = {'single': runs['single'].draw_posterior, 'g4': runs['g4'].draw, 'g4_i': runs['g4_i'].draw}
    for f in step.values():                # warm-up: module loads, the draws' inputs, workspaces
        f()
    torch.cuda.synchronize()
    ms = {k: [] for k in step}
    for _ in range(a.reps):
        for k, f in step.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    jumps = {k: float(r.ev_total.double().mean()) for k, r in runs.items()}
    name, power = card()
    print(json.dumps(dict(
        workload='C4: 4-state HKY, 64-leaf tree, %d chains x %d sites = %d trajectories, one draw each'
                 % (a.chains, a.sites, a.chains * a.sites),
        gpu=name, power_limit=power, draw_ms=med, draw_ms_all=ms,
        ratio_to_single=dict(g4=med['g4'] / med['single'], g4_i=med['g4_i'] / med['single']),
        mean_real_jumps_per_trajectory=jumps)))


if __name__ == '__main__':
    main()
