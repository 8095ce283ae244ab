"""Site-class mixtures (raoteh_b200.mixture.SiteMixtureMJP.expected_history_statistics) against K
single-class evaluations (TreeMJP.expected_history_statistics) on the same sites, in one process:
    C2: synth.config_c2, 1e6 sites, HKY+G4 (alpha = 0.5, mean rates);
    C3: synth.config_c3, 1e5 sites, three MG94 omega classes (0.1, 1, 2.5).
The mixture runs 2K up passes (K log-likelihood-only, K with stored partials), K weighted down
passes and K contractions; the single class one up pass with stored partials, one down pass and
one contraction.  After a warm-up, the mixture and K single-class calls are timed in turn with
CUDA events, `--reps` times.  Prints one JSON line per case: the card and its power limit, the
median times and their ratio.

    python tools/time_mixture.py [--reps 5] [--c2-sites 1000000] [--c3-sites 100000]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))

from time_posterior_draw import card  # noqa: E402


def time_case(name, cfg, Qs, rates, weights, reps):
    from raoteh_b200 import engine
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.mixture import SiteMixtureMJP
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    mix = SiteMixtureMJP(sched, np.stack(Qs), root_distn=cfg['pi'], rates=rates, weights=weights)
    single = engine.TreeMJP(sched, Qs[0], root_distn=cfg['pi'])
    K = len(rates)

    def run_single():
        for _ in range(K):
            single.expected_history_statistics(obs)

    ev = lambda: torch.cuda.Event(enable_timing=True)
    mix.expected_history_statistics(obs)
    run_single()
    torch.cuda.synchronize()
    ms_mix, ms_single = [], []
    for _ in range(reps):
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        mix.expected_history_statistics(obs)
        e1.record()
        run_single()
        e2.record()
        torch.cuda.synchronize()
        ms_mix.append(e0.elapsed_time(e1))
        ms_single.append(e1.elapsed_time(e2))
    m, s = float(np.median(ms_mix)), float(np.median(ms_single))
    gpu, power = card()
    return dict(workload=name, gpu=gpu, power_limit=power, n_sites=obs.n_sites, K=K,
                mixture_ms=m, k_single_class_ms=s, mixture_over_k_single=m / s,
                mixture_ms_all=ms_mix, k_single_class_ms_all=ms_single)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--c2-sites', type=int, default=1_000_000)
    ap.add_argument('--c3-sites', type=int, default=100_000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    from raoteh_b200 import synth
    from raoteh_b200.mixture import discrete_gamma_rates
    c2 = synth.config_c2(n_sites=a.c2_sites)
    rates = discrete_gamma_rates(0.5, 4)
    print(json.dumps(time_case('C2: HKY+G4 (alpha 0.5), 32-leaf tree', c2, [c2['Q']] * 4, rates,
                               np.full(4, 0.25), a.reps)))
    c3 = synth.config_c3(n_sites=a.c3_sites)
    Qs = [synth.mg94(omega=om)[0] for om in (0.1, 1.0, 2.5)]
    print(json.dumps(time_case('C3: three MG94 omega classes (0.1, 1, 2.5), 128-leaf tree', c3, Qs,
                               np.ones(3), np.array([0.6, 0.3, 0.1]), a.reps)))


if __name__ == '__main__':
    main()
