"""Forward simulation (rt_forward_simulate) against the host simulator and the exact posterior draw.

  NODES   C2 shape (synth.config_c2 tree: 4-state HKY, 32 leaves, 1e6 sites) and C3 shape (config_c3
          tree: 61-state MG94, 128 leaves, 1e5 sites; also as three omega classes): the native call
          alone (arguments built once) and the whole simulate_sites() call, against
          synth.simulate_leaf_codes on the host; the leaf-code bytes written over the kernel time.
  HISTORY C4 shape (config_c4 tree: 4-state HKY, 64 leaves; 4096 chains x 1e4 sites = 4.1e7
          trajectories): one ForwardHistories.draw() against one RaoTehChains.draw_posterior() of the
          same chains, both with statistics.

After warm-up every GPU case is timed with CUDA events `--reps` times, the cases alternating; the host
simulator once.  Prints one JSON line with the card, its power limit and SM clock, and the medians.

    python tools/time_simulate.py [--reps 5] [--c4-chains 4096]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.sm,clocks.max.sm',
                            '--format=csv,noheader', '-i', '0'], capture_output=True, text=True, timeout=30)
        info = q.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        info = 'unknown'
    return name, info


def timed(f):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--c4-chains', type=int, default=4096)
    ap.add_argument('--c4-sites', type=int, default=10_000)
    ap.add_argument('--cap', type=int, default=112)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    from raoteh_b200 import engine, simulate, synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains

    cases, host_ms, info = {}, {}, {}
    for name, cfg_fn, n_sites in (('C2', synth.config_c2, 1_000_000), ('C3', synth.config_c3, 100_000)):
        cfg = cfg_fn(n_sites=16)              # the tree and model; the 16 sites are not used
        parent, length, leaves, Q, pi = (cfg[k] for k in ('parent', 'length', 'leaves', 'Q', 'pi'))
        sched = TreeSchedule(parent, length)
        mjp = engine.TreeMJP(sched, Q)
        P = mjp.transition_matrices()[None].contiguous()
        A, out, keep = simulate._nodes_call(sched, P, None, pi, n_sites, 1, 0, None, None, False, 0, None,
                                            mjp.device)
        cases[name + '_nodes_kernel'] = (lambda A=A: simulate._call(A))
        cases[name + '_simulate_sites'] = (lambda sched=sched, Q=Q, pi=pi, n=n_sites:
                                          simulate.simulate_sites(sched, Q, n, root_distn=pi, seed=1))
        info[name] = dict(n_sites=n_sites, n_leaves=len(leaves), S=int(Q.shape[0]),
                          leaf_code_bytes=len(leaves) * n_sites,
                          table_bytes=4 * sched.n * Q.shape[0] ** 2, _keep=(A, out, keep))
        t0 = time.perf_counter()
        synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, np.random.default_rng(1))
        host_ms[name] = 1e3 * (time.perf_counter() - t0)
        if name == 'C3':
            Qs = np.stack([synth.mg94(omega=om)[0] for om in (0.1, 1.0, 3.0)])
            from raoteh_b200.mixture import SiteMixtureMJP
            mix = SiteMixtureMJP(sched, Qs, root_distn=pi, weights=[0.6, 0.3, 0.1])
            Pk = torch.stack([m.transition_matrices() for m in mix.classes])
            w = torch.tensor([0.6, 0.3, 0.1], dtype=torch.float64, device=mjp.device)
            A3, out3, keep3 = simulate._nodes_call(sched, Pk, w, pi, n_sites, 1, 0, None, None, False, 0, None,
                                                   mjp.device)
            cases['C3_3omega_nodes_kernel'] = (lambda A=A3: simulate._call(A))
            info['C3_3omega'] = dict(table_bytes=4 * 3 * sched.n * 61 ** 2, _keep=(A3, out3, keep3))

    cfg = synth.config_c4(n_sites=a.c4_sites)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    n_traj = a.c4_chains * a.c4_sites
    fh = simulate.ForwardHistories(sched, cfg['Q'], n_traj, root_distn=cfg['pi'], seed=1, cap=a.cap)
    ch = RaoTehChains(sched, cfg['Q'], obs, n_chains=a.c4_chains, root_distn=cfg['pi'], seed=1, cap=a.cap)
    cases['C4_history_draw'] = fh.draw
    cases['C4_draw_posterior'] = ch.draw_posterior

    for f in cases.values():                   # warm-up: module loads, inputs, workspaces
        f()
    torch.cuda.synchronize()
    ms = {k: [] for k in cases}
    for _ in range(a.reps):
        for k, f in cases.items():
            ms[k].append(timed(f))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    for name in ('C2', 'C3'):
        info[name]['leaf_code_write_GBps'] = info[name]['leaf_code_bytes'] / (med[name + '_nodes_kernel'] * 1e6)
        info[name]['host_simulate_leaf_codes_ms'] = host_ms[name]
        info[name]['speedup_kernel_vs_host'] = host_ms[name] / med[name + '_nodes_kernel']
    info['C4'] = dict(n_traj=n_traj, mean_jumps_forward=float(fh.ev_total.double().mean()),
                      mean_jumps_posterior=float(ch.ev_total.double().mean()),
                      ratio_forward_to_posterior=med['C4_history_draw'] / med['C4_draw_posterior'])
    for v in info.values():
        v.pop('_keep', None)
    name, clocks = card()
    print(json.dumps(dict(gpu=name, power_limit_sm_clock_max_sm_clock=clocks, median_ms=med, all_ms=ms,
                          info=info)))


if __name__ == '__main__':
    main()
