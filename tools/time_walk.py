"""The S <= 8 down walk alone (rt_posterior_stats on the stored partials of one up pass) at C2
shape: 4 states, 32-leaf tree, uint8 leaf codes, 1e6 sites by default.  CUDA events around each
call; a 256 MiB buffer is overwritten between calls so that the stored partials are read from
HBM, as in a step where the up pass has streamed 1 GB through L2 since writing them.
Prints one JSON line: per-call times (ms), their median, min and max, the card and its power limit.
usage: python tools/time_walk.py [--sites N] [--reps R] [--codes4]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from raoteh_b200 import engine, synth
from raoteh_b200.lowering import TreeSchedule


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=1_000_000)
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--codes4', action='store_true', help='4-bit packed leaf codes')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_walk.py needs a CUDA device')
    cfg = synth.config_c2(n_sites=args.sites)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    make = engine.Observations.from_leaf_codes4 if args.codes4 else engine.Observations.from_leaf_codes
    obs = make(sched, cfg['codes'], cfg['leaves'])
    mjp = engine.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'])
    up = mjp.log_likelihood(obs, keep_partials=True)
    prog = mjp._programs(obs)
    S, n = mjp.S, sched.n
    W = torch.zeros((n, S, S), dtype=torch.float64, device='cuda')
    rps = torch.zeros(S, dtype=torch.float64, device='cuda')
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')

    def walk():
        mjp._down(obs, prog, 0, obs.n_sites, None, up['partials'], up['status'], None, W, rps)

    for _ in range(5):
        walk()
    torch.cuda.synchronize()
    ts = []
    for _ in range(args.reps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        walk()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().split('\n')[0]
    print(json.dumps(dict(walk_ms_median=float(np.median(ts)), walk_ms_min=float(np.min(ts)),
                          walk_ms_max=float(np.max(ts)), reps=args.reps, sites=args.sites,
                          codes4=args.codes4, gpu=smi)))


if __name__ == '__main__':
    main()
