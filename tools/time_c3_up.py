"""C3 (61 states, 128 leaves, 1e5 sites): time of the DMMA pruning kernel alone (log-lik only)
and with stored partials."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, numpy as np
from raoteh_b200 import engine, synth
from raoteh_b200.lowering import TreeSchedule
dev = torch.device('cuda:0')
cfg = synth.config_c3(n_sites=100_000)
sched = TreeSchedule(cfg['parent'], cfg['length'])
mjp = engine.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'], device=dev)
obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'], device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
def timed(fn, n=8):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(n):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); r = fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), r
t_ll, r = timed(lambda: mjp.log_likelihood(obs))
mjp.events = {}
t_ex, r2 = timed(lambda: mjp.expected_history_statistics(obs), n=4)
print(json.dumps(dict(loglik_ms=t_ll, expectations_ms=t_ex, loglik_sum=float(r['loglik'].sum()))))
