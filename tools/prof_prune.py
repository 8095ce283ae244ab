"""Per-phase cycle breakdown of the DMMA pruning kernel (library built with
RT_EXTRA_NVCC_FLAGS=-DRT_PD_PROFILE=1)."""
import ctypes
import sys
import torch
sys.path.insert(0, '.')
from raoteh_b200 import engine, synth, _native
from raoteh_b200.lowering import TreeSchedule
cfg = synth.config_c3(n_sites=100_000)
sched = TreeSchedule(cfg['parent'], cfg['length'])
obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
mjp = engine.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'])
L = ctypes.CDLL(_native.LIB_PATH)
buf = (ctypes.c_ulonglong * 11)()
for _ in range(2):
    mjp.log_likelihood(obs)
L.rt_debug_prune_profile(buf)
mjp.log_likelihood(obs)
L.rt_debug_prune_profile(buf)
v = list(buf)
names = ['total', 'leaf gather', 'B fill', 'wait P', None, 'DMMA loop', 'release+product', 'store/root', 'code staging', 'other ops', 'warps']
tot = v[0]
for n, x in zip(names, v):
    if n is None:       # slot 4: unused
        continue
    print('%-16s %14d  %5.1f%%  per warp %.0f' % (n, x, 100.0 * x / tot, x / max(1, v[10])))
