#!/usr/bin/env python
"""
bench.py -- headline benchmark of the raoteh_b200 hot path.

Workload (BASELINE.json configs[1], "C2"): 4-state HKY MJP on a 32-leaf random
binary tree, 1M synthetic sites per GPU: per-site log-likelihood + site-summed
expected dwell times / transition counts.  One step = one full evaluation for
one batch of sites: per-edge expm, upward pass (partials stored), downward
pass + per-edge weights, Frechet contraction, (N > 1) one NCCL allreduce of
[1 + S + S*S] doubles.  Metric: site.edge messages / s = n_sites * n_edges / t.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

`value`   : inputs resident in HBM, CUDA-event time, max over ranks.
`e2e`     : same step through the public API with HOST buffers: H2D of the leaf
            codes from pinned memory and D2H of log-likelihoods, status and the
            statistics inside the timed region.
`roofline`: dominant kernel of the step (downward pass), algorithmic bytes /
            CUDA-event duration against MEASURED_PEAKS.json hbm_gbs.
`extra`   : C3 (61-state DMMA pruning), C4 (Rao-Teh sweeps), C5 (tolerance model:
            likelihood + blocked Gibbs sampler + summary) and 61-state Rao-Teh figures.
`--impl reference`: the oracle port of the reference's CPU path (numpy/scipy,
            one process per host core) on a bounded sample of the same workload.
`--dump-outputs DIR`: what the step behind `value` returned in its last timed step,
            as DIR/<name>.npy (rank 0), so that two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

C2_SITES = 1_000_000
E2E_CHUNKS = int(os.environ.get('RT_E2E_CHUNKS', '8'))
E2E_PACKED = os.environ.get('RT_E2E_PACKED', '1') != '0'         # 4-bit leaf codes on the host side
USE_GRAPH = os.environ.get('RT_STEP_GRAPH', '1') != '0'       # device-resident arm: replay the step as one CUDA graph
DEV_CHUNKS = int(os.environ.get('RT_DEV_CHUNKS', '0'))     # device-resident arm: two-stream chunk overlap   # site chunks of the pipelined host-buffer call
C2_LEAVES = 32
# what a caller of the C2 step receives: per-site log-likelihoods and status, the site-summed
# statistics, the per-edge weights and contractions, and the packed (allreduced) vector
# [loglik sum, dwell, trans, root posterior sum]
DUMP_KEYS = ('loglik', 'status', 'dwell', 'trans', 'root_post_sum', 'W', 'M_edges', 'stats')


# ----------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------
def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), 'measured'
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0), 'fallback'


def fp64_peak(which='dmma'):
    """FP64 tensor (DMMA) peak measured on this pool's B200 with tools/fp64_peak.cu
    (profiles/r1_fp64_peak.jsonl): 37.0 TFLOP/s; DFMA 33.5 TFLOP/s."""
    path = os.path.join(ROOT, 'profiles', 'r1_fp64_peak.jsonl')
    best = 37.0 if which == 'dmma' else 33.5
    if os.path.exists(path):
        vals = []
        for line in open(path):
            try:
                d = json.loads(line)
            except ValueError:
                continue
            if d.get('probe', '').startswith('dmma' if which == 'dmma' else 'dfma'):
                vals.append(d['tflops'])
        if vals:
            best = max(vals)
    return best


class ClockSampler(object):
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None,
                    sm_max_mhz=float(max(mx)) if mx else None,
                    samples=len(sm), reasons=sorted(reasons))


def c2_config(n_edges, S, world, scaling='weak'):
    """`config` of the JSON line: the same object for the GPU arm and the reference arm."""
    return dict(workload='C2: 4-state HKY MJP, 32-leaf random binary tree, 1e6 synthetic sites per GPU '
                         '(uint8 leaf codes, 1% missing): per-site log-lik + site-summed expected '
                         'dwell/transition counts',
                sites_per_gpu=C2_SITES, n_edges=n_edges, n_states=S,
                parallelism='site-sharded x%d, one allreduce of %d doubles' % (world, 1 + 2 * S + S * S),
                l2='256 MiB flush buffer written between timed iterations')


def c2_workload(rank, n_sites=C2_SITES):
    from raoteh_b200 import synth
    return synth.config_c2(n_sites=n_sites, seed=20260201 + 1000 * rank, n_leaves=C2_LEAVES) \
        if rank else synth.config_c2(n_sites=n_sites, n_leaves=C2_LEAVES)


def step_outputs(r, stats):
    """Host copies of the step's outputs (float64; the int8 site status as float32), about
    12 MB for the 1e6 C2 sites."""
    r = dict(r, stats=stats)
    out = {}
    for k in DUMP_KEYS:
        a = r[k].detach().cpu().numpy()
        out[k] = a if a.dtype == np.float64 else a.astype(np.float32)
    return out


def c2_bytes_per_site(sched, S):
    """Algorithmic HBM bytes per site (DESIGN.md section 4)."""
    n_int = sched.n_store
    n_leaf = len(sched.leaves)
    up = n_leaf * 1 + n_int * S * 8 + 8 + 1
    # down (fused walk): every stored partial read once, leaf codes and status read once;
    # node marginals never leave the chip, W is S*S*n_edges doubles per CTA (negligible)
    down = n_int * S * 8 + n_leaf * 1 + 1
    return up, down


def ncu_traffic(kernel_substr):
    """dram read+write bytes per launch from the committed `ncu --set full` capture."""
    path = os.path.join(ROOT, 'profiles', 'r1_ncu_full_summary.json')
    if not os.path.exists(path):
        return None
    mult = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
    ks = []
    for name in ('r2_ncu_full_summary.json', 'r1_ncu_full_summary.json'):
        pth = os.path.join(ROOT, 'profiles', name)
        if os.path.exists(pth):
            ks += json.load(open(pth))
    for k in ks:
        if kernel_substr in k['kernel']:
            tot = 0.0
            for key in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                v, u = k[key].split()
                tot += float(v) * mult[u]
            return tot
    return None


# ----------------------------------------------------------------------------
# reference arm / cpu baseline: oracle port on host cores
# ----------------------------------------------------------------------------
def _cpu_chunk(args):
    from oracle import np_oracle
    cfg, lo, hi = args
    S = cfg['S']
    P = np_oracle.expm_edges(cfg['Q'], cfg['length'])
    obs = np_oracle.Obs('codes', S, hi - lo, leaf_nodes=cfg['leaves'], codes=cfg['codes'][:, lo:hi])
    r = np_oracle.expected_history_statistics(cfg['parent'], cfg['length'], cfg['Q'], P, obs, cfg['pi'])
    return float(r['loglik'].sum()), r['dwell'], r['trans']


def cpu_reference_step(cfg, n_sample, pool, cores):
    """One step of the oracle port (log-lik + expectations) on n_sample sites."""
    per = (n_sample + cores - 1) // cores
    jobs = [(cfg, lo, min(n_sample, lo + per)) for lo in range(0, n_sample, per)]
    t0 = time.perf_counter()
    out = pool.map(_cpu_chunk, jobs)
    dt = time.perf_counter() - t0
    return dt, sum(o[0] for o in out)


def cpu_per_site_reference_style(cfg, n_sites=3):
    """The reference's own structure: expm of every edge redone for every site
    (raoteh/sampler/_mjp_dense.py:352-358), one site per call."""
    from oracle import np_oracle
    S = cfg['S']
    t0 = time.perf_counter()
    for i in range(n_sites):
        P = np_oracle.expm_edges(cfg['Q'], cfg['length'])
        obs = np_oracle.Obs('codes', S, 1, leaf_nodes=cfg['leaves'], codes=cfg['codes'][:, i:i + 1])
        np_oracle.log_likelihood(cfg['parent'], P, obs, cfg['pi'])
    return (time.perf_counter() - t0) / n_sites


def physical_cores():
    """One logical CPU per physical core of this process's affinity mask (hyper-thread siblings
    share the FP units the numpy port lives on, and make the figure swing between boxes)."""
    allowed = sorted(os.sched_getaffinity(0))
    seen, picked = set(), []
    for c in allowed:
        try:
            with open('/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list' % c) as f:
                key = f.read().strip()
        except OSError:
            key = str(c)
        if key not in seen:
            seen.add(key)
            picked.append(c)
    return picked or allowed


def _pin_worker(cpu_queue):
    try:
        os.sched_setaffinity(0, {cpu_queue.get(timeout=5)})
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass


def cpu_pool(cpus):
    import multiprocessing as mp
    ctx = mp.get_context('fork')
    q = ctx.Queue()
    for c in cpus:
        q.put(c)
    return ctx.Pool(len(cpus), initializer=_pin_worker, initargs=(q,))


def reference_as_is_record():
    """The UNMODIFIED reference called one site at a time (shimmed `_mjp_dense.get_likelihood` +
    `get_expected_history_statistics`, /root/reference exists only in the build container):
    measured there by oracle/time_reference_as_is.py and committed under profiles/."""
    path = os.path.join(ROOT, 'profiles', 'r2_reference_as_is.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    cpus = physical_cores()
    cores = len(cpus)
    n_sample = 200_000
    cfg = c2_workload(0, n_sample)
    n_edges = len(cfg['parent']) - 1
    with cpu_pool(cpus) as pool:
        for _ in range(max(1, args.warmup)):
            cpu_reference_step(cfg, n_sample, pool, cores)
        times = [cpu_reference_step(cfg, n_sample, pool, cores)[0] for _ in range(args.steps)]
    # best-of-k: the CPU arm shares the host with whatever else runs on it; the fastest step is
    # the machine's capability, the spread is reported beside it
    dt = float(np.min(times))
    value = n_sample * n_edges / dt
    line = dict(
        impl='reference', metric='site_edge_messages_per_sec', value=value, unit='messages/s',
        n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=dt * 1e3,
        higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f64', data='synthetic',
        config=c2_config(n_edges, cfg['S'], max(1, args.gpus)),
        cpu_baseline=dict(value=value, unit='messages/s', cores=cores, kind='port',
                          timing='best of %d steps; mean %.1f ms, max %.1f ms' % (
                              len(times), 1e3 * float(np.mean(times)), 1e3 * float(np.max(times))),
                          spread=dict(min_ms=1e3 * float(np.min(times)), mean_ms=1e3 * float(np.mean(times)),
                                      max_ms=1e3 * float(np.max(times))),
                          logical_cpus=os.cpu_count(),
                          sample='%d of the 1e6 C2 sites per step (same tree, model and seed), '
                                 'oracle/np_oracle.py: numpy/scipy restatement with expm hoisted out of '
                                 'the site loop -- a STRONGER baseline than the reference as it is '
                                 '(see reference_as_is) -- one process pinned to each physical core'
                                 % n_sample,
                          reference_as_is=reference_as_is_record()),
        e2e=dict(value=value, unit='messages/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from raoteh_b200 import engine
    from raoteh_b200 import dist as rdist
    from raoteh_b200.lowering import TreeSchedule

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    # stdout carries exactly ONE JSON line: library chatter (e.g. NCCL's version
    # banner) is diverted to stderr while the benchmark runs
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    if world > 1:
        # one rank per GPU on a multi-socket host: keep the rank (and the pinned buffers it is
        # about to allocate) on the CPU cores local to its GPU
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
            if cpus:
                os.sched_setaffinity(0, cpus)
        except Exception:
            pass
    cfg = c2_workload(rank)
    S = cfg['S']
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    n_edges = sched.n_edges
    N = cfg['codes'].shape[1]
    codes_pinned = torch.from_numpy(cfg['codes']).pin_memory()
    codes4_pinned = torch.from_numpy(engine.pack_codes4(cfg['codes'])).pin_memory()   # RT_OBS_CODES4
    codes_dev = codes_pinned.to(dev)
    obs_slot = np.full(sched.n, -1, dtype=np.int32)
    obs_slot[cfg['leaves']] = np.arange(len(cfg['leaves']), dtype=np.int32)
    obs = engine.Observations(engine.OBS_CODES, codes_dev, obs_slot, N)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    out_ll = torch.empty(N, dtype=torch.float64).pin_memory()
    out_st = torch.empty(N, dtype=torch.int8).pin_memory()
    out_stats = torch.empty(1 + S + S * S + S, dtype=torch.float64).pin_memory()

    ev = lambda: torch.cuda.Event(enable_timing=True)
    mjp = engine.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'], device=dev)
    state = {}

    def step(record=False):
        """New rate matrix -> expm + up + down + Frechet contraction (+ allreduce);
        observations resident in HBM.  record=True: one launch per kernel on the current
        stream with CUDA events around the up and the down kernel (roofline accounting);
        otherwise the production schedule (DEV_CHUNKS site chunks alternating between two
        streams when > 1)."""
        mjp.events = sub if record else None
        mjp.set_rate_matrix(cfg['Q'])
        if USE_GRAPH and not record:
            # production schedule: the whole evaluation replayed as one CUDA graph
            r = mjp.expected_history_statistics_graphed(obs)
            stats = r['stats']
        else:
            r = mjp.expected_history_statistics(obs, overlap_chunks=0 if record else DEV_CHUNKS)
            ll_sum = r['loglik_sum'] if 'loglik_sum' in r else r['loglik'].sum()
            stats = rdist.pack_stats(ll_sum, r['dwell'], r['trans'], r['root_post_sum'])
        rdist.allreduce_stats(stats)      # the path's only collective (NCCL, 1+S+S*S+S doubles)
        state['n_levels'] = r['n_levels']
        state['last'] = r, stats
        return r, stats
    sub = {}

    def step_e2e(packed=E2E_PACKED):
        """Same step through the public host-buffer API: H2D of the leaf codes from pinned
        memory (two 4-bit codes per byte by default, one byte per code with packed=False),
        D2H of per-site log-lik / status and of the statistics, all inside."""
        mjp.events = None
        mjp.set_rate_matrix(cfg['Q'])
        r = mjp.expected_history_statistics_from_host(
            codes4_pinned if packed else codes_pinned, cfg['leaves'], out_ll, out_st,
            n_chunks=E2E_CHUNKS, packed=packed)
        stats = rdist.pack_stats(r['loglik_sum'], r['dwell'], r['trans'], r['root_post_sum'])
        rdist.allreduce_stats(stats)
        out_stats.copy_(stats, non_blocking=True)

    def timed(fn, steps, warmup, record=False):
        for _ in range(warmup):
            flush.fill_(1)
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total = 0.0
        evs = []
        for _ in range(steps):
            flush.fill_(1)            # evict L2 between timed iterations
            a, b = ev(), ev()
            a.record()
            fn(record) if record else fn()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([total], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]) / steps

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_plain = timed(step, args.steps, args.warmup, record=True)   # per-kernel events (roofline)
    ms = timed(step, args.steps, args.warmup) if (DEV_CHUNKS > 1 or USE_GRAPH) else ms_plain
    if args.dump_outputs and rank == 0:
        # copied now: the legs below reuse the engine's workspaces
        for name, a in step_outputs(*state['last']).items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    clocks = sampler.stop() if rank == 0 else None
    ms_e2e = timed(step_e2e, args.steps, args.warmup)
    ms_e2e_u8 = timed(lambda: step_e2e(False), args.steps, args.warmup) if E2E_PACKED else ms_e2e

    total_sites = N * world
    value = total_sites * n_edges / (ms * 1e-3)
    e2e_value = total_sites * n_edges / (ms_e2e * 1e-3)

    # roofline of the dominant kernel
    peaks, peak_kind = measured_peaks()
    torch.cuda.synchronize()
    pair = lambda L: [(L[i], L[i + 1]) for i in range(0, len(L) - 1, 2)]
    n_int, n_leaf = sched.n_store, len(sched.leaves)
    n_int_edges = n_edges - n_leaf
    if 'fused' in sub:
        # ONE kernel does the up pass, root combine, down walk and W accumulation of a site tile;
        # the partials stay in an L2-resident per-CTA scratch, so the algorithmic HBM bytes are the
        # leaf codes + status + log-lik: (L + 1 + 8) per site
        f_ms = float(np.mean([a.elapsed_time(b) for a, b in pair(sub['fused'])]))
        b_site = n_leaf + 9
        gbs = N * b_site / (f_ms * 1e-3) / 1e9
        # algorithmic FP64 work per site (DESIGN.md section 4): up 2S^2+S per internal edge, S per leaf
        # edge, S per rescale, 2S root; down 6S^2+2S per internal edge (m, G, D_child, W), 2S per leaf
        flop_site = (n_int_edges * (2 * S * S + S) + n_leaf * S + n_int * S + 2 * S +
                     n_int_edges * (6 * S * S + 2 * S) + n_leaf * 2 * S)
        tfl = N * flop_site / (f_ms * 1e-3) / 1e12
        fma_peak = fp64_peak('dfma')
        roofline = dict(bound='hbm', kernel='fused_small_kernel<4,codes> (1 launch/step, %.0f%% of the step)'
                        % (100 * f_ms / ms), achieved=gbs, peak=peaks['hbm_gbs'], unit='GB/s',
                        frac=gbs / peaks['hbm_gbs'], peak_source='%s (MEASURED_PEAKS.json hbm_gbs)' % peak_kind,
                        traffic=ncu_traffic('fused_small_kernel<4, 0'),
                        algorithmic_bytes_per_launch=N * b_site, ms=f_ms,
                        fp64_pipe=dict(achieved=tfl, peak=fma_peak, unit='TFLOP/s', frac=tfl / fma_peak,
                                       algorithmic_flop_per_site=flop_site,
                                       peak_source='tools/fp64_peak.cu DFMA probe (profiles/r1_fp64_peak.jsonl)'),
                        note='the S=4 evaluation is bound by issue slots / the FP64 pipe, not by HBM: '
                             'fusing the up pass and the down walk removed the 2 x %d B/site of stored '
                             'partials from HBM (they live in an L2-resident per-CTA scratch), which '
                             'LOWERS the HBM fraction while making the step faster; the HBM-bound form of '
                             '4-state pruning is the dense-emission input (extra.c2_loglik_only)'
                             % (n_int * S * 8))
    else:
        up_ms = float(np.mean([a.elapsed_time(b) for a, b in pair(sub['up'])]))
        down_ms = float(np.mean([a.elapsed_time(b) for a, b in pair(sub['down'])]))
        up_b, down_b = c2_bytes_per_site(sched, S)
        down_gbs = N * down_b / (down_ms * 1e-3) / 1e9
        up_gbs = N * up_b / (up_ms * 1e-3) / 1e9
        # algorithmic FP64 work of the walk per site: 6S^2+2S per internal edge (m, G, D_child, W),
        # S^2+2S per leaf edge (G from a column of P, W)
        walk_flop = n_int_edges * (6 * S * S + 2 * S) + n_leaf * (S * S + 2 * S)
        walk_tfl = N * walk_flop / (down_ms * 1e-3) / 1e12
        fma_peak = fp64_peak('dfma')
        roofline = dict(bound='hbm', kernel='down_walk_kernel<4,codes> (1 launch/step, %.0f%% of the step)'
                        % (100 * down_ms / ms), achieved=down_gbs, peak=peaks['hbm_gbs'], unit='GB/s',
                        frac=down_gbs / peaks['hbm_gbs'], peak_source='%s (MEASURED_PEAKS.json hbm_gbs)' % peak_kind,
                        traffic=ncu_traffic('down_walk_kernel<4, 0'),
                        algorithmic_bytes_per_launch=N * down_b, ms=down_ms,
                        fp64_pipe=dict(achieved=walk_tfl, peak=fma_peak, unit='TFLOP/s', frac=walk_tfl / fma_peak,
                                       algorithmic_flop_per_site=walk_flop,
                                       peak_source='tools/fp64_peak.cu DFMA probe (profiles/r1_fp64_peak.jsonl)',
                                       ncu='fp64 pipe 34 %, issue slots 52 % (profiles/r2_ncu_full_summary.json)'),
                        note='the S=4 walk reads every stored partial exactly once (ncu dram read = algorithmic '
                             'bytes) but is bound by latency / issue slots, not by HBM; the fused up+down kernel '
                             'that removes these bytes altogether was built and measured slower '
                             '(profiles/r2_fused_small.md)',
                        also=dict(kernel='prune_small_kernel<4,codes,store>', achieved=up_gbs,
                                  frac=up_gbs / peaks['hbm_gbs'], ms=up_ms,
                                  algorithmic_bytes_per_launch=N * up_b,
                                  traffic=ncu_traffic('prune_small_kernel<4, 0, 1')))

    # ---- strong scaling beside the weak figure: 1e6 sites IN TOTAL, 1/N of them on this rank
    strong = None
    if world > 1 or args.scaling == 'strong':
        lo, hi = rdist.shard_range(C2_SITES, rank, world)
        obs_w, N_w = obs, N
        obs = engine.Observations(engine.OBS_CODES, codes_dev[:, lo:hi].contiguous(), obs_slot, hi - lo)
        ms_strong = timed(step, args.steps, args.warmup)
        strong = dict(scaling='strong', sites_total=C2_SITES, sites_this_rank=hi - lo, ms_per_step=ms_strong,
                      value=C2_SITES * n_edges / (ms_strong * 1e-3), unit='messages/s')
        obs = obs_w

    # ---- the other half of the metric: Rao-Teh sweeps/s, every rank, configured sizes
    sweeps = {}
    if not args.no_samplers:
        import bench_legs
        del flush
        torch.cuda.empty_cache()
        for name, fn in (('c4', lambda: bench_legs.bench_c4_sharded(
                              dev, rank, world, n_chains=args.c4_chains, timed_sweeps=args.c4_sweeps,
                              cpu_leg=not args.no_cpu)),
                         ('c5', lambda: bench_legs.bench_c5_sharded(
                              dev, rank, world, n_sites=args.c5_sites, cpu_leg=not args.no_cpu))):
            try:
                sweeps[name] = fn()
            except Exception as e:     # keep the headline line; all ranks fail alike (same sizes)
                sweeps[name] = dict(error=repr(e))
                torch.cuda.empty_cache()

    extra = {}
    if rank == 0 and not args.no_extra:
        try:
            extra['c3_61state_pruning'] = bench_c3(dev, args)
        except Exception as e:   # keep the headline line even if an extra fails
            extra['c3_61state_pruning'] = dict(error=repr(e))
        try:
            extra['c2_loglik_only'] = bench_c2_loglik(dev, cfg, sched, obs, args, peaks)
        except Exception as e:
            extra['c2_loglik_only'] = dict(error=repr(e))
        try:
            import bench_legs as raoteh_bench
            extra['codon_raoteh_sweeps'] = raoteh_bench.bench_codon_raoteh(dev, args)
        except Exception as e:
            extra['codon_raoteh_sweeps'] = dict(error=repr(e))
        try:
            import bench_legs as raoteh_bench
            extra['next_rows'] = raoteh_bench.bench_next_rows(dev, args)
        except Exception as e:
            extra['next_rows'] = dict(error=repr(e))

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpus = physical_cores()
        cores = len(cpus)
        n_sample = 200_000
        small = c2_workload(0, n_sample)
        with cpu_pool(cpus) as pool:
            cpu_reference_step(small, n_sample, pool, cores)
            dts = [cpu_reference_step(small, n_sample, pool, cores)[0] for _ in range(3)]
        dt = min(dts)
        per_site = cpu_per_site_reference_style(small, 3)
        cpu_baseline = dict(value=n_sample * n_edges / dt, unit='messages/s', cores=cores, kind='port',
                            timing='best of 3 steps (%.0f / %.0f / %.0f ms)' % tuple(1e3 * x for x in dts),
                            sample='%d of 1e6 C2 sites, oracle/np_oracle.py (numpy/scipy, expm hoisted '
                                   'out of the site loop), one process pinned to each physical core; '
                                   'the port in the reference\'s per-site structure (expm per edge per '
                                   'site, log-lik only): %.4f s/site = %.0f messages/s on 1 core'
                                   % (n_sample, per_site, n_edges / per_site),
                            reference_as_is=reference_as_is_record())

    if rank == 0:
        # expm (2), fused up+down (1; or up + down walk), Frechet contraction (3) + edge accumulation (1)
        launches_per_step = 2 + (1 if 'fused' in sub else 2) + 4
        line = dict(
            metric='site_edge_messages_per_sec', value=value, unit='messages/s', n_gpus=world,
            steps=args.steps, warmup=args.warmup, ms_per_step=ms, higher_is_better=True,
            ms_per_step_with_per_kernel_events=ms_plain,
            schedule=('one CUDA graph replay per step (TreeMJP.expected_history_statistics_graphed) + the '
                      'H2D copy of the rate matrix + the allreduce' if USE_GRAPH else 'eager launches'),
            scaling='weak', vs_baseline=None, dtype='f64', data='synthetic',
            config=c2_config(n_edges, S, world),
            # headline e2e: uint8 leaf codes exactly as a caller holds them, nothing prepared outside
            # the timed region; `packed_codes4` = the same call fed two 4-bit codes per byte, the
            # packing done once at data-load time (outside the timed region)
            e2e=dict(value=total_sites * n_edges / (ms_e2e_u8 * 1e-3), unit='messages/s',
                     ms_per_step=ms_e2e_u8, input='leaf codes, uint8',
                     h2d_bytes_per_step=int(codes_pinned.numel()),
                     d2h_bytes_per_step=int(out_ll.numel() * 8 + out_st.numel() + out_stats.numel() * 8),
                     pcie_gbs_per_rank=(codes_pinned.numel() + out_ll.numel() * 8 + out_st.numel())
                     / (ms_e2e_u8 * 1e-3) / 1e9,
                     packed_codes4=dict(ms_per_step=ms_e2e, value=e2e_value,
                                        h2d_bytes_per_step=int(codes4_pinned.numel()),
                                        note='RT_OBS_CODES4, packed by the caller before the timed region')),
            strong_scaling=strong, sweeps=sweeps,
            gpu_launches=launches_per_step * args.steps,
            roofline=roofline, cpu_baseline=cpu_baseline, clocks=clocks, extra=extra)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + '\n').encode())
    if world > 1:
        dist.destroy_process_group()
    return 0


def bench_c2_loglik(dev, cfg, sched, obs, args, peaks):
    """K2 alone: log-likelihood only (no stored partials), codes and dense-emission input."""
    import torch
    from raoteh_b200 import engine
    S = cfg['S']
    N = obs.n_sites
    mjp = engine.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'], device=dev)
    mjp.transition_matrices()
    res = {}
    ll = torch.empty(N, dtype=torch.float64, device=dev)
    st = torch.empty(N, dtype=torch.int8, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def time_it(o):
        for _ in range(3):
            mjp.log_likelihood(o, out=(ll, st))
        ts = []
        for _ in range(args.steps):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            mjp.log_likelihood(o, out=(ll, st))
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.mean(ts))
    ms = time_it(obs)
    b_site = len(sched.leaves) + 9
    # with hard codes the input is 41 B per site, so the honest roof is the FP64 FMA pipe / issue slots:
    # a mat-vec per internal edge (2 S^2 flop), one product per message (S), a leaf message is a gather
    n_leaf = len(sched.leaves)
    flop_site = (sched.n_edges - n_leaf) * 2 * S * S + sched.n_edges * S
    fp64_peak = 33.55        # TFLOP/s, tools/fp64_peak.cu DFMA probe (profiles/r1_fp64_peak.jsonl)
    res['codes'] = dict(ms=ms, messages_per_sec=N * sched.n_edges / (ms * 1e-3), bytes_per_site=b_site,
                        hbm_gbs=N * b_site / (ms * 1e-3) / 1e9, hbm_frac=N * b_site / (ms * 1e-3) / 1e9 / peaks['hbm_gbs'],
                        bound='fp64 pipe / issue slots', fp64_flop_per_site=flop_site,
                        fp64_tflops=N * flop_site / (ms * 1e-3) / 1e12,
                        fp64_frac=N * flop_site / (ms * 1e-3) / 1e12 / fp64_peak,
                        ncu='issue slots 60 %, fp64 pipe 24 % (profiles/r2_ncu_full_summary.json)')
    # dense emission likelihoods (obs type z): [n_leaves, S, N] fp64 = 1 KiB / site
    codes = obs.data.long()
    lik = torch.zeros((len(sched.leaves), S, N), dtype=torch.float64, device=dev)
    miss = codes == 255
    lik.scatter_(1, codes.clamp(max=S - 1).unsqueeze(1), 1.0)
    lik[miss.unsqueeze(1).expand(-1, S, -1)] = 1.0
    dobs = engine.Observations(engine.OBS_DENSE, lik, obs.obs_slot, N)
    ms = time_it(dobs)
    b_site = len(sched.leaves) * S * 8 + 9
    res['dense_emissions'] = dict(ms=ms, messages_per_sec=N * sched.n_edges / (ms * 1e-3), bytes_per_site=b_site,
                                  hbm_gbs=N * b_site / (ms * 1e-3) / 1e9,
                                  hbm_frac=N * b_site / (ms * 1e-3) / 1e9 / peaks['hbm_gbs'])
    return res


def bench_c3(dev, args):
    """C3: 61-state codon model, 128-leaf tree, 1e5 sites, log-likelihood (DMMA)."""
    import torch
    from raoteh_b200 import engine, synth
    from raoteh_b200.lowering import TreeSchedule
    cfg = synth.config_c3(n_sites=100_000)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    mjp = engine.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'], device=dev)
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'], device=dev)
    N = obs.n_sites
    ll = torch.empty(N, dtype=torch.float64, device=dev)
    st = torch.empty(N, dtype=torch.int8, device=dev)
    mjp.transition_matrices()
    for _ in range(3):
        mjp.log_likelihood(obs, out=(ll, st))
    torch.cuda.synchronize()
    ts = []
    for _ in range(args.steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        mjp.log_likelihood(obs, out=(ll, st))
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ms = float(np.mean(ts))
    E = sched.n_edges
    n_int_edges = int((~sched.is_leaf[1:]).sum())
    flops_nominal = N * E * 7503.0
    flops_dmma = N * n_int_edges * 2.0 * 64 * 64
    peak = fp64_peak()
    # expm alone
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    mjp._P_valid = False
    a.record()
    mjp.transition_matrices()
    b.record()
    torch.cuda.synchronize()
    # expectations at the same size: up pass with stored partials + level-synchronous DMMA down pass
    # (three contractions per internal edge; a leaf edge with hard codes is a column sum of the parent
    # marginals segmented by the code -- down_leaf_scatter_kernel, HBM-bound, no DMMA)
    exp = {}
    try:
        mjp.events = {}
        for _ in range(2):
            mjp.expected_history_statistics(obs)
        torch.cuda.synchronize()
        mjp.events = sub = {}
        te = []
        for _ in range(3):
            a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a2.record()
            mjp.expected_history_statistics(obs)
            b2.record()
            torch.cuda.synchronize()
            te.append(a2.elapsed_time(b2))
        pair = lambda L: [(L[i], L[i + 1]) for i in range(0, len(L) - 1, 2)]
        up_ms = float(np.mean([x.elapsed_time(y) for x, y in pair(sub['up'])]))
        down_ms = float(np.mean([x.elapsed_time(y) for x, y in pair(sub['down'])]))
        n_leaf_edges = E - n_int_edges
        flops_down = N * 3.0 * n_int_edges * 2.0 * 64 * 64
        # the floor of the whole evaluation on the FP64 tensor pipe: 1 (up) + 3 (down) padded 64 x 64
        # contractions per internal edge and site at the measured DMMA peak
        floor_ms = N * 4.0 * n_int_edges * 2.0 * 64 * 64 / (peak * 1e12) * 1e3
        exp = dict(expectations_ms=float(np.mean(te)), up_store_ms=up_ms, down_ms=down_ms,
                   down_tflops_executed_on_tensor_pipe=flops_down / (down_ms * 1e-3) / 1e12,
                   down_frac_executed=flops_down / (down_ms * 1e-3) / 1e12 / peak,
                   leaf_edges_bytes=float(N) * n_leaf_edges * 61 * 8,
                   tensor_pipe_floor_ms=floor_ms,
                   frac_of_tensor_pipe_floor=floor_ms / float(np.mean(te)))
        mjp.events = None
        # the same evaluation with the spectral scheme for this time-reversible model: P(t) and the
        # Frechet contraction in the eigenbasis (host eigh once per rate matrix, batched products)
        mjp.use_spectral(cfg['pi'])
        for _ in range(2):
            mjp._P_valid = False
            mjp.expected_history_statistics(obs)
        ts = []
        for _ in range(3):
            a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            mjp._P_valid = False
            a2.record()
            mjp.expected_history_statistics(obs)
            b2.record()
            torch.cuda.synchronize()
            ts.append(a2.elapsed_time(b2))
        exp['expectations_ms_spectral_scheme'] = float(np.mean(ts))
        mjp.use_spectral(None)
    except Exception as e:  # pragma: no cover
        exp = dict(expectations_error=repr(e))
    flops_useful = N * n_int_edges * (2.0 * 61 * 61 + 61)      # S = 61, internal edges only
    return dict(workload='C3: 61-state MG94 codon MJP, 128-leaf tree, 1e5 sites, log-lik',
                expectations=exp,
                # headline C3 fraction: USEFUL flops (S = 61 not the padded 64; internal edges only --
                # a leaf message with a hard code is a column gather, not a mat-vec) over the measured
                # DMMA peak; frac_executed counts the padded 64 x 64 contractions the pipe really ran,
                # frac_nominal SURVEY 8(d)'s 2S^2+S per message on EVERY edge
                tflops_useful=flops_useful / (ms * 1e-3) / 1e12,
                frac_useful=flops_useful / (ms * 1e-3) / 1e12 / peak,
                ms=ms, messages_per_sec=N * E / (ms * 1e-3),
                tflops_nominal=flops_nominal / (ms * 1e-3) / 1e12,
                tflops_executed_on_tensor_pipe=flops_dmma / (ms * 1e-3) / 1e12,
                fp64_tensor_peak_tflops=peak,
                frac_nominal=flops_nominal / (ms * 1e-3) / 1e12 / peak,
                frac_executed=flops_dmma / (ms * 1e-3) / 1e12 / peak,
                expm_ms=a.elapsed_time(b), finite=bool(torch.isfinite(ll).all()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-extra', action='store_true')
    ap.add_argument('--no-samplers', action='store_true')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='strong: also time 1e6 C2 sites IN TOTAL split over the ranks (always done for N > 1)')
    ap.add_argument('--c4-chains', type=int, default=4096)
    ap.add_argument('--c4-sweeps', type=int, default=100)
    ap.add_argument('--c5-sites', type=int, default=1_000_000)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the arrays the timed C2 step returned in its last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs:
        if args.impl != 'b200':
            ap.error('--dump-outputs needs --impl b200')
        os.makedirs(args.dump_outputs, exist_ok=True)
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference':
        return run_reference(args)
    return run_gpu(args)


if __name__ == '__main__':
    sys.exit(main())
