"""ctypes binding of librt_b200.so (include/rt_b200.h).

There is no CPU fallback: if the library is missing or a call fails, the
product raises.  Building is explicit (`python -m raoteh_b200._build` or
`__graft_entry__.build()`); importing never compiles.
"""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'librt_b200.so')

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_int64 = ctypes.c_int64

EXPORTS = {
    'rt_version': ([], c_int),
    'rt_release_workspace': ([], c_int),
    'rt_last_error_string': ([], ctypes.c_char_p),
    'rt_expm_batched': ([c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p], c_int),
    'rt_frechet_contract': ([c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p,
                             c_void_p], c_int),
    'rt_expm_spectral': ([c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p,
                          c_void_p], c_int),
    'rt_lb_transition': ([c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p], c_int),
    'rt_history_statistics': ([c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                               c_void_p, c_void_p, c_void_p], c_int),
    'rt_support_sets': ([c_int, c_int, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                         c_void_p], c_int),
    'rt_joint_distn': ([c_int, c_int, c_int64, c_int64, c_void_p, c_int, c_void_p, c_int, c_void_p,
                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p], c_int),
    'rt_prune_loglik': ([c_int, c_int, c_int64, c_int64, c_void_p, c_int, c_int, c_void_p,
                         c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                         c_void_p, c_void_p], c_int),
    'rt_posterior_stats': ([c_int, c_int, c_int64, c_int64, c_void_p, c_int, c_int,
                            c_void_p, c_void_p, c_int, c_void_p,
                            c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                            c_void_p, c_void_p], c_int),
    'rt_posterior_weighted_stats': ([c_int, c_int, c_int64, c_int64, c_void_p, c_int, c_int,
                                     c_void_p, c_void_p, c_int, c_void_p,
                                     c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p], c_int),
    'rt_posterior_branch_stats': ([c_int, c_int, c_int64, c_int64, c_void_p, c_int, c_int,
                                   c_void_p, c_void_p, c_int, c_void_p,
                                   c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p], c_int),
    'rt_copy2d_async': ([c_void_p, ctypes.c_size_t, c_void_p, ctypes.c_size_t, ctypes.c_size_t,
                         ctypes.c_size_t, c_int, c_void_p], c_int),
    'rt_raoteh_sweeps': ([c_int, c_int, c_int64, c_int64, c_int64, c_int64, c_void_p, c_int, c_int,
                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64,
                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, ctypes.c_uint64,
                          c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p], c_int),
}


class RaotehArgs(ctypes.Structure):
    """Mirror of `rt_raoteh_args` (include/rt_b200.h)."""
    _fields_ = [
        ('S', ctypes.c_int32), ('n_nodes', ctypes.c_int32), ('n_ops', ctypes.c_int32),
        ('n_slots', ctypes.c_int32), ('obs_kind', ctypes.c_int32), ('cap', ctypes.c_int32),
        ('n_sweeps', ctypes.c_int32), ('init_k', ctypes.c_int32),
        ('time_f64', ctypes.c_int32), ('reserved', ctypes.c_int32),
        ('n_traj', c_int64), ('traj_stride', c_int64), ('n_sites', c_int64), ('traj0', c_int64),
        ('obs_stride', c_int64), ('sweep0', c_int64),
        ('seed', ctypes.c_uint64),
        ('program', c_void_p), ('parent', c_void_p), ('length', c_void_p), ('B', c_void_p),
        ('rate', c_void_p), ('root_distn', c_void_p), ('obs', c_void_p),
        ('node_state', c_void_p), ('ev_time', c_void_p), ('ev_sb', c_void_p),
        ('ev_count', c_void_p), ('ev_total', c_void_p), ('sweep_count', c_void_p),
        ('dwell_sum', c_void_p), ('trans_sum', c_void_p), ('status', c_void_p),
    ]


EXPORTS['rt_raoteh_run'] = ([ctypes.POINTER(RaotehArgs), c_void_p], c_int)


class TmjpArgs(ctypes.Structure):
    """Mirror of `rt_tmjp_args` (include/rt_b200.h)."""
    _fields_ = [
        ('S', ctypes.c_int32), ('n_parts', ctypes.c_int32), ('n_nodes', ctypes.c_int32),
        ('n_ops', ctypes.c_int32), ('n_slots', ctypes.c_int32),
        ('cap_p', ctypes.c_int32), ('cap_t', ctypes.c_int32), ('obs_kind', ctypes.c_int32),
        ('program', c_void_p), ('parent', c_void_p), ('length', c_void_p),
        ('B', c_void_p), ('rate_p', c_void_p), ('pi_p', c_void_p),
        ('part', c_void_p), ('absorb', c_void_p),
        ('rate_on', ctypes.c_double), ('rate_off', ctypes.c_double), ('omega_t', ctypes.c_double),
        ('omega_p', ctypes.c_double),
        ('obs', c_void_p), ('obs_stride', c_int64),
        ('tol_obs', c_void_p), ('tol_obs_slot', c_void_p), ('tol_obs_stride', c_int64),
        ('n_traj', c_int64), ('n_sites', c_int64), ('traj0', c_int64),
        ('p_node', c_void_p), ('p_cnt', c_void_p),
        ('pn_traj_stride', c_int64), ('pn_node_stride', c_int64),
        ('p_total', c_void_p), ('p_time', c_void_p), ('p_sb', c_void_p),
        ('t_node', c_void_p), ('t_cnt', c_void_p), ('t_total', c_void_p), ('t_time', c_void_p),
        ('status', c_void_p),
        ('seed', ctypes.c_uint64), ('sweep0', c_int64),
        ('n_sweeps', ctypes.c_int32), ('mode', ctypes.c_int32), ('init_k', ctypes.c_int32),
        ('flags', ctypes.c_int32),
        ('prim_dwell', c_void_p), ('prim_trans', c_void_p), ('tol_stats', c_void_p),
        ('summary_sum', c_void_p), ('summary_out', c_void_p), ('traj_loglik', c_void_p), ('p_time64', c_void_p),
    ]


EXPORTS['rt_tmjp_run'] = ([ctypes.POINTER(TmjpArgs), c_void_p], c_int)


class PosteriorDrawArgs(ctypes.Structure):
    """Mirror of `rt_posterior_draw_args` (include/rt_b200.h)."""
    _fields_ = [
        ('S', ctypes.c_int32), ('n_nodes', ctypes.c_int32), ('n_ops', ctypes.c_int32),
        ('cap', ctypes.c_int32), ('obs_kind', ctypes.c_int32), ('time_f64', ctypes.c_int32),
        ('n_traj', c_int64), ('traj_stride', c_int64), ('n_sites', c_int64), ('traj0', c_int64),
        ('obs_stride', c_int64), ('site_stride', c_int64),
        ('seed', ctypes.c_uint64), ('k', c_int64),
        ('program', c_void_p), ('parent', c_void_p), ('length', c_void_p), ('Q', c_void_p),
        ('P', c_void_p), ('root_distn', c_void_p), ('obs', c_void_p), ('partials', c_void_p),
        ('site_status', c_void_p),
        ('node_state', c_void_p), ('ev_time', c_void_p), ('ev_sb', c_void_p),
        ('ev_count', c_void_p), ('ev_total', c_void_p), ('sweep_count', c_void_p),
        ('dwell_sum', c_void_p), ('trans_sum', c_void_p), ('status', c_void_p),
    ]


EXPORTS['rt_posterior_draw'] = ([ctypes.POINTER(PosteriorDrawArgs), c_void_p], c_int)


class PosteriorDrawMixtureArgs(ctypes.Structure):
    """Mirror of `rt_posterior_draw_mixture_args` (include/rt_b200.h)."""
    _fields_ = [
        ('base', PosteriorDrawArgs),
        ('K', ctypes.c_int32), ('reserved', ctypes.c_int32),
        ('partials_class_stride', c_int64), ('class_post_stride', c_int64),
        ('class_post', c_void_p), ('site_class', c_void_p),
    ]


EXPORTS['rt_posterior_draw_mixture'] = ([ctypes.POINTER(PosteriorDrawMixtureArgs), c_void_p], c_int)

SIM_NODES, SIM_HISTORY = 0, 1


class ForwardArgs(ctypes.Structure):
    """Mirror of `rt_forward_args` (include/rt_b200.h)."""
    _fields_ = [
        ('S', ctypes.c_int32), ('n_nodes', ctypes.c_int32), ('n_ops', ctypes.c_int32),
        ('K', ctypes.c_int32), ('mode', ctypes.c_int32), ('cap', ctypes.c_int32),
        ('time_f64', ctypes.c_int32), ('reserved', ctypes.c_int32),
        ('n_traj', c_int64), ('traj_stride', c_int64), ('traj0', c_int64), ('obs_stride', c_int64),
        ('tmpl_stride', c_int64), ('tmpl_n_sites', c_int64),
        ('seed', ctypes.c_uint64), ('k', c_int64),
        ('program', c_void_p), ('parent', c_void_p), ('length', c_void_p), ('obs_slot', c_void_p),
        ('class_weight', c_void_p), ('Q', c_void_p), ('P', c_void_p), ('root_distn', c_void_p),
        ('tmpl', c_void_p), ('obs', c_void_p), ('site_class', c_void_p), ('node_state', c_void_p),
        ('ev_time', c_void_p), ('ev_sb', c_void_p), ('ev_count', c_void_p), ('ev_total', c_void_p),
        ('dwell_sum', c_void_p), ('trans_sum', c_void_p), ('status', c_void_p),
    ]


EXPORTS['rt_forward_simulate'] = ([ctypes.POINTER(ForwardArgs), c_void_p], c_int)


class NativeError(RuntimeError):
    pass


_lib = None


def lib():
    """Load librt_b200.so once; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                'librt_b200.so not found at %s -- build it with '
                '`python -m raoteh_b200._build` (needs nvcc); there is no CPU fallback'
                % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, sig in EXPORTS.items():
            if sig is None:
                continue
            fn = getattr(L, name)
            fn.argtypes, fn.restype = sig
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().rt_last_error_string()
        raise NativeError('%s failed with code %d: %s'
                          % (what, rc, msg.decode() if msg else ''))


def declared_symbols():
    """Symbols include/rt_b200.h declares (parsed, for the export test)."""
    import re
    hdr = os.path.join(HERE, '..', 'include', 'rt_b200.h')
    text = open(hdr).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(rt_[a-z0-9_]+)\s*\(', text)))
