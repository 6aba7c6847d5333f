"""Tensor-level wrapper of the RL loss kernel (`vpt_rl_heads_bwd`, csrc/rl_heads.cuh), re-exported as `ops.rl_heads_bwd`.

It lives in its own module because its CPU emulation does too: tests/test_rl_training.py carries it and patches it into `ops`
in that module's fixture, next to the emulation of the other ops in tests/emu_ops.py."""
import ctypes as C

import torch

from . import _native as nat
from . import ops
from .ops import F32, _cuda, _p, _stream


def rl_heads_bwd(logp, logp_teacher, idx, cols, old_logp, adv, ret, vpred, mu_rsig, clip_eps, kl_coef, ent_coef, vf_coef, inv_temp, inv_n,
                 dlog, col_v):
    """Per head h: logp[h] fp32 [rows, n_h] (student log-softmax), logp_teacher[h] the teacher's (logp_teacher None: no KL term),
    idx[h] int64 [rows] (taken action), cols[h] its first column in dlog.  old_logp, adv, ret, vpred: fp32 [rows]; mu_rsig: fp32 [2]
    on the device, (mean, 1/std) of the return normaliser.  Writes the bf16 gradient wrt the head GEMM outputs into dlog (columns
    cols[h] + [0, n_h) and col_v); returns the fp32 per-row statistics [rows, 5] = (lp, kl, entropy, (vpred - tn)^2, clipped)."""
    nh = len(logp)
    rows = logp[0].shape[0]
    heads = list(logp) + list(idx) + ([] if logp_teacher is None else list(logp_teacher))
    _cuda(*heads, old_logp, adv, ret, vpred, mu_rsig, dlog)
    for t in heads:
        assert t.is_contiguous() and t.shape[0] == rows
    assert all(t.dtype == torch.int64 for t in idx) and all(t.dtype == F32 for t in logp)
    for t in (old_logp, adv, ret, vpred):
        assert t.dtype == F32 and t.is_contiguous() and t.numel() == rows
    assert mu_rsig.dtype == F32 and mu_rsig.numel() == 2 and dlog.stride(1) == 1
    stats = torch.empty((rows, 5), dtype=F32, device=dlog.device)
    P = C.c_void_p * nh
    lp_arr = P(*[_p(t) for t in logp])
    lt_arr = None if logp_teacher is None else P(*[_p(t) for t in logp_teacher])
    idx_arr = P(*[_p(t) for t in idx])
    n_arr = (C.c_int32 * nh)(*[t.shape[1] for t in logp])
    c_arr = (C.c_int32 * nh)(*[int(c) for c in cols])
    nat.check(nat.lib().vpt_rl_heads_bwd(lp_arr, lt_arr, idx_arr, n_arr, c_arr, nh, _p(old_logp), _p(adv), _p(ret), _p(vpred), _p(mu_rsig),
                                         float(clip_eps), float(kl_coef), float(ent_coef), float(vf_coef), float(inv_temp), float(inv_n),
                                         _p(dlog), dlog.stride(0), int(col_v), _p(stats), rows, _stream()), "vpt_rl_heads_bwd")
    ops._count()
    return stats
