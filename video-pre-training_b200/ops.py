"""Tensor-level wrappers of the C ABI: torch tensors in, torch tensors out, everything enqueued on torch's current
CUDA stream.  torch is used for device memory and streams only -- all arithmetic happens in libvpt_b200.so."""
import ctypes as C

import torch

from . import _native as nat

BF16, F32 = torch.bfloat16, torch.float32


LAUNCHES = 0        # kernels launched through this module since import (bench.py reports the per-step delta)
GEMM_PROFILE = None  # set to a list to record (start_event, end_event, flops, tag) around every GEMM/conv launch


def _count(n=1):
    global LAUNCHES
    LAUNCHES += n


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t):
    if not t.is_cuda:
        raise nat.NativeError("vpt_b200 runs on CUDA (sm_100a) only; there is no CPU fallback")


def _cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise nat.NativeError("vpt_b200 ops need CUDA tensors (there is no CPU fallback)")


def gemm(A, Bw, out, M, N, K, *, conv=None, mr=None, rows_per_group=1, S1=None, S2=None, relu=0, out_scale=1.0,
         residual=None, ld_out=None, seg=None, stat_part=None, stat_mode=0, cluster=0, dsts=None):
    """out = epilogue(A @ Bw^T); see struct vpt_gemm_args.  dsts: up to 4 column segments [(n0, tensor, ld, remap)] with their own
    destination buffer (then `out` is only used for its device / may be the first segment's tensor)."""
    _cuda(A, Bw, out)
    a = nat.GemmArgs()
    a.A, a.B, a.M, a.N, a.K = _p(A), _p(Bw), M, N, K
    if conv is not None:
        a.conv, (a.H, a.W, a.Cin) = 1, conv
    a.mr, a.rows_per_group, a.S1, a.S2 = _p(mr), rows_per_group, _p(S1), _p(S2)
    a.relu, a.out_scale = relu, out_scale
    if residual is not None:
        a.residual, a.residual_f32, a.ld_res = _p(residual), int(residual.dtype == F32), residual.stride(-2)
    a.out, a.out_f32 = _p(out), int(out.dtype == F32)
    a.ld_out = ld_out if ld_out is not None else out.stride(-2)
    if seg is not None:
        a.seg_len, a.seg_stride, a.seg_off = seg
    a.stat_part, a.stat_mode, a.cluster = _p(stat_part), stat_mode, cluster
    if dsts:
        a.ndst = len(dsts)
        for i, (n0, t, ld, remap) in enumerate(dsts):
            _cuda(t)
            a.dst_n0[i], a.dst_out[i], a.dst_ld[i], a.dst_f32[i], a.dst_remap[i] = n0, _p(t), ld, int(t.dtype == F32), int(remap)
    prof = GEMM_PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    nat.check(nat.lib().vpt_gemm_bf16(C.byref(a), _stream()), "vpt_gemm_bf16")
    if prof is not None:
        e1.record()
        prof.append((e0, e1, 2.0 * M * N * K, "conv" if conv is not None else "linear", (M, N, K)))
    _count()
    return out


def set_default_cluster(cs):
    nat.check(nat.lib().vpt_set_default_cluster(cs), "vpt_set_default_cluster")


def gemm_stat_parts(N):
    return nat.lib().vpt_gemm_stat_parts(N)


def stats_finalize(part, G, n_per_group, count, eps=1e-5):
    mr = torch.empty((G, 2), dtype=F32, device=part.device)
    nat.check(nat.lib().vpt_stats_finalize(_p(part), _p(mr), G, n_per_group, float(count), eps, _stream()), "vpt_stats_finalize")
    _count()
    return mr


def conv3x3_zp(x, Wb, H, W, *, mr=None, S1=None, S2=None, relu=1, residual=None, want_stats=True, out=None, Ef=None, res_scale=None,
               res_shift=None):
    """GroupNorm(1)->conv3x3->ReLU[+residual] on a ZP tensor x bf16 [F,H+1,W+1,Cin]; returns (ZP out, per-frame (mean, rstd))."""
    _cuda(x, Wb)
    F_, Cin = x.shape[0], x.shape[3]
    Cout = Wb.shape[0]
    assert tuple(x.shape[1:3]) == (H + 1, W + 1) and Wb.shape[1] == 9 * Cin
    if out is None:
        out = torch.empty((F_, H + 1, W + 1, Cout), dtype=BF16, device=x.device)
    assert out.is_contiguous() and tuple(out.shape) == (F_, H + 1, W + 1, Cout)
    P = nat.lib().vpt_conv_zp_stat_parts(F_, H, W, Cout)
    tfl = nat.lib().vpt_conv_zp_t_stat_floats(F_, H, W, Cout)  # > 0: the swapped kernel's fragment epilogue (per-tile partials)
    part = None
    if want_stats:
        part = torch.empty((tfl,) if tfl > 0 else (F_ * (H + 1) * (W + 1), P, 2), dtype=F32, device=x.device)
    a = nat.ConvZpArgs()
    a.x, a.w, a.F, a.H, a.W, a.Cin, a.Cout = _p(x), _p(Wb), F_, H, W, Cin, Cout
    a.mr, a.S1, a.S2, a.relu, a.residual, a.out, a.stat_part = _p(mr), _p(S1), _p(S2), relu, _p(residual), _p(out), _p(part)
    a.Ef, a.res_scale, a.res_shift = _p(Ef), _p(res_scale), _p(res_shift)  # two-norm composition (vpt_norm2_fold)
    prof = GEMM_PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    nat.check(nat.lib().vpt_conv3x3_zp(C.byref(a), _stream()), "vpt_conv3x3_zp")
    if prof is not None:
        e1.record()
        prof.append((e0, e1, 2.0 * F_ * H * W * Cout * 9 * Cin, "conv", (F_ * H * W, Cout, 9 * Cin)))  # algorithmic FLOPs (no halo rows)
    _count()
    mr_out = None
    if want_stats and tfl > 0:
        mr_out = torch.empty((F_, 2), dtype=F32, device=x.device)
        nat.check(nat.lib().vpt_conv_zp_t_stats_finalize(_p(part), _p(mr_out), F_, H, W, 1e-5, _stream()), "vpt_conv_zp_t_stats_finalize")
        _count()
    elif want_stats:
        mr_out = stats_finalize(part, F_, (H + 1) * (W + 1) * P, H * W * Cout)
    return out, mr_out


def firstconv_pool(img, w, bias, C0, zp=True, out_f32=False, want_chan=False):
    """img u8 [F,H,W,3] -> (bf16 (fp32 with out_f32) [F,H/2(+1),W/2(+1),C0] (ZP layout when zp), per-frame (mean, rstd)).
    want_chan: also return the per-channel (sum, sumsq) partials [F, NP, C0, 2] of the pooled tensor (None if the kernel that ran does
    not produce them), for `norm2_fold`."""
    _cuda(img, w, bias)
    F_, H, W, _ = img.shape
    z = int(zp)
    out = torch.empty((F_, H // 2 + z, W // 2 + z, C0), dtype=F32 if out_f32 else BF16, device=img.device)
    P = nat.lib().vpt_firstconv_stat_parts(F_, H, W, C0)
    part = torch.empty((F_, P, 2), dtype=F32, device=img.device)
    nat.check(nat.lib().vpt_firstconv_pool(_p(img), _p(w), _p(bias), _p(out), _p(part), F_, H, W, C0, z, int(out_f32), _stream()), "vpt_firstconv_pool")
    _count()
    mr = stats_finalize(part, F_, P, (H // 2) * (W // 2) * C0)
    if want_chan:  # the tcgen05 kernel's partials are per (8 pooled rows, column half, channel)
        return out, mr, (part.view(F_, P // C0, C0, 2) if P % C0 == 0 and P >= C0 else None)
    return out, mr


def conv3d_t5(img, w, bias, C, out_f32=False):
    """img u8 [B,T,H,W,3] -> (bf16 (fp32 with out_f32) ZP [B*T,H+1,W+1,C], per-frame (mean, rstd)); lib/policy.py:394-403."""
    _cuda(img, w, bias)
    B, T, H, W, _ = img.shape
    out = torch.empty((B * T, H + 1, W + 1, C), dtype=F32 if out_f32 else BF16, device=img.device)
    P = nat.lib().vpt_conv3d_stat_parts(H, W, C)
    part = torch.empty((B * T, P, 2), dtype=F32, device=img.device)
    nat.check(nat.lib().vpt_conv3d_t5(_p(img), _p(w), _p(bias), _p(out), _p(part), B, T, H, W, C, int(out_f32), _stream()), "vpt_conv3d_t5")
    _count()
    return out, stats_finalize(part, B * T, P, H * W * C)


# ---- fp32-parity precision mode (csrc/precise.cuh) ----------------------------------------------------------------------
def group_stats_f32(x, groups, eps=1e-5):
    """(mean, rstd) [groups, 2] over equal consecutive slices of the fp32 tensor x."""
    _cuda(x)
    assert x.dtype == F32 and x.is_contiguous() and x.numel() % groups == 0
    mr = torch.empty((groups, 2), dtype=F32, device=x.device)
    nat.check(nat.lib().vpt_group_stats_f32(_p(x), _p(mr), groups, x.numel() // groups, eps, _stream()), "vpt_group_stats_f32")
    _count()
    return mr


def norm_split_f32(x, mr=None, gamma=None, beta=None, groups=1, split=True, want_f32=False):
    """u = [(x - mean_g) rstd_g] gamma[c] + beta[c] on fp32 x [..., C] -> (hi bf16, lo bf16, u fp32) (None where not requested)."""
    _cuda(x, mr, gamma, beta)
    assert x.dtype == F32 and x.is_contiguous()
    C = x.shape[-1]
    hi = torch.empty(x.shape, dtype=BF16, device=x.device) if split else None
    lo = torch.empty(x.shape, dtype=BF16, device=x.device) if split else None
    u = torch.empty_like(x) if want_f32 else None
    nat.check(nat.lib().vpt_norm_split_f32(_p(x), _p(mr), _p(gamma), _p(beta), _p(hi), _p(lo), _p(u), x.numel(), C, x.numel() // groups, _stream()),
              "vpt_norm_split_f32")
    _count()
    return hi, lo, u


def add_f32(a, b=None, relu=False, out=None):
    _cuda(a, b)
    assert a.dtype == F32 and a.is_contiguous() and (b is None or (b.dtype == F32 and b.is_contiguous() and b.shape == a.shape))
    if out is None:
        out = torch.empty_like(a)
    nat.check(nat.lib().vpt_add_f32(_p(a), _p(b), _p(out), a.numel(), int(relu), _stream()), "vpt_add_f32")
    _count()
    return out


def maxpool3s2_f32(x):
    """fp32 NHWC [F,H,W,C] -> [F,H/2,W/2,C] (max_pool2d(3, 2, 1))."""
    _cuda(x)
    assert x.dtype == F32 and x.is_contiguous()
    F_, H, W, Cc = x.shape
    out = torch.empty((F_, H // 2, W // 2, Cc), dtype=F32, device=x.device)
    nat.check(nat.lib().vpt_maxpool3s2_f32(_p(x), _p(out), F_, H, W, Cc, _stream()), "vpt_maxpool3s2_f32")
    _count()
    return out


def attention_f32(q, full_k, full_v, R, b_nd, first_u8, smask_u8, B, t, maxlen, heads, causal=True):
    _cuda(q, full_k, full_v)
    out = torch.empty_like(q)
    nat.check(nat.lib().vpt_attention_f32(_p(q), _p(full_k), _p(full_v), _p(R), _p(b_nd), _p(first_u8), _p(smask_u8), _p(out), B, t, maxlen, heads,
                                          int(causal), _stream()), "vpt_attention_f32")
    _count()
    return out


def maxpool3s2(x, zp=True, want_chan=False):
    """bf16 [F,H,W,C] (>= 0) -> (bf16 [F,H/2,W/2,C], per-frame (mean, rstd)); with zp both tensors are ZP ([F,H+1,W+1,C]).
    want_chan: also the per-channel (sum, sumsq) partials [F, NP, C, 2] of the pooled tensor (None when C/8 does not divide 256)."""
    _cuda(x)
    z = int(zp)
    F_, H, W, Cc = x.shape[0], x.shape[1] - z, x.shape[2] - z, x.shape[3]
    out = torch.empty((F_, H // 2 + z, W // 2 + z, Cc), dtype=BF16, device=x.device)
    with_chan = want_chan and Cc >= 8 and 256 % (Cc // 8) == 0
    P = nat.lib().vpt_pool_chan_parts(F_, H, W, Cc) if with_chan else nat.lib().vpt_pool_stat_parts(F_, H, W, Cc)
    part = torch.empty((F_, P, 2), dtype=F32, device=x.device)
    chan = torch.empty((F_, P, Cc, 2), dtype=F32, device=x.device) if with_chan else None
    nat.check(nat.lib().vpt_maxpool3s2(_p(x), _p(out), _p(part), _p(chan), F_, H, W, Cc, z, _stream()), "vpt_maxpool3s2")
    _count()
    mr = stats_finalize(part, F_, P, (H // 2) * (W // 2) * Cc)
    return (out, mr, chan) if want_chan else (out, mr)


def norm2_fold(chan_part, npix, gamma_n, beta_n, tabs):
    """Two-norm composition tables (vpt_norm2_fold): chan_part fp32 [F, NP, C, 2]; tabs = (Ta, Tb, Tc, Td) each fp32 [9, Cout] ->
    (mrE [F, 2], Ef [F, 9, Cout], res_scale [F, C], res_shift [F, C])."""
    _cuda(chan_part, gamma_n, beta_n, *tabs)
    F_, NP, Cc, _ = chan_part.shape
    Cout = tabs[0].shape[1]
    dev = chan_part.device
    mrE = torch.empty((F_, 2), dtype=F32, device=dev)
    Ef = torch.empty((F_, 9, Cout), dtype=F32, device=dev)
    rs = torch.empty((F_, Cc), dtype=F32, device=dev)
    rb = torch.empty((F_, Cc), dtype=F32, device=dev)
    nat.check(nat.lib().vpt_norm2_fold(_p(chan_part), NP, Cc, npix, _p(gamma_n), _p(beta_n), _p(tabs[0]), _p(tabs[1]), _p(tabs[2]), _p(tabs[3]), Cout, 1e-5,
                                       _p(mrE), _p(Ef), _p(rs), _p(rb), F_, _stream()), "vpt_norm2_fold")
    _count()
    return mrE, Ef, rs, rb


def affine_norm(x, mr, gamma, beta, rows_per_group, want_stats=False, want_f32=False):
    """(x - mean_g) * rstd_g * gamma + beta on [M, C] rows; returns (bf16 out, fp32 out | None, (mean, rstd) of out | None)."""
    _cuda(x, mr, gamma, beta)
    Cc = x.shape[-1]
    M = x.numel() // Cc
    out = torch.empty_like(x)
    out32 = torch.empty(x.shape, dtype=F32, device=x.device) if want_f32 else None
    part, P = None, 0
    G = M // rows_per_group
    if want_stats:
        P = nat.lib().vpt_norm_stat_parts(rows_per_group, Cc)
        part = torch.empty((G, P, 2), dtype=F32, device=x.device)
    nat.check(nat.lib().vpt_affine_norm(_p(x), _p(mr), _p(gamma), _p(beta), _p(out), _p(out32), _p(part), M, Cc, rows_per_group,
                                        _stream()), "vpt_affine_norm")
    _count()
    mr_out = stats_finalize(part, G, P, rows_per_group * Cc) if want_stats else None
    return out, out32, mr_out


def affine_norm_zp(x, mr, gamma, beta):
    """GroupNorm(1) application on a ZP tensor [F,H+1,W+1,C] (one group per frame); returns (ZP out, (mean, rstd) of out)."""
    _cuda(x, mr, gamma, beta)
    F_, H, W, Cc = x.shape[0], x.shape[1] - 1, x.shape[2] - 1, x.shape[3]
    out = torch.empty_like(x)
    P = nat.lib().vpt_norm_stat_parts((H + 1) * (W + 1), Cc)
    part = torch.empty((F_, P, 2), dtype=F32, device=x.device)
    nat.check(nat.lib().vpt_affine_norm_zp(_p(x), _p(mr), _p(gamma), _p(beta), _p(out), _p(part), F_, H, W, Cc, _stream()), "vpt_affine_norm_zp")
    _count()
    return out, stats_finalize(part, F_, P, H * W * Cc)


def copy_rows(src, src_off, dst, dst_off, rows):
    """dst[:, dst_off:dst_off+rows, :] = src[:, src_off:src_off+rows, :] for [B, L, C] tensors (fp32 <-> bf16)."""
    _cuda(src, dst)
    if rows == 0:
        return
    B, _, Cc = src.shape
    nat.check(nat.lib().vpt_copy_rows(_p(src), int(src.dtype == F32), src.stride(0), src.stride(1), src_off, _p(dst),
                                      int(dst.dtype == F32), dst.stride(0), dst.stride(1), dst_off, B, rows, Cc, _stream()),
              "vpt_copy_rows")
    _count()


def copy_rows2(src_a, src_b, src_off, dst_a, dst_b, dst_off, rows):
    """copy_rows for two (source, destination) pairs of identical shape / strides / dtypes in ONE launch (K and V of a layer)."""
    _cuda(src_a, src_b, dst_a, dst_b)
    if rows == 0:
        return
    assert src_a.shape == src_b.shape and src_a.stride() == src_b.stride() and src_a.dtype == src_b.dtype
    assert dst_a.shape == dst_b.shape and dst_a.stride() == dst_b.stride() and dst_a.dtype == dst_b.dtype
    B, _, Cc = src_a.shape
    nat.check(nat.lib().vpt_copy_rows2(_p(src_a), _p(src_b), int(src_a.dtype == F32), src_a.stride(0), src_a.stride(1), src_off, _p(dst_a), _p(dst_b),
                                       int(dst_a.dtype == F32), dst_a.stride(0), dst_a.stride(1), dst_off, B, rows, Cc, _stream()), "vpt_copy_rows2")
    _count()


def state_mask_update(mask_in, first_u8, t, maxlen):
    """mask_in: bool (B,1,maxlen) or None; first_u8: u8 view of first (B,T); returns new bool (B,1,maxlen)."""
    B = first_u8.shape[0]
    out = torch.empty((B, 1, maxlen), dtype=torch.bool, device=first_u8.device)
    if maxlen > 0:
        nat.check(nat.lib().vpt_state_mask_update(_p(mask_in), _p(first_u8), first_u8.stride(0), _p(out), B, t, maxlen, _stream()),
                  "vpt_state_mask_update")
    _count()
    return out


def attention(Q, Kf, Vf, R, b_nd, first_u8, smask, B, t, maxlen, heads, causal=True):
    _cuda(Q, Kf, Vf)
    out = torch.empty_like(Q)
    nbasis = b_nd.shape[0] if (causal and b_nd is not None) else 0
    nat.check(nat.lib().vpt_attention(_p(Q), _p(Kf), _p(Vf), _p(R), R.stride(-2) if R is not None else 0, _p(b_nd),
                                      _p(first_u8), first_u8.stride(0) if first_u8 is not None else 0, _p(smask), _p(out), B, t,
                                      maxlen, heads, nbasis, int(causal), _stream()), "vpt_attention")
    _count()
    return out


def log_softmax(raw, col0, n):
    """raw fp32 [rows, ld] -> fp32 [rows, n] = log_softmax(raw[:, col0:col0+n])."""
    rows = raw.shape[0]
    out = torch.empty((rows, n), dtype=F32, device=raw.device)
    nat.check(nat.lib().vpt_log_softmax(_p(raw), raw.stride(0), col0, n, _p(out), rows, _stream()), "vpt_log_softmax")
    _count()
    return out


def gumbel_argmax(logits, u=None):
    """logits fp32 [..., n] contiguous, u same shape or None -> int64 [...]."""
    _cuda(logits)
    logits = logits.contiguous()
    n = logits.shape[-1]
    rows = logits.numel() // n
    idx = torch.empty(logits.shape[:-1], dtype=torch.int64, device=logits.device)
    nat.check(nat.lib().vpt_gumbel_argmax(_p(logits), _p(u), _p(idx), rows, n, _stream()), "vpt_gumbel_argmax")
    _count()
    return idx


def gather_logprob(logits, idx, lp=None):
    logits = logits.contiguous()
    idx = idx.contiguous()
    n = logits.shape[-1]
    rows = logits.numel() // n
    acc = lp is not None
    if lp is None:
        lp = torch.empty(logits.shape[:-1], dtype=F32, device=logits.device)
    nat.check(nat.lib().vpt_gather_logprob(_p(logits), _p(idx), _p(lp), rows, n, int(acc), _stream()), "vpt_gather_logprob")
    _count()
    return lp


# ---------------------------------------------------------------------------------------------------------------------
# backward ops of the BC step (training.py; behavioural_cloning.py:101-123)
# ---------------------------------------------------------------------------------------------------------------------
def relu_mask(dout, out):
    """dz = dout where the ReLU was open (out > 0), else 0 (bf16, any shape)."""
    _cuda(dout, out)
    dz = torch.empty_like(dout)
    nat.check(nat.lib().vpt_relu_mask(_p(dout), _p(out), _p(dz), dout.numel(), _stream()), "vpt_relu_mask")
    _count()
    return dz


def add_zp(a, b, H, W, out=None):
    """ZP a + b -> (bf16 ZP sum, per-frame (mean, rstd) of the sum): the residual add of a training forward."""
    _cuda(a, b)
    F_, Cc = a.shape[0], a.shape[3]
    if out is None:
        out = torch.empty_like(a)
    per = (H + 1) * (W + 1) * Cc
    P = nat.lib().vpt_add_stat_parts(per)
    part = torch.empty((F_, P, 2), dtype=F32, device=a.device)
    nat.check(nat.lib().vpt_add_stats(_p(a), _p(b), _p(out), _p(part), F_, per, _stream()), "vpt_add_stats")
    _count()
    return out, stats_finalize(part, F_, P, H * W * Cc)


def wgrad(a, b, shifts=(0,), out=None):
    """fp32 out[m][tap*N + n] = sum_k a[k][m] * b[k + shifts[tap]][n]: a bf16 [R][M] = output gradient, b bf16 [R][N] = layer input
    (row strides allowed; rows outside [0, R) count as zero)."""
    _cuda(a, b)
    R, M = a.shape
    N = b.shape[1]
    assert b.shape[0] == R and a.stride(1) == 1 and b.stride(1) == 1
    nt = len(shifts)
    if out is None:
        out = torch.empty((M, nt * N), dtype=F32, device=a.device)
    ws_bytes = nat.lib().vpt_wgrad_workspace_bytes(M, N, nt, R)
    ws = torch.empty((max(ws_bytes, 4) // 4,), dtype=F32, device=a.device)
    sh = (C.c_int32 * nt)(*[int(s) for s in shifts])
    prof = GEMM_PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    nat.check(nat.lib().vpt_wgrad_bf16(_p(a), a.stride(0), _p(b), b.stride(0), M, N, R, sh, nt, _p(out), _p(ws), ws_bytes, _stream()),
              "vpt_wgrad_bf16")
    if prof is not None:
        e1.record()
        prof.append((e0, e1, 2.0 * M * N * nt * R, "wgrad", (M, nt * N, R)))
    _count(2)
    return out


def group_sums(du, x, mr, gamma, rows_per_group, count):
    """fp32 [G][2]: per statistics group (mean of gamma*du, mean of gamma*du*n), n = (x - mean) * rstd; du, x bf16 [rows][C]."""
    _cuda(du, x, mr, gamma)
    rows, Cc = x.shape
    G = rows // rows_per_group
    P = nat.lib().vpt_group_sums_parts(rows_per_group, Cc)
    part = torch.empty((G, P, 2), dtype=F32, device=x.device)
    ms = torch.empty((G, 2), dtype=F32, device=x.device)
    nat.check(nat.lib().vpt_group_sums(_p(du), _p(x), _p(mr), _p(gamma), _p(part), _p(ms), rows, Cc, rows_per_group, float(count),
                                       _stream()), "vpt_group_sums")
    _count(2)
    return ms


def col_sums(du, x=None, mr=None, rows_per_group=1):
    """fp32 [2][C]: (sum_rows du*n, sum_rows du); without x row 0 is zero.  du (and x) bf16 [rows][C] (row stride allowed)."""
    _cuda(du, x, mr)
    rows, Cc = du.shape
    out = torch.empty((2, Cc), dtype=F32, device=du.device)
    S = nat.lib().vpt_col_sums_parts(rows, Cc)
    ws = torch.empty((S, 2, Cc), dtype=F32, device=du.device)
    nat.check(nat.lib().vpt_col_sums(_p(du), du.stride(0), _p(x), _p(mr), rows, Cc, rows_per_group, _p(out), _p(ws), _stream()), "vpt_col_sums")
    _count(2)
    return out


def norm_sums(du, x, mr, gamma, rows_per_group, count):
    """(col_sums(du, x, mr), group_sums(du, x, mr, gamma)) in one pass over the data; for groups of many rows (GroupNorm frames)."""
    _cuda(du, x, mr, gamma)
    rows, Cc = x.shape
    G = rows // rows_per_group
    out = torch.empty((2, Cc), dtype=F32, device=x.device)
    ms = torch.empty((G, 2), dtype=F32, device=x.device)
    ws = torch.empty((nat.lib().vpt_norm_sums_workspace(rows, Cc, rows_per_group),), dtype=F32, device=x.device)
    nat.check(nat.lib().vpt_norm_sums(_p(du), _p(x), _p(mr), _p(gamma), rows, Cc, rows_per_group, float(count), _p(out), _p(ms), _p(ws), _stream()),
              "vpt_norm_sums")
    _count(3)
    return out, ms


def norm_bwd_apply(du, x, mr, gamma, ms, rows_per_group, zp=None, add=None, relu_x=False):
    """dx = rstd * (gamma*du - m1 - n*m2) [+ add] (bf16 [rows][C]); zp = (H, W, Cch): groups are ZP frames, pads written as 0;
    relu_x: x is a ReLU output and dx is zeroed where x == 0 (the producer's ReLU backward, fused)."""
    _cuda(du, x, mr, gamma, ms, add)
    rows, Cc = x.shape
    dx = torch.empty_like(x)
    H, W, Cch = zp if zp is not None else (0, 0, 0)
    nat.check(nat.lib().vpt_norm_bwd_apply(_p(du), _p(x), _p(mr), _p(gamma), _p(ms), _p(add), _p(dx), rows, Cc, rows_per_group, H, W, Cch,
                                           int(relu_x), _stream()), "vpt_norm_bwd_apply")
    _count()
    return dx


def maxpool3s2_bwd(dy, x):
    """Gradient of ReLU -> max_pool2d(3, 2, 1) on ZP tensors: dy [F,H/2+1,W/2+1,C], x (post-ReLU pool input) [F,H+1,W+1,C]."""
    _cuda(dy, x)
    F_, H, W, Cc = x.shape[0], x.shape[1] - 1, x.shape[2] - 1, x.shape[3]
    dx = torch.empty_like(x)
    ws = torch.empty((F_ * (H // 2) * (W // 2) * Cc,), dtype=torch.uint8, device=x.device)
    nat.check(nat.lib().vpt_maxpool3s2_bwd(_p(dy), _p(x), _p(dx), _p(ws), F_, H, W, Cc, _stream()), "vpt_maxpool3s2_bwd")
    _count(2)
    return dx


def firstconv_bwd(img, w, bias, dy, C0):
    """Weight / bias gradient of the fused first conv + ReLU + max-pool: (fp32 [C0][27] in (ky,kx,c) order, fp32 [C0])."""
    _cuda(img, w, bias, dy)
    F_, H, W, _ = img.shape
    S = nat.lib().vpt_firstconv_bwd_parts(F_, H, W)
    ws = torch.empty((S, C0, 28), dtype=F32, device=img.device)
    dW = torch.empty((C0, 27), dtype=F32, device=img.device)
    db = torch.empty((C0,), dtype=F32, device=img.device)
    nat.check(nat.lib().vpt_firstconv_bwd(_p(img), _p(w), _p(bias), _p(dy), _p(dW), _p(db), _p(ws), F_, H, W, C0, _stream()), "vpt_firstconv_bwd")
    _count(2)
    return dW, db


def attention_bwd(Q, Kf, Vf, R, b_nd, first_u8, smask, dO, out, B, t, maxlen, heads, causal=True):
    """Backward of `attention`: d q | d k | d v | d R written side by side into out[:, 0:h | h:2h | 2h:3h | 3h:3h+10*heads]
    (bf16, chunk rows only: the KV memory is detached state); returns d b_nd fp32 [nbasis][maxlen]."""
    _cuda(Q, Kf, Vf, R, b_nd, dO, out)
    if not causal:
        raise NotImplementedError("attention_bwd: only the causal policy attention is trained")
    nbasis = b_nd.shape[0]
    ws = torch.empty((2, B * heads, t, maxlen), dtype=F32, device=Q.device)  # P and dS by relative distance d
    db = torch.empty((nbasis, maxlen), dtype=F32, device=Q.device)
    nat.check(nat.lib().vpt_attention_bwd(_p(Q), _p(Kf), _p(Vf), _p(R), R.stride(-2), _p(b_nd), _p(first_u8), first_u8.stride(0), _p(smask),
                                          _p(dO), _p(out), out.stride(0), _p(db), _p(ws), B, t, maxlen, heads, nbasis, _stream()),
              "vpt_attention_bwd")
    _count(3)
    return db


def softmax_bwd(logp, idx, scale, out, col0):
    """out[:, col0:col0+n] = (exp(logp) - onehot(idx)) * scale  (bf16): d loss / d logits of a categorical NLL head."""
    _cuda(logp, idx, out)
    rows, n = logp.shape
    nat.check(nat.lib().vpt_softmax_bwd(_p(logp.contiguous()), _p(idx.contiguous()), float(scale), _p(out), out.stride(0), col0, rows, n, _stream()),
              "vpt_softmax_bwd")
    _count()
    return out


# ---- on-device action codec (csrc/codec.cuh) -----------------------------------------------------------------------------
def codec_to_env(buttons, camera, lut_btn, lut_cam_off, cam_lut, nbins):
    """int64 [n] joint indices -> int64 [n, 22] words (20 button flags + 2 float64 camera angles as bit patterns)."""
    _cuda(buttons, camera, lut_btn, lut_cam_off, cam_lut)
    n = buttons.numel()
    out = torch.empty((n, 22), dtype=torch.int64, device=buttons.device)
    bad = torch.zeros(1, dtype=torch.int32, device=buttons.device)
    nat.check(nat.lib().vpt_codec_to_env(_p(buttons), _p(camera), _p(lut_btn), _p(lut_cam_off), _p(cam_lut), nbins, lut_cam_off.numel(), n, _p(out), _p(bad),
                                         _stream()), "vpt_codec_to_env")
    _count()
    return out, bad


def codec_from_env(buttons, camera, thresholds, nbins, strides, inventory_idx):
    """int64 [n, 20] button flags + float64 [n, 2] camera angles -> int64 [n, 3] (buttons index, camera index, is-null flag)."""
    _cuda(buttons, camera, thresholds, strides)
    n = buttons.shape[0]
    out = torch.empty((n, 3), dtype=torch.int64, device=buttons.device)
    nat.check(nat.lib().vpt_codec_from_env(_p(buttons), _p(camera), _p(thresholds), nbins, _p(strides), inventory_idx, n, _p(out), _stream()),
              "vpt_codec_from_env")
    _count()
    return out


# ---- RL fine-tuning step (csrc/rl_heads.cuh; training.RLTrainer) --------------------------------------------------------
from .rl_ops import rl_heads_bwd  # noqa: E402,F401
