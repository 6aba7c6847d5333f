"""TEST-ONLY torch emulation of the C ABI ops (same signatures as video-pre-training_b200/ops.py).

Purpose: check the HOST logic (weight re-layout, GroupNorm/LayerNorm folds, border-class tables, dense column
permutation, KV-memory bookkeeping, launch order) against the oracle on CPU, where no GPU exists.  It mirrors what each
kernel computes, including where values are rounded to bf16.  It is never importable from the product package."""
import torch
import torch.nn.functional as F

BF16, F32 = torch.bfloat16, torch.float32


def require_cuda(t):
    pass


def gemm_stat_parts(N):
    nt = (N + 255) // 256
    bn = (-(-N // nt) + 15) // 16 * 16
    return -(-N // bn) * 2


def _row_stats(v, rows_per_group):
    """(mean, rstd) per group of rows from the stored values."""
    G = v.shape[0] // rows_per_group
    x = v.float().reshape(G, -1).double()
    mean = x.mean(1)
    var = (x * x).mean(1) - mean * mean
    return torch.stack([mean, 1.0 / torch.sqrt(var.clamp(min=0) + 1e-5)], 1).float()


def gemm(A, Bw, out, M, N, K, *, conv=None, mr=None, rows_per_group=1, S1=None, S2=None, relu=0, out_scale=1.0,
         residual=None, ld_out=None, seg=None, stat_part=None, stat_mode=0, cluster=0, dsts=None):
    if dsts:  # column segments with their own destination: emulate as one GEMM per segment
        assert stat_part is None
        bounds = [d[0] for d in dsts] + [N]
        for i, (n0, t, ld, remap) in enumerate(dsts):
            n1 = bounds[i + 1]
            sl = lambda v: None if v is None else v.reshape(-1, N)[:, n0:n1].contiguous()
            gemm(A, Bw[n0:n1], t, M, n1 - n0, K, conv=conv, mr=mr, rows_per_group=rows_per_group, S1=sl(S1), S2=sl(S2), relu=relu,
                 out_scale=out_scale, residual=residual, ld_out=ld, seg=seg if remap else None)
        return out
    Af = A.float()
    # products summed in fp64 and rounded once to fp32 here and in conv3x3_zp / wgrad: an fp32 sum's order (and with it
    # which outputs round to the other bf16 neighbour) depends on the host CPU's vector width; this does not
    if conv is not None:
        H, W, Cin = conv
        x = Af.double().reshape(-1, H, W, Cin).permute(0, 3, 1, 2)
        w = Bw.double().reshape(N, 3, 3, Cin).permute(0, 3, 1, 2)
        acc = F.conv2d(x, w, padding=1).float().permute(0, 2, 3, 1).reshape(M, N)
        pix = torch.arange(M) % (H * W)
        y, xx = pix // W, pix % W
        cy = torch.where(y == 0, 0, torch.where(y == H - 1, 2, 1))
        cx = torch.where(xx == 0, 0, torch.where(xx == W - 1, 2, 1))
        cls = cy * 3 + cx
    else:
        acc = (Af.double().reshape(M, K) @ Bw.double().T).float()
        cls = torch.zeros(M, dtype=torch.long)
    v = acc
    s1 = S1.reshape(-1, N)[cls] if S1 is not None else 0.0
    s2 = S2.reshape(-1, N)[cls] if S2 is not None else 0.0
    if mr is not None:
        g = torch.arange(M) // rows_per_group
        a, b = mr[g, 1:2], (mr[g, 1] * mr[g, 0])[:, None]
        v = a * acc - b * s1 + s2
    else:
        v = acc + s2
    if relu == 1:
        v = v.relu()
    if residual is not None:
        v = v + residual.reshape(M, -1)[:, :N].float()
    if relu == 2:
        v = v.relu()
    v = v * out_scale
    v = v.to(out.dtype)
    o2 = out.reshape(-1, out.shape[-1])
    if seg is not None:
        sl, ss, so = seg
        m = torch.arange(M)
        rows = (m // sl) * ss + so + m % sl
        o2[rows, :N] = v
    else:
        o2[:M, :N] = v
    if stat_part is not None:
        vf = v.float()
        P = gemm_stat_parts(N)
        if stat_mode == 1:
            pp = stat_part.reshape(-1, P, 2)
            pp[:M] = 0
            pp[:M, 0, 0] = vf.sum(1)
            pp[:M, 0, 1] = (vf * vf).sum(1)
        else:
            r32 = (M + 31) // 32
            pad = torch.zeros(r32 * 32, N)
            pad[:M] = vf
            pp = stat_part.reshape(-1, P, 2)
            pp[:r32] = 0
            pp[:r32, 0, 0] = pad.reshape(r32, -1).sum(1)
            pp[:r32, 0, 1] = (pad * pad).reshape(r32, -1).sum(1)
    return out


def stats_finalize(part, G, n_per_group, count, eps=1e-5):
    p = part.reshape(G, n_per_group, 2).double().sum(1)
    mean = p[:, 0] / count
    var = (p[:, 1] / count - mean * mean).clamp(min=0)
    return torch.stack([mean, 1.0 / torch.sqrt(var + eps)], 1).float()


def to_zp(x):
    """[F,H,W,C] -> ZP [F,H+1,W+1,C] with a zero last row / column."""
    return F.pad(x, (0, 0, 0, 1, 0, 1))


def from_zp(x):
    return x[:, :-1, :-1, :]


def _frame_stats(x_interior):
    return _row_stats(x_interior.reshape(x_interior.shape[0], -1), 1)


def conv3x3_zp(x, Wb, H, W, *, mr=None, S1=None, S2=None, relu=1, residual=None, want_stats=True, out=None, Ef=None, res_scale=None,
               res_shift=None):
    if Ef is not None or res_scale is not None:  # two-norm composition: per-frame fold table / affine residual
        F_, Cin = x.shape[0], x.shape[3]
        Cout = Wb.shape[0]
        xi = from_zp(x).float().permute(0, 3, 1, 2)
        acc = F.conv2d(xi.double(), Wb.double().reshape(Cout, 3, 3, Cin).permute(0, 3, 1, 2), padding=1).float().permute(0, 2, 3, 1)  # [F,H,W,Cout]
        yy, xx = torch.arange(H)[:, None], torch.arange(W)[None, :]
        cls = (torch.where(yy == 0, 0, torch.where(yy == H - 1, 2, 1)) * 3 + torch.where(xx == 0, 0, torch.where(xx == W - 1, 2, 1)))  # [H,W]
        if Ef is not None:
            v = mr[:, 1, None, None, None] * acc + Ef[:, cls]           # Ef [F,9,Cout] -> [F,H,W,Cout]
        else:
            s1 = S1[cls] if S1 is not None else 0.0
            s2 = S2[cls] if S2 is not None else 0.0
            v = mr[:, 1, None, None, None] * acc - (mr[:, 1] * mr[:, 0])[:, None, None, None] * s1 + s2 if mr is not None else acc + s2
        if relu == 1:
            v = v.relu()
        if residual is not None:
            r = from_zp(residual).float()
            if res_scale is not None:
                r = res_scale[:, None, None, :] * r + res_shift[:, None, None, :]
            v = v + r
        if relu == 2:
            v = v.relu()
        o = v.to(BF16)
        res = to_zp(o)
        if out is not None:
            out.copy_(res)
            res = out
        return res, (_frame_stats(o) if want_stats else None)
    F_, Cin = x.shape[0], x.shape[3]
    Cout = Wb.shape[0]
    assert (x[:, -1] == 0).all() and (x[:, :, -1] == 0).all(), "ZP invariant violated on the conv input"
    xi = from_zp(x).contiguous()
    M = F_ * H * W
    out_buf = out
    out = torch.zeros((M, Cout), dtype=BF16)
    gemm(xi, Wb, out, M, Cout, 9 * Cin, conv=(H, W, Cin), mr=mr, rows_per_group=H * W, S1=S1, S2=S2, relu=relu,
         residual=None if residual is None else from_zp(residual).contiguous())
    o = out.reshape(F_, H, W, Cout)
    res = to_zp(o)
    if out_buf is not None:
        out_buf.copy_(res)
        res = out_buf
    return res, (_frame_stats(o) if want_stats else None)


def _chan_parts(y):
    """[F,H,W,C] -> per-channel (sum, sumsq) [F, 1, C, 2] (one partial)"""
    yf = y.float()
    return torch.stack([yf.sum((1, 2)), (yf * yf).sum((1, 2))], -1)[:, None]


def firstconv_pool(img, w, bias, C0, zp=True, out_f32=False, want_chan=False):
    F_, H, W, _ = img.shape
    x = img.float().permute(0, 3, 1, 2)
    wt = w.reshape(C0, 3, 3, 3).permute(0, 3, 1, 2)  # [C0][ky][kx][c] -> OIHW
    y = F.relu(F.conv2d(x, wt, bias, padding=1))
    y = F.max_pool2d(y, 3, 2, 1).permute(0, 2, 3, 1).contiguous().to(F32 if out_f32 else BF16)
    r = ((to_zp(y) if zp else y), _frame_stats(y))
    return r + (_chan_parts(y),) if want_chan else r


def conv3d_t5(img, w, bias, C, out_f32=False):
    B, T, H, W, _ = img.shape
    x = img.float().permute(0, 4, 1, 2, 3)                       # b c t h w
    wt = w.reshape(C, 5, 3).permute(0, 2, 1).reshape(C, 3, 5, 1, 1)  # [C][dt][c] -> [C][c][dt][1][1]
    y = F.relu(F.conv3d(x, wt, bias, padding=(2, 0, 0)))         # per-sample zero padding in time == batched conv3d
    y = y.permute(0, 2, 3, 4, 1).reshape(B * T, H, W, C).contiguous().to(F32 if out_f32 else BF16)
    return to_zp(y), _frame_stats(y)


# ---- fp32-parity precision mode (csrc/precise.cuh) ----
def group_stats_f32(x, groups, eps=1e-5):
    v = x.reshape(groups, -1).double()
    mean = v.mean(1)
    var = ((v * v).mean(1) - mean * mean).clamp(min=0)
    return torch.stack([mean, 1.0 / torch.sqrt(var + eps)], 1).float()


def norm_split_f32(x, mr=None, gamma=None, beta=None, groups=1, split=True, want_f32=False):
    u = x
    if mr is not None:
        v = x.reshape(groups, -1)
        u = ((v - mr[:, 0:1]) * mr[:, 1:2]).reshape(x.shape)
    if gamma is not None:
        u = u * gamma
    if beta is not None:
        u = u + beta
    hi = u.to(BF16) if split else None
    lo = (u - hi.float()).to(BF16) if split else None
    return hi, lo, (u.clone() if want_f32 else None)


def add_f32(a, b=None, relu=False, out=None):
    v = a if b is None else a + b
    return v.relu() if relu else v.clone()


def maxpool3s2_f32(x):
    return F.max_pool2d(x.permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1).contiguous()


def attention_f32(q, full_k, full_v, R, b_nd, first_u8, smask_u8, B, t, maxlen, heads, causal=True):
    smask = smask_u8
    h = q.shape[-1]
    D = h // heads
    T = maxlen + t
    qq = q.reshape(B, t, heads, D).permute(0, 2, 1, 3)
    k = full_k.reshape(B, T, heads, D).permute(0, 2, 1, 3)
    v = full_v.reshape(B, T, heads, D).permute(0, 2, 1, 3)
    logit = qq @ k.transpose(-1, -2) / D
    if causal:
        i = torch.arange(t)[:, None]
        j = torch.arange(T)[None, :]
        d = maxlen + i - j
        band = (d >= 0) & (d < maxlen)
        memok = torch.zeros(B, maxlen, dtype=torch.bool) if smask is None else (smask.reshape(B, maxlen) != 0)
        memok = memok & (first_u8[:, 0] == 0)[:, None]
        colok = torch.cat([memok, torch.ones(B, t, dtype=torch.bool)], 1)
        allowed = band[None] & colok[:, None, :]
        E = R.reshape(B, t, heads, -1).permute(0, 2, 1, 3) @ b_nd
        extra = torch.gather(E, 3, d.clamp(0, maxlen - 1)[None, None].expand(B, heads, t, T)) * band[None, None]
        logit = logit + extra + (~allowed[:, None]).float() * -1e9
    w = torch.softmax(logit, -1)
    return (w @ v).permute(0, 2, 1, 3).reshape(B * t, h)


def maxpool3s2(x, zp=True, want_chan=False):
    xi = from_zp(x) if zp else x
    y = F.max_pool2d(xi.float().permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1).contiguous().to(BF16)
    r = ((to_zp(y) if zp else y), _frame_stats(y))
    return r + (_chan_parts(y),) if want_chan else r


def norm2_fold(chan_part, npix, gamma_n, beta_n, tabs):
    Ta, Tb, Tc, Td = [t.double() for t in tabs]
    cp = chan_part.double().sum(1)                      # [F, C, 2]
    S, Q = cp[..., 0], cp[..., 1]
    Cc = S.shape[1]
    cnt = float(npix) * Cc
    mu1 = S.sum(1) / cnt
    rstd1 = 1.0 / torch.sqrt((Q.sum(1) / cnt - mu1 * mu1).clamp(min=0) + 1e-5)
    a = rstd1[:, None] * gamma_n.double()[None]
    b = beta_n.double()[None] - mu1[:, None] * a
    m0 = (a * S + npix * b).sum(1) / cnt
    e0 = (a * a * Q + 2 * a * b * S + npix * b * b).sum(1) / cnt
    rstd0 = 1.0 / torch.sqrt((e0 - m0 * m0).clamp(min=0) + 1e-5)
    R = rstd0 * rstd1
    Ef = rstd0[:, None, None] * Ta[None] - (R * mu1)[:, None, None] * Tb[None] - (rstd0 * m0)[:, None, None] * Tc[None] + Td[None]
    mrE = torch.stack([torch.zeros_like(R), R], 1)
    return mrE.float(), Ef.float(), a.float(), b.float()


def affine_norm_zp(x, mr, gamma, beta):
    xi = from_zp(x).float()
    o = ((xi - mr[:, 0, None, None, None]) * mr[:, 1, None, None, None]) * gamma + beta
    ob = o.to(BF16)
    return to_zp(ob), _frame_stats(ob)


def affine_norm(x, mr, gamma, beta, rows_per_group, want_stats=False, want_f32=False):
    Cc = x.shape[-1]
    xf = x.float().reshape(-1, Cc)
    g = torch.arange(xf.shape[0]) // rows_per_group
    o = ((xf - mr[g, 0:1]) * mr[g, 1:2]) * gamma[None] + beta[None]
    ob = o.to(BF16).reshape(x.shape)
    mr_out = _row_stats(ob.reshape(-1, Cc), rows_per_group) if want_stats else None
    return ob, (o.reshape(x.shape) if want_f32 else None), mr_out


def copy_rows(src, src_off, dst, dst_off, rows):
    if rows:
        dst[:, dst_off:dst_off + rows] = src[:, src_off:src_off + rows].to(dst.dtype)


def copy_rows2(src_a, src_b, src_off, dst_a, dst_b, dst_off, rows):
    copy_rows(src_a, src_off, dst_a, dst_off, rows)
    copy_rows(src_b, src_off, dst_b, dst_off, rows)


def state_mask_update(mask_in, first_u8, t, maxlen):
    B = first_u8.shape[0]
    if mask_in is None:
        mask_in = torch.zeros((B, 1, maxlen), dtype=torch.uint8)
    nf = (first_u8[:, 0] == 0)[:, None, None]
    keep = maxlen - min(t, maxlen)
    old = (mask_in.reshape(B, 1, maxlen)[:, :, t:t + keep] != 0) & nf
    return torch.cat([old, torch.ones((B, 1, maxlen - keep), dtype=torch.bool)], -1)


def attention(Q, Kf, Vf, R, b_nd, first_u8, smask, B, t, maxlen, heads, causal=True):
    h = Q.shape[-1]
    D = h // heads
    T = maxlen + t
    q = Q.float().reshape(B, t, heads, D).permute(0, 2, 1, 3)
    k = Kf.float().reshape(B, T, heads, D).permute(0, 2, 1, 3)
    v = Vf.float().reshape(B, T, heads, D).permute(0, 2, 1, 3)
    logit = q @ k.transpose(-1, -2) / D
    if causal:
        i = torch.arange(t)[:, None]
        j = torch.arange(T)[None, :]
        d = maxlen + i - j
        band = (d >= 0) & (d < maxlen)
        memok = torch.zeros(B, maxlen, dtype=torch.bool) if smask is None else (smask.reshape(B, maxlen) != 0)
        memok = memok & (first_u8[:, 0] == 0)[:, None]
        colok = torch.cat([memok, torch.ones(B, t, dtype=torch.bool)], 1)  # [B, T]
        allowed = band[None] & colok[:, None, :]
        E = R.float().reshape(B, t, heads, -1).permute(0, 2, 1, 3) @ b_nd.float()  # [B, heads, t, maxlen]
        dd = d.clamp(0, maxlen - 1)[None, None].expand(B, heads, t, T)
        extra = torch.gather(E, 3, dd)
        logit = torch.where(allowed[:, None], logit + extra, torch.tensor(-float("inf")))
    w = torch.softmax(logit, -1)
    o = (w.to(BF16).float() @ v).permute(0, 2, 1, 3).reshape(B * t, h)
    return o.to(BF16).reshape(Q.shape)


def log_softmax(raw, col0, n):
    return F.log_softmax(raw[:, col0:col0 + n].float(), -1)


def gumbel_argmax(logits, u=None):
    if u is None:
        return torch.argmax(logits, -1)
    u = u.clone()
    u[u == 1.0] = 0.999
    return torch.argmax(logits - torch.log(-torch.log(u)), -1)


def gather_logprob(logits, idx, lp=None):
    r = logits.gather(-1, idx.long().unsqueeze(-1)).squeeze(-1)
    return r if lp is None else lp + r


# ---------------------------------------------------------------------------------------------------------------------
# backward ops of the BC step (training.py)
# ---------------------------------------------------------------------------------------------------------------------
def relu_mask(dout, out):
    return torch.where(out.float() > 0, dout, torch.zeros_like(dout))


def add_zp(a, b, H, W, out=None):
    """ZP a + b (bf16) with the per-frame statistics of the sum."""
    s = (a.float() + b.float()).to(BF16)
    if out is not None:
        out.copy_(s)
        s = out
    return s, _frame_stats(from_zp(s))


def wgrad(a, b, shifts=(0,), out=None):
    """out[m][tap*N + n] = sum_k a[k][m] * b[k + shifts[tap]][n]  (rows k + shift outside [0, R) are zero); fp32."""
    R = a.shape[0]
    af, bf = a.float(), b.float()
    cols = []
    for s in shifts:
        bs = torch.zeros_like(bf)
        if s >= 0:
            bs[:R - s] = bf[s:]
        else:
            bs[-s:] = bf[:R + s]
        cols.append((af.double().T @ bs.double()).float())
    res = torch.cat(cols, 1)
    if out is not None:
        out.copy_(res)
        return out
    return res


def _norm_n(x, mr, rows_per_group):
    Cc = x.shape[-1]
    xf = x.float().reshape(-1, Cc)
    g = torch.arange(xf.shape[0]) // rows_per_group
    return (xf - mr[g, 0:1]) * mr[g, 1:2], g


def group_sums(du, x, mr, gamma, rows_per_group, count):
    """per group: (mean of gamma*du, mean of gamma*du*n) with n = (x - mean) * rstd; `count` = real elements per group."""
    Cc = x.shape[-1]
    n, g = _norm_n(x, mr, rows_per_group)
    dn = du.float().reshape(-1, Cc) * gamma[None]
    G = n.shape[0] // rows_per_group
    s1 = dn.double().reshape(G, -1).sum(1) / count
    s2 = (dn * n).double().reshape(G, -1).sum(1) / count
    return torch.stack([s1, s2], 1).float()


def col_sums(du, x=None, mr=None, rows_per_group=1):
    """fp32 [2][C]: (sum_rows du*n, sum_rows du); without x only row 1 is meaningful (row 0 = 0)."""
    Cc = du.shape[-1]
    d = du.float().reshape(-1, Cc)
    out = torch.zeros((2, Cc), dtype=F32)
    out[1] = d.double().sum(0).float()
    if x is not None:
        n, _ = _norm_n(x, mr, rows_per_group)
        out[0] = (d * n).double().sum(0).float()
    return out


def norm_sums(du, x, mr, gamma, rows_per_group, count):
    return col_sums(du, x, mr, rows_per_group), group_sums(du, x, mr, gamma, rows_per_group, count)


def norm_bwd_apply(du, x, mr, gamma, ms, rows_per_group, zp=None, add=None, relu_x=False):
    """dx = rstd * (gamma*du - m1 - n*m2) [+ add] on [rows][C]; with zp = (H, W, Cch) every group is a ZP frame
    [(H+1)(W+1)][Cch] (flattened over rows_per_group rows of C) whose pad row / column is written as zero."""
    Cc = x.shape[-1]
    n, g = _norm_n(x, mr, rows_per_group)
    dn = du.float().reshape(-1, Cc) * gamma[None]
    dx = mr[g, 1:2] * (dn - ms[g, 0:1] - n * ms[g, 1:2])
    if add is not None:
        dx = dx + add.float().reshape(-1, Cc)
    dx = dx.to(BF16)
    if relu_x:
        dx = torch.where(x.float().reshape(-1, Cc) > 0, dx, torch.zeros((), dtype=BF16))
    if zp is not None:
        H, W, Cch = zp
        e = torch.arange(rows_per_group * Cc) // Cch          # pixel row inside the frame
        pad = ((e // (W + 1)) == H) | ((e % (W + 1)) == W)
        dx = torch.where(pad.reshape(1, -1), torch.zeros((), dtype=BF16), dx.reshape(-1, rows_per_group * Cc))
    return dx.reshape(x.shape)


def maxpool3s2_bwd(dy, x):
    """Gradient of max_pool2d(3,2,1) (+ the ReLU in front of it: x is post-ReLU) on ZP tensors; first maximum wins ties."""
    xi = from_zp(x).float().permute(0, 3, 1, 2).requires_grad_(True)
    yo = F.max_pool2d(xi, 3, 2, 1)
    (g,) = torch.autograd.grad(yo, xi, from_zp(dy).float().permute(0, 3, 1, 2))
    g = torch.where(xi > 0, g, torch.zeros_like(g))
    return to_zp(g.permute(0, 2, 3, 1).contiguous().to(BF16))


def firstconv_bwd(img, w, bias, dy, C0):
    """(dW fp32 [C0][27] in the kernel's (ky,kx,c) order for the /255-scaled weights, db [C0])."""
    x = img.float().permute(0, 3, 1, 2)
    wt = w.reshape(C0, 3, 3, 3).permute(0, 3, 1, 2).clone().requires_grad_(True)
    b = bias.clone().requires_grad_(True)
    y = F.max_pool2d(F.relu(F.conv2d(x, wt, b, padding=1)), 3, 2, 1)
    gw, gb = torch.autograd.grad(y, (wt, b), from_zp(dy).float().permute(0, 3, 1, 2))
    return gw.permute(0, 2, 3, 1).reshape(C0, 27).contiguous(), gb


def attention_bwd(Q, Kf, Vf, R, b_nd, first_u8, smask, dO, out, B, t, maxlen, heads, causal=True):
    """Gradients of `attention` wrt Q, the chunk rows of K / V and R, written side by side into out[:, 0:h | h:2h | 2h:3h |
    3h:3h+10*heads] (bf16); returns d b_nd (fp32).  The memory rows of K / V are detached state and get no gradient."""
    h = Q.shape[-1]
    D = h // heads
    T = maxlen + t
    q = Q.float().reshape(B, t, heads, D).permute(0, 2, 1, 3).requires_grad_(True)
    kf = Kf.float().requires_grad_(True)
    vf = Vf.float().requires_grad_(True)
    k = kf.reshape(B, T, heads, D).permute(0, 2, 1, 3)
    v = vf.reshape(B, T, heads, D).permute(0, 2, 1, 3)
    Rf = R.float().requires_grad_(True) if R is not None else None
    bf = b_nd.float().requires_grad_(True) if causal else None
    logit = q @ k.transpose(-1, -2) / D
    if causal:
        i = torch.arange(t)[:, None]
        j = torch.arange(T)[None, :]
        d = maxlen + i - j
        band = (d >= 0) & (d < maxlen)
        memok = torch.zeros(B, maxlen, dtype=torch.bool) if smask is None else (smask.reshape(B, maxlen) != 0)
        memok = memok & (first_u8[:, 0] == 0)[:, None]
        colok = torch.cat([memok, torch.ones(B, t, dtype=torch.bool)], 1)
        allowed = band[None] & colok[:, None, :]
        E = Rf.reshape(B, t, heads, -1).permute(0, 2, 1, 3) @ bf
        dd = d.clamp(0, maxlen - 1)[None, None].expand(B, heads, t, T)
        extra = torch.gather(E, 3, dd)
        logit = torch.where(allowed[:, None], logit + extra, torch.tensor(-float("inf")))
    w = torch.softmax(logit, -1)
    o = (w @ v).permute(0, 2, 1, 3).reshape(B * t, h)
    ins = [q, kf, vf] + ([Rf, bf] if causal else [])
    gs = torch.autograd.grad(o, ins, dO.float().reshape(B * t, h))
    out[:, 0:h] = gs[0].permute(0, 2, 1, 3).reshape(B * t, h).to(BF16)
    out[:, h:2 * h] = gs[1][:, maxlen:].reshape(B * t, h).to(BF16)
    out[:, 2 * h:3 * h] = gs[2][:, maxlen:].reshape(B * t, h).to(BF16)
    if causal:
        nr = R.shape[-1]
        out[:, 3 * h:3 * h + nr] = gs[3].reshape(B * t, nr).to(BF16)
        return gs[4].contiguous()
    return None


def softmax_bwd(logp, idx, scale, out, col0):
    """out[:, col0:col0+n] = (exp(logp) - onehot(idx)) * scale   (bf16)."""
    n = logp.shape[-1]
    g = torch.exp(logp.float().reshape(-1, n))
    g[torch.arange(g.shape[0]), idx.reshape(-1).long()] -= 1.0
    out[:, col0:col0 + n] = (g * scale).to(out.dtype)
    return out


# ---- on-device action codec (csrc/codec.cuh) ----
def codec_to_env(buttons, camera, lut_btn, lut_cam_off, cam_lut, nbins):
    b, c = buttons.reshape(-1).long(), camera.reshape(-1).long()
    cy, cx = c // nbins, c % nbins
    off = lut_cam_off[b] != 0
    cy = torch.where(off, torch.full_like(cy, nbins // 2), cy)
    cx = torch.where(off, torch.full_like(cx, nbins // 2), cx)
    out = torch.empty((b.numel(), 22), dtype=torch.int64)
    out[:, :20] = lut_btn.reshape(-1, 20)[b].long()
    out[:, 20] = cam_lut[cy].view(torch.int64)
    out[:, 21] = cam_lut[cx].view(torch.int64)
    return out, torch.zeros(1, dtype=torch.int32)


def codec_from_env(buttons, camera, thresholds, nbins, strides, inventory_idx):
    on = buttons != 0
    n = buttons.shape[0]
    hot = torch.zeros(n, dtype=torch.int64)
    for k in range(9):
        hot = torch.where(on[:, 11 + k], torch.full_like(hot, k + 1), hot)

    def pair(a, b, cancel):
        r = torch.where(on[:, b], 2, torch.where(on[:, a], 1, 0))
        return torch.where(on[:, a] & on[:, b], 0, r) if cancel else r

    binv = (camera[:, :, None] >= thresholds[None, None, :]).sum(-1)
    null = nbins // 2
    cam_null = (binv == null).all(1)
    parts = [hot, pair(2, 1, True), pair(4, 5, True), pair(7, 6, False), on[:, 8].long(), on[:, 9].long(), on[:, 0].long(), on[:, 3].long(), (~cam_null).long()]
    joint = sum(p_ * s_ for p_, s_ in zip(parts, strides.tolist()))
    cidx = binv[:, 0] * nbins + binv[:, 1]
    inv = buttons[:, 10] == 1
    joint = torch.where(inv, torch.full_like(joint, inventory_idx), joint)
    cidx = torch.where(inv, torch.full_like(cidx, null * nbins + null), cidx)
    return torch.stack([joint, cidx, ((~on.any(1)) & cam_null).long()], 1)
