"""Drop-in replacements for the reference's policy classes (lib/policy.py) whose forward pass runs entirely in the
hand-written sm_100a kernels of libvpt_b200.so.

    MinecraftPolicy        lib/policy.py:83-224    forward(ob, state_in, context) / initial_state / output_latent_size
    MinecraftAgentPolicy   lib/policy.py:227-339   forward / act / get_output_for_observation / get_logprob_of_action /
                                                   get_kl_of_action_dists / v / initial_state
    InverseActionPolicy    lib/policy.py:406-467   (see idm.py)

Same constructor kwargs, same state pytree (list over layers of (state_mask bool (B,1,maxlen) | None, (K, V) fp32
(B,maxlen,hidsize))), same `state_dict()` keys / shapes (SURVEY.md App. B), so reference weight files load with
`load_state_dict`.  Parameters are kept in fp32 exactly as the reference stores them; at first use (and whenever a
parameter changes) they are re-laid-out for the kernels (`_Prepared`): conv weights OIHW -> [Cout][tap][Cin] bf16 with
the input GroupNorm gamma folded in plus the 9 border-class fold tables, linear weights with LayerNorm folded, the
`dense` columns permuted from C,H,W to H,W,C order.

`forward` runs under no_grad and returns detached tensors; the BC step has its own hand-written backward (training.py).
There is no CPU path: CPU tensors raise.
"""
import math
from collections import OrderedDict
from typing import Dict, Optional

import torch
from torch import nn

from . import _native as nat
from . import ops
from .types import DictType

BF16, F32 = torch.bfloat16, torch.float32
NBASIS = 10  # lib/xf.py:259


# ---------------------------------------------------------------------------------------------------------------
# parameter schema + init (names / shapes / init scales of the reference)
# ---------------------------------------------------------------------------------------------------------------
class _Node(nn.Module):
    """Bare container so that `state_dict()` keys nest exactly like the reference's module tree."""


def _set(root: nn.Module, name: str, tensor: torch.Tensor, requires_grad=True):
    parts = name.split(".")
    m = root
    for p in parts[:-1]:
        if p not in m._modules:
            m.add_module(p, _Node())
        m = m._modules[p]
    m.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=requires_grad))


def _fanin(shape, scale):
    """lib/util.py:67-73 / lib/torch_util.py:79: default torch init, then every output row L2-normalised to `scale`."""
    w = torch.empty(shape)
    nn.init.kaiming_uniform_(w, a=math.sqrt(5))
    flat = w.reshape(shape[0], -1)
    flat *= scale / flat.norm(dim=1, p=2, keepdim=True)
    return w


def _default_linear(out_f, in_f):
    """nn.Linear default init (lib/action_head.py:150, lib/scaled_mse_head.py:24)."""
    w = torch.empty(out_f, in_f)
    nn.init.kaiming_uniform_(w, a=math.sqrt(5))
    bound = 1 / math.sqrt(in_f)
    return w, torch.empty(out_f).uniform_(-bound, bound)


class NetConfig:
    """The kwargs of lib/policy.py:96-126 that the transformer models use (agent.py:16-36)."""

    def __init__(self, recurrence_type="transformer", impala_width=1, impala_chans=(16, 32, 32), obs_processing_width=256,
                 hidsize=512, single_output=False, img_shape=None, scale_input_img=True, only_img_input=False,
                 init_norm_kwargs=None, impala_kwargs=None, input_shape=None, active_reward_monitors=None, img_statistics=None,
                 first_conv_norm=False, diff_mlp_embedding=False, attention_mask_style="clipped_causal", attention_heads=8,
                 attention_memory_size=2048, use_pointwise_layer=True, pointwise_ratio=4, pointwise_use_activation=False,
                 n_recurrence_layers=1, recurrence_is_residual=True, timesteps=None, use_pre_lstm_ln=True, conv3d_params=None,
                 **unused_kwargs):
        init_norm_kwargs = init_norm_kwargs or {}
        impala_kwargs = impala_kwargs or {}
        # Only the configuration family of the released models is implemented in CUDA; anything else is refused loudly.
        if recurrence_type != "transformer":
            raise NotImplementedError("vpt_b200: only recurrence_type='transformer' (all released VPT models, agent.py:32)")
        if init_norm_kwargs.get("group_norm_groups", None) != 1 or init_norm_kwargs.get("batch_norm", False):
            raise NotImplementedError("vpt_b200: init_norm_kwargs must be {'batch_norm': False, 'group_norm_groups': 1} (agent.py:26)")
        if impala_kwargs.get("post_pool_groups", None) != 1:
            raise NotImplementedError("vpt_b200: impala_kwargs must be {'post_pool_groups': 1} (agent.py:24)")
        if img_statistics is not None or not scale_input_img or diff_mlp_embedding or use_pre_lstm_ln:
            raise NotImplementedError("vpt_b200: img_statistics / scale_input_img=False / diff_mlp_embedding / use_pre_lstm_ln unsupported")
        if not (use_pointwise_layer and recurrence_is_residual) or pointwise_use_activation:
            raise NotImplementedError("vpt_b200: needs use_pointwise_layer, recurrence_is_residual, no pointwise activation")
        if attention_mask_style not in ("clipped_causal", "none"):
            raise AssertionError("mask must be 'none' or 'clipped_causal'")  # lib/masked_attention.py:134
        assert attention_memory_size >= 0  # lib/masked_attention.py:135
        self.chans = tuple(int(impala_width * c) for c in impala_chans)
        self.hidsize = hidsize
        self.heads = attention_heads
        self.timesteps = timesteps
        self.maxlen = attention_memory_size - timesteps
        self.mask_style = attention_mask_style
        self.n_layers = n_recurrence_layers
        self.img_shape = tuple(img_shape)
        self.pointwise_ratio = pointwise_ratio
        self.single_output = single_output
        # IDM (lib/policy.py:342-372): a temporal conv3d pre-stage feeds the CNN, whose first conv is then normalised too
        self.conv3d_out = None
        if conv3d_params is not None:
            ks, pad = list(conv3d_params.get("kernel_size", [])), list(conv3d_params.get("padding", []))
            if conv3d_params.get("inchan") != 3 or ks != [5, 1, 1] or pad != [2, 0, 0]:
                raise NotImplementedError("vpt_b200: conv3d_params must be inchan=3, kernel_size=[5,1,1], padding=[2,0,0] (the IDM)")
            self.conv3d_out = int(conv3d_params["outchan"])
            first_conv_norm = True
        self.first_conv_norm = first_conv_norm
        self.cnn_outsize = 256
        assert hidsize % attention_heads == 0, "Embsize must be divisible by number of heads"  # lib/xf.py:98
        if hidsize // attention_heads != 128:
            raise NotImplementedError("vpt_b200: head_dim must be 128 (true of every VPT width)")
        assert self.maxlen > 0 or self.mask_style == "none"  # lib/xf.py:256
        H, W, Cin = self.img_shape
        want_cin = 3 if self.conv3d_out is None else self.conv3d_out
        if Cin != want_cin or H % 16 or W % 16 or any(c % 64 for c in self.chans) or (self.conv3d_out or 64) % 64:
            raise NotImplementedError("vpt_b200: img must be (H,W,3) [(H,W,conv3d outchan) for the IDM] with H,W % 16 == 0 and channels % 64 == 0")
        if self.first_conv_norm and self.conv3d_out is None:
            raise NotImplementedError("vpt_b200: first_conv_norm without the conv3d pre-stage is not implemented")
        self.final_hw = (H // 8, W // 8)

    def forward_flops_per_frame(self, head_outputs: int = 121 + 8641 + 1) -> float:
        """Algorithmic work of one frame through the forward path (SURVEY.md section 8d): 2 x MAC; clipped-causal attention counts
        `maxlen` keys per query (the band), unmasked attention (IDM) every key of the chunk.  bench.py's roofline uses this."""
        H, W = self.img_shape[0], self.img_shape[1]
        fl, cin = 0.0, 3
        if self.conv3d_out is not None:
            fl += 2 * H * W * 15 * self.conv3d_out
            cin = self.conv3d_out
        for c in self.chans:
            fl += 2 * H * W * 9 * cin * c
            H, W = (H + 1) // 2, (W + 1) // 2
            fl += 4 * 2 * H * W * 9 * c * c
            cin = c
        h = self.hidsize
        fl += 2 * (cin * H * W) * self.cnn_outsize + 2 * self.cnn_outsize * h
        keys = self.maxlen if self.mask_style == "clipped_causal" else self.maxlen + (self.timesteps or 0)
        nb = NBASIS if self.mask_style == "clipped_causal" else 0
        per_layer = 2 * h * h * 4 + 2 * h * nb * self.heads + 2 * 2 * h * h * self.pointwise_ratio
        per_layer += 4 * keys * h + 2 * nb * keys * self.heads
        fl += self.n_layers * per_layer + (2 * h * h if self.conv3d_out is None else 0) + 2 * h * head_outputs
        return fl


def _net_schema(cfg: NetConfig) -> "OrderedDict[str, torch.Tensor]":
    """Freshly initialised parameters in the reference's registration order (lib/impala_cnn.py, lib/util.py, lib/xf.py)."""
    sd = OrderedDict()
    p = "img_process.cnn"
    cin = cfg.img_shape[2]
    nstack = len(cfg.chans)
    for i, c in enumerate(cfg.chans):
        s = f"{p}.stacks.{i}"
        has_norm = cfg.first_conv_norm if i == 0 else True
        if has_norm:
            sd[f"{s}.firstconv.norm.weight"], sd[f"{s}.firstconv.norm.bias"] = torch.ones(cin), torch.zeros(cin)
        sd[f"{s}.firstconv.layer.weight"] = _fanin((c, cin, 3, 3), 1.0)
        if not has_norm:
            sd[f"{s}.firstconv.layer.bias"] = torch.zeros(c)
        sd[f"{s}.n.weight"], sd[f"{s}.n.bias"] = torch.ones(c), torch.zeros(c)
        bs = math.sqrt(math.sqrt(nstack) / math.sqrt(2))  # impala_cnn.py:164,105,30
        for j in range(2):
            for k in range(2):
                q = f"{s}.blocks.{j}.conv{k}"
                sd[f"{q}.norm.weight"], sd[f"{q}.norm.bias"] = torch.ones(c), torch.zeros(c)
                sd[f"{q}.layer.weight"] = _fanin((c, c, 3, 3), bs)
        cin = c
    kd = cin * cfg.final_hw[0] * cfg.final_hw[1]
    sd[f"{p}.dense.norm.weight"], sd[f"{p}.dense.norm.bias"] = torch.ones(kd), torch.zeros(kd)
    sd[f"{p}.dense.layer.weight"] = _fanin((cfg.cnn_outsize, kd), 1.4)
    sd["img_process.linear.norm.weight"], sd["img_process.linear.norm.bias"] = torch.ones(256), torch.zeros(256)
    sd["img_process.linear.layer.weight"] = _fanin((cfg.hidsize, 256), 1.0)
    h = cfg.hidsize
    s_blk = cfg.n_layers ** -0.5 * 2 ** -0.5  # lib/util.py:101,154-155
    s_att = math.sqrt(s_blk)                  # lib/xf.py:246
    for l in range(cfg.n_layers):
        b = f"recurrent_layer.blocks.{l}"
        sd[f"{b}.mlp0.norm.weight"], sd[f"{b}.mlp0.norm.bias"] = torch.ones(h), torch.zeros(h)
        sd[f"{b}.mlp0.layer.weight"] = _fanin((h * cfg.pointwise_ratio, h), 1.0)
        sd[f"{b}.mlp1.layer.weight"] = _fanin((h, h * cfg.pointwise_ratio), s_blk)
        sd[f"{b}.mlp1.layer.bias"] = torch.zeros(h)
        sd[f"{b}.pre_r_ln.weight"], sd[f"{b}.pre_r_ln.bias"] = torch.ones(h), torch.zeros(h)
        o = f"{b}.r.orc_block"
        sd[f"{o}.b_nd"] = torch.randn(NBASIS, cfg.maxlen) * 0.2
        sd[f"{o}.q_layer.weight"], sd[f"{o}.q_layer.bias"] = _fanin((h, h), 0.1), torch.zeros(h)
        sd[f"{o}.k_layer.weight"] = _fanin((h, h), 0.2)
        sd[f"{o}.v_layer.weight"] = _fanin((h, h), 1.0 * s_att)
        sd[f"{o}.proj_layer.weight"], sd[f"{o}.proj_layer.bias"] = _fanin((h, h), 1.0 * s_att), torch.zeros(h)
        sd[f"{o}.r_layer.weight"], sd[f"{o}.r_layer.bias"] = _fanin((NBASIS * cfg.heads, h), 0.1), torch.zeros(NBASIS * cfg.heads)
    sd["lastlayer.norm.weight"], sd["lastlayer.norm.bias"] = torch.ones(h), torch.zeros(h)
    sd["lastlayer.layer.weight"] = _fanin((h, h), 1.0)
    sd["final_ln.weight"], sd["final_ln.bias"] = torch.ones(h), torch.zeros(h)
    if cfg.conv3d_out is not None:  # lib/policy.py:362-372 (registered after the base class's modules)
        sd["conv3d_layer.layer.weight"] = _fanin((cfg.conv3d_out, 3, 5, 1, 1), 1.0)
        sd["conv3d_layer.layer.bias"] = torch.zeros(cfg.conv3d_out)
    return sd


# ---------------------------------------------------------------------------------------------------------------
# kernel-side weight layouts
# ---------------------------------------------------------------------------------------------------------------
_CLASS_TAPS = None


def _class_taps(device):
    """[9 border classes][9 taps] 0/1 matrix (float64): which taps of a 3x3 pad-1 convolution read inside the image for an output
    pixel of border class (cy, cx), cy / cx in {first row / column, interior, last row / column}."""
    global _CLASS_TAPS
    if _CLASS_TAPS is None or _CLASS_TAPS.device != device:
        valid = {0: [1, 2], 1: [0, 1, 2], 2: [0, 1]}
        m = torch.zeros(9, 9, dtype=torch.float64)
        for cy in range(3):
            for cx in range(3):
                for ky in valid[cy]:
                    for kx in valid[cx]:
                        m[cy * 3 + cx, ky * 3 + kx] = 1.0
        _CLASS_TAPS = m.to(device)
    return _CLASS_TAPS


def _fold_conv(W, gamma, beta):
    """GroupNorm(1) -> conv3x3(pad 1) fold (SURVEY.md section 7.2):
    conv(GN(x))[o,p] = rstd*conv_{W*gamma}(x)[o,p] - rstd*mean*S1[cls(p)][o] + S2[cls(p)][o].
    S1 is summed from the bf16-ROUNDED weights (the ones the tensor cores multiply) so the mean term cancels exactly.
    (Runs after every optimizer step of a BC run, hence a handful of batched ops rather than a loop over the 9 classes.)"""
    Cout = W.shape[0]
    Wg = (W * gamma[None, :, None, None]).permute(0, 2, 3, 1).contiguous()  # [Cout, ky, kx, Cin]
    Wb = Wg.to(BF16)
    tg = Wb.sum(-1, dtype=torch.float64).reshape(Cout, 9)                                  # per-tap sums of W*gamma
    tb = (W * beta[None, :, None, None]).sum(1, dtype=torch.float64).reshape(Cout, 9)      # per-tap sums of W*beta
    M = _class_taps(W.device)
    S1 = (M @ tg.t()).float().contiguous()  # [9, Cout]
    S2 = (M @ tb.t()).float().contiguous()
    return Wb.reshape(Cout, -1).contiguous(), S1, S2


def _fold_conv2(W, gamma0, beta0, gamma_n, beta_n):
    """Two-norm composition for block 0's conv0 (x0 = GN_n(y1) is not materialised; the conv reads y1):
    conv(GN_0(GN_n(y1))) = R * conv_{W g0 gn}(y1) + rstd0*Ta - R*mu1*Tb - rstd0*mu0*Tc + Td   per border class (see vpt_norm2_fold).
    Returns (bf16 weights [Cout, 9*Cin], (Ta, Tb, Tc, Td) fp32 [9, Cout]); Tb is summed from the bf16-rounded weights."""
    Cout = W.shape[0]
    Wb = (W * (gamma0 * gamma_n)[None, :, None, None]).permute(0, 2, 3, 1).contiguous().to(BF16)  # [Cout, ky, kx, Cin]
    M = _class_taps(W.device)
    per_tap = lambda v: v.reshape(Cout, 9)
    tb = per_tap(Wb.sum(-1, dtype=torch.float64))
    ta = per_tap((W * (gamma0 * beta_n)[None, :, None, None]).sum(1, dtype=torch.float64))
    tc = per_tap((W * gamma0[None, :, None, None]).sum(1, dtype=torch.float64))
    td = per_tap((W * beta0[None, :, None, None]).sum(1, dtype=torch.float64))
    tabs = tuple((M @ t.t()).float().contiguous() for t in (ta, tb, tc, td))
    return Wb.reshape(Cout, -1).contiguous(), tabs


def _fold_linear(W, gamma=None, beta=None, bias=None):
    """[LayerNorm ->] Linear fold: out = rstd*(x @ (W*gamma)^T) - rstd*mean*S1 + S2, S2 = W @ beta (+ bias)."""
    Wg = W if gamma is None else W * gamma[None, :]
    Wb = Wg.to(BF16).contiguous()
    S1 = Wb.sum(1, dtype=torch.float64).float().contiguous() if gamma is not None else None
    S2 = None
    if beta is not None:
        S2 = (W * beta[None, :]).sum(1, dtype=torch.float64)
    if bias is not None:
        S2 = bias.double() if S2 is None else S2 + bias.double()
    return Wb, S1, (S2.float().contiguous() if S2 is not None else None)


class _Prepared:
    """Device-side, kernel-layout copy of the parameters of one MinecraftPolicy (+ optional heads)."""

    def __init__(self, cfg: NetConfig, sd: Dict[str, torch.Tensor], prefix: str = ""):
        g = lambda k: sd[prefix + k].detach()
        p = "img_process.cnn"
        self.conv3d = None
        if cfg.conv3d_out is not None:  # [C, 3, dt, 1, 1] -> [C][dt][c] / 255
            w3 = g("conv3d_layer.layer.weight").double().reshape(cfg.conv3d_out, 3, 5).permute(0, 2, 1).reshape(cfg.conv3d_out, 15) / 255.0
            self.conv3d = (w3.float().contiguous(), g("conv3d_layer.layer.bias").float().contiguous())
        self.stacks = []
        for i, c in enumerate(cfg.chans):
            s = f"{p}.stacks.{i}"
            st = {}
            if i == 0 and not cfg.first_conv_norm:
                w = g(f"{s}.firstconv.layer.weight")  # [C0, 3, ky, kx] -> [C0][ky][kx][c] / 255 (lib/policy.py:44)
                st["fc_w"] = (w.double().permute(0, 2, 3, 1).reshape(c, 27) / 255.0).float().contiguous()
                st["fc_b"] = g(f"{s}.firstconv.layer.bias").float().contiguous()
            else:
                st["first"] = _fold_conv(g(f"{s}.firstconv.layer.weight"), g(f"{s}.firstconv.norm.weight"), g(f"{s}.firstconv.norm.bias"))
            st["n_g"], st["n_b"] = g(f"{s}.n.weight").float().contiguous(), g(f"{s}.n.bias").float().contiguous()
            q0 = f"{s}.blocks.0.conv0"
            st["conv0n"] = _fold_conv2(g(f"{q0}.layer.weight"), g(f"{q0}.norm.weight"), g(f"{q0}.norm.bias"), g(f"{s}.n.weight"), g(f"{s}.n.bias"))
            st["convs"] = []
            for j in range(2):
                for k in range(2):
                    q = f"{s}.blocks.{j}.conv{k}"
                    st["convs"].append(_fold_conv(g(f"{q}.layer.weight"), g(f"{q}.norm.weight"), g(f"{q}.norm.bias")))
            self.stacks.append(st)
        C2 = cfg.chans[-1]
        Hf, Wf = cfg.final_hw
        # dense: reference flatten order is c*H*W + h*W + w (lib/impala_cnn.py:192-193); ours is the ZP layout
        # [Hf+1][Wf+1][C2] -> permute to (h, w, c) and insert zero columns where the layout holds its zero row / column
        def perm(v):
            v = v.reshape(*v.shape[:-1], C2, Hf, Wf).movedim(-3, -1)          # (..., Hf, Wf, C2)
            v = torch.nn.functional.pad(v, (0, 0, 0, 1, 0, 1))                # (..., Hf+1, Wf+1, C2)
            return v.reshape(*v.shape[:-3], -1)
        self.dense = _fold_linear(perm(g(f"{p}.dense.layer.weight")), perm(g(f"{p}.dense.norm.weight")), perm(g(f"{p}.dense.norm.bias")))
        self.linear = _fold_linear(g("img_process.linear.layer.weight"), g("img_process.linear.norm.weight"), g("img_process.linear.norm.bias"))
        self.layers = []
        for l in range(cfg.n_layers):
            b = f"recurrent_layer.blocks.{l}"
            o = f"{b}.r.orc_block"
            L = {}
            L["ln_g"], L["ln_b"] = g(f"{b}.pre_r_ln.weight").float().contiguous(), g(f"{b}.pre_r_ln.bias").float().contiguous()
            L["q"] = _fold_linear(g(f"{o}.q_layer.weight"), bias=g(f"{o}.q_layer.bias"))
            L["k"] = _fold_linear(g(f"{o}.k_layer.weight"))
            L["v"] = _fold_linear(g(f"{o}.v_layer.weight"))
            L["r"] = _fold_linear(g(f"{o}.r_layer.weight"), bias=g(f"{o}.r_layer.bias"))
            # fused projection (lib/xf.py:334-365: Q(+bias) | K | V | R(+bias) of the same x_hat): one GEMM over the concatenated weight with
            # four column segments, each with its own destination (csrc/gemm_tc.cuh, vpt_gemm_args.dst_*)
            causal = cfg.mask_style == "clipped_causal"
            ws = [g(f"{o}.q_layer.weight"), g(f"{o}.k_layer.weight"), g(f"{o}.v_layer.weight")] + ([g(f"{o}.r_layer.weight")] if causal else [])
            zb = torch.zeros_like(g(f"{o}.q_layer.bias"))
            bs = [g(f"{o}.q_layer.bias"), zb, zb] + ([g(f"{o}.r_layer.bias")] if causal else [])
            L["qkvr"] = _fold_linear(torch.cat(ws, 0), bias=torch.cat(bs, 0))
            L["b_nd"] = g(f"{o}.b_nd").float().contiguous()
            L["proj"] = _fold_linear(g(f"{o}.proj_layer.weight"), bias=g(f"{o}.proj_layer.bias"))
            L["mlp0"] = _fold_linear(g(f"{b}.mlp0.layer.weight"), g(f"{b}.mlp0.norm.weight"), g(f"{b}.mlp0.norm.bias"))
            L["mlp1"] = _fold_linear(g(f"{b}.mlp1.layer.weight"), bias=g(f"{b}.mlp1.layer.bias"))
            self.layers.append(L)
        self.last = _fold_linear(g("lastlayer.layer.weight"), g("lastlayer.norm.weight"), g("lastlayer.norm.bias"))
        self.fin_g, self.fin_b = g("final_ln.weight").float().contiguous(), g("final_ln.bias").float().contiguous()


def _fingerprint(module: nn.Module):
    return tuple((p.data_ptr(), p._version) for p in module.parameters())


# ---------------------------------------------------------------------------------------------------------------
# MinecraftPolicy
# ---------------------------------------------------------------------------------------------------------------
class MinecraftPolicy(nn.Module):
    """lib/policy.py:83-224.  `forward(ob, state_in, context)` -> ((pi_latent, vf_latent), state_out)."""

    cnn_chunk_frames = 2048  # frames per CNN pass (bounds the activation workspace: ~5 MiB/frame at 2x width)
    fold_stack_norm = True   # inference: fold the post-pool GroupNorm of every stack into block 0 (no `affine_norm_zp` pass)
    idm_chunk_frames = 512   # IDM: ~13 MiB/frame at 4x width (conv3d output + full-resolution first conv)

    def __init__(self, **policy_kwargs):
        super().__init__()
        self.cfg = NetConfig(**policy_kwargs)
        self.hidsize = self.cfg.hidsize
        self.single_output = self.cfg.single_output
        for name, t in _net_schema(self.cfg).items():
            _set(self, name, t)
        self._prep = None
        self._prep_fp = None
        self.precision = "bf16"  # "fp32": the fp32-parity mode (precise.py): bf16 hi/lo split operands, fp32 activations
        self._pprep = None
        self._pprep_fp = None
        self.debug_taps = None  # set to a dict to capture intermediate activations (tests)
        self._tape = None       # set to a dict by training.BCTrainer: the forward then records what the backward needs

    def output_latent_size(self):
        return self.hidsize

    def initial_state(self, batchsize):
        """lib/policy.py:220-224 -> lib/xf.py:393-397: zeros on the module's device; state_mask None."""
        dev = self.final_ln.weight.device
        mk = lambda: torch.zeros((batchsize, self.cfg.maxlen, self.hidsize), dtype=F32, device=dev)
        return [(None, (mk(), mk())) for _ in range(self.cfg.n_layers)]

    # -- weights -------------------------------------------------------------------------------------------
    def prepared(self) -> _Prepared:
        fp = _fingerprint(self)
        if self._prep is None or fp != self._prep_fp:
            with torch.no_grad():
                self._prep = _Prepared(self.cfg, dict(self.named_parameters()))
            self._prep_fp = fp
        return self._prep

    def prepared_precise(self):
        from .precise import PreparedPrecise
        fp = _fingerprint(self)
        if self._pprep is None or fp != self._pprep_fp:
            with torch.no_grad():
                self._pprep = PreparedPrecise(self.cfg, dict(self.named_parameters()))
            self._pprep_fp = fp
        return self._pprep

    def _tap(self, name, t):
        if self.debug_taps is not None:
            self.debug_taps[name] = t

    # -- CNN -----------------------------------------------------------------------------------------------
    # Activations are kept in the "ZP" layout [F][H+1][W+1][C] (zero last row / column; include/vpt_b200.h): it lets the
    # conv kernel address every 3x3 neighbour linearly and reuse one shared-memory input span for all nine taps.
    def _cnn_chunk(self, img, prep: _Prepared, out, pfx="img_process.cnn"):
        """lib/impala_cnn.py:187-195 for a chunk of frames; writes the last stack's output (ZP [F, Hf+1, Wf+1, C2] bf16) into
        `out` and returns (out, per-frame stats)."""
        cfg = self.cfg
        H, W = cfg.img_shape[0], cfg.img_shape[1]
        x, mr = None, None
        tape = self._tape
        if prep.conv3d is not None:  # IDM: img is (b, T, H, W, 3), whole sequences (the temporal conv needs its neighbours)
            x, mr = ops.conv3d_t5(img, prep.conv3d[0], prep.conv3d[1], cfg.conv3d_out)
            self._tap("conv3d", x)
        for i, c in enumerate(cfg.chans):
            st = prep.stacks[i]
            rec = dict(x_in=x, mr_in=mr, H_in=H, W_in=W, full=None, blocks=[]) if tape is not None else None
            fold = self.fold_stack_norm and rec is None  # inference: the post-pool GroupNorm is folded into its two consumers
            if i == 0 and "fc_w" in st:
                y1, mr1, chan = ops.firstconv_pool(img, st["fc_w"], st["fc_b"], c, zp=True, want_chan=True)
            else:
                Wb, S1, S2 = st["first"]
                full, _ = ops.conv3x3_zp(x, Wb, H, W, mr=mr, S1=S1, S2=S2, relu=1, want_stats=False)
                y1, mr1, chan = ops.maxpool3s2(full, zp=True, want_chan=True)
                if rec is not None:
                    rec["full"] = full
                del full
            H, W = H // 2, W // 2
            self._tap(f"{pfx}.stacks.{i}.pool", y1)
            if fold and chan is not None:
                # two-norm composition (vpt_norm2_fold): x0 = n(y1) is never written; block 0 reads y1 with per-frame fold tables
                Wb0, tabs = st["conv0n"]
                mrE, Ef, rs, rb = ops.norm2_fold(chan, H * W, st["n_g"], st["n_b"], tabs)
                del chan
                hmid, mrh = ops.conv3x3_zp(y1, Wb0, H, W, mr=mrE, Ef=Ef, relu=1)
                self._tap(f"{pfx}.stacks.{i}.blocks.0.conv0", hmid)
                Wb, S1, S2 = st["convs"][1]
                x, mr = ops.conv3x3_zp(hmid, Wb, H, W, mr=mrh, S1=S1, S2=S2, relu=1, residual=y1, res_scale=rs, res_shift=rb)
                del y1, hmid
                self._tap(f"{pfx}.stacks.{i}.blocks.0", x)
                first_block = 1
            else:
                # post-pool GroupNorm `n` (lib/impala_cnn.py:119) as a pass: the training tape needs x0, and so do shapes whose pool
                # kernel cannot produce per-channel sums
                x, mr = ops.affine_norm_zp(y1, mr1, st["n_g"], st["n_b"])
                if rec is not None:
                    rec.update(y1=y1, mr1=mr1, x0=x, mr0=mr)
                del y1
                self._tap(f"{pfx}.stacks.{i}.n", x)
                first_block = 0
            for j in range(first_block, 2):
                Wb, S1, S2 = st["convs"][2 * j]
                hmid, mrh = ops.conv3x3_zp(x, Wb, H, W, mr=mr, S1=S1, S2=S2, relu=1)
                self._tap(f"{pfx}.stacks.{i}.blocks.{j}.conv0", hmid)
                Wb, S1, S2 = st["convs"][2 * j + 1]
                last = (i == len(cfg.chans) - 1) and j == 1
                if rec is None:
                    x, mr = ops.conv3x3_zp(hmid, Wb, H, W, mr=mrh, S1=S1, S2=S2, relu=1, residual=x, out=out if last else None)
                else:
                    # training: the branch output r = relu(conv1(..)) is kept on its own (its sign pattern IS the ReLU mask the
                    # backward needs; x + r rounded to bf16 no longer shows which small r were positive), then added
                    r, _ = ops.conv3x3_zp(hmid, Wb, H, W, mr=mrh, S1=S1, S2=S2, relu=1, want_stats=False)
                    x, mr = ops.add_zp(x, r, H, W, out=out if last else None)
                    rec["blocks"].append(dict(h=hmid, mrh=mrh, r=r, x=x, mr=mr))
                self._tap(f"{pfx}.stacks.{i}.blocks.{j}", x)
            if rec is not None:
                tape["stacks"].append(rec)
        return x, mr

    # -- transformer -----------------------------------------------------------------------------------------
    def _linear(self, x, fold, N, *, mr=None, relu=0, residual=None, out=None, out_dtype=None, seg=None, want_stats=False,
                out_scale=1.0, ld_out=None):
        Wb, S1, S2 = fold
        M, K = x.shape[0], x.shape[1]
        if out is None:
            out = torch.empty((M, N), dtype=out_dtype or BF16, device=x.device)
        part, P = None, ops.gemm_stat_parts(N)
        if want_stats:
            part = torch.empty((M, P, 2), dtype=F32, device=x.device)
        ops.gemm(x, Wb, out, M, N, K, mr=mr, rows_per_group=1, S1=S1 if mr is not None else None, S2=S2, relu=relu,
                 residual=residual, seg=seg, stat_part=part, stat_mode=1 if want_stats else 0, out_scale=out_scale, ld_out=ld_out)
        mr_out = ops.stats_finalize(part, M, P, N) if want_stats else None
        return out, mr_out

    def _block(self, l, x, mr_x, first_u8, state, B, t, prep: _Prepared, last: bool):
        """lib/util.py:193-211: x_hat = LN(x); y = x_hat + Proj(Attn(x_hat)); z = y + mlp1(relu(mlp0(LN(y))))."""
        cfg, L = self.cfg, prep.layers[l]
        h, heads, maxlen = cfg.hidsize, cfg.heads, cfg.maxlen
        causal = cfg.mask_style == "clipped_causal"
        state_mask, (mem_k, mem_v) = state
        xhat, _, _ = ops.affine_norm(x, mr_x, L["ln_g"], L["ln_b"], rows_per_group=1)
        T = maxlen + t
        full_k = torch.empty((B, T, h), dtype=BF16, device=x.device)
        full_v = torch.empty((B, T, h), dtype=BF16, device=x.device)
        if maxlen > 0:
            if mem_k.shape != (B, maxlen, h):
                raise AssertionError(f"KV memory shape {tuple(mem_k.shape)} != {(B, maxlen, h)}")
            if mem_k.stride() == mem_v.stride() and mem_k.dtype == mem_v.dtype:
                ops.copy_rows2(mem_k, mem_v, 0, full_k, full_v, 0, maxlen)  # lib/xf.py:378-379  full = cat(prev, new), K and V in one launch
            else:
                ops.copy_rows(mem_k, 0, full_k, 0, maxlen)
                ops.copy_rows(mem_v, 0, full_v, 0, maxlen)
        R = None
        if h % 256 == 0:
            # Q | K | V | R as ONE GEMM: K / V land in the rows of `full` after the memory (row remap), R in fp32
            q = torch.empty((B * t, h), dtype=BF16, device=x.device)
            dsts = [(0, q, h, False), (h, full_k, h, True), (2 * h, full_v, h, True)]
            if causal:
                R = torch.empty((B * t, NBASIS * heads), dtype=F32, device=x.device)
                dsts.append((3 * h, R, NBASIS * heads, False))
            Wc, _, bc = L["qkvr"]
            ops.gemm(xhat, Wc, q, B * t, Wc.shape[0], h, S2=bc, seg=(t, T, maxlen), dsts=dsts)
        else:  # hidsize not a multiple of the N tile: four launches
            q, _ = self._linear(xhat, L["q"], h)
            self._linear(xhat, L["k"], h, out=full_k, seg=(t, T, maxlen), ld_out=h)
            self._linear(xhat, L["v"], h, out=full_v, seg=(t, T, maxlen), ld_out=h)
            if causal:
                R, _ = self._linear(xhat, L["r"], NBASIS * heads, out_dtype=F32)
        smask_u8 = state_mask.contiguous().view(torch.uint8) if state_mask is not None else None
        a = ops.attention(q, full_k, full_v, R, L["b_nd"], first_u8, smask_u8, B, t, maxlen, heads, causal=causal)
        # new state (lib/xf.py:380-381: last `maxlen` rows of full; lib/masked_attention.py:86-92)
        new_k = torch.empty((B, maxlen, h), dtype=F32, device=x.device)
        new_v = torch.empty((B, maxlen, h), dtype=F32, device=x.device)
        ops.copy_rows2(full_k, full_v, T - maxlen, new_k, new_v, 0, maxlen)
        new_mask = ops.state_mask_update(smask_u8, first_u8, t, maxlen) if causal else state_mask
        y, mr_y = self._linear(a, L["proj"], h, residual=xhat, want_stats=True)
        self._tap(f"recurrent_layer.blocks.{l}.attn", y)
        hmid, _ = self._linear(y, L["mlp0"], h * cfg.pointwise_ratio, mr=mr_y, relu=1)
        # the F.relu of lib/policy.py:211 is fused into the last block's epilogue (relu after the residual add)
        z, mr_z = self._linear(hmid, L["mlp1"], h, residual=y, relu=2 if last else 0, want_stats=True)
        if not last:
            self._tap(f"recurrent_layer.blocks.{l}", z)
        if self._tape is not None:
            self._tape["blocks"].append(dict(x=x, mr_x=mr_x, xhat=xhat, q=q, full_k=full_k, full_v=full_v, R=R, smask=smask_u8, a=a, y=y,
                                             mr_y=mr_y, hmid=hmid, z=z, mr_z=mr_z))
        return z, mr_z, (new_mask, (new_k, new_v))

    # -- whole net -------------------------------------------------------------------------------------------
    @torch.no_grad()
    def _forward_impl(self, img, first, state_in, use_lastlayer=True):
        cfg = self.cfg
        ops.require_cuda(img)
        if img.dtype != torch.uint8:
            raise TypeError("ob['img'] must be uint8 (B,T,H,W,3) as in the reference (lib/policy.py:39-45)")
        B, t = img.shape[:2]
        frame_shape = (cfg.img_shape[0], cfg.img_shape[1], 3)
        assert tuple(img.shape[2:]) == frame_shape, f"img shape {tuple(img.shape[2:])} != {frame_shape}"
        assert len(state_in) == cfg.n_layers, \
            f"Length of state {len(state_in)} did not match length of blocks {cfg.n_layers}"  # lib/util.py:117-119
        if self.precision == "fp32":
            if self._tape is not None:
                raise NotImplementedError("the BC step runs in the bf16 mode only")
            from . import precise
            return precise.forward(self, img, first, state_in, use_lastlayer)
        if self.precision != "bf16":
            raise ValueError(f"unknown precision {self.precision!r} (use 'bf16' or 'fp32')")
        prep = self.prepared()
        N = B * t
        frames = img.reshape(N, *frame_shape).contiguous()
        first_u8 = first.to(device=img.device, dtype=torch.bool).contiguous().view(torch.uint8)
        Hf, Wf = cfg.final_hw
        C2 = cfg.chans[-1]
        # ---- ImpalaCNN in frame chunks (bounds the activation workspace), then ONE dense GEMM over all frames
        cnn_out = torch.empty((N, Hf + 1, Wf + 1, C2), dtype=BF16, device=img.device)
        mrs = []
        if cfg.conv3d_out is None:
            step = self.cnn_chunk_frames
        else:  # chunks of whole sequences; the IDM's 128-channel full-resolution stage is ~13 MiB/frame
            step = max(1, self.idm_chunk_frames // t) * t
        for f0 in range(0, N, step):
            F_ = min(step, N - f0)
            chunk = frames[f0:f0 + F_] if cfg.conv3d_out is None else frames[f0:f0 + F_].view(F_ // t, t, *frame_shape)
            _, mr = self._cnn_chunk(chunk, prep, cnn_out[f0:f0 + F_])
            mrs.append(mr)
        mr_c = mrs[0] if len(mrs) == 1 else torch.cat(mrs, 0)
        Kd = (Hf + 1) * (Wf + 1) * C2  # ZP rows flattened; the zero row / column meets zero weight columns
        xd, mr_d = self._linear(cnn_out.view(N, Kd), prep.dense, cfg.cnn_outsize, mr=mr_c, relu=1, want_stats=True)
        tape = self._tape
        if tape is not None:
            if len(mrs) != 1:
                raise NotImplementedError(f"training forward: at most {step} frames per call (got {N})")
            tape.update(frames=frames, first_u8=first_u8, cnn_out=cnn_out, mr_c=mr_c, xd=xd, mr_d=mr_d)
        del cnn_out
        self._tap("img_process.cnn.dense", xd)
        x, mr_x = self._linear(xd, prep.linear, cfg.hidsize, mr=mr_d, relu=1, want_stats=True)
        self._tap("img_process", x)
        if tape is not None:
            tape.update(x0=x, mr_x0=mr_x)
        # ---- transformer
        state_out = []
        for l in range(cfg.n_layers):
            x, mr_x, s = self._block(l, x, mr_x, first_u8, state_in[l], B, t, prep, last=(l == cfg.n_layers - 1))
            state_out.append(s)
        # x is relu(recurrent output) here
        if use_lastlayer:
            z_last, mr_zl = x, mr_x
            x, mr_x = self._linear(x, prep.last, cfg.hidsize, mr=mr_x, relu=1, want_stats=True)
            if tape is not None:
                tape.update(z_last=z_last, mr_zl=mr_zl, xl=x, mr_xl=mr_x)
        lat_bf16, lat_f32, _ = ops.affine_norm(x, mr_x, prep.fin_g, prep.fin_b, rows_per_group=1, want_f32=True)
        return lat_bf16, lat_f32.view(B, t, cfg.hidsize), state_out

    def forward(self, ob, state_in, context):
        """lib/policy.py:193-218."""
        first = context["first"]
        _, latent, state_out = self._forward_impl(ob["img"], first, state_in)
        if self.single_output:
            return latent, state_out
        return (latent, latent), state_out


class InverseActionNet(MinecraftPolicy):
    """lib/policy.py:342-403: conv3d pre-stage -> ImpalaCNN (first conv normalised) -> unmasked transformer ->
    relu -> final_ln.  `lastlayer` keeps its parameters (state_dict schema) but its output is discarded by the reference
    (lib/policy.py:390-391), so it is not computed."""

    def __init__(self, hidsize=512, conv3d_params=None, **MCPoliy_kwargs):
        super().__init__(hidsize=hidsize, conv3d_params=conv3d_params, **MCPoliy_kwargs)

    def forward(self, ob, state_in, context):
        """lib/policy.py:374-392 -> ((pi_latent, None), state_out)."""
        first = context["first"]
        _, latent, state_out = self._forward_impl(ob["img"], first, state_in, use_lastlayer=False)
        return (latent, None), state_out


# ---------------------------------------------------------------------------------------------------------------
# heads + MinecraftAgentPolicy
# ---------------------------------------------------------------------------------------------------------------
class _PolicyBase(nn.Module):
    """Shared head plumbing of MinecraftAgentPolicy and InverseActionPolicy (lib/action_head.py:136-260)."""

    has_value_head = True

    def _init_heads(self, action_space, pi_head_kwargs):
        self.action_space = action_space
        self.temperature = float((pi_head_kwargs or {}).get("temperature", 1.0))
        h = self.net.output_latent_size()
        if self.has_value_head:  # lib/scaled_mse_head.py:24 + lib/normalize_ewma.py:18-20
            w, b = _default_linear(1, h)
            _set(self, "value_head.linear.weight", w)
            _set(self, "value_head.linear.bias", b)
            _set(self, "value_head.normalizer.running_mean", torch.zeros(1), requires_grad=False)
            _set(self, "value_head.normalizer.running_mean_sq", torch.zeros(1), requires_grad=False)
            _set(self, "value_head.normalizer.debiasing_term", torch.tensor(0.0), requires_grad=False)
        # pi head: lib/action_head.py:263-275 -> one CategoricalActionHead per Discrete TensorType, in dict order
        self.head_specs = OrderedDict()
        for name, space in action_space.items():
            n = space.eltype.n
            shape = tuple(space.shape)
            cnt = 1
            for s_ in shape:
                cnt *= s_
            w, b = _default_linear(cnt * n, h)
            _set(self, f"pi_head.{name}.linear_layer.weight", w)
            _set(self, f"pi_head.{name}.linear_layer.bias", b)
            self.head_specs[name] = (shape, n)
        self._hprep = None
        self._hprep_fp = None

    def initial_state(self, batch_size: int):
        return self.net.initial_state(batch_size)

    def set_precision(self, precision: str):
        """"bf16" (default, production: bf16 operands, 1e-2 tolerance) or "fp32" (fp32-parity mode, precise.py: 1e-3 tolerance)."""
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.net.precision = precision
        return self

    def _heads_prepared_precise(self):
        from .precise import _f, _split_w
        params = [p for n, p in self.named_parameters() if not n.startswith("net.")]
        fp = tuple((p.data_ptr(), p._version) for p in params)
        if getattr(self, "_hpprep", None) is None or fp != self._hpprep_fp:
            with torch.no_grad():
                ws, bs, cols, c0 = [], [], OrderedDict(), 0
                for name in self.head_specs:
                    lin = getattr(self.pi_head, name).linear_layer
                    ws.append(lin.weight.detach())
                    bs.append(lin.bias.detach())
                    cols[name] = (c0, lin.weight.shape[0])
                    c0 += lin.weight.shape[0]
                self._hpprep = dict(pi=(_split_w(torch.cat(ws, 0)), _f(torch.cat(bs, 0))), cols=cols, ntot=c0)
                if self.has_value_head:
                    self._hpprep["v"] = (_split_w(self.value_head.linear.weight), _f(self.value_head.linear.bias))
            self._hpprep_fp = fp
        return self._hpprep

    def _heads_fp(self):  # (the return normaliser is not part of the heads' kernel-side weights)
        return tuple((p.data_ptr(), p._version) for n, p in self.named_parameters() if not n.startswith(("net.", "value_head.normalizer.")))

    def _build_heads_prepared(self):
        ws, bs, cols, c0 = [], [], OrderedDict(), 0
        for name, (shape, n) in self.head_specs.items():
            lin = getattr(self.pi_head, name).linear_layer
            ws.append(lin.weight.detach())
            bs.append(lin.bias.detach())
            cols[name] = (c0, lin.weight.shape[0])
            c0 += lin.weight.shape[0]
        hp = dict(pi=_fold_linear(torch.cat(ws, 0), bias=torch.cat(bs, 0)), cols=cols, ntot=c0)
        if self.has_value_head:
            hp["v"] = _fold_linear(self.value_head.linear.weight.detach(), bias=self.value_head.linear.bias.detach())
        return hp

    def _heads_prepared(self):
        fp = self._heads_fp()
        if self._hprep is None or fp != self._hprep_fp:
            with torch.no_grad():
                self._hprep = self._build_heads_prepared()
            self._hprep_fp = fp
        return self._hprep

    @torch.no_grad()
    def _heads(self, lat_bf16, B, t, mask=None):
        """lib/action_head.py:163-174 for every head + lib/scaled_mse_head.py:34-35."""
        if isinstance(lat_bf16, tuple):  # fp32-parity mode: (latent hi, latent lo)
            from . import precise
            return precise.heads(self, lat_bf16, B, t, mask)
        hp = self._heads_prepared()
        N = lat_bf16.shape[0]
        ntot = hp["ntot"]
        ld = (ntot + 7) // 8 * 8
        raw = torch.empty((N, ld), dtype=F32, device=lat_bf16.device)
        self.net._linear(lat_bf16, hp["pi"], ntot, out=raw, out_scale=1.0 / self.temperature, ld_out=ld)
        pd = OrderedDict()
        for name, (shape, n) in self.head_specs.items():
            c0, width = hp["cols"][name]
            cnt = width // n
            if mask is not None and mask.get(name) is not None:
                # lib/action_head.py:170-171: shaped_out[~mask] = LOG0 (-100) before the log-softmax.  Rare side input:
                # applied as a masked fill on the raw (already temperature-scaled) logits.
                view = raw[:, c0:c0 + width].view(B, t, *shape, n)
                view.masked_fill_(~mask[name].to(device=raw.device, dtype=torch.bool).expand_as(view), -100.0)
            if cnt == 1:
                lp = ops.log_softmax(raw, c0, n)
            else:  # several sub-actions per head (IDM): softmax over each group of n columns
                lp = torch.cat([ops.log_softmax(raw, c0 + i * n, n) for i in range(cnt)], dim=1)
            pd[name] = lp.view(B, t, *shape, n)
        if not self.has_value_head:
            return pd, None
        vpred, _ = self.net._linear(lat_bf16, hp["v"], 1, out_dtype=F32)
        return pd, vpred.view(B, t, 1)
    # -- distribution helpers (lib/action_head.py:176-220, 250-260) ---------------------------------------------
    def sample(self, pd, deterministic: bool = False):
        """DictActionHead.sample: per head in dict order; `torch.rand_like` supplies the uniforms so the Philox stream
        is consumed exactly like the reference's (lib/action_head.py:200)."""
        ac = OrderedDict()
        for name in self.head_specs:
            lg = pd[name].contiguous()
            u = None if deterministic else torch.rand_like(lg)
            ac[name] = ops.gumbel_argmax(lg, u)
        return ac

    def logprob(self, ac, pd):
        tot = None
        for name, (shape, n) in self.head_specs.items():
            lg = pd[name].contiguous()
            lp = ops.gather_logprob(lg, ac[name].to(torch.int64))
            for _ in shape:
                lp = lp.sum(dim=-1)
            tot = lp if tot is None else tot + lp
        return tot



class MinecraftAgentPolicy(_PolicyBase):
    """lib/policy.py:227-339."""

    def __init__(self, action_space, policy_kwargs, pi_head_kwargs):
        super().__init__()
        self.net = MinecraftPolicy(**policy_kwargs)
        self._init_heads(action_space, pi_head_kwargs)

    def forward(self, obs, first: torch.Tensor, state_in):
        """lib/policy.py:252-269 -> ((pi_logits, vpred, None), state_out)."""
        if isinstance(obs, dict):
            obs = obs.copy()
            mask = obs.pop("mask", None)
        else:
            mask = None
        lat_bf16, _, state_out = self.net._forward_impl(obs["img"], first, state_in)
        B, t = obs["img"].shape[:2]
        pi_logits, vpred = self._heads(lat_bf16, B, t, mask)
        return (pi_logits, vpred, None), state_out

    def denormalize(self, v):
        """lib/normalize_ewma.py:31-35,57-60 (a 3-scalar affine map; host-side glue)."""
        nz = self.value_head.normalizer
        bufs = (nz.debiasing_term, nz.running_mean, nz.running_mean_sq)
        key = tuple((b.data_ptr(), b._version) for b in bufs)
        if getattr(self, "_denorm_key", None) != key:  # the three scalars only change when the normaliser is updated / reloaded:
            deb = nz.debiasing_term.clamp(min=1e-5)    # 7 of the 9 tiny launches per rollout step were this recomputation
            mean = nz.running_mean / deb
            var = (nz.running_mean_sq / deb - mean ** 2).clamp(min=1e-2)
            self._denorm = (torch.sqrt(var)[None, None], mean[None, None])
            self._denorm_key = key
        std, mean = self._denorm
        return v * std + mean

    def get_logprob_of_action(self, pd, action):
        """lib/policy.py:271-279."""
        ac = {k: v.unsqueeze(1) for k, v in action.items()}
        log_prob = self.logprob(ac, pd)
        assert not torch.isnan(log_prob).any()
        return log_prob[:, 0]

    def get_kl_of_action_dists(self, pd1, pd2):
        """lib/policy.py:281-285 / lib/action_head.py:209-220 (diagnostic, not on the hot path: torch ops)."""
        tot = 0
        for name, (shape, n) in self.head_specs.items():
            kl = (torch.exp(pd1[name]) * (pd1[name] - pd2[name])).sum(-1, keepdim=True)
            for _ in shape:
                kl = kl.sum(dim=-2)
            tot = tot + kl
        return tot

    def get_output_for_observation(self, obs, state_in, first):
        """lib/policy.py:287-305."""
        obs = {k: v.unsqueeze(1) for k, v in obs.items()}
        first = first.unsqueeze(1)
        (pd, vpred, _), state_out = self(obs=obs, first=first, state_in=state_in)
        return pd, self.denormalize(vpred)[:, 0], state_out

    @torch.no_grad()
    def act(self, obs, first, state_in, stochastic: bool = True, taken_action=None, return_pd=False):
        """lib/policy.py:307-328."""
        obs = {k: v.unsqueeze(1) for k, v in obs.items()}
        first = first.unsqueeze(1)
        (pd, vpred, _), state_out = self(obs=obs, first=first, state_in=state_in)
        if taken_action is None:
            ac = self.sample(pd, deterministic=not stochastic)
        else:
            ac = {k: v.unsqueeze(1) for k, v in taken_action.items()}
        log_prob = self.logprob(ac, pd)
        if not (log_prob.is_cuda and torch.cuda.is_current_stream_capturing()):  # the check synchronises: not inside a graph capture
            assert not torch.isnan(log_prob).any()
        result = {"log_prob": log_prob[:, 0], "vpred": self.denormalize(vpred)[:, 0]}
        if return_pd:
            result["pd"] = {k: v[:, 0] for k, v in pd.items()}
        ac = {k: v[:, 0] for k, v in ac.items()}
        return ac, state_out, result

    def make_graphed_act(self, batch_size: int, pdl: bool = False):
        """Rollout-latency path (agent.py:190-206, SURVEY f-1): returns a callable with the signature of `act` whose whole
        step (forward + heads + sampling + log-prob + KV-memory roll) is ONE captured CUDA graph replay (pdl: captured with
        programmatic dependent launch between its kernels -- bit-identical, and measured neutral on B200: 0.953 vs 0.957 ms/step)."""
        return GraphedAct(self, batch_size, pdl=pdl)

    @torch.no_grad()
    def v(self, obs, first, state_in):
        """lib/policy.py:330-339."""
        obs = {k: v.unsqueeze(1) for k, v in obs.items()}
        first = first.unsqueeze(1)
        (pd, vpred, _), state_out = self(obs=obs, first=first, state_in=state_in)
        return self.denormalize(vpred)[:, 0]


class InverseActionPolicy(_PolicyBase):
    """lib/policy.py:406-467 (the IDM): InverseActionNet + factored categorical heads, no value head."""

    has_value_head = False

    def __init__(self, action_space, pi_head_kwargs=None, idm_net_kwargs=None):
        super().__init__()
        self.net = InverseActionNet(**idm_net_kwargs)
        self._init_heads(action_space, pi_head_kwargs)

    def forward(self, obs, first: torch.Tensor, state_in, **kwargs):
        """lib/policy.py:432-446 -> ((pi_logits, None, None), state_out)."""
        if isinstance(obs, dict):
            obs = obs.copy()
            mask = obs.pop("mask", None)
        else:
            mask = None
        lat_bf16, _, state_out = self.net._forward_impl(obs["img"], first, state_in, use_lastlayer=False)
        B, t = obs["img"].shape[:2]
        pi_logits, _ = self._heads(lat_bf16, B, t, mask)
        return (pi_logits, None, None), state_out

    @torch.no_grad()
    def predict(self, obs, deterministic: bool = True, **kwargs):
        """lib/policy.py:448-464."""
        (pd, _, _), state_out = self(obs=obs, **kwargs)
        ac = self.sample(pd, deterministic=deterministic)
        log_prob = self.logprob(ac, pd)
        assert not torch.isnan(log_prob).any()
        return ac, state_out, {"log_prob": log_prob, "pd": pd}


class GraphedAct:
    """`MinecraftAgentPolicy.act` for a fixed batch size as a CUDA graph: ~170 kernel launches become one graph launch,
    which is what bounds the B=1, T=1 rollout step (the arithmetic itself is ~0.1 ms of weight streaming at 2x width).

    The recurrent state lives in static buffers owned by the graph; the state object returned by a call is a handle to
    them (valid until the next call).  Passing any other state (e.g. `policy.initial_state(B)` after an episode reset)
    copies it in.  Sampling uses torch's graph-safe Philox generator, i.e. the same `rand_like` draws as eager mode."""

    def __init__(self, policy: "MinecraftAgentPolicy", batch_size: int, pdl: bool = False):
        self.policy = policy
        self.pdl = pdl
        cfg = policy.net.cfg
        dev = policy.net.final_ln.weight.device
        B, self.B = batch_size, batch_size
        H, W = cfg.img_shape[0], cfg.img_shape[1]
        self.img = torch.zeros((B, H, W, 3), dtype=torch.uint8, device=dev)
        self.first = torch.zeros((B,), dtype=torch.bool, device=dev)
        self.state = [(torch.zeros((B, 1, cfg.maxlen), dtype=torch.bool, device=dev),
                       (torch.zeros((B, cfg.maxlen, cfg.hidsize), dtype=F32, device=dev),
                        torch.zeros((B, cfg.maxlen, cfg.hidsize), dtype=F32, device=dev))) for _ in range(cfg.n_layers)]
        policy.net.prepared()
        policy._heads_prepared()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):  # warm-up outside capture (lazy function attributes, allocator pools)
            for _ in range(2):
                policy.act({"img": self.img}, self.first, self.state)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graphs = {}
        self._pin()

    def _weights_fp(self):
        return _fingerprint(self.policy)

    def _pin(self):
        """The captured graph holds RAW device pointers into the kernel-layout weight copies: keep those copies alive and remember
        which parameter versions they were made from (a later load_weights / optimizer step invalidates the graph)."""
        self._fp = self._weights_fp()
        self._held = (self.policy.net.prepared(), self.policy._heads_prepared())
        if self.policy.has_value_head:  # refresh the cached de-normalisation scalars OUTSIDE the capture (they must not live in the graph's pool)
            with torch.no_grad():
                self.policy.denormalize(torch.zeros((1, 1, 1), device=self.img.device))

    def _capture(self, stochastic: bool):
        g = torch.cuda.CUDAGraph()
        # optional programmatic dependent launch: with the attribute the next kernel is scheduled while the previous one drains
        # (csrc/common.cuh pdl_sync).  Measured neutral for this graph (0.953 vs 0.957 ms), hence off by default.
        nat.lib().vpt_set_pdl(1 if self.pdl else 0)
        try:
            with torch.cuda.graph(g):
                ac, st, res = self.policy.act({"img": self.img}, self.first, self.state, stochastic=stochastic, return_pd=True)
                for (m_in, (k_in, v_in)), (m_out, (k_out, v_out)) in zip(self.state, st):  # roll the state inside the graph
                    m_in.copy_(m_out)
                    if k_in.shape[1] > 0:
                        ops.copy_rows2(k_out, v_out, 0, k_in, v_in, 0, k_in.shape[1])  # K and V in one launch
        finally:
            nat.lib().vpt_set_pdl(0)
        self.graphs[stochastic] = (g, ac, res)
        return self.graphs[stochastic]

    @torch.no_grad()
    def __call__(self, obs, first, state_in, stochastic: bool = True, taken_action=None, return_pd: bool = False):
        if taken_action is not None:
            raise NotImplementedError("GraphedAct: taken_action is only supported by the eager act()")
        self.img.copy_(obs["img"])
        self.first.copy_(first)
        if state_in is not self.state:
            for (m_in, (k_in, v_in)), (m, (k, v)) in zip(self.state, state_in):
                if m is None:
                    m_in.zero_()  # lib/masked_attention.py:75-76: None == all-False
                else:
                    m_in.copy_(m)
                k_in.copy_(k)
                v_in.copy_(v)
        if self._weights_fp() != self._fp:  # parameters changed since capture: re-layout the weights and re-capture
            self.graphs = {}
            self._pin()
        g, ac, res = self.graphs.get(stochastic) or self._capture(stochastic)
        g.replay()
        out = {"log_prob": res["log_prob"], "vpred": res["vpred"]}
        if return_pd:
            out["pd"] = res["pd"]
        return ac, self.state, out
