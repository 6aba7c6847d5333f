"""Behavioural-cloning step of `MinecraftAgentPolicy` (behavioural_cloning.py:101-123): forward with a tape, the
negative log-likelihood loss of the demonstrated actions, and a hand-written backward through the same CUDA ops the forward
uses -- no autograd graph.  Gradients land in `param.grad` (fp32, reference parameter layout), so `parallel.FlatAdamDP`
(one NCCL all-reduce over the flat gradient bucket + one fused Adam launch) finishes the step.

    loss = -(1 / (B*T)) * sum_{b,t} sum_heads log_softmax(logits_head / temperature)[action]      (lib/action_head.py:176-184)

What each layer type needs (u = gamma * n + beta is the normalised layer input, n = (x - mean) * rstd):

    NormConv / NormLinear   dz = dout * [out > 0]              ReLU (residual convs keep their branch output r for this)
                            du = dz (*) W^T                    the forward conv / GEMM kernel on flipped / transposed weights
                            dW = dz^T (*) u                    `wgrad`: tcgen05 GEMM over the pixel / token dimension
                            dgamma, dbeta = sum du*n, sum du   `col_sums`
                            dx = rstd * (gamma*du - mean(gamma*du) - n * mean(gamma*du*n))      `group_sums` + `norm_bwd_apply`
    max-pool, first conv, attention, softmax heads: their own backward kernels (see include/vpt_b200.h).

The KV memory carried in `state_in` is detached exactly like behavioural_cloning.py:111 (`tree_map(lambda x: x.detach())`),
and `value_head.*` receives no gradient (None in the reference: the BC loss never touches it).

`RLTrainer` shares the taped forward, the backward and the weight re-layout; only its loss block differs (clipped policy gradient,
KL to a frozen teacher, entropy, value loss -- one kernel, csrc/rl_heads.cuh), and it also trains `value_head.linear.*`.
"""
import torch
import torch.distributed as dist

from . import ops
from .policy import BF16, F32, MinecraftAgentPolicy


def _rot(W):
    """conv weight [Cout, Cin, 3, 3] -> dgrad weight bf16 [Cin][tap'][Cout] with tap' = 8 - tap (180-degree rotation)."""
    return W.detach().flip(2, 3).permute(1, 2, 3, 0).reshape(W.shape[1], -1).to(BF16).contiguous()


def _tr(W, pad_to=None):
    """linear weight [out, in] -> dgrad weight bf16 [in][out] (optionally zero-padded along `out` to `pad_to` columns)."""
    Wt = W.detach().t().to(BF16)
    if pad_to is not None and pad_to != Wt.shape[1]:
        Wt = torch.nn.functional.pad(Wt, (0, pad_to - Wt.shape[1]))
    return Wt.contiguous()


def _relayout_fp(policy):
    """Fingerprint of the parameters the weight re-layout reads: not the return normaliser, which every RL step updates."""
    return tuple((p.data_ptr(), p._version) for n, p in policy.named_parameters() if not n.startswith("value_head.normalizer."))


def _acc(p, g):
    """p.grad += g (allocating on first use), like autograd's accumulation."""
    g = g.reshape(p.shape)
    if p.grad is None:
        p.grad = g.to(F32).clone()
    else:
        p.grad.add_(g)


class BCTrainer:
    """`loss, state_out = trainer.loss_and_grad(img, first, state_in, actions)` accumulates d loss / d param into `.grad`."""

    value_column = False  # RLTrainer: the value head rides in column ntot of the heads' dgrad / wgrad GEMMs

    def __init__(self, policy: MinecraftAgentPolicy):
        if not isinstance(policy, MinecraftAgentPolicy):
            raise TypeError("BCTrainer trains a MinecraftAgentPolicy (behavioural_cloning.py:54-62)")
        cfg = policy.net.cfg
        if cfg.conv3d_out is not None or cfg.first_conv_norm or cfg.mask_style != "clipped_causal":
            raise NotImplementedError("BCTrainer: only the causal policy models are trained by the reference")
        self.policy = policy
        self._wprep = None
        self._wprep_fp = None
        self.debug_grads = None  # set to a dict to capture d loss / d activation under the forward's tap names (tests)
        self.keep_tape = False   # tests: keep the last forward's tape in `self.last_tape` (tests/forced_replica.py)
        self.last_tape = None
        self.graph_relayout = True  # re-layout of the kernel-side weights after an optimizer step as one CUDA graph replay
        self._rl_graph = None
        self._rl_seen = 0

    def _dbg(self, name, g):
        if self.debug_grads is not None:
            self.debug_grads[name] = g

    # -- backward-side weight layouts (re-made whenever a parameter changes, like policy._Prepared) -------------------
    def _weights(self):
        fp = _relayout_fp(self.policy)
        if self._wprep is not None and fp == self._wprep_fp:
            return self._wprep
        with torch.no_grad():
            self._wprep = self._build_weights()
        self._wprep_fp = fp
        return self._wprep

    def refresh_weights(self):
        """Re-layout of every kernel-side weight copy (forward folds of policy._Prepared + the heads, backward transposes of
        `_build_weights`) after an optimizer step.  Eagerly this is ~500 small torch launches (12 ms at 3x width, profiles/bc_step_r1.md);
        the parameters live at fixed addresses (FlatAdamDP's flat bucket), so from the second refresh on the whole re-layout is ONE captured
        CUDA graph replay writing the same kernel-layout tensors in place.  Called by `loss_and_grad`; a no-op when nothing changed."""
        pol, net = self.policy, self.policy.net
        from .policy import _Prepared, _fingerprint
        fp_net, fp_heads = _fingerprint(net), pol._heads_fp()
        fp_all = _relayout_fp(pol)
        if net._prep is not None and net._prep_fp == fp_net and pol._hprep is not None and pol._hprep_fp == fp_heads and self._wprep is not None \
                and self._wprep_fp == fp_all:
            return
        ptrs = tuple(p.data_ptr() for p in pol.parameters())
        if not self.graph_relayout or not all(p.is_cuda for p in pol.parameters()):
            return  # the lazy eager paths (prepared() / _heads_prepared() / _weights()) rebuild on use
        if self._rl_graph is not None and self._rl_graph[0] != ptrs:
            self._rl_graph = None  # the parameters moved (e.g. .to(), a new optimizer bucket): capture again
        if self._rl_graph is None:
            self._rl_seen += 1
            if self._rl_seen < 2:
                return  # first change: eager (also warms up every lazily initialised helper before capture)
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.no_grad(), torch.cuda.graph(g):
                prep = _Prepared(net.cfg, dict(net.named_parameters()))
                hprep = pol._build_heads_prepared()
                wprep = self._build_weights()
            self._rl_graph = (ptrs, g, prep, hprep, wprep)
        _, g, prep, hprep, wprep = self._rl_graph
        g.replay()
        net._prep, net._prep_fp = prep, fp_net
        pol._hprep, pol._hprep_fp = hprep, fp_heads
        self._wprep, self._wprep_fp = wprep, fp_all

    def _build_weights(self):
        pol, net = self.policy, self.policy.net
        cfg = net.cfg
        P = dict(net.named_parameters())
        w = dict(stacks=[], layers=[])
        pfx = "img_process.cnn"
        for i in range(len(cfg.chans)):
            s = f"{pfx}.stacks.{i}"
            st = dict(convs=[_rot(P[f"{s}.blocks.{j}.conv{k}.layer.weight"]) for j in range(2) for k in range(2)])
            if i > 0:
                st["first"] = _rot(P[f"{s}.firstconv.layer.weight"])
            w["stacks"].append(st)
        Hf, Wf = cfg.final_hw
        C2 = cfg.chans[-1]

        def perm(v):  # reference C,H,W flatten order -> ZP (h, w, c) order with zero columns at the pad row / column
            v = v.reshape(*v.shape[:-1], C2, Hf, Wf).movedim(-3, -1)
            v = torch.nn.functional.pad(v, (0, 0, 0, 1, 0, 1))
            return v.reshape(*v.shape[:-3], -1)

        w["dense_t"] = _tr(perm(P[f"{pfx}.dense.layer.weight"].detach()))
        w["dense_g"] = perm(P[f"{pfx}.dense.norm.weight"].detach()).float().contiguous()
        w["dense_b"] = perm(P[f"{pfx}.dense.norm.bias"].detach()).float().contiguous()
        w["linear_t"] = _tr(P["img_process.linear.layer.weight"])
        h, heads = cfg.hidsize, cfg.heads
        nr = 10 * heads
        self.kcat = (3 * h + nr + 7) // 8 * 8
        for l in range(cfg.n_layers):
            o = f"recurrent_layer.blocks.{l}.r.orc_block"
            b = f"recurrent_layer.blocks.{l}"
            cat = torch.cat([P[f"{o}.q_layer.weight"], P[f"{o}.k_layer.weight"], P[f"{o}.v_layer.weight"], P[f"{o}.r_layer.weight"]], 0)
            w["layers"].append(dict(qkvr_t=_tr(cat, self.kcat), proj_t=_tr(P[f"{o}.proj_layer.weight"]), mlp0_t=_tr(P[f"{b}.mlp0.layer.weight"]),
                                    mlp1_t=_tr(P[f"{b}.mlp1.layer.weight"])))
        w["last_t"] = _tr(P["lastlayer.layer.weight"])
        self.ntot = sum(getattr(pol.pi_head, name).linear_layer.weight.shape[0] for name in pol.head_specs)
        rows = [getattr(pol.pi_head, name).linear_layer.weight for name in pol.head_specs]
        if self.value_column:  # value weight as row ntot: dlat, its wgrad row and col_sums column come out of the heads' GEMMs
            rows.append(pol.value_head.linear.weight)
        self.ld_logits = (len(rows) - len(pol.head_specs) + self.ntot + 7) // 8 * 8
        assert not self.value_column or self.ntot < self.ld_logits
        w["heads_t"] = _tr(torch.cat(rows, 0), self.ld_logits)
        return w

    # -- generic pieces -------------------------------------------------------------------------------------------------
    @staticmethod
    def _gemm(A, Bt, N, residual=None):
        """bf16 [M][N] = A [M][K] @ Bt[N][K]^T (+ residual)."""
        M, K = A.shape
        out = torch.empty((M, N), dtype=BF16, device=A.device)
        ops.gemm(A, Bt, out, M, N, K, residual=residual)
        return out

    @staticmethod
    def _wgrad_linear(dz, u, weight_param=None):
        """dW [out][in] = dz^T u (tcgen05 GEMM over the token dimension); accumulated into `weight_param.grad` when given."""
        dW = ops.wgrad(dz, u)
        if weight_param is not None:
            _acc(weight_param, dW)
        return dW

    @staticmethod
    def _norm_bwd(du, x, mr, gamma, rows_per_group, count, g_param, b_param, zp=None, add=None, relu_x=False):
        """Backward of n = (x - mean) * rstd, u = gamma * n + beta given du: accumulates dgamma / dbeta, returns dx (+ add).
        relu_x: x is the output of a ReLU whose backward is applied to the result in the same pass."""
        if rows_per_group > 1:  # GroupNorm frames: column sums and group sums share one pass over (du, x)
            cs, ms = ops.norm_sums(du, x, mr, gamma, rows_per_group, count)
        else:
            cs = ops.col_sums(du, x, mr, rows_per_group)
            ms = ops.group_sums(du, x, mr, gamma, rows_per_group, count)
        if g_param is not None:
            _acc(g_param[0], g_param[1](cs[0]))
            _acc(b_param[0], b_param[1](cs[1]))
        return ops.norm_bwd_apply(du, x, mr, gamma, ms, rows_per_group, zp=zp, add=add, relu_x=relu_x)

    def _normconv_bwd(self, dz, x, mr, H, W, W_rot, names, P, add=None, relu_x=False):
        """dz: gradient wrt the conv output (ReLU already applied), ZP [F,H+1,W+1,Cout]; x: the layer input (ZP, pre-norm).
        Accumulates the weight / norm gradients and returns the gradient wrt x (+ add)."""
        Fn, Cin, Cout = x.shape[0], x.shape[3], dz.shape[3]
        R = Fn * (H + 1) * (W + 1)
        gam, bet = P[names + ".norm.weight"], P[names + ".norm.bias"]
        g32 = gam.detach().float().contiguous()
        du, _ = ops.conv3x3_zp(dz, W_rot, H, W, relu=0, want_stats=False)
        u, _ = ops.affine_norm_zp(x, mr, g32, bet.detach().float().contiguous())
        shifts = [(ky - 1) * (W + 1) + (kx - 1) for ky in range(3) for kx in range(3)]
        dWk = ops.wgrad(dz.view(R, Cout), u.view(R, Cin), shifts)  # [Cout][tap][Cin]
        del u
        _acc(P[names + ".layer.weight"], dWk.view(Cout, 3, 3, Cin).permute(0, 3, 1, 2))
        ident = lambda v: v
        return self._norm_bwd(du.view(R, Cin), x.view(R, Cin), mr, g32, (H + 1) * (W + 1), H * W * Cin, (gam, ident), (bet, ident),
                              zp=(H, W, Cin), add=None if add is None else add.view(R, Cin), relu_x=relu_x).view(x.shape)

    def _normlinear_bwd(self, dz, x, mr, Wt, names, P, add=None, relu_x=False):
        """[LayerNorm ->] Linear backward; dz [rows][out] is the gradient wrt the GEMM output (after ReLU masking)."""
        gam, bet = P[names + ".norm.weight"], P[names + ".norm.bias"]
        g32, b32 = gam.detach().float().contiguous(), bet.detach().float().contiguous()
        du = self._gemm(dz, Wt, Wt.shape[0])
        u, _, _ = ops.affine_norm(x, mr, g32, b32, rows_per_group=1)
        self._wgrad_linear(dz, u, P[names + ".layer.weight"])
        del u
        ident = lambda v: v
        return self._norm_bwd(du, x, mr, g32, 1, x.shape[1], (gam, ident), (bet, ident), add=add, relu_x=relu_x)

    # -- the step ---------------------------------------------------------------------------------------------------------
    def loss_and_grad(self, img, first, state_in, actions, upper_grads_ready=None):
        """`upper_grads_ready()` is called once every gradient except those of `img_process.cnn.stacks.*` is final (the ImpalaCNN
        backward, most of the step's time, is still to come): the hook for `FlatAdamDP.reduce_async`."""
        return self._step(img, first, state_in, lambda pd, vpred, N: self._nll_dlog(pd, actions, N), upper_grads_ready)

    def _nll_dlog(self, pd, actions, N):
        """BC loss block: -mean joint log-prob of the taken actions -> (d loss / d head GEMM outputs, loss)."""
        pol = self.policy
        hp = pol._heads_prepared()
        dlog = torch.zeros((N, self.ld_logits), dtype=BF16, device=pd[next(iter(pd))].device)
        scale = 1.0 / (pol.temperature * N)
        logp = None
        for name, (shape, n) in pol.head_specs.items():
            c0, width = hp["cols"][name]
            if width != n:
                raise NotImplementedError("BCTrainer: heads with several sub-actions are not trained by the reference")
            idx = actions[name].reshape(N).to(torch.int64)
            lp = ops.gather_logprob(pd[name].reshape(N, n), idx)
            logp = lp if logp is None else logp + lp
            ops.softmax_bwd(pd[name].reshape(N, n), idx, scale, dlog, c0)
        loss = -logp.sum() / N
        return dlog, loss

    def _step(self, img, first, state_in, loss_block, upper_grads_ready):
        """Taped forward, `loss_block(pd, vpred, N) -> (dlog, result)` (d loss / d head GEMM outputs, bf16 [N][ld_logits]), then the
        hand-written backward from dlog to every parameter gradient.  Returns (result, state_out)."""
        pol, net = self.policy, self.policy.net
        cfg = net.cfg
        self.refresh_weights()
        wts = self._weights()
        P = dict(net.named_parameters())
        B, t = img.shape[:2]
        N = B * t
        h = cfg.hidsize
        # ---------------- forward (the inference kernels, recording what the backward needs) ----------------
        state_in = [(m, (k.detach(), v.detach())) for (m, (k, v)) in state_in]  # behavioural_cloning.py:111
        tape = dict(stacks=[], blocks=[])
        net._tape = tape
        try:
            lat_bf16, _, state_out = net._forward_impl(img, first, state_in)
        finally:
            net._tape = None
        if self.keep_tape:
            tape["latent"] = lat_bf16
            self.last_tape = tape
        pd, vpred = pol._heads(lat_bf16, B, t)
        # ---------------- loss + d logits ----------------
        dlog, result = loss_block(pd, vpred, N)
        hp = pol._heads_prepared()
        # ---------------- heads ----------------
        nrow = self.ntot + (1 if self.value_column else 0)
        dWh = ops.wgrad(dlog, lat_bf16)[:nrow]
        dbh = ops.col_sums(dlog)[1]
        for name in pol.head_specs:
            c0, width = hp["cols"][name]
            lin = getattr(pol.pi_head, name).linear_layer
            _acc(lin.weight, dWh[c0:c0 + width])
            _acc(lin.bias, dbh[c0:c0 + width])
        if self.value_column:
            _acc(pol.value_head.linear.weight, dWh[self.ntot:nrow])
            _acc(pol.value_head.linear.bias, dbh[self.ntot:nrow])
        dlat = self._gemm(dlog, wts["heads_t"], h)
        self._dbg("latent", dlat)
        del dlog
        # ---------------- final_ln (plain norm) + lastlayer ----------------
        ident = lambda v: v
        fg = P["final_ln.weight"]
        # (xl, z_last, x0, xd and the convs' h are ReLU outputs that feed a norm: their ReLU backward rides on that norm's apply pass)
        dz = self._norm_bwd(dlat, tape["xl"], tape["mr_xl"], fg.detach().float().contiguous(), 1, h, (fg, ident), (P["final_ln.bias"], ident),
                            relu_x=True)
        dx = self._normlinear_bwd(dz, tape["z_last"], tape["mr_zl"], wts["last_t"], "lastlayer", P, relu_x=True)
        # ---------------- transformer blocks, last to first ----------------
        for l in reversed(range(cfg.n_layers)):
            self._dbg(f"recurrent_layer.blocks.{l}" if l < cfg.n_layers - 1 else "recurrent_out", dx)
            dx = self._block_bwd(l, dx, tape["blocks"][l], tape["first_u8"], wts["layers"][l], P, B, t, last=(l == cfg.n_layers - 1))
        # ---------------- img_process.linear, dense ----------------
        dz = self._normlinear_bwd(dx, tape["xd"], tape["mr_d"], wts["linear_t"], "img_process.linear", P, relu_x=True)
        dcnn = self._dense_bwd(dz, tape, wts, P)
        if upper_grads_ready is not None:
            upper_grads_ready()
        # ---------------- ImpalaCNN, last stack to first ----------------
        self._cnn_bwd(dcnn, tape, wts, P)
        return result, state_out

    def _dense_bwd(self, dz, tape, wts, P):
        cfg = self.policy.net.cfg
        Hf, Wf = cfg.final_hw
        C2 = cfg.chans[-1]
        N = dz.shape[0]
        Kd = (Hf + 1) * (Wf + 1) * C2
        x = tape["cnn_out"].view(N, Kd)
        pfx = "img_process.cnn.dense"
        du = self._gemm(dz, wts["dense_t"], Kd)
        u, _, _ = ops.affine_norm(x, tape["mr_c"], wts["dense_g"], wts["dense_b"], rows_per_group=1)
        dWz = self._wgrad_linear(dz, u)  # [out][Kd] in ZP column order
        del u

        def unperm(v):  # ZP (h, w, c) order -> the reference's C,H,W flatten order (dropping the pad row / column)
            v = v.reshape(*v.shape[:-1], Hf + 1, Wf + 1, C2)[..., :Hf, :Wf, :]
            return v.movedim(-1, -3).reshape(*v.shape[:-3], -1)

        _acc(P[pfx + ".layer.weight"], unperm(dWz))
        del dWz
        return self._norm_bwd(du, x, tape["mr_c"], wts["dense_g"], 1, Hf * Wf * C2, (P[pfx + ".norm.weight"], unperm),
                              (P[pfx + ".norm.bias"], unperm), zp=(Hf, Wf, C2)).view(N, Hf + 1, Wf + 1, C2)

    def _block_bwd(self, l, dzo, S, first_u8, W, P, B, t, last):
        """Backward of lib/util.py:193-211 (see policy.MinecraftPolicy._block for the forward in the same notation)."""
        cfg = self.policy.net.cfg
        h, heads, maxlen = cfg.hidsize, cfg.heads, cfg.maxlen
        b = f"recurrent_layer.blocks.{l}"
        o = f"{b}.r.orc_block"
        N = B * t
        nr = 10 * heads
        dz = dzo  # (last block: z is relu(..) (lib/policy.py:211 fused into its epilogue); lastlayer's norm backward already masked dzo)
        # mlp1: z = y + hmid W1^T + b1
        dh = self._gemm(dz, W["mlp1_t"], h * cfg.pointwise_ratio)
        self._wgrad_linear(dz, S["hmid"], P[f"{b}.mlp1.layer.weight"])
        _acc(P[f"{b}.mlp1.layer.bias"], ops.col_sums(dz)[1])
        # mlp0: hmid = relu(LN(y) W0^T)
        dzh = ops.relu_mask(dh, S["hmid"])
        del dh
        dy = self._normlinear_bwd(dzh, S["y"], S["mr_y"], W["mlp0_t"], f"{b}.mlp0", P, add=dz)
        del dzh
        # proj: y = xhat + a Wp^T + bp
        da = self._gemm(dy, W["proj_t"], h)
        self._wgrad_linear(dy, S["a"], P[f"{o}.proj_layer.weight"])
        _acc(P[f"{o}.proj_layer.bias"], ops.col_sums(dy)[1])
        # attention: gradients wrt q | k | v | R side by side (one buffer = one dgrad GEMM + one wgrad GEMM for all four)
        dqkvr = torch.zeros((N, self.kcat), dtype=BF16, device=dy.device)
        db_nd = ops.attention_bwd(S["q"], S["full_k"], S["full_v"], S["R"], P[f"{o}.b_nd"].detach().float().contiguous(), first_u8, S["smask"],
                                  da, dqkvr, B, t, maxlen, heads)
        _acc(P[f"{o}.b_nd"], db_nd)
        dxhat = self._gemm(dqkvr, W["qkvr_t"], h, residual=dy)
        dWc = self._wgrad_linear(dqkvr, S["xhat"])
        dbc = ops.col_sums(dqkvr)[1]
        _acc(P[f"{o}.q_layer.weight"], dWc[0:h])
        _acc(P[f"{o}.k_layer.weight"], dWc[h:2 * h])
        _acc(P[f"{o}.v_layer.weight"], dWc[2 * h:3 * h])
        _acc(P[f"{o}.r_layer.weight"], dWc[3 * h:3 * h + nr])
        _acc(P[f"{o}.q_layer.bias"], dbc[0:h])
        _acc(P[f"{o}.r_layer.bias"], dbc[3 * h:3 * h + nr])
        # pre_r_ln (plain norm of the block input)
        ident = lambda v: v
        g = P[f"{b}.pre_r_ln.weight"]
        return self._norm_bwd(dxhat, S["x"], S["mr_x"], g.detach().float().contiguous(), 1, h, (g, ident), (P[f"{b}.pre_r_ln.bias"], ident),
                              relu_x=(l == 0))  # block 0's input is relu(img_process.linear)

    def _cnn_bwd(self, dout, tape, wts, P):
        """Backward of lib/impala_cnn.py:187-195; `dout` is the gradient wrt the last stack's output (ZP)."""
        cfg = self.policy.net.cfg
        pfx = "img_process.cnn"
        ident = lambda v: v
        dx = dout
        for i in reversed(range(len(cfg.chans))):
            rec = tape["stacks"][i]
            s = f"{pfx}.stacks.{i}"
            H, W = rec["H_in"] // 2, rec["W_in"] // 2
            C = cfg.chans[i]
            R = dx.shape[0] * (H + 1) * (W + 1)
            for j in (1, 0):
                blk = rec["blocks"][j]
                self._dbg(f"{s}.blocks.{j}", dx)
                x_in = rec["blocks"][j - 1]["x"] if j == 1 else rec["x0"]
                mr_in = rec["blocks"][j - 1]["mr"] if j == 1 else rec["mr0"]
                # x_out = x_in + relu(conv1(GN(h)));  h = relu(conv0(GN(x_in)))
                dz1 = ops.relu_mask(dx, blk["r"])
                dz0 = self._normconv_bwd(dz1, blk["h"], blk["mrh"], H, W, wts["stacks"][i]["convs"][2 * j + 1], f"{s}.blocks.{j}.conv1", P,
                                         relu_x=True)
                del dz1
                dx = self._normconv_bwd(dz0, x_in, mr_in, H, W, wts["stacks"][i]["convs"][2 * j], f"{s}.blocks.{j}.conv0", P, add=dx)
                del dz0
            self._dbg(f"{s}.n", dx)
            # x0 = GN_n(y1) (plain norm)
            g = P[f"{s}.n.weight"]
            dy1 = self._norm_bwd(dx.view(R, C), rec["y1"].view(R, C), rec["mr1"], g.detach().float().contiguous(), (H + 1) * (W + 1), H * W * C,
                                 (g, ident), (P[f"{s}.n.bias"], ident), zp=(H, W, C)).view(rec["y1"].shape)
            self._dbg(f"{s}.pool", dy1)
            if i == 0:
                st = self.policy.net.prepared().stacks[0]
                dWk, db = ops.firstconv_bwd(tape["frames"], st["fc_w"], st["fc_b"], dy1, C)
                # kernel weights are W[c0][ky][kx][c] / 255 (lib/policy.py:44 folded in)
                _acc(P[f"{s}.firstconv.layer.weight"], (dWk / 255.0).view(C, 3, 3, 3).permute(0, 3, 1, 2))
                _acc(P[f"{s}.firstconv.layer.bias"], db)
            else:
                dfull = ops.maxpool3s2_bwd(dy1, rec["full"])  # includes the ReLU in front of the pool
                del dy1
                dx = self._normconv_bwd(dfull, rec["x_in"], rec["mr_in"], rec["H_in"], rec["W_in"], wts["stacks"][i]["first"],
                                        f"{s}.firstconv", P)
                del dfull


class RLTrainer(BCTrainer):
    """RL fine-tuning step of `MinecraftAgentPolicy`: clipped policy gradient, KL to a frozen pretrained teacher, entropy bonus and
    the value head's loss in normalised space (lib/action_head.py:176-220, lib/scaled_mse_head.py:37-43, lib/normalize_ewma.py:26-55).

        stats, state_out, teacher_state_out = tr.loss_and_grad(img, first, state_in, teacher_state_in, actions,
                                                               old_logp, advantages, returns, upper_grads_ready=None)

    One call covers N = B*T frames.  Per frame i: the taken action a_i (one index per head), old_logp_i (the joint log-prob recorded at
    rollout), the advantage A_i and the return R_i, all computed by the caller.  pd is the student's per-head log-softmax of the
    logits divided by the temperature (what `forward` returns), pd_t the teacher's, q = exp(pd):

        lp_i  = sum_h pd_h[i, a_h,i]                                          (joint, as `logprob`)
        r_i   = exp(lp_i - old_logp_i)
        pg_i  = -min(r_i A_i, clip(r_i, 1 - clip_eps, 1 + clip_eps) A_i)
        kl_i  = sum_h sum_j q_h,j (pd_h,j - pd_t,h,j)                          (= get_kl_of_action_dists(pd, pd_teacher): student first)
        ent_i = sum_h -sum_j q_h,j pd_h,j
        tn_i  = (R_i - mu) / sigma    with (mu, sigma^2) = running_mean_var() AFTER this batch's EWMA update (norm_axes = 2)
        loss  = mean_i pg_i + kl_coef mean_i kl_i - ent_coef mean_i ent_i + vf_coef mean_i (vpred_i - tn_i)^2

    vpred is the raw (normalised-space) value output.  Gradients wrt the temperature-scaled logits z of head h (times 1/temperature
    for the GEMM output): g_i (delta_ja - q_j) with g_i = -r_i A_i / N, or 0 where the clipped term is the minimum (r > 1 + clip_eps
    with A > 0, r < 1 - clip_eps with A < 0); (kl_coef/N) q_j ((pd_j - pd_t,j) - kl_h,i); (ent_coef/N) q_j (pd_j + H_h,i); and
    d/dvpred_i = 2 vf_coef (vpred_i - tn_i) / N.  All of it is one kernel (ops.rl_heads_bwd).  The value head sits in column ntot
    of the heads' gradient buffer, so its backward rides in the heads' dgrad / wgrad / bias-sum launches.

    The return normaliser (`value_head.normalizer.*`) is updated in place by every call with the batch mean and mean square of R,
    averaged over the ranks of an initialised torch.distributed group (one all-reduce of two floats), so every replica holds the
    normaliser a single process would hold for the global batch.  No step synchronises with the host.  The teacher (a frozen
    `MinecraftAgentPolicy` with the same heads) runs its bf16 inference forward on the same frames with its own KV memory; its
    parameters are never written.  `stats` holds 0-d device tensors: loss, pg, kl, entropy, value, clipfrac (the fraction of frames
    whose clipped term is the minimum, i.e. that pass no policy gradient).  bf16 only; heads with several sub-actions are refused."""

    value_column = True
    norm_beta = 0.99999  # NormalizeEwma defaults (lib/normalize_ewma.py:9): beta, epsilon, per_element_update=False
    norm_eps = 1e-5

    def __init__(self, policy: MinecraftAgentPolicy, teacher=None, *, clip_eps=0.2, kl_coef=0.0, ent_coef=0.0, vf_coef=1.0):
        super().__init__(policy)
        if policy.net.precision != "bf16":
            raise NotImplementedError("RLTrainer: bf16 precision only")
        if teacher is not None:
            if not isinstance(teacher, MinecraftAgentPolicy):
                raise TypeError("RLTrainer: the teacher is a MinecraftAgentPolicy")
            if teacher is policy:
                raise ValueError("RLTrainer: the teacher must be a separate, frozen policy (e.g. a copy of the pretrained weights)")
            if dict(teacher.head_specs) != dict(policy.head_specs):
                raise ValueError("RLTrainer: the teacher's action heads differ from the student's")
            if teacher.net.precision != "bf16":
                raise NotImplementedError("RLTrainer: bf16 precision only (teacher)")
        if kl_coef != 0 and teacher is None:
            raise ValueError("RLTrainer: kl_coef != 0 needs a teacher")
        self.teacher = teacher
        self.clip_eps, self.kl_coef, self.ent_coef, self.vf_coef = float(clip_eps), float(kl_coef), float(ent_coef), float(vf_coef)

    def _update_normalizer(self, returns):
        """EWMA update of value_head.normalizer with this batch (lib/normalize_ewma.py:37-52) -> fp32 [2] (mean, 1/std) after it."""
        nz = self.policy.value_head.normalizer
        R = returns.reshape(-1)
        mom = torch.stack([R.mean(), (R * R).mean()])
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(mom, op=dist.ReduceOp.SUM)  # equal shards: the mean of the rank means is the global batch mean
            mom = mom / dist.get_world_size()
        w = self.norm_beta
        with torch.no_grad():
            nz.running_mean.mul_(w).add_(mom[0:1] * (1.0 - w))
            nz.running_mean_sq.mul_(w).add_(mom[1:2] * (1.0 - w))
            nz.debiasing_term.mul_(w).add_(1.0 * (1.0 - w))
            deb = nz.debiasing_term.clamp(min=self.norm_eps)
            mean = nz.running_mean / deb
            var = (nz.running_mean_sq / deb - mean ** 2).clamp(min=1e-2)
            return torch.cat([mean, torch.rsqrt(var)]).to(F32).contiguous()

    def loss_and_grad(self, img, first, state_in, teacher_state_in, actions, old_logp, advantages, returns, upper_grads_ready=None):
        """`upper_grads_ready()`: as in BCTrainer.loss_and_grad (the value head's gradient is final by then)."""
        B, t = img.shape[:2]
        N = B * t
        for name, x in (("old_logp", old_logp), ("advantages", advantages), ("returns", returns)):
            if tuple(x.shape) != (B, t) or x.dtype != F32 or x.device != img.device:
                raise ValueError(f"RLTrainer: {name} must be a float32 ({B}, {t}) tensor on {img.device}, got {x.dtype} {tuple(x.shape)} on {x.device}")
        pd_t, teacher_state_out = None, None
        if self.teacher is not None:
            with torch.no_grad():
                (pd_t, _, _), st = self.teacher({"img": img}, first, teacher_state_in)
            teacher_state_out = [(m, (k.detach(), v.detach())) for (m, (k, v)) in st]
        mu_rsig = self._update_normalizer(returns)
        old, adv, ret = old_logp.reshape(N).contiguous(), advantages.reshape(N).contiguous(), returns.reshape(N).contiguous()

        def loss_block(pd, vpred, n_rows):
            pol = self.policy
            hp = pol._heads_prepared()
            dlog = torch.zeros((N, self.ld_logits), dtype=BF16, device=img.device)
            lps, lts, idx, cols = [], [], [], []
            for name, (shape, n) in pol.head_specs.items():
                c0, width = hp["cols"][name]
                if width != n:
                    raise NotImplementedError("RLTrainer: heads with several sub-actions are not trained")
                lps.append(pd[name].reshape(N, n))
                if pd_t is not None:
                    lts.append(pd_t[name].reshape(N, n))
                idx.append(actions[name].reshape(N).to(torch.int64).contiguous())
                cols.append(c0)
            rs = ops.rl_heads_bwd(lps, lts if pd_t is not None else None, idx, cols, old, adv, ret, vpred.reshape(N).contiguous(), mu_rsig,
                                  self.clip_eps, self.kl_coef, self.ent_coef, self.vf_coef, 1.0 / pol.temperature, 1.0 / N, dlog, self.ntot)
            m = rs.mean(0)  # (lp, kl, entropy, value loss, clipped)
            r = torch.exp(rs[:, 0] - old)
            pg = -torch.minimum(r * adv, r.clamp(1.0 - self.clip_eps, 1.0 + self.clip_eps) * adv).mean()
            loss = pg + self.kl_coef * m[1] - self.ent_coef * m[2] + self.vf_coef * m[3]
            return dlog, dict(loss=loss, pg=pg, kl=m[1], entropy=m[2], value=m[3], clipfrac=m[4])

        stats, state_out = self._step(img, first, state_in, loss_block, upper_grads_ready)
        return stats, state_out, teacher_state_out
