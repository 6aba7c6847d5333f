"""RL fine-tuning step on the GPU (training.RLTrainer): the loss kernel against its emulation at the real head widths, the new part of
the backward (heads + value head) against fp32 autograd from the taped latent, the whole step against the emulated step, the reduction
to BC, a few optimizer steps, and one step at the 3x production shapes."""
import copy

import pytest
import torch

import vpt_b200
from common import emulation, make_policy, small_kwargs
from test_rl_training import EPS, emu_rl_heads_bwd
from video_pre_training_b200 import _native as nat
from video_pre_training_b200 import ops
from video_pre_training_b200.parallel import FlatAdamDP
from video_pre_training_b200.training import BCTrainer, RLTrainer

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF16 = torch.bfloat16
WIDTHS = (121, 8641)


def rel(a, b):
    return ((a.float().cpu() - b.float().cpu()).norm() / b.float().cpu().norm().clamp(min=1e-20)).item()


def _branch_ratios(g, shape):
    """Ratios in all three clip branches, >= 0.05 from a boundary; advantages of both signs, away from 0."""
    k = torch.arange(shape[0] * shape[1]).reshape(shape) % 3
    u = torch.rand(shape, generator=g)
    r = torch.where(k == 0, 0.55 + 0.2 * u, torch.where(k == 1, 0.85 + 0.3 * u, 1.25 + 0.3 * u))
    adv = torch.randn(shape, generator=g)
    return r, adv + 0.2 * torch.sign(adv)


@pytest.mark.parametrize("N", [37, 2048])
@pytest.mark.parametrize("teacher", [False, True])
def test_rl_heads_kernel_matches_emulation(N, teacher):
    g = torch.Generator().manual_seed(N + teacher)
    logp = [torch.log_softmax(torch.randn(N, n, generator=g) * 2, -1) for n in WIDTHS]
    logp_t = [torch.log_softmax(torch.randn(N, n, generator=g) * 2, -1) for n in WIDTHS] if teacher else None
    idx = [torch.randint(0, n, (N,), generator=g) for n in WIDTHS]
    lp = (logp[0].gather(1, idx[0][:, None]) + logp[1].gather(1, idx[1][:, None]))[:, 0]
    r, adv = _branch_ratios(g, (N, 1))
    old = (lp - torch.log(r[:, 0])).float()
    adv = adv[:, 0].contiguous()
    ret = torch.randn(N, generator=g) * 3 + 1
    vpred = torch.randn(N, generator=g)
    mu_rsig = torch.tensor([0.7, 1.0 / 2.5])
    cols, ld, col_v = [0, 121], 8768, 8762
    args = (0.2, 0.3 if teacher else 0.0, 0.05, 0.5, 0.5, 1.0 / N)
    out_e = torch.zeros(N, ld, dtype=BF16)
    st_e = emu_rl_heads_bwd(logp, logp_t, idx, cols, old, adv, ret, vpred, mu_rsig, *args, out_e, col_v)
    out = torch.zeros(N, ld, dtype=BF16, device=DEV)
    cu = lambda ts: None if ts is None else [t.to(DEV) for t in ts]
    st = ops.rl_heads_bwd(cu(logp), cu(logp_t), cu(idx), cols, old.to(DEV), adv.to(DEV), ret.to(DEV), vpred.to(DEV), mu_rsig.to(DEV), *args, out,
                          col_v)
    nat.device_check()
    assert set(st_e[:, 4].tolist()) == {0.0, 1.0}
    out, st = out.cpu(), st.cpu()
    # bf16 outputs: the kernel rounds an fp32 value, the emulation an fp64 one
    assert rel(out, out_e) < 4e-3 and (out.float() - out_e.float()).abs().max() <= 2 ** -7 * out_e.float().abs().max()
    assert (out[:, 8763:] == 0).all()
    assert torch.equal(st[:, 4], st_e[:, 4])
    for c in range(4):
        assert torch.allclose(st[:, c], st_e[:, c], rtol=1e-5, atol=1e-5 * st_e[:, c].abs().max().item()), c


def _case(seed, B, T, hw=32):
    g = torch.Generator().manual_seed(seed)
    img = torch.randint(0, 256, (B, T, hw, hw, 3), dtype=torch.uint8, generator=g)
    first = torch.zeros(B, T, dtype=torch.bool)
    actions = {"camera": torch.randint(0, 121, (B, T, 1), generator=g), "buttons": torch.randint(0, 8641, (B, T, 1), generator=g)}
    return g, img, first, actions


def _to(d, x):
    return {k: v.to(d) for k, v in x.items()} if isinstance(x, dict) else x.to(d)


def _joint_logprob(pol, img, first, state, actions):
    """This forward's joint log-prob of the actions, as the trainer's loss kernel sees it (recorded from its statistics)."""
    rec = []
    orig = ops.rl_heads_bwd

    def spy(*a):
        rec.append(orig(*a))
        return rec[-1]

    B, T = img.shape[:2]
    z = torch.zeros(B, T, device=img.device)
    nz = pol.value_head.normalizer
    bufs = [t.detach().clone() for t in (nz.running_mean, nz.running_mean_sq, nz.debiasing_term)]
    ops.rl_heads_bwd = spy
    try:
        RLTrainer(pol, vf_coef=0.0).loss_and_grad(img, first, state, None, actions, z, z, z)
    finally:
        ops.rl_heads_bwd = orig
        with torch.no_grad():  # leave the normaliser as it was
            for t, b in zip((nz.running_mean, nz.running_mean_sq, nz.debiasing_term), bufs):
                t.copy_(b)
    for p in pol.parameters():
        p.grad = None
    return rec[0][:, 0].view(B, T).clone()


def test_heads_and_value_backward_match_autograd_from_the_taped_latent():
    """The new part of the backward, pinned tightly: fp32 autograd of the objective through the heads and the value head, from the
    taped bf16 latent and the bf16 head weights the GEMMs use, against the trainer's d latent and its pi_head.* / value_head.linear.*
    gradients (rel-L2 < 1e-2, TF32 off).  The trunk below the latent is pinned by test_gpu_training.py."""
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        kc, ec, vc = 0.3, 0.05, 0.5
        pol, _, _ = make_policy(small_kwargs(), seed=0)
        teacher, _, _ = make_policy(small_kwargs(), seed=5)
        pol, teacher = pol.to(DEV), teacher.to(DEV)
        B, T = 3, 8
        g, img, first, actions = _case(1, B, T)
        img, first, actions = img.to(DEV), first.to(DEV), _to(DEV, actions)
        lp = _joint_logprob(pol, img, first, pol.initial_state(B), actions)
        r, adv = _branch_ratios(g, (B, T))
        old = lp - torch.log(r).to(DEV)
        adv = adv.to(DEV)
        ret = (torch.randn(B, T, generator=g) * 3 + 1).to(DEV)
        tr = RLTrainer(pol, teacher, clip_eps=EPS, kl_coef=kc, ent_coef=ec, vf_coef=vc)
        tr.keep_tape, tr.debug_grads = True, {}
        stats, _, _ = tr.loss_and_grad(img, first, pol.initial_state(B), teacher.initial_state(B), actions, old, adv, ret)
        nat.device_check()
        with torch.no_grad():
            (pd_t, _, _), _ = teacher({"img": img}, first, teacher.initial_state(B))
        nz = pol.value_head.normalizer
        deb = nz.debiasing_term.clamp(min=1e-5)
        mean = nz.running_mean / deb
        std = torch.sqrt((nz.running_mean_sq / deb - mean ** 2).clamp(min=1e-2))
        lat = tr.last_tape["latent"].float().requires_grad_(True)
        # the GEMMs read bf16 weights and fp32 biases
        leaf = {n: (p.detach().to(BF16).float() if n.endswith("weight") else p.detach().clone()).requires_grad_(True)
                for n, p in pol.named_parameters() if n.startswith(("pi_head", "value_head.linear"))}
        N = B * T
        lp_a, kl, ent = 0, 0, 0
        for name, (_, n) in pol.head_specs.items():
            z = (lat @ leaf[f"pi_head.{name}.linear_layer.weight"].T + leaf[f"pi_head.{name}.linear_layer.bias"]) / pol.temperature
            pd = torch.log_softmax(z, -1)
            q = torch.exp(pd)
            lp_a = lp_a + pd.gather(1, actions[name].reshape(N, 1))[:, 0]
            kl = kl + (q * (pd - pd_t[name].reshape(N, n))).sum(-1)
            ent = ent - (q * pd).sum(-1)
        vpred = (lat @ leaf["value_head.linear.weight"].T + leaf["value_head.linear.bias"])[:, 0]
        rr = torch.exp(lp_a - old.reshape(N))
        A = adv.reshape(N)
        pg = -torch.minimum(rr * A, rr.clamp(1 - EPS, 1 + EPS) * A).mean()
        vl = ((vpred - (ret.reshape(N) - mean) / std) ** 2).mean()
        loss = pg + kc * kl.mean() - ec * ent.mean() + vc * vl
        loss.backward()
        parts = dict(pg=pg, kl=kc * kl.mean(), entropy=-ec * ent.mean(), value=vc * vl)
        scale = sum(abs(v.item()) for v in parts.values())
        for k, v in parts.items():
            got = stats[k].item() * {"pg": 1.0, "kl": kc, "entropy": -ec, "value": vc}[k]
            assert abs(got - v.item()) < 1e-3 * scale, (k, got, v.item())
        assert abs(stats["loss"].item() - loss.item()) < 1e-3 * scale, (stats["loss"].item(), loss.item())
        errs = {"latent": rel(tr.debug_grads["latent"], lat.grad)}
        for n, t in leaf.items():
            errs[n] = rel(pol.get_parameter(n).grad, t.grad)
        print("rel-L2 vs fp32 autograd from the taped latent:", {k: f"{v:.2e}" for k, v in errs.items()})
        for n, e in errs.items():
            assert e < 1e-2, (n, e)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old_tf32


def test_rl_step_matches_emulated_step():
    """The whole step through the kernels against the same step through the emulated ops (same bf16 rounding points), at the BC
    step's tolerances (tests/test_gpu_training.py: top-of-network parameters 5 %, the rest 60 %, loss 2e-3)."""
    pol, _, _ = make_policy(small_kwargs(), seed=0)
    teacher, _, _ = make_policy(small_kwargs(), seed=5)
    B, T = 2, 8
    g, img, first, actions = _case(2, B, T)
    # ratios >= 0.1 inside their clip branch (a frame whose branch flips between the two bf16 forwards moves the head gradient like a
    # flipped ReLU mask): the emulated forward's joint log-prob minus log of a target ratio
    with emulation(), torch.no_grad():
        (pd, _, _), _ = pol({"img": img}, first, pol.initial_state(B))
        lp = pol.logprob(actions, pd)
    k = torch.arange(B * T).reshape(B, T) % 3
    u = torch.rand(B, T, generator=g)
    old = lp - torch.log(torch.where(k == 0, 0.5 + 0.15 * u, torch.where(k == 1, 0.9 + 0.2 * u, 1.3 + 0.2 * u)))
    adv = torch.randn(B, T, generator=g)
    ret = torch.randn(B, T, generator=g) * 2
    kw = dict(kl_coef=0.2, ent_coef=0.02, vf_coef=0.5)
    pol_e = copy.deepcopy(pol)
    saved = ops.rl_heads_bwd
    with emulation():
        ops.rl_heads_bwd = emu_rl_heads_bwd
        try:
            stats_e, _, _ = RLTrainer(pol_e, copy.deepcopy(teacher), **kw).loss_and_grad(img, first, pol_e.initial_state(B), teacher.initial_state(B),
                                                                                        actions, old, adv, ret)
        finally:
            ops.rl_heads_bwd = saved
    pol, teacher = pol.to(DEV), teacher.to(DEV)
    stats, _, _ = RLTrainer(pol, teacher, **kw).loss_and_grad(img.to(DEV), first.to(DEV), pol.initial_state(B), teacher.initial_state(B),
                                                              _to(DEV, actions), old.to(DEV), adv.to(DEV), ret.to(DEV))
    nat.device_check()
    # kl, entropy: the BC loss's 2e-3.  pg (and the loss) moves by |r A| per unit of joint log-prob, and the BC tolerance lets
    # the log-prob of the two bf16 forwards differ by 2e-3 of the NLL (~0.03 here): an absolute bound of 0.03 * 2 mean|A|.
    tol_pg = 0.03 * 2 * adv.abs().mean().item()
    print({k: (round(stats[k].item(), 5), round(stats_e[k].item(), 5)) for k in stats})
    for k in ("kl", "entropy"):
        assert abs(stats[k].item() - stats_e[k].item()) < 2e-3 * abs(stats_e[k].item()) + 1e-5, (k, stats[k].item(), stats_e[k].item())
    # vpred is one projection of the latent, which two bf16 forwards give to ~1 % (measured: value loss 0.75 % apart on B200)
    assert abs(stats["value"].item() - stats_e["value"].item()) < 2e-2 * stats_e["value"].item()
    for k in ("pg", "loss"):
        assert abs(stats[k].item() - stats_e[k].item()) < tol_pg, (k, stats[k].item(), stats_e[k].item())
    errs = {}
    for (n, p), (_, p_e) in zip(pol.named_parameters(), pol_e.named_parameters()):
        if n.startswith("value_head.normalizer"):
            assert torch.allclose(p.cpu(), p_e, rtol=1e-6), n
            continue
        assert p.grad is not None and torch.isfinite(p.grad).all(), n
        errs[n] = rel(p.grad, p_e.grad)
    print("rel-L2 vs emulated step:", " ".join(f"{e:.3f}" for e in errs.values()))
    for n, e in errs.items():
        top = n.startswith(("pi_head", "value_head", "net.final_ln"))
        assert e < (0.05 if top else 0.6), (n, e)


def test_rl_reduces_to_bc_on_the_gpu():
    """A = 1, old_logp = this forward's joint log-prob, all coefficients 0: every gradient equals BCTrainer's (rel-L2 <= 1e-6), the
    value head's is zero."""
    pol, _, _ = make_policy(small_kwargs(), seed=3)
    pol = pol.to(DEV)
    B, T = 2, 8
    g, img, first, actions = _case(3, B, T)
    img, first, actions = img.to(DEV), first.to(DEV), _to(DEV, actions)
    old = _joint_logprob(pol, img, first, pol.initial_state(B), actions)
    BCTrainer(pol).loss_and_grad(img, first, pol.initial_state(B), actions)
    g_bc = {n: p.grad.clone() for n, p in pol.named_parameters() if p.grad is not None}
    for p in pol.parameters():
        p.grad = None
    tr = RLTrainer(pol, kl_coef=0.0, ent_coef=0.0, vf_coef=0.0)
    stats, _, _ = tr.loss_and_grad(img, first, pol.initial_state(B), None, actions, old, torch.ones(B, T, device=DEV),
                                   torch.randn(B, T, device=DEV))
    nat.device_check()
    assert stats["clipfrac"].item() == 0.0
    bitwise, worst = True, 0.0
    for n, p in pol.named_parameters():
        if n.startswith("value_head.normalizer"):
            continue
        if n.startswith("value_head"):
            assert (p.grad == 0).all(), n
            continue
        bitwise &= bool(torch.equal(p.grad, g_bc[n]))
        worst = max(worst, rel(p.grad, g_bc[n]))
    print(f"RL(A=1, coefficients 0) vs BC: worst rel-L2 {worst:.2e}, bitwise equal: {bitwise}")
    assert worst <= 1e-6


def test_rl_training_learns_and_leaves_the_teacher_alone():
    """FlatAdamDP steps on one fixed batch with positive advantages on its actions raise their log-prob and lower the value loss; with
    the teacher a copy of the student the first step's KL is the bf16 rounding difference of the two forward paths only (the student's
    taped training forward normalises stack.n in a pass of its own, the teacher's inference forward folds it into the next conv;
    measured 1.0e-4 on B200, where a pd difference of one percent would give ~1e-2); the teacher's parameters are bitwise unchanged."""
    pol, _, _ = make_policy(small_kwargs(), seed=1)
    teacher = copy.deepcopy(pol)
    pol, teacher = pol.to(DEV), teacher.to(DEV)
    t0 = {n: p.detach().clone() for n, p in teacher.state_dict().items()}
    B, T = 4, 8
    g, img, first, actions = _case(4, B, T)
    img, first, actions = img.to(DEV), first.to(DEV), _to(DEV, actions)
    old = _joint_logprob(pol, img, first, pol.initial_state(B), actions)
    adv = torch.ones(B, T, device=DEV)
    ret = (torch.randn(B, T, generator=g) * 2 + 3).to(DEV)
    tr = RLTrainer(pol, teacher, kl_coef=0.1, ent_coef=0.01, vf_coef=1.0)
    opt = FlatAdamDP(list(pol.parameters()), lr=5e-4)
    hist = []
    for _ in range(10):
        opt.zero_grad()
        stats, _, _ = tr.loss_and_grad(img, first, pol.initial_state(B), teacher.initial_state(B), actions, old, adv, ret)
        opt.step()
        hist.append({k: v.item() for k, v in stats.items()})
    nat.device_check()
    lp_after = _joint_logprob(pol, img, first, pol.initial_state(B), actions)
    print("kl / value / pg per step:", [(round(h["kl"], 6), round(h["value"], 4), round(h["pg"], 4)) for h in hist])
    assert abs(hist[0]["kl"]) < 1e-3 and hist[-1]["kl"] > 10 * abs(hist[0]["kl"])
    assert hist[-1]["value"] < hist[0]["value"]
    assert (lp_after - old).mean().item() > 0.05, (lp_after - old).mean().item()
    assert all(torch.equal(p, t0[n]) for n, p in teacher.state_dict().items())


def test_rl_step_at_3x_width_shapes():
    """BASELINE configs[3] shapes (3x width, 128x128 frames, 128-frame memory) with a 3x teacher, B = 2, T = 128: the step finishes with
    finite gradients and no device-side error."""
    torch.manual_seed(0)
    mk = lambda: vpt_b200.MinecraftAgentPolicy(vpt_b200.minecraft_action_space(), vpt_b200.policy_kwargs("3x"), vpt_b200.PI_HEAD_KWARGS).to(DEV)
    pol, teacher = mk(), mk()
    B, T = 2, 128
    g, img, first, actions = _case(7, B, T, hw=128)
    img, first, actions = img.to(DEV), first.to(DEV), _to(DEV, actions)
    tr = RLTrainer(pol, teacher, kl_coef=0.1, ent_coef=0.01, vf_coef=0.5)
    opt = FlatAdamDP(list(pol.parameters()), lr=1e-4)
    opt.zero_grad()
    old = -12.0 + torch.randn(B, T, generator=g).to(DEV)
    stats, st, st_t = tr.loss_and_grad(img, first, pol.initial_state(B), teacher.initial_state(B), actions, old, torch.randn(B, T, device=DEV),
                                       torch.randn(B, T, device=DEV))
    assert torch.isfinite(opt.flat_g).all() and opt.flat_g.abs().sum() > 0
    assert pol.value_head.linear.weight.grad.abs().sum() > 0
    opt.step()
    nat.device_check()
    assert all(torch.isfinite(v) for v in stats.values())
    assert len(st) == len(st_t) == 4 and st_t[0][1][0].shape == (B, 128, 3072)
