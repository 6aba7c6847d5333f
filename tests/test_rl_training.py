"""RL fine-tuning step (training.RLTrainer) on CPU: the hand-written step against autograd through the oracle of the objective in
the trainer's docstring, the return normaliser against a restatement of lib/normalize_ewma.py:26-55, the reduction to BC, and the
data-parallel step (gloo, world 2).  The loss kernel's CPU emulation lives here (`emu_rl_heads_bwd`) and is patched into `ops` by
the `rl_emulated` fixture, on top of the tests/emu_ops.py emulation of every other op."""
import inspect
import os
import socket
import sys

import pytest
import torch

import vpt_oracle as O
from common import make_policy, small_kwargs
from test_host_logic import emulated  # noqa: F401  (fixture)
from test_training import exact  # noqa: F401  (fixture)
from video_pre_training_b200 import ops
from video_pre_training_b200.training import BCTrainer, RLTrainer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 0.2


def emu_rl_heads_bwd(logp, logp_teacher, idx, cols, old_logp, adv, ret, vpred, mu_rsig, clip_eps, kl_coef, ent_coef, vf_coef, inv_temp, inv_n,
                     dlog, col_v):
    """fp64 emulation of vpt_rl_heads_bwd (include/vpt_b200.h), rounded once to dlog's dtype / fp32 statistics."""
    rows = logp[0].shape[0]
    ar = torch.arange(rows)
    lp = torch.zeros(rows, dtype=torch.float64)
    kls, ents, qs, pds, pts = [], [], [], [], []
    for h, a in enumerate(logp):
        a = a.double()
        q = torch.exp(a)
        b = logp_teacher[h].double() if logp_teacher is not None else a
        lp = lp + a[ar, idx[h].long()]
        kls.append((q * (a - b)).sum(1))
        ents.append(-(q * a).sum(1))
        qs.append(q), pds.append(a), pts.append(b)
    A = adv.double()
    r = torch.exp(lp - old_logp.double())
    clipped = ((A > 0) & (r > 1 + clip_eps)) | ((A < 0) & (r < 1 - clip_eps))
    g = torch.where(clipped, torch.zeros_like(r), -r * A * inv_n)
    kc, ec = kl_coef * inv_n, ent_coef * inv_n
    for h in range(len(logp)):
        gz = qs[h] * (kc * (pds[h] - pts[h] - kls[h][:, None]) + ec * (pds[h] + ents[h][:, None]) - g[:, None])
        gz[ar, idx[h].long()] += g
        dlog[:, cols[h]:cols[h] + gz.shape[1]] = (gz * inv_temp).to(dlog.dtype)
    mu, rsig = mu_rsig.double()
    dv = vpred.double() - (ret.double() - mu) * rsig
    dlog[:, col_v] = (2 * vf_coef * dv * inv_n).to(dlog.dtype)
    return torch.stack([lp, sum(kls), sum(ents), dv * dv, clipped.double()], 1).float()


@pytest.fixture()
def rl_emulated(emulated, monkeypatch):
    monkeypatch.setattr(ops, "rl_heads_bwd", emu_rl_heads_bwd)
    yield


def test_emulation_mirrors_the_rl_op():
    assert list(inspect.signature(ops.rl_heads_bwd).parameters) == list(inspect.signature(emu_rl_heads_bwd).parameters)


def ewma(norm, R, beta=0.99999):
    """lib/normalize_ewma.py:37-55 restated: (running_mean, running_mean_sq, debiasing_term) after the batch R, and (mean, std)."""
    m, msq, deb = [t.clone() for t in norm]
    bm, bsq = R.mean(dim=(0, 1)), (R ** 2).mean(dim=(0, 1))
    m = m * beta + bm * (1.0 - beta)
    msq = msq * beta + bsq * (1.0 - beta)
    deb = deb * beta + 1.0 * (1.0 - beta)
    mean = m / deb.clamp(min=1e-5)
    var = (msq / deb.clamp(min=1e-5) - mean ** 2).clamp(min=1e-2)
    return (m, msq, deb), (mean, torch.sqrt(var))


def norm_bufs(pol):
    nz = pol.value_head.normalizer
    return tuple(t.detach().clone() for t in (nz.running_mean, nz.running_mean_sq, nz.debiasing_term))


def oracle_rl(sd, sd_t, cfg, img, first, state, state_t, actions, old, adv, ret, mean, std, kl_coef, ent_coef, vf_coef):
    """The objective of the RLTrainer docstring by autograd through the oracle -> (parts, grads, state_out, teacher state_out)."""
    leaf = {k: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in sd.items()}
    (pd, vpred, _), st = O.agent_policy_forward(leaf, cfg, img, first, state)
    with torch.no_grad():
        (pd_t, _, _), st_t = O.agent_policy_forward(sd_t, cfg, img, first, state_t)
    lp = O.logprob(pd, actions)
    r = torch.exp(lp - old)
    pg = -torch.minimum(r * adv, r.clamp(1 - EPS, 1 + EPS) * adv).mean()
    kl = sum((torch.exp(pd[k]) * (pd[k] - pd_t[k])).sum(-1).sum(-1) for k in pd).mean()
    ent = sum(-(torch.exp(pd[k]) * pd[k]).sum(-1).sum(-1) for k in pd).mean()
    vl = ((vpred[..., 0] - (ret - mean) / std) ** 2).mean()
    loss = pg + kl_coef * kl - ent_coef * ent + vf_coef * vl
    loss.backward()
    parts = dict(loss=loss, pg=pg, kl=kl, entropy=ent, value=vl)
    return {k: v.detach() for k, v in parts.items()}, {k: v.grad for k, v in leaf.items()}, st, st_t


def _batch(g, B, T):
    img = torch.randint(0, 256, (B, T, 32, 32, 3), dtype=torch.uint8, generator=g)
    actions = {"camera": torch.randint(0, 121, (B, T, 1), generator=g), "buttons": torch.randint(0, 8641, (B, T, 1), generator=g)}
    return img, actions


def _ratios(g, B, T):
    """Target ratios in the three clip branches, each >= 0.05 from a boundary (1 -/+ EPS), and advantages of both signs."""
    k = torch.randint(0, 3, (B, T), generator=g)
    u = torch.rand(B, T, generator=g)
    r = torch.where(k == 0, 0.55 + 0.2 * u, torch.where(k == 1, 0.85 + 0.3 * u, 1.25 + 0.3 * u))
    adv = torch.randn(B, T, generator=g)
    adv = adv + 0.2 * torch.sign(adv)
    return r, adv


def test_rl_step_is_the_exact_gradient(rl_emulated, exact):
    """fp32 in place of bf16: RLTrainer's gradient of every parameter (value_head.linear.* included) and its loss parts equal autograd
    through the oracle, over two chunks with carried student and teacher KV memory, an episode reset in the second chunk, advantages
    of both signs and frames in all three clip branches."""
    kc, ec, vc = 0.3, 0.05, 0.5
    pol, sd, cfg = make_policy(small_kwargs(), seed=0)
    teacher, sd_t, _ = make_policy(small_kwargs(), seed=5)
    B, T = 2, 8
    tr = RLTrainer(pol, teacher, clip_eps=EPS, kl_coef=kc, ent_coef=ec, vf_coef=vc)
    g = torch.Generator().manual_seed(0)
    st, st_t = pol.initial_state(B), teacher.initial_state(B)
    st_o, st_to = O.initial_state(cfg, B), O.initial_state(cfg, B)
    norm = norm_bufs(pol)
    branches = set()
    for c in range(2):
        img, actions = _batch(g, B, T)
        first = torch.zeros(B, T, dtype=torch.bool)
        if c == 1:
            first[1, 0] = True
        with torch.no_grad():
            (pd_o, _, _), _ = O.agent_policy_forward(sd, cfg, img, first, st_o)
        lp = O.logprob(pd_o, actions)
        r, adv = _ratios(g, B, T)
        old = (lp - torch.log(r)).float()
        ret = torch.randn(B, T, generator=g) * 3 + 1.5
        branches |= set(torch.where(r < 1 - EPS, 0, torch.where(r > 1 + EPS, 2, 1)).flatten().tolist())
        norm, (mean, std) = ewma(norm, ret[..., None])
        for p in pol.parameters():
            p.grad = None
        stats, st, st_t = tr.loss_and_grad(img, first, st, st_t, actions, old, adv, ret)
        parts, grads_o, st_o, st_to = oracle_rl(sd, sd_t, cfg, img, first, st_o, st_to, actions, old, adv, ret, mean, std, kc, ec, vc)
        st_o = [(m, (k.detach(), v.detach())) for (m, (k, v)) in st_o]
        for k, v in parts.items():
            assert abs(stats[k].item() - v.item()) < 1e-3 * abs(v.item()) + 1e-6, (k, stats[k].item(), v.item())
        assert 0 < stats["clipfrac"].item() < 1
        for t_in, t_o in zip(st_t, st_to):
            assert torch.allclose(t_in[1][0], t_o[1][0], rtol=1e-4, atol=1e-5)
        bad = {}
        for n, p in pol.named_parameters():
            g_o = grads_o[n]
            if g_o is None:
                assert p.grad is None, n
                continue
            assert p.grad is not None, n
            e = ((p.grad - g_o).norm() / g_o.norm().clamp(min=1e-12)).item()
            if e > 5e-2:
                bad[n] = e
        assert not bad, bad
        for n in ("value_head.linear.weight", "value_head.linear.bias", "pi_head.buttons.linear_layer.weight"):
            assert ((pol.get_parameter(n).grad - grads_o[n]).norm() / grads_o[n].norm()).item() < 1e-3, n
    assert branches == {0, 1, 2}
    for a, b in zip(norm_bufs(pol), norm):
        assert torch.allclose(a, b, rtol=1e-6, atol=0)


def test_normalizer_follows_normalize_ewma(rl_emulated):
    """After two steps the normaliser buffers equal lib/normalize_ewma.py:37-52 restated; `denormalize` reads the new values."""
    pol, _, _ = make_policy(small_kwargs())
    tr = RLTrainer(pol)
    g = torch.Generator().manual_seed(3)
    B, T = 2, 8
    norm = norm_bufs(pol)
    st = pol.initial_state(B)
    for _ in range(2):
        img, actions = _batch(g, B, T)
        ret = torch.randn(B, T, generator=g) * 5 - 2
        zeros = torch.zeros(B, T)
        _, st, _ = tr.loss_and_grad(img, torch.zeros(B, T, dtype=torch.bool), st, None, actions, zeros, zeros, ret)
        norm, (mean, std) = ewma(norm, ret[..., None])
    for a, b in zip(norm_bufs(pol), norm):
        assert a.shape == b.shape and torch.allclose(a, b, rtol=1e-6, atol=0)
    v = torch.tensor([[[0.7]]])
    assert torch.allclose(pol.denormalize(v), v * std + mean, rtol=1e-6)


def test_one_relayout_per_parameter_change(rl_emulated):
    """The normaliser update bumps its buffers' versions, but the kernel-side weights are re-laid out only when a parameter changed."""
    pol, _, _ = make_policy(small_kwargs())
    tr = RLTrainer(pol)
    counts = {"bwd": 0, "heads": 0}

    def counted(key, fn):
        def f(*a, **k):
            counts[key] += 1
            return fn(*a, **k)
        return f

    tr._build_weights = counted("bwd", tr._build_weights)
    pol._build_heads_prepared = counted("heads", pol._build_heads_prepared)
    g = torch.Generator().manual_seed(4)
    img, actions = _batch(g, 1, 8)
    first, z = torch.zeros(1, 8, dtype=torch.bool), torch.zeros(1, 8)
    ret = torch.randn(1, 8, generator=g)
    seen = []
    for change in (False, False, True, False):
        if change:
            with torch.no_grad():
                pol.value_head.linear.weight.mul_(1.01)  # what an optimizer step does to the versions
        tr.loss_and_grad(img, first, pol.initial_state(1), None, actions, z, z, ret)
        seen.append(dict(counts))
    assert seen == [{"bwd": 1, "heads": 1}, {"bwd": 1, "heads": 1}, {"bwd": 2, "heads": 2}, {"bwd": 2, "heads": 2}], seen


def test_rl_reduces_to_bc(rl_emulated, exact):
    """A = 1, old_logp = this forward's joint log-prob, all three coefficients 0: the policy-gradient term's gradient is the NLL's,
    so every gradient equals BCTrainer's and the value head's is zero."""
    pol, _, _ = make_policy(small_kwargs(), seed=2)
    g = torch.Generator().manual_seed(5)
    B, T = 2, 8
    img, actions = _batch(g, B, T)
    first = torch.zeros(B, T, dtype=torch.bool)
    (pd, _, _), _ = pol({"img": img}, first, pol.initial_state(B))
    old = pol.logprob(actions, pd).float()
    loss_bc, _ = BCTrainer(pol).loss_and_grad(img, first, pol.initial_state(B), actions)
    g_bc = {n: p.grad.clone() for n, p in pol.named_parameters() if p.grad is not None}
    for p in pol.parameters():
        p.grad = None
    tr = RLTrainer(pol, clip_eps=EPS, kl_coef=0.0, ent_coef=0.0, vf_coef=0.0)
    stats, _, _ = tr.loss_and_grad(img, first, pol.initial_state(B), None, actions, old, torch.ones(B, T), torch.randn(B, T, generator=g))
    assert abs(stats["pg"].item() + 1.0) < 1e-6 and stats["clipfrac"].item() == 0.0
    for n, p in pol.named_parameters():
        if n.startswith("value_head.normalizer"):
            continue
        if n.startswith("value_head"):
            assert p.grad is not None and (p.grad == 0).all(), n
            continue
        assert ((p.grad - g_bc[n]).norm() / g_bc[n].norm()).item() < 1e-5, n


def test_rl_trainer_input_checks(rl_emulated):
    pol, _, _ = make_policy(small_kwargs())
    with pytest.raises(ValueError):
        RLTrainer(pol, kl_coef=0.1)  # the KL term needs a teacher
    with pytest.raises(ValueError):
        RLTrainer(pol, pol)
    tr = RLTrainer(pol)
    g = torch.Generator().manual_seed(6)
    img, actions = _batch(g, 1, 8)
    first, z = torch.zeros(1, 8, dtype=torch.bool), torch.zeros(1, 8)
    for bad in (torch.zeros(8), torch.zeros(1, 8, dtype=torch.float64), torch.zeros(1, 7)):
        with pytest.raises(ValueError):
            tr.loss_and_grad(img, first, pol.initial_state(1), None, actions, z, bad, z)


# ---- data parallel (gloo, world 2) ------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rl_case():
    """Identical replicas of the student and the teacher, and the global batch."""
    pol, _, _ = make_policy(small_kwargs(), seed=0)
    teacher, _, _ = make_policy(small_kwargs(), seed=5)
    tr = RLTrainer(pol, teacher, kl_coef=0.2, ent_coef=0.01, vf_coef=0.5)
    B, T = 4, 8
    g = torch.Generator().manual_seed(0)
    img, actions = _batch(g, B, T)
    first = torch.zeros(B, T, dtype=torch.bool)
    old = -14.0 + 0.3 * torch.randn(B, T, generator=g)
    adv = torch.randn(B, T, generator=g)
    ret = torch.randn(B, T, generator=g) * 2 + 1
    return pol, tr, (img, first, actions, old, adv, ret)


def _rl_worker(rank, world, port, q):
    for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(2)
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    import vpt_b200  # noqa: F401
    from common import emulation
    from test_rl_training import _rl_case, emu_rl_heads_bwd, norm_bufs
    from video_pre_training_b200 import ops, parallel

    pol, tr, (img, first, actions, old, adv, ret) = _rl_case()
    B = img.shape[0]
    opt = parallel.FlatAdamDP(list(pol.parameters()), lr=1e-3)  # value_head.linear.* included; the normaliser is not a parameter
    split = opt.offset_of(pol.net.img_process.cnn.dense.norm.weight)
    assert 0 < split < opt.offset_of(pol.value_head.linear.weight) < opt.n
    lo, hi = parallel.shard_range(B, rank, world)
    sh = lambda x: x[lo:hi]
    with emulation():
        ops.rl_heads_bwd = emu_rl_heads_bwd  # (restored with the other ops when the context exits)
        opt.zero_grad()
        tr.loss_and_grad(sh(img), sh(first), pol.initial_state(hi - lo), pol.initial_state(hi - lo), {k: sh(v) for k, v in actions.items()},
                         sh(old), sh(adv), sh(ret), upper_grads_ready=lambda: opt.reduce_async(split, opt.n))
        w = opt.reduce_gradients()
    q.put((rank, w, (opt.flat_g / w).numpy(), torch.cat([t.reshape(-1) for t in norm_bufs(pol)]).numpy()))  # by value, not shared memory
    dist.destroy_process_group()


def test_rl_data_parallel_equals_the_global_batch_gloo(rl_emulated):
    """RL step over 2 ranks (clips sharded, one all-reduce of the flat gradient bucket overlapped with the CNN backward): the averaged
    gradient equals the global batch's in one process; the normaliser, updated with the all-reduced batch moments, is identical on
    both ranks and equal to the single-process update."""
    import torch.multiprocessing as mp

    from video_pre_training_b200.parallel import FlatAdamDP

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_rl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted((q.get(timeout=600) for _ in ps), key=lambda r: r[0])
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    pol, tr, (img, first, actions, old, adv, ret) = _rl_case()
    opt = FlatAdamDP(list(pol.parameters()), lr=1e-3)
    opt.zero_grad()
    B = img.shape[0]
    tr.loss_and_grad(img, first, pol.initial_state(B), pol.initial_state(B), actions, old, adv, ret)
    bufs1 = torch.cat([t.reshape(-1) for t in norm_bufs(pol)])
    (_, w0, g0, b0), (_, w1, g1, b1) = [(r, w, torch.from_numpy(g), torch.from_numpy(b)) for r, w, g, b in res]
    assert w0 == w1 == 2 and torch.equal(g0, g1)
    err = ((g0 - opt.flat_g).norm() / opt.flat_g.norm()).item()
    sl = slice(opt.offset_of(pol.value_head.linear.weight), opt.offset_of(pol.value_head.linear.weight) + pol.value_head.linear.weight.numel())
    v_err = ((g0[sl] - opt.flat_g[sl]).norm() / opt.flat_g[sl].norm()).item()
    assert err < 2e-2 and v_err < 2e-2, (err, v_err)
    assert torch.equal(b0, b1)
    assert torch.allclose(b0, bufs1, rtol=1e-6, atol=0), (b0, bufs1)
