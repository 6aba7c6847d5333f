"""Generates tests/golden/ from the UNMODIFIED reference (run where a checkout of openai/Video-Pre-Training is present,
see oracle/refshim.py):

    python oracle/make_golden.py

`tiny_*.pt`: each fixture = {policy_kwargs, temperature, state_dict (fp32, reference schema), chunks: [{img u8, first bool,
camera log-probs, buttons log-probs of the chunk's last frame, vpred, state_out K/V of layer 0, state masks}], sample: indices under manual_seed(1234)}.
`tiny_*` use the smallest config the unmodified reference accepts (SURVEY.md section 4) so the files stay small; they pin
`oracle/vpt_oracle.py` on machines where the reference is absent (the GPU box).  The `perturbed` variant randomises every
norm affine / bias and scales q weights x30 so that layout mistakes that plain init hides (gamma=1, beta=0, near-uniform
attention) show up.

`reference/*`: what the reference computed in the comparisons of tests/test_oracle.py, tests/test_idm.py and
tests/test_agent.py, so that those tests need nothing outside the repository.  To keep the files small, the weights are not
stored: `weight_spec` keeps each tensor's shape, mean and spread, and the reference is run on `synth_state_dict(spec)`, which
the tests rebuild bit for bit; frames come from seeded generators in both places; large outputs are stored as `digest`s.
"""
import math
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import refshim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
REC = os.path.join(OUT, "reference")


def perturb(pol, seed=1):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in pol.named_parameters():
            if ".norm." in n or n.endswith(".bias") or "_ln." in n or ".n." in n:
                p.add_(torch.randn(p.shape, generator=g) * 0.1)
            if "q_layer.weight" in n:
                p.mul_(30.0)


def make(name, pkw, chunks, B, pert, seed=0):
    pol = refshim.make_reference_agent_policy(pkw, temperature=2.0, seed=seed)
    if pert:
        perturb(pol)
    g = torch.Generator().manual_seed(seed + 100)
    H, W, _ = pkw["img_shape"]
    st = pol.initial_state(B)
    rec = []
    with torch.no_grad():
        for ci, T in enumerate(chunks):
            img = torch.randint(0, 256, (B, T, H, W, 3), dtype=torch.uint8, generator=g)
            first = torch.zeros(B, T, dtype=torch.bool)
            if ci == 2:
                first[B - 1, 0] = True
            (pd, v, _), st = pol({"img": img}, first, st)
            rec.append(dict(img=img, first=first, camera=pd["camera"].clone(), buttons_last=pd["buttons"][:, -1:].clone(), vpred=v.clone(),
                            k0=st[0][1][0].clone(), v0=st[0][1][1].clone(), masks=[s[0].clone() for s in st]))
        torch.manual_seed(1234)
        ac = pol.pi_head.sample(pd)
        lp = pol.pi_head.logprob(ac, pd)
    fx = dict(policy_kwargs=pkw, temperature=2.0, B=B, state_dict={k: v.clone() for k, v in pol.state_dict().items()},
              chunks=rec, sample={k: v.clone() for k, v in ac.items()}, sample_logprob=lp.clone())
    os.makedirs(OUT, exist_ok=True)
    torch.save(fx, os.path.join(OUT, name + ".pt"))
    print(name, os.path.getsize(os.path.join(OUT, name + ".pt")) // 1024, "KiB")


# ------------------------------------------------------------------------------------------------------------------
# compact fixtures: synthetic weights, digests of large outputs (shared with the tests that read them)
# ------------------------------------------------------------------------------------------------------------------
def hashed_uniform(n, seed):
    """n float64 values in [-1, 1) from an integer hash of (seed, index): the same on every machine and torch version."""
    x = (torch.arange(n, dtype=torch.int64) * 0x9E3779B1 + (seed + 1) * 0x85EBCA77) & 0xFFFFFFFF
    x = ((x ^ (x >> 15)) * 0x2C1B3C6D) & 0xFFFFFFFF
    x = ((x ^ (x >> 12)) * 0x297A2D39) & 0xFFFFFFFF
    x = x ^ (x >> 15)
    return x.double() / 2.0 ** 31 - 1.0


def weight_spec(sd):
    """name -> (shape, mean, half-width) of every tensor: a uniform distribution with the tensor's mean and standard deviation."""
    spec = {}
    for k, v in sd.items():
        d = v.detach().double()
        spec[k] = (tuple(v.shape), float(d.mean()), float(d.std(unbiased=False)) * math.sqrt(3.0) if d.numel() > 1 else 0.0)
    return spec


def synth_state_dict(spec):
    """fp32 state_dict from `weight_spec` output; a constant tensor (norm gains, zero biases) comes back exactly."""
    return {k: (mean + half * hashed_uniform(math.prod(shape), i)).float().reshape(shape)
            for i, (k, (shape, mean, half)) in enumerate(spec.items())}


def sample_index(n, k):
    return ((hashed_uniform(k, n) + 1.0) * (n / 2.0)).long().clamp_(max=n - 1)


def digest(t, k=256):
    """A tensor of up to k entries as is; a larger one as k fixed entries plus its sum and absolute sum (float64)."""
    t = t.detach()
    if t.numel() <= k:
        return dict(full=t.clone())
    f = t.flatten().double()
    return dict(shape=tuple(t.shape), sample=t.flatten()[sample_index(f.numel(), k)].clone(), sum=float(f.sum()), abs_sum=float(f.abs().sum()))


def assert_digest(t, d, rtol, atol, what=""):
    """`t` against `digest` output: the kept entries elementwise, the whole tensor through its two sums, to the same tolerance."""
    t = t.detach().cpu()
    if "full" in d:
        assert t.shape == d["full"].shape and torch.allclose(t, d["full"], rtol=rtol, atol=atol), what
        return
    assert tuple(t.shape) == d["shape"], (what, tuple(t.shape), d["shape"])
    f = t.flatten().double()
    assert torch.allclose(t.flatten()[sample_index(f.numel(), len(d["sample"]))], d["sample"], rtol=rtol, atol=atol), what
    slack = rtol * d["abs_sum"] + atol * f.numel()
    assert abs(float(f.sum()) - d["sum"]) <= slack and abs(float(f.abs().sum()) - d["abs_sum"]) <= slack, what


def _reference_policy(pkw, pert):
    """The reference policy with `synth_state_dict` weights shaped like its own init (perturbed like `perturb` if asked)."""
    pol = refshim.make_reference_agent_policy(pkw)
    if pert:
        perturb(pol)
    spec = weight_spec(pol.state_dict())
    pol.load_state_dict(synth_state_dict(spec))
    return pol, spec


def _save(name, obj):
    os.makedirs(REC, exist_ok=True)
    path = os.path.join(REC, name)
    torch.save(obj, path)
    print(os.path.relpath(path, OUT), os.path.getsize(path) // 1024, "KiB")


def record_forward(pert):
    """tests/test_oracle.py::test_oracle_matches_live_reference: 5 chunks (one with a reset) and a seeded sample."""
    pkw = refshim.policy_kwargs("2x", **refshim.TINY)
    pol, spec = _reference_policy(pkw, pert)
    B = 3
    g = torch.Generator().manual_seed(0)
    st = pol.initial_state(B)
    chunks = []
    for ci, T in enumerate([8, 8, 3, 8, 1]):
        img = torch.randint(0, 256, (B, T, 32, 32, 3), dtype=torch.uint8, generator=g)
        first = torch.zeros(B, T, dtype=torch.bool)
        if ci == 3:
            first[1, 0] = True
        with torch.no_grad():
            (pd, v, _), st = pol({"img": img}, first, st)
        chunks.append(dict(pd={k: digest(x) for k, x in pd.items()}, v=digest(v),
                           state=[(m.clone(), digest(kk), digest(vv)) for m, (kk, vv) in st]))
    torch.manual_seed(7)
    a = pol.pi_head.sample(pd)
    _save(f"forward_{'perturbed' if pert else 'plain'}.pt",
          dict(policy_kwargs=pkw, weights=spec, B=B, chunks=chunks, sample={k: x.clone() for k, x in a.items()},
               logprob=pol.pi_head.logprob(a, pd).detach().clone()))


def record_forward_128px():
    """tests/test_oracle.py::test_oracle_matches_live_reference_128px: one 128x128 frame, 1x width, one transformer layer."""
    pkw = refshim.policy_kwargs("1x", n_recurrence_layers=1)
    pol, spec = _reference_policy(pkw, False)
    img = torch.randint(0, 256, (1, 1, 128, 128, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        (pd, v, _), _ = pol({"img": img}, torch.zeros(1, 1, dtype=torch.bool), pol.initial_state(1))
    _save("forward_128px.pt", dict(policy_kwargs=pkw, weights=spec, pd={k: digest(x) for k, x in pd.items()}, v=digest(v)))


def record_gradient():
    """tests/test_oracle.py::test_oracle_gradient_matches_live_reference_autograd: BC loss and per-parameter gradients."""
    pkw = refshim.policy_kwargs("2x", **refshim.TINY)
    pol, spec = _reference_policy(pkw, True)
    pol.train()
    B, T = 2, 8
    g = torch.Generator().manual_seed(3)
    st = pol.initial_state(B)
    chunks = []
    for _ in range(2):
        img = torch.randint(0, 256, (B, T, 32, 32, 3), dtype=torch.uint8, generator=g)
        first = torch.zeros(B, T, dtype=torch.bool)
        actions = {"camera": torch.randint(0, 121, (B, T, 1), generator=g), "buttons": torch.randint(0, 8641, (B, T, 1), generator=g)}
        for p in pol.parameters():
            p.grad = None
        (pd, _, _), st = pol({"img": img}, first, st)
        loss = -pol.pi_head.logprob(actions, pd).mean()
        loss.backward()
        st = [(m, (k.detach(), v.detach())) for (m, (k, v)) in st]
        chunks.append(dict(loss=loss.detach().clone(),
                           grads={n: None if p.grad is None else digest(p.grad, 64) for n, p in pol.named_parameters()}))
    _save("gradient.pt", dict(policy_kwargs=pkw, weights=spec, chunks=chunks))


def _idm_kwargs(**kw):
    import vpt_b200

    return vpt_b200.idm_net_kwargs(**kw)


def record_idm():
    """tests/test_idm.py::test_idm_schema_and_oracle_match_live_reference: IDM forward, and the reference's parameter schema at
    a config the CUDA path supports."""
    sys.path.insert(0, os.path.dirname(HERE))
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
    from test_idm import SMALL_IDM

    ns = refshim.load()
    kw = _idm_kwargs(impala_width=1, hidsize=64, attention_heads=2, img_shape=[32, 32, 16],
                     conv3d_params=dict(inchan=3, outchan=16, kernel_size=[5, 1, 1], padding=[2, 0, 0]), timesteps=8,
                     attention_memory_size=8)
    mapper = ns.action_mapping.IDMActionMapping(n_camera_bins=11)
    space = ns.DictType(**mapper.get_action_space_update())
    torch.manual_seed(0)
    ref = ns.policy.InverseActionPolicy(action_space=space, pi_head_kwargs=dict(temperature=2.0), idm_net_kwargs=kw)
    ref.eval()
    spec = weight_spec(ref.state_dict())
    ref.load_state_dict(synth_state_dict(spec))
    img = torch.randint(0, 256, (2, 8, 32, 32, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        (pd, _, _), _ = ref(obs={"img": img}, first=torch.zeros(2, 8), state_in=ref.initial_state(2))
    ref2 = ns.policy.InverseActionPolicy(action_space=space, pi_head_kwargs=dict(temperature=2.0), idm_net_kwargs=_idm_kwargs(**SMALL_IDM))
    _save("idm.pt", dict(idm_net_kwargs=kw, weights=spec, pd={k: digest(x) for k, x in pd.items()},
                         schema_small=[(k, tuple(v.shape)) for k, v in ref2.state_dict().items()]))


def record_codec():
    """tests/test_agent.py::test_codec_matches_live_reference: the reference's action mapping and transformer on seeded inputs."""
    import numpy as np

    sys.path.insert(0, os.path.dirname(HERE))
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
    from test_agent import _random_factored, A

    ns = refshim.load()
    import lib.actions as ref_actions

    mapper = ns.action_mapping.CameraHierarchicalMapping(n_camera_bins=11)
    tr = ref_actions.ActionTransformer(**A.ACTION_TRANSFORMER_KWARGS)
    rng = np.random.default_rng(0)
    out = dict(n_combinations=len(mapper.BUTTONS_COMBINATIONS), idx_to_factored=mapper.BUTTON_IDX_TO_FACTORED,
               idx_camera_off=mapper.BUTTON_IDX_TO_CAMERA_META_OFF, null_buttons_idx=mapper.get_zero_action()["buttons"],
               camera_null_idx=mapper.camera_null_idx)
    joint = dict(buttons=rng.integers(0, 8641, (500, 1)), camera=rng.integers(0, 121, (500, 1)))
    out.update({"to_factored." + k: v for k, v in mapper.to_factored({k: v.copy() for k, v in joint.items()}).items()})
    fac = _random_factored(2000, rng)
    out.update({"from_factored." + k: v for k, v in mapper.from_factored({k: v.copy() for k, v in fac.items()}).items()})
    out.update({"policy2env." + k: v for k, v in tr.policy2env({k: v.copy() for k, v in fac.items()}).items()})
    env = {"camera": rng.uniform(-15, 15, (300, 2)), "attack": rng.integers(0, 2, 300), "hotbar.3": rng.integers(0, 2, 300)}
    out.update({"env2policy." + k: v for k, v in tr.env2policy(env).items()})
    os.makedirs(REC, exist_ok=True)
    path = os.path.join(REC, "codec.npz")
    np.savez_compressed(path, **{k: np.asarray(v) for k, v in out.items()})
    print(os.path.relpath(path, OUT), os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    tiny = refshim.policy_kwargs("2x", impala_width=1, hidsize=32, attention_heads=2, img_shape=[32, 32, 3], timesteps=8,
                                 attention_memory_size=16, n_recurrence_layers=2)
    make("tiny_plain", tiny, [8, 3, 8, 1], B=2, pert=False)
    make("tiny_perturbed", tiny, [8, 3, 8, 1], B=2, pert=True)
    record_forward(False)
    record_forward(True)
    record_forward_128px()
    record_gradient()
    record_idm()
    record_codec()
