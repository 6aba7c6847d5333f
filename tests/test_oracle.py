"""CPU: pins oracle/vpt_oracle.py against (a) fixtures generated from the unmodified reference, (b) the reference's own
outputs recorded under tests/golden/reference/ for the comparisons below, (c) the invariants of SURVEY.md section 4."""
import glob
import os

import pytest
import torch

import make_golden
import vpt_oracle as O

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.pt")))


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p) for p in GOLD])
def test_oracle_matches_golden(path):
    fx = torch.load(path)
    cfg = O.Cfg(**fx["policy_kwargs"])
    sd = fx["state_dict"]
    st = O.initial_state(cfg, fx["B"])
    with torch.no_grad():
        for ch in fx["chunks"]:
            (pd, v, _), st = O.agent_policy_forward(sd, cfg, ch["img"], ch["first"], st)
            # same torch ops in the same order as the reference -> bit exact on the same machine; 1e-5 across machines
            assert torch.allclose(pd["camera"], ch["camera"], rtol=1e-5, atol=1e-5)
            assert torch.allclose(pd["buttons"][:, -1:], ch["buttons_last"], rtol=1e-5, atol=1e-5)
            assert torch.allclose(v, ch["vpred"], rtol=1e-5, atol=1e-5)
            assert torch.allclose(st[0][1][0], ch["k0"], rtol=1e-5, atol=1e-6)
            assert torch.allclose(st[0][1][1], ch["v0"], rtol=1e-5, atol=1e-6)
            for s, m in zip(st, ch["masks"]):
                assert torch.equal(s[0], m)
    if torch.equal(pd["camera"], fx["chunks"][-1]["camera"]):  # identical logits -> sampling must be bit exact
        torch.manual_seed(1234)
        ac = O.sample(pd)
        assert torch.equal(ac["camera"], fx["sample"]["camera"]) and torch.equal(ac["buttons"], fx["sample"]["buttons"])
        assert torch.allclose(O.logprob(pd, ac), fx["sample_logprob"])


def test_golden_fixtures_exist():
    assert len(GOLD) >= 2


def _record(name):
    """What the unmodified reference computed for the comparison, recorded by oracle/make_golden.py."""
    return torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference", name))


@pytest.mark.parametrize("pert", [False, True])
def test_oracle_matches_live_reference(pert):
    """B=3, 5 chunks of uneven length with a reset in the 4th: log-probs, vpred and every layer's state after each chunk, then
    seeded sampling, against the reference run on the same weights and frames (bit exact on the machine that recorded them)."""
    rec = _record(f"forward_{'perturbed' if pert else 'plain'}.pt")
    pkw = rec["policy_kwargs"]
    sd = make_golden.synth_state_dict(rec["weights"])
    cfg = O.Cfg(**pkw)
    B = rec["B"]
    g = torch.Generator().manual_seed(0)
    st_o = O.initial_state(cfg, B)
    for ci, (T, ch) in enumerate(zip([8, 8, 3, 8, 1], rec["chunks"])):
        img = torch.randint(0, 256, (B, T, 32, 32, 3), dtype=torch.uint8, generator=g)
        first = torch.zeros(B, T, dtype=torch.bool)
        if ci == 3:
            first[1, 0] = True
        with torch.no_grad():
            (pd2, v2, _), st_o = O.agent_policy_forward(sd, cfg, img, first, st_o)
        for k in pd2:
            make_golden.assert_digest(pd2[k], ch["pd"][k], rtol=1e-5, atol=1e-5, what=(ci, k))
        make_golden.assert_digest(v2, ch["v"], rtol=1e-5, atol=1e-5, what=(ci, "vpred"))
        for (m, dk, dv), (m2, (k2, v2_)) in zip(ch["state"], st_o):
            assert torch.equal(m, m2)
            make_golden.assert_digest(k2, dk, rtol=1e-5, atol=1e-6, what=(ci, "K"))
            make_golden.assert_digest(v2_, dv, rtol=1e-5, atol=1e-6, what=(ci, "V"))
    torch.manual_seed(7)
    a2 = O.sample(pd2)
    assert all(torch.equal(rec["sample"][k], a2[k]) for k in a2)
    assert torch.allclose(rec["logprob"], O.logprob(pd2, a2), rtol=1e-5, atol=1e-5)


def test_oracle_matches_live_reference_128px():
    """One full-size 128x128 frame through the 1x-width CNN path with reduced transformer (config C1 shape)."""
    rec = _record("forward_128px.pt")
    pkw = rec["policy_kwargs"]
    sd = make_golden.synth_state_dict(rec["weights"])
    cfg = O.Cfg(**pkw)
    img = torch.randint(0, 256, (1, 1, 128, 128, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    first = torch.zeros(1, 1, dtype=torch.bool)
    with torch.no_grad():
        (pd2, v2, _), _ = O.agent_policy_forward(sd, cfg, img, first, O.initial_state(cfg, 1))
    for k in ("buttons", "camera"):
        make_golden.assert_digest(pd2[k], rec["pd"][k], rtol=1e-5, atol=1e-5, what=k)
    make_golden.assert_digest(v2, rec["v"], rtol=1e-5, atol=1e-5, what="vpred")


def _tiny():
    fx = torch.load(GOLD[0])
    return fx["state_dict"], O.Cfg(**fx["policy_kwargs"])


def test_chunk_size_invariance():
    """SURVEY.md section 4 (i): N frames fed as chunks of 1/4/8 give the same logits."""
    sd, cfg = _tiny()
    img = torch.randint(0, 256, (2, 16, 32, 32, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(5))
    outs = []
    with torch.no_grad():
        for cs in (1, 4, 8):
            st, acc = O.initial_state(cfg, 2), []
            for t0 in range(0, 16, cs):
                (pd, _, _), st = O.agent_policy_forward(sd, cfg, img[:, t0:t0 + cs], torch.zeros(2, cs, dtype=torch.bool), st)
                acc.append(pd["camera"])
            outs.append(torch.cat(acc, 1))
    assert torch.allclose(outs[0], outs[1], atol=2e-5) and torch.allclose(outs[0], outs[2], atol=2e-5)


def test_reset_equals_fresh():
    """SURVEY.md section 4 (ii): first[b,0]=True at a chunk start == a fresh initial_state for that row."""
    sd, cfg = _tiny()
    g = torch.Generator().manual_seed(6)
    a = torch.randint(0, 256, (2, 8, 32, 32, 3), dtype=torch.uint8, generator=g)
    b = torch.randint(0, 256, (2, 8, 32, 32, 3), dtype=torch.uint8, generator=g)
    with torch.no_grad():
        _, st = O.agent_policy_forward(sd, cfg, a, torch.zeros(2, 8, dtype=torch.bool), O.initial_state(cfg, 2))
        first = torch.zeros(2, 8, dtype=torch.bool)
        first[:, 0] = True
        (pd1, _, _), _ = O.agent_policy_forward(sd, cfg, b, first, st)
        (pd2, _, _), _ = O.agent_policy_forward(sd, cfg, b, torch.zeros(2, 8, dtype=torch.bool), O.initial_state(cfg, 2))
    assert torch.allclose(pd1["buttons"], pd2["buttons"], atol=2e-5)


def test_flop_model_matches_survey():
    for w, gf in (("1x", 3.8213), ("2x", 15.0973), ("3x", 33.8278)):
        assert abs(O.forward_flops_per_frame(O.Cfg(**O.widths(w))) / 1e9 - gf) < 1e-3


def test_oracle_gradient_matches_live_reference_autograd():
    """The BC step's parity target is autograd through the oracle (tests/test_training.py); this pins that target itself: the
    gradient of the BC loss (behavioural_cloning.py:101-123: -log-prob of the demonstrated action, KV memory detached between
    chunks) through the unmodified reference equals the gradient through the oracle, parameter by parameter."""
    rec = _record("gradient.pt")
    pkw = rec["policy_kwargs"]
    sd = make_golden.synth_state_dict(rec["weights"])
    cfg = O.Cfg(**pkw)
    B, T = 2, 8
    g = torch.Generator().manual_seed(3)
    st_o = O.initial_state(cfg, B)
    for ch in rec["chunks"]:
        img = torch.randint(0, 256, (B, T, 32, 32, 3), dtype=torch.uint8, generator=g)
        first = torch.zeros(B, T, dtype=torch.bool)
        actions = {"camera": torch.randint(0, 121, (B, T, 1), generator=g), "buttons": torch.randint(0, 8641, (B, T, 1), generator=g)}
        leaf = {k: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in sd.items()}
        (pd_o, _, _), st_o = O.agent_policy_forward(leaf, cfg, img, first, st_o)
        loss_o = -O.logprob(pd_o, actions).mean()
        loss_o.backward()
        st_o = [(m, (k.detach(), v.detach())) for (m, (k, v)) in st_o]
        assert torch.allclose(ch["loss"], loss_o.detach(), rtol=1e-6, atol=0)
        n_checked = 0
        for name, d in ch["grads"].items():
            if d is None:
                assert leaf[name].grad is None, name  # value head: untouched by the BC loss in both
                continue
            # a recorded gradient comes from another machine, where fp32 sums run in another order: entries far below the
            # parameter's largest one carry that rounding, so the absolute slack is 1e-5 of the largest recorded entry
            scale = (d["full"] if "full" in d else d["sample"]).abs().max().item()
            make_golden.assert_digest(leaf[name].grad, d, rtol=1e-5, atol=1e-5 * scale, what=name)
            n_checked += 1
        assert n_checked > 80
