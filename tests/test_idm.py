"""IDM (BASELINE config 5, SURVEY a19): InverseActionPolicy = conv3d pre-stage + ImpalaCNN (first conv normalised) +
unmasked transformer + factored heads.  CPU: host logic through the emulated ops vs the oracle (itself pinned to the
reference, tests/test_idm.py::test_idm_schema_and_oracle_match_live_reference).  GPU: the CUDA path vs the oracle."""
import os

import pytest
import torch

import emu_ops
import make_golden
import vpt_b200
import vpt_oracle as O
from common import perturb
from video_pre_training_b200 import ops

SMALL_IDM = dict(impala_width=4, hidsize=256, attention_heads=2, img_shape=[32, 32, 64],
                 conv3d_params=dict(inchan=3, outchan=64, kernel_size=[5, 1, 1], padding=[2, 0, 0]), timesteps=8, attention_memory_size=8)


def _make(kw, pert=True):
    torch.manual_seed(0)
    pol = vpt_b200.InverseActionPolicy(vpt_b200.idm_action_space(), dict(temperature=2.0), kw)
    if pert:
        perturb(pol)
    sd = {k: v.detach().clone() for k, v in pol.state_dict().items()}
    cfg = O.Cfg(conv3d=True, **{k: v for k, v in kw.items() if k != "conv3d_params"})
    return pol, sd, cfg


def _compare(pol, sd, cfg, dev, B=2, T=8, hw=32):
    img = torch.randint(0, 256, (B, T, hw, hw, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    first = torch.zeros(B, T, dtype=torch.bool)
    ac, st, res = pol.predict({"img": img.to(dev)}, first=first.to(dev), state_in=pol.initial_state(B), deterministic=True)
    with torch.no_grad():
        (pd_o, _, _), st_o = O.idm_policy_forward(sd, cfg, img, first, O.initial_state(cfg, B))
    for k in pd_o:
        got = res["pd"][k].float().cpu()
        assert got.shape == pd_o[k].shape
        # binary / 11-way heads: log-probs approach 0, so a pure relative bound is ill-conditioned.  Measured bf16 error of
        # this path: rel-L2 0.4-0.9 %, max |err| 0.03-0.045 on log-probs of magnitude ~0.7-2.4 -> the 1e-2 bf16 tolerance
        # holds in the L2 sense only; the max-norm gap is recorded in DESIGN.md section 6 (precision).
        err = (got - pd_o[k]).abs()
        l2 = ((got - pd_o[k]).norm() / pd_o[k].norm()).item()
        print(f"IDM {k}: rel-L2 {l2:.3g}, max abs err {err.max().item():.3g}")
        assert l2 < 1e-2 and err.max() < 6e-2, (k, l2, err.max().item())
    assert ac["buttons"].shape == (B, T, 20) and ac["camera"].shape == (B, T, 2) and res["log_prob"].shape == (B, T)
    assert st[0][0] is None and tuple(st[0][1][0].shape) == (B, 0, cfg.hidsize)   # mask "none": empty KV state forever
    ac_o = O.sample(pd_o, deterministic=True)
    agree = sum((ac[k].cpu() == ac_o[k]).float().mean().item() for k in ac_o) / 2
    # random-init binary heads are nearly tied (p ~ 0.5), so the argmax flips under bf16 noise; bit-exactness of the sampler
    # itself given identical logits is tested in test_gpu_kernels.py::test_heads_tail
    assert agree > 0.85, agree


@pytest.fixture()
def emulated(monkeypatch):
    for name in dir(emu_ops):
        if not name.startswith("_") and callable(getattr(emu_ops, name)) and hasattr(ops, name):
            monkeypatch.setattr(ops, name, getattr(emu_ops, name))
    yield


def test_idm_host_logic_matches_oracle(emulated):
    pol, sd, cfg = _make(vpt_b200.idm_net_kwargs(**SMALL_IDM), pert=False)
    _compare(pol, sd, cfg, "cpu")


def test_idm_schema_and_oracle_match_live_reference():
    """The oracle's IDM forward against the reference's, recorded by oracle/make_golden.py on the same weights and frames, and
    the product's parameter schema against the reference's at a config the CUDA path supports."""
    rec = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference", "idm.pt"))
    kw = rec["idm_net_kwargs"]
    sd = make_golden.synth_state_dict(rec["weights"])
    cfg = O.Cfg(conv3d=True, **{k: v for k, v in kw.items() if k != "conv3d_params"})
    img = torch.randint(0, 256, (2, 8, 32, 32, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        (pd2, _, _), _ = O.idm_policy_forward(sd, cfg, img, torch.zeros(2, 8, dtype=torch.bool), O.initial_state(cfg, 2))
    assert set(pd2) == set(rec["pd"])
    for k in pd2:
        make_golden.assert_digest(pd2[k], rec["pd"][k], rtol=1e-5, atol=1e-5, what=k)
    # product schema == reference schema at a config the CUDA path supports
    ours, _, _ = _make(vpt_b200.idm_net_kwargs(**SMALL_IDM), pert=False)
    assert [(k, tuple(v.shape)) for k, v in ours.state_dict().items()] == rec["schema_small"]


@pytest.mark.gpu
def test_idm_small_gpu():
    from video_pre_training_b200 import _native as nat
    pol, sd, cfg = _make(vpt_b200.idm_net_kwargs(**SMALL_IDM), pert=False)
    _compare(pol.to("cuda"), sd, cfg, "cuda")
    nat.device_check()


@pytest.mark.gpu
def test_idm_fullsize_frames_gpu():
    """128x128 frames, conv3d 3->128, 1x-width CNN behind it (the full 4x IDM is exercised by tools/idm_bench.py)."""
    from video_pre_training_b200 import _native as nat
    kw = vpt_b200.idm_net_kwargs(impala_width=4, hidsize=1024, attention_heads=8, timesteps=6, attention_memory_size=6)
    pol, sd, cfg = _make(kw, pert=False)
    _compare(pol.to("cuda"), sd, cfg, "cuda", B=1, T=6, hw=128)
    nat.device_check()


@pytest.mark.gpu
def test_conv3d_kernel():
    from video_pre_training_b200 import _native as nat
    g = torch.Generator().manual_seed(2)
    for (B, T, H, W, C) in [(2, 5, 16, 16, 64), (1, 3, 32, 32, 128), (3, 1, 16, 16, 64)]:
        img = torch.randint(0, 256, (B, T, H, W, 3), dtype=torch.uint8, generator=g)
        w = torch.randn(C, 15, generator=g) / 255.0 * 0.3
        b = torch.randn(C, generator=g) * 0.1
        got, gmr = ops.conv3d_t5(img.cuda(), w.cuda(), b.cuda(), C)
        nat.device_check()
        ref, rmr = emu_ops.conv3d_t5(img, w, b, C)
        assert (got.float().cpu() - ref.float()).abs().max() < 2e-2 and torch.allclose(gmr.cpu(), rmr, rtol=2e-3, atol=2e-3)
        gc = got.cpu()
        assert (gc[:, -1] == 0).all() and (gc[:, :, -1] == 0).all()


def test_idm_agent_predict_actions_emulated(emulated, monkeypatch):
    """inverse_dynamics_model.py:75-95 mirror: frames in, MineRL action dict out (host glue around InverseActionPolicy.predict)."""
    import numpy as np

    from video_pre_training_b200 import agent as A

    monkeypatch.setattr(A, "AGENT_RESOLUTION", (32, 32))  # the small test model sees 32x32 frames: no resize on the CPU
    kw = vpt_b200.idm_net_kwargs(**SMALL_IDM)
    torch.manual_seed(0)
    ag = vpt_b200.IDMAgent(kw, dict(temperature=2.0), device="cpu")
    frames = np.random.default_rng(0).integers(0, 256, (8, 32, 32, 3), dtype=np.uint8)
    act = ag.predict_actions(frames)
    assert set(act) == set(A.BUTTONS) | {"camera"}
    assert act["camera"].shape == (1, 8, 2) and act["attack"].shape == (1, 8) and set(np.unique(act["attack"])) <= {0, 1}
    assert np.all(np.abs(act["camera"]) <= 10.0)
    # same heads through the policy API
    ac, _, _ = ag.policy.predict({"img": torch.from_numpy(frames)[None]}, first=torch.zeros(1, 8, dtype=torch.bool),
                                 state_in=ag.policy.initial_state(1), deterministic=True)
    assert np.array_equal(act["attack"], ac["buttons"][..., A.BUTTONS.index("attack")].numpy())
    assert np.allclose(act["camera"], ag.codec.undiscretize_camera(ac["camera"].numpy()))
    ag.reset()
    assert ag.hidden_state[0][0] is None
