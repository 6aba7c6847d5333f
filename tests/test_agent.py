"""Caller-side rows f-2 (frame ingest) and f-3 (action codec) + the MineRLAgent mirror.
CPU: the codec against recorded outputs of the reference (lib/action_mapping.py, lib/actions.py), codec
properties, the resize oracle against cv2.  GPU: the resize kernel bit-exact against the oracle / cv2, agent smoke."""
import os

import numpy as np
import pytest
import torch

import resize_oracle
import vpt_b200
from video_pre_training_b200 import agent as A

try:
    import cv2
except Exception:  # pragma: no cover
    cv2 = None


def _random_factored(n, rng):
    btn = (rng.random((n, 20)) < 0.25).astype(np.int64)
    cam = rng.integers(0, 11, (n, 2))
    cam[rng.random(n) < 0.4] = 5
    return dict(buttons=btn, camera=cam)


def test_codec_matches_live_reference():
    """The codec against the reference's action mapping and action transformer on the same seeded inputs (outputs recorded by
    oracle/make_golden.py)."""
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference", "codec.npz"))
    codec = A.ActionCodec(**A.ACTION_TRANSFORMER_KWARGS)
    assert codec.n_buttons_joint == ref["n_combinations"] == 8641
    assert np.array_equal(codec.idx_to_factored, ref["idx_to_factored"])
    assert np.array_equal(codec.idx_camera_off, ref["idx_camera_off"])

    def same(out, prefix):
        keys = sorted(k[len(prefix):] for k in ref.files if k.startswith(prefix))
        assert sorted(out) == keys and all(np.array_equal(out[k], ref[prefix + k]) for k in keys), prefix

    rng = np.random.default_rng(0)
    joint = dict(buttons=rng.integers(0, 8641, (500, 1)), camera=rng.integers(0, 121, (500, 1)))
    same(codec.to_factored(joint), "to_factored.")
    fac = _random_factored(2000, rng)
    same(codec.from_factored(fac), "from_factored.")
    same(codec.policy2env(fac), "policy2env.")
    env = {"camera": rng.uniform(-15, 15, (300, 2)), "attack": rng.integers(0, 2, 300), "hotbar.3": rng.integers(0, 2, 300)}
    same(codec.env2policy(env), "env2policy.")
    assert codec.null_buttons_idx == ref["null_buttons_idx"] and codec.camera_null_idx == ref["camera_null_idx"]


def test_codec_properties():
    codec = A.ActionCodec(**A.ACTION_TRANSFORMER_KWARGS)
    # every joint index survives joint -> factored -> joint, except that a non-null camera choice is dropped when the
    # button combination has the camera meta action off (lib/action_mapping.py:222-223)
    b = np.arange(8641)[:, None]
    for cam in (60, 0, 120, 37):
        fac = codec.to_factored(dict(buttons=b, camera=np.full_like(b, cam)))
        back = codec.from_factored(fac)
        off = codec.idx_camera_off[b[:, 0]]
        assert np.array_equal(back["camera"][off, 0], np.full(off.sum(), 60))
        assert np.array_equal(back["buttons"][off, 0], b[off, 0])          # meta-off combinations are fixed points
        on = ~off
        on[codec.inventory_idx] = False                                    # inventory is exclusive with the camera (:204-208)
        if cam != 60:  # (a camera-meta-ON combination whose camera choice is null maps back to its meta-OFF twin)
            assert np.array_equal(back["buttons"][on, 0], b[on, 0]) and np.all(back["camera"][on, 0] == cam)
        assert back["buttons"][codec.inventory_idx, 0] == codec.inventory_idx and back["camera"][codec.inventory_idx, 0] == 60
    # mu-law quantiser: bins 0..10 <-> [-10, 10], null bin 5 <-> 0, monotone, inverse on the bin centres
    centres = codec.undiscretize_camera(np.arange(11))
    assert centres[5] == 0 and np.all(np.diff(centres) > 0) and abs(centres[0] + 10) < 1e-9 and abs(centres[10] - 10) < 1e-9
    assert np.array_equal(codec.discretize_camera(centres), np.arange(11))


@pytest.mark.skipif(cv2 is None, reason="cv2 not importable")
def test_resize_oracle_is_bit_exact_with_cv2():
    rng = np.random.default_rng(0)
    for (H, W) in [(360, 640), (720, 1280), (128, 128), (200, 300), (431, 777), (129, 1399)]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        ref = cv2.resize(img, (128, 128), interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(resize_oracle.resize_linear_u8(img, 128, 128), ref), (H, W)


@pytest.mark.skipif(cv2 is None, reason="cv2 not importable")
def test_product_resize_tables_match_cv2_on_many_source_sizes():
    """ADVICE round 1: the product's coefficient tables (agent._linear_tables, fx computed in float like resize.cpp) driven through the
    oracle's integer arithmetic == cv2 for source sizes beyond the reference's 640x360 / 1280x720; exact 2x downscales are refused."""
    rng = np.random.default_rng(2)
    for (H, W) in [(360, 640), (720, 1280), (240, 320), (150, 200), (211, 333), (300, 500), (129, 129), (700, 1000), (300, 257)]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        xi, xa = A._linear_tables(128, W)
        yi, ya = A._linear_tables(128, H)
        src = img.astype(np.int64)
        hor = src[:, xi, :] * xa[None, :, 0, None].astype(np.int64) + src[:, np.minimum(xi + 1, W - 1), :] * xa[None, :, 1, None].astype(np.int64)
        out = ((ya[:, 0, None, None].astype(np.int64) * (hor[yi] >> 4)) >> 16) + ((ya[:, 1, None, None].astype(np.int64) * (hor[np.minimum(yi + 1, H - 1)] >> 4)) >> 16)
        got = np.clip((out + 2) >> 2, 0, 255).astype(np.uint8)
        assert np.array_equal(got, cv2.resize(img, (128, 128), interpolation=cv2.INTER_LINEAR)), (H, W)


@pytest.mark.gpu
def test_resize_kernel_bit_exact():
    rng = np.random.default_rng(1)
    for (F_, H, W) in [(3, 360, 640), (1, 720, 1280), (2, 431, 777)]:
        img = rng.integers(0, 256, (F_, H, W, 3), dtype=np.uint8)
        got = A.resize_frames(torch.from_numpy(img).cuda()).cpu().numpy()
        for f in range(F_):
            assert np.array_equal(got[f], resize_oracle.resize_linear_u8(img[f], 128, 128))
            if cv2 is not None:
                assert np.array_equal(got[f], cv2.resize(img[f], (128, 128), interpolation=cv2.INTER_LINEAR))
    with pytest.raises(NotImplementedError):  # exact 2x: OpenCV switches to INTER_AREA
        A.resize_frames(torch.zeros((1, 256, 256, 3), dtype=torch.uint8, device="cuda"))


@pytest.mark.gpu
def test_minerl_agent_rollout_smoke():
    kw = vpt_b200.policy_kwargs("1x", n_recurrence_layers=1)
    torch.manual_seed(0)
    agent = A.MineRLAgent(device="cuda", policy_kwargs=kw, pi_head_kwargs=vpt_b200.PI_HEAD_KWARGS)
    rng = np.random.default_rng(2)
    for _ in range(3):
        act = agent.get_action({"pov": rng.integers(0, 256, (360, 640, 3), dtype=np.uint8)})
        assert set(act) == set(A.BUTTONS) | {"camera"} and act["camera"].shape == (1, 2) and act["attack"].shape == (1,)
    agent.reset()
    back = agent._env_action_to_agent({k: (np.asarray(v) if k == "camera" else np.asarray(v)) for k, v in act.items()})
    assert back["buttons"].shape == (1, 1) and back["camera"].shape == (1, 1)


def test_checkpoint_io_roundtrip(tmp_path):
    """f-4: `.model` pickle -> constructor kwargs (run_agent.py:11-14), `.weights` round trip on the reference schema
    (agent.py:132-135, behavioural_cloning.py:131-132), optimizer state save / resume."""
    import pickle

    import vpt_b200
    from common import make_policy, small_kwargs
    from video_pre_training_b200.parallel import FlatAdamDP

    kw = small_kwargs()
    model_file = tmp_path / "tiny.model"
    with open(model_file, "wb") as fh:  # the layout of the released .model files
        pickle.dump({"model": {"args": {"net": {"args": kw}, "pi_head_opts": {"temperature": "2.0"}}}}, fh)
    pk, hk = vpt_b200.load_model_parameters(str(model_file))
    assert pk == kw and hk == {"temperature": 2.0} and isinstance(hk["temperature"], float)

    pol, sd, _ = make_policy(kw, seed=3)
    opt = FlatAdamDP([p for n, p in pol.named_parameters() if not n.startswith("value_head")], lr=1e-3, weight_decay=0.01)
    assert pol.net.final_ln.weight.data_ptr() >= opt.flat_p.data_ptr()  # parameters now live in the flat bucket
    vpt_b200.save_weights(pol, str(tmp_path / "a.weights"))
    loaded = torch.load(tmp_path / "a.weights")
    assert list(loaded.keys()) == list(sd.keys()) and all(torch.equal(loaded[k], sd[k]) for k in sd)
    assert all(v.is_contiguous() and v.untyped_storage().nbytes() == v.numel() * v.element_size() for v in loaded.values())

    pol2, _, _ = make_policy(kw, seed=4)
    opt2 = FlatAdamDP([p for n, p in pol2.named_parameters() if not n.startswith("value_head")], lr=5e-4)
    opt.exp_avg.normal_(); opt.exp_avg_sq.uniform_(); opt.t = 17
    vpt_b200.save_training_state(str(tmp_path / "run.pt"), pol, opt)
    vpt_b200.load_training_state(str(tmp_path / "run.pt"), pol2, opt2)
    assert all(torch.equal(a, b) for a, b in zip(pol.state_dict().values(), pol2.state_dict().values()))
    assert torch.equal(opt.exp_avg, opt2.exp_avg) and torch.equal(opt.exp_avg_sq, opt2.exp_avg_sq)
    assert opt2.t == 17 and opt2.lr == 1e-3 and opt2.weight_decay == 0.01
    assert pol2.net.final_ln.weight.data_ptr() >= opt2.flat_p.data_ptr()  # still aliased after the in-place load


def _cursor(rng):
    png = rng.integers(0, 256, (16, 16, 4), dtype=np.uint8)  # stand-in for cursors/mouse_cursor_white_16x16.png (BGRA)
    png[:4, :4, 3] = 0
    png[4:8, 4:8, 3] = 255
    return np.ascontiguousarray(png[:, :, :3]), png[:, :, 3:] / 255.0  # data_loader.py:78-83


def test_ingest_oracle_matches_reference_arithmetic():
    """The oracle's cursor overlay is the reference's numpy expression (data_loader.py:34-45), incl. clipping at the border, and
    its ingest = overlay -> cv2.cvtColor(BGR2RGB) -> cv2.resize, checked against cv2 where it is importable."""
    rng = np.random.default_rng(5)
    cur, alpha = _cursor(rng)
    frame = rng.integers(0, 256, (360, 640, 3), dtype=np.uint8)
    for (x, y) in [(0, 0), (100, 37), (630, 350), (639, 359), (700, 10)]:
        got = resize_oracle.composite_cursor(frame.copy(), cur, alpha, x, y)
        exp = frame.copy()
        ch, cw = max(0, min(360 - y, 16)), max(0, min(640 - x, 16))
        if ch and cw:
            a = alpha[:ch, :cw]
            exp[y:y + ch, x:x + cw, :] = (exp[y:y + ch, x:x + cw, :] * (1 - a) + cur[:ch, :cw, :] * a).astype(np.uint8)
        assert np.array_equal(got, exp)
        if cv2 is not None:
            ref = exp.copy()
            cv2.cvtColor(ref, code=cv2.COLOR_BGR2RGB, dst=ref)
            ref = cv2.resize(ref, (128, 128), interpolation=cv2.INTER_LINEAR)
            assert np.array_equal(resize_oracle.ingest(frame, (128, 128), cur, alpha, (x, y)), ref)


@pytest.mark.gpu
def test_ingest_kernels_bit_exact():
    rng = np.random.default_rng(6)
    cur, alpha = _cursor(rng)
    F_, H, W = 6, 360, 640
    frames = rng.integers(0, 256, (F_, H, W, 3), dtype=np.uint8)
    xy = np.array([[0, 0], [100, 37], [-1, -1], [630, 350], [639, 359], [700, 10]], dtype=np.int32)
    got = A.ingest_frames(torch.from_numpy(frames).cuda(), torch.from_numpy(cur).cuda(), torch.from_numpy(alpha[:, :, 0].copy()).cuda(),
                          torch.from_numpy(xy).cuda()).cpu().numpy()
    for f in range(F_):
        exp = resize_oracle.ingest(frames[f], (128, 128), cur, alpha, xy[f])
        assert np.array_equal(got[f], exp), f


def _codec_cases(c, n=50000, seed=0):
    """Every joint action (x3 random cameras) for to_env; random env actions + camera angles exactly at / next to every quantiser
    threshold, null actions and inventory presses for from_env."""
    g = torch.Generator().manual_seed(seed)
    b = torch.arange(8641).repeat_interleave(3)[:, None]
    cam = torch.randint(0, 121, (b.shape[0], 1), generator=g)
    rng = np.random.default_rng(seed)
    btn = (rng.random((n, 20)) < 0.15).astype(np.int64)
    btn[:500] = 0
    camv = rng.uniform(-12, 12, (n, 2))
    camv[:250] = 0.0
    thr = c._device_tables("cpu")["thr"].numpy()
    k = len(thr)
    camv[1000:1000 + k, 0] = thr
    camv[2000:2000 + k, 0] = np.nextafter(thr, -np.inf)
    camv[3000:3000 + k, 1] = np.nextafter(thr, np.inf)
    return b, cam, btn, camv


def _check_codec(c, dev):
    b, cam, btn, camv = _codec_cases(c)
    got = c.to_env_device({"buttons": b.to(dev), "camera": cam.to(dev)}) if dev != "cpu" else None
    ref = c.policy2env(c.to_factored({"buttons": b.numpy(), "camera": cam.numpy()}))
    if got is None:  # CPU: through the emulated op (the wrapper's .cpu() path is the same)
        got = c.to_env_device({"buttons": b, "camera": cam})
    for name in A.BUTTONS:
        assert got[name].dtype == np.int64 and np.array_equal(got[name], ref[name]), name
    assert got["camera"].dtype == np.float64 and np.array_equal(got["camera"], ref["camera"])  # bit-exact float64 angles
    env = {name: btn[:, i] for i, name in enumerate(A.BUTTONS)}
    env["camera"] = camv
    a = c.env2policy(env)
    ref2 = c.from_factored(a)
    null_ref = (a["buttons"] == 0).all(1) & (a["camera"] == c.null_bin).all(1)
    ac, is_null = c.from_env_device(torch.from_numpy(btn).to(dev), torch.from_numpy(camv).to(dev))
    assert np.array_equal(ac["buttons"].cpu().numpy(), ref2["buttons"]) and np.array_equal(ac["camera"].cpu().numpy(), ref2["camera"])
    assert np.array_equal(is_null.cpu().numpy(), null_ref) and null_ref.sum() >= 250


def test_device_codec_tables_match_the_host_codec():
    """SURVEY f-3: the tables / thresholds the on-device codec uses, checked through the test-only emulation of the two kernels against
    the numpy codec (which test_codec_matches_live_reference pins to the reference)."""
    from common import emulation
    with emulation():
        _check_codec(A.ActionCodec(**A.ACTION_TRANSFORMER_KWARGS), "cpu")


@pytest.mark.gpu
def test_device_codec_kernels_bit_exact():
    """vpt_codec_to_env / vpt_codec_from_env on the GPU == the numpy codec on every joint action and on 50k env actions incl. camera
    angles at the quantiser thresholds (integer + float64 bit patterns, so: exact)."""
    _check_codec(A.ActionCodec(**A.ACTION_TRANSFORMER_KWARGS), "cuda")
