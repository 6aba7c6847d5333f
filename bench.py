#!/usr/bin/env python
"""bench.py -- frames/s through MinecraftAgentPolicy.forward (ImpalaCNN -> transformer with KV memory -> action heads)
on synthetic 128x128x3 uint8 video, B x T = 128 x 128 per GPU (BASELINE.json metric; agent.py default 2x width).

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA path through the C ABI)
    python bench.py --impl reference ...                     # the reference algorithm on the host CPU (oracle port)

One "step" = one forward over a (B, T) = (128, 128) chunk per GPU = 16384 frames, KV memory carried from the previous
step (so the 128-frame memory is full in the timed region).  Inputs (805 MB of u8 frames per step) are far larger than the
126 MB L2, so no explicit flush is needed.  Multi-GPU: batch rows are independent -> each rank runs its own (128, 128)
chunk, no data-path collective (weak scaling); timing = max over ranks of CUDA-event time.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "frames/sec MinecraftPolicy fwd, 128x128x3 BxT=128x128"
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel (conv3x3_zp_kernel, 128->128 @64x64, 2048 frames)
# from the committed ncu capture (profiles/conv_zp_r2.md, profiles/kernels_r2.csv)
TRAFFIC_NCU = 2.307e9  # 1.171 GB read + 1.136 GB written (conv3x3_zp_kernel<pair>, 256->256 @32x32, 2048 frames; algorithmic 2.28 GB; profiles/conv_zp_r2.md)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--width", default="2x", choices=["1x", "2x", "3x"])
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--timesteps", type=int, default=128)
    ap.add_argument("--cpu-baseline-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra blocks (gpu_eager_baseline, configs, bc, sample_agreement)")
    ap.add_argument("--bc-width", default="3x", choices=["1x", "2x", "3x"])
    ap.add_argument("--bc-batch", type=int, default=16)
    ap.add_argument("--bc-steps", type=int, default=4)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def dump_outputs(path, pd, vpred, ac, state, limit=1 << 20, budget=64 << 20):
    """Writes the timed forward's results (log-probs, vpred, sampled actions, state out) to path/<name>.npy as float32, so that two
    builds can be compared output for output.  An array of more than `limit` entries is written as a fixed sample of `limit` of
    them: the indices come from a generator seeded with the array's name, so every run with the same arguments picks the same ones."""
    import numpy as np

    arrays = {f"pd_{k}": v for k, v in pd.items()}
    arrays["vpred"] = vpred
    arrays.update({f"action_{k}": v for k, v in ac.items()})
    for i, (mask, (k, v)) in enumerate(state):
        if mask is not None:
            arrays[f"state{i}_mask"] = mask
        arrays[f"state{i}_k"], arrays[f"state{i}_v"] = k, v
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > limit:
            idx = torch.randint(0, t.numel(), (limit,), generator=torch.Generator().manual_seed(zlib.crc32(name.encode())))
            t = t.reshape(-1)[idx.to(t.device)]
        a = t.float().cpu().numpy()  # integer actions (< 2^24) and masks are exact in float32
        total += a.nbytes
        if total > budget:
            raise RuntimeError(f"--dump-outputs: more than {budget >> 20} MB")
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return dict(tflops=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json, sustained bf16)")
    return dict(tflops=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md: ~1.4 PF sustained, 6.65 TB/s)")


# ------------------------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], None, set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm),
                    power_w_max=max(pw) if pw else None)


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline: the reference algorithm (oracle port, torch CPU fp32, all host threads) on a bounded sample
# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_fps(width, seconds, T=128, passes_max=4):
    import vpt_oracle as O
    import vpt_b200

    ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)
    kw = vpt_b200.policy_kwargs(width)
    torch.manual_seed(0)
    pol = vpt_b200.MinecraftAgentPolicy(vpt_b200.minecraft_action_space(), kw, vpt_b200.PI_HEAD_KWARGS)
    sd = {k: v.detach() for k, v in pol.state_dict().items()}
    cfg = O.Cfg(**kw)
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (1, T, 128, 128, 3), dtype=torch.uint8, generator=g)
    first = torch.zeros(1, T, dtype=torch.bool)
    st = O.initial_state(cfg, 1)
    with torch.no_grad():
        _, st = O.agent_policy_forward(sd, cfg, img[:, :16], first[:, :16], st)  # warm-up (thread pool, oneDNN primitives)
        # "all the host threads it can use": torch's CPU kernels do not always scale to every hardware thread of a big host,
        # so the thread count is picked by a short probe (16 frames each) and the best one is used for the timed passes
        probe = {}
        for nt in sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
            torch.set_num_threads(nt)
            O.agent_policy_forward(sd, cfg, img[:, :16], first[:, :16], O.initial_state(cfg, 1))
            t0 = time.perf_counter()
            O.agent_policy_forward(sd, cfg, img[:, :16], first[:, :16], O.initial_state(cfg, 1))
            probe[nt] = time.perf_counter() - t0
        best_nt = min(probe, key=probe.get)
        torch.set_num_threads(best_nt)
        st = O.initial_state(cfg, 1)
        _, st = O.agent_policy_forward(sd, cfg, img, first, st)                   # fills the KV memory (untimed)
        times = []
        t_begin = time.perf_counter()
        while len(times) < passes_max and (time.perf_counter() - t_begin < seconds or not times):
            t0 = time.perf_counter()
            _, st = O.agent_policy_forward(sd, cfg, img, first, st)
            times.append(time.perf_counter() - t0)
    best = min(times)
    return dict(value=T / best, unit="frames/s", cores=torch.get_num_threads(), kind="port",
                sample=f"oracle/vpt_oracle.py (torch {torch.__version__} CPU fp32), {width} width, B=1 T={T} with full KV memory, "
                       f"best of {len(times)} passes ({best:.2f} s/pass) at {best_nt} threads (best of a probe over "
                       f"{sorted(probe)} threads on {ncpu} hardware threads); B x T = 128 x 128 cannot be materialised on the host "
                       f"(>=137 GB of fp32 activations), per-frame cost is batch independent")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_reference_fps(args.width, seconds=max(10.0, 4.0 * (args.steps + args.warmup)))
    T = 128
    out = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1000.0 * T / cb["value"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"VPT {args.width} policy forward + heads, reference algorithm on host CPU, B=1 T=128 sample of the B x T = 128 x 128 chunk"},
           "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))



# ------------------------------------------------------------------------------------------------------------------
# extra blocks of the JSON line (VERDICT round 1, item 2): every number that used to be prose in DESIGN.md
# ------------------------------------------------------------------------------------------------------------------
def _free():
    import gc
    gc.collect()
    torch.cuda.empty_cache()


def _event_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def gpu_eager_baseline(width, dev, B=4, T=128, seconds=6.0):
    """The honest GPU bar (SURVEY 8d / BASELINE.md 4): the reference ALGORITHM run eagerly by PyTorch on the same B200 -- the oracle
    port (same torch ops in the same order as lib/policy.py; the reference itself cannot travel to the GPU box) dispatched to
    cuDNN / cuBLAS / ATen, fp32 with TF32 off and on.  B x T = 128 x 128 does not fit (8 MiB of fp32 per frame for the first conv
    alone), so it runs B sequences of T frames with the KV memory full; per-frame cost is batch independent."""
    import vpt_oracle as O
    import vpt_b200

    kw = vpt_b200.policy_kwargs(width)
    torch.manual_seed(0)
    pol = vpt_b200.MinecraftAgentPolicy(vpt_b200.minecraft_action_space(), kw, vpt_b200.PI_HEAD_KWARGS)
    sd = {k: v.detach().to(dev) for k, v in pol.state_dict().items()}
    del pol
    cfg = O.Cfg(**kw)
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (B, T, 128, 128, 3), dtype=torch.uint8, generator=g).to(dev)
    first = torch.zeros(B, T, dtype=torch.bool, device=dev)
    out = {"kind": "port", "sample": f"oracle/vpt_oracle.py on cuda (torch {torch.__version__} eager: cuDNN/cuBLAS/ATen), {width} width, fp32, "
                                      f"B={B} T={T} with full KV memory, best of the passes that fit in {seconds:.0f} s per mode",
           "unit": "frames/s"}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        with torch.device(dev), torch.no_grad():
            for name, tf32 in (("fp32_tf32_off", False), ("fp32_tf32_on", True)):
                torch.backends.cuda.matmul.allow_tf32 = tf32
                torch.backends.cudnn.allow_tf32 = tf32
                st = O.initial_state(cfg, B)
                for _ in range(2):  # warm-up (cuDNN heuristics) + fills the KV memory
                    _, st = O.agent_policy_forward(sd, cfg, img, first, st)
                torch.cuda.synchronize()
                best, t_begin = None, time.perf_counter()
                while time.perf_counter() - t_begin < seconds:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    (pd, v, _), st = O.agent_policy_forward(sd, cfg, img, first, st)
                    e1.record()
                    torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1)
                    best = ms if best is None else min(best, ms)
                out[name] = B * T / (best / 1000.0)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    del sd, img
    _free()
    return out


def sample_agreement(pol, kw, dev, B=2, T=64, seed=1234):
    """End-to-end agreement of the SAMPLED action indices with the oracle (north_star: 'bit-exact on sampled action indices under a
    fixed seed'; lib/action_head.py:195-207): the CUDA policy (bf16 operands) and the fp32 oracle (host CPU) see the same frames, the
    same weights and the same uniforms (the CUDA Philox stream after torch.manual_seed(seed), drawn camera-then-buttons like
    DictActionHead.sample).  The sampler itself is bit exact given logits (tests/test_gpu_policy.py); a mismatch here is a Gumbel
    arg-max whose top-two gap is below the bf16 logit error."""
    import vpt_oracle as O

    sd = {k: v.detach().cpu().float() for k, v in pol.state_dict().items()}
    cfg = O.Cfg(**kw)
    g = torch.Generator().manual_seed(7)
    img = torch.randint(0, 256, (B, T, 128, 128, 3), dtype=torch.uint8, generator=g)
    first = torch.zeros(B, T, dtype=torch.bool)
    (pd, _, _), _ = pol({"img": img.to(dev)}, first.to(dev), pol.initial_state(B))
    torch.manual_seed(seed)
    ac = pol.sample(pd)
    ac_det = pol.sample(pd, deterministic=True)
    torch.manual_seed(seed)  # replay the same Philox stream for the oracle
    us = {name: torch.rand_like(pd[name].contiguous()).cpu() for name in pd}
    nthr = torch.get_num_threads()
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    with torch.no_grad():
        (pd_o, _, _), _ = O.agent_policy_forward(sd, cfg, img, first, O.initial_state(cfg, B))
    torch.set_num_threads(nthr)
    # the same in the fp32-parity mode (precise.py): the mode in which "bit-exact sampled indices" is a meaningful target
    pol.set_precision("fp32")
    try:
        (pd32, _, _), _ = pol({"img": img.to(dev)}, first.to(dev), pol.initial_state(B))
        torch.manual_seed(seed)
        ac32 = pol.sample(pd32)
        ac32_det = pol.sample(pd32, deterministic=True)
    finally:
        pol.set_precision("bf16")
    out = {"frames": B * T, "seed": seed, "rng": "CUDA Philox, torch.manual_seed(seed), camera then buttons"}
    for name in pd:
        so = O.gumbel_sample(pd_o[name], us[name])
        do = torch.argmax(pd_o[name], dim=-1)
        n = so.numel()
        agree = lambda a, ref: int((a.cpu().view_as(ref) == ref).sum()) / n
        out[name] = {"stochastic_agree": agree(ac[name], so), "deterministic_agree": agree(ac_det[name], do),
                     "logprob_max_rel_err": float(((pd[name].cpu() - pd_o[name]).abs() / pd_o[name].abs()).max()),
                     "fp32_mode": {"stochastic_agree": agree(ac32[name], so), "deterministic_agree": agree(ac32_det[name], do),
                                   "logprob_max_rel_err": float(((pd32[name].cpu() - pd_o[name]).abs() / pd_o[name].abs()).max())}}
    return out


def config_blocks(dev, pk):
    """BASELINE configs C2 (1x, B=64, T=128), C5 (IDM 4x, B=64, T=128) and the f-1 rollout step, each with its own roofline fraction."""
    import vpt_b200
    from video_pre_training_b200 import _native as nat

    out = {}
    # ---- C2: 1x width, B=64, T=128, bf16 inference-only forward
    kw = vpt_b200.policy_kwargs("1x")
    torch.manual_seed(0)
    pol = vpt_b200.MinecraftAgentPolicy(vpt_b200.minecraft_action_space(), kw, vpt_b200.PI_HEAD_KWARGS).to(dev)
    B, T = 64, 128
    img = torch.randint(0, 256, (B, T, 128, 128, 3), dtype=torch.uint8, device=dev)
    first = torch.zeros(B, T, dtype=torch.bool, device=dev)
    box = {"st": pol.initial_state(B)}

    def step_c2():
        (_, _, _), box["st"] = pol({"img": img}, first, box["st"])

    ms = _event_ms(step_c2, 5, 3)
    fl = pol.net.cfg.forward_flops_per_frame()
    fps = B * T / ms * 1000.0
    out["C2_1x_B64_T128"] = {"frames_per_s": fps, "ms_per_step": ms, "gflop_per_frame": fl / 1e9,
                             "frac_of_flop_roofline": fps * fl / 1e12 / pk["tflops"]}
    nat.device_check()
    del pol, img, box
    _free()
    # ---- C5: IDM 4x, B=64, T=128 (bidirectional attention, conv3d pre-stage)
    ikw = vpt_b200.idm_net_kwargs()
    torch.manual_seed(0)
    idm = vpt_b200.InverseActionPolicy(vpt_b200.idm_action_space(), dict(temperature=2.0), ikw).to(dev)
    img = torch.randint(0, 256, (B, T, 128, 128, 3), dtype=torch.uint8, device=dev)

    def step_c5():
        idm.predict({"img": img}, first=first, state_in=idm.initial_state(B))

    ms = _event_ms(step_c5, 2, 1)
    fl = idm.net.cfg.forward_flops_per_frame(idm._heads_prepared()["ntot"])  # 68.59 GFLOP (SURVEY 8d: 68.62 incl. the discarded lastlayer)
    fps = B * T / ms * 1000.0
    out["C5_idm4x_B64_T128"] = {"frames_per_s": fps, "ms_per_step": ms, "gflop_per_frame": fl / 1e9,
                                "frac_of_flop_roofline": fps * fl / 1e12 / pk["tflops"]}
    nat.device_check()
    del idm, img
    _free()
    # ---- f-1: rollout step, 2x, B=1, T=1 (agent.py:190-206): one CUDA graph per step; bound = streaming the bf16 weights once
    kw = vpt_b200.policy_kwargs("2x")
    torch.manual_seed(0)
    pol = vpt_b200.MinecraftAgentPolicy(vpt_b200.minecraft_action_space(), kw, vpt_b200.PI_HEAD_KWARGS).to(dev)
    step = pol.make_graphed_act(1)
    img1 = torch.randint(0, 256, (1, 128, 128, 3), dtype=torch.uint8, device=dev)
    first1 = torch.zeros(1, dtype=torch.bool, device=dev)
    box = {"st": pol.initial_state(1)}

    def step_f1():
        ac, box["st"], _ = step({"img": img1}, first1, box["st"])
        return ac

    for _ in range(5):
        step_f1()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n = 200
    for _ in range(n):
        ac = step_f1()
        ac["buttons"].cpu()  # the env needs the action on the host every step
    wall_ms = (time.perf_counter() - t0) / n * 1000.0
    dev_ms = _event_ms(step_f1, 200, 5)
    wbytes = sum(p.numel() for p in pol.parameters()) * 2
    bound_ms = wbytes / (pk["hbm"] * 1e9) * 1000.0
    out["f1_rollout_2x_B1_T1"] = {"ms_per_step_device": dev_ms, "ms_per_step_wall_with_d2h": wall_ms, "weight_bytes_bf16": wbytes,
                                  "hbm_bound_ms": bound_ms, "frac_of_hbm_bound": bound_ms / dev_ms}
    nat.device_check()
    del pol, step, box
    _free()
    return out


def bc_block(args, dev, world, rank, pk):
    """BASELINE configs[3]: BC fine-tune step (fwd + hand-written bwd + ONE NCCL all-reduce over the flat fp32 gradient bucket + fused
    Adam) at `world` ranks, B clips per GPU, T=128 (behavioural_cloning.py:101-123).  The only path with a collective."""
    import torch.distributed as dist
    import vpt_b200
    from video_pre_training_b200 import _native as nat
    from video_pre_training_b200.parallel import FlatAdamDP
    from video_pre_training_b200.training import BCTrainer

    kw = vpt_b200.policy_kwargs(args.bc_width)
    torch.manual_seed(0)
    pol = vpt_b200.MinecraftAgentPolicy(vpt_b200.minecraft_action_space(), kw, vpt_b200.PI_HEAD_KWARGS).to(dev)
    B, T = args.bc_batch, 128
    g = torch.Generator(device=dev).manual_seed(rank)
    img = torch.randint(0, 256, (B, T, 128, 128, 3), dtype=torch.uint8, device=dev, generator=g)
    first = torch.zeros(B, T, dtype=torch.bool, device=dev)
    actions = {"camera": torch.randint(0, 121, (B, T, 1), device=dev, generator=g),
               "buttons": torch.randint(0, 8641, (B, T, 1), device=dev, generator=g)}
    tr = BCTrainer(pol)
    opt = FlatAdamDP([p for n, p in pol.named_parameters() if not n.startswith("value_head")], lr=0.000181, weight_decay=0.039428)
    split = opt.offset_of(pol.net.img_process.cnn.dense.norm.weight)
    hook = lambda: opt.reduce_async(split, opt.n)
    box = {"st": pol.initial_state(B)}
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def step(marks=None):
        opt.zero_grad()
        if marks:
            marks[0].record()
        loss, box["st"] = tr.loss_and_grad(img, first, box["st"], actions, upper_grads_ready=hook)
        if marks:
            marks[1].record()
        opt.step()
        if marks:
            marks[2].record()
        return loss

    losses = [float(step()) for _ in range(2)]
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    marks = [(ev(), ev(), ev()) for _ in range(args.bc_steps)]
    for m in marks:
        losses.append(step(m))
    torch.cuda.synchronize()
    nat.device_check()
    t = torch.tensor([marks[0][0].elapsed_time(marks[-1][2]) / args.bc_steps,
                      sum(m[0].elapsed_time(m[1]) for m in marks) / args.bc_steps,
                      sum(m[1].elapsed_time(m[2]) for m in marks) / args.bc_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, fb, ad = [float(x) for x in t.tolist()]
    # the collective alone (not overlapped): bus bandwidth = 2 (N-1)/N x bytes / time
    ar_ms, bus = None, None
    if world > 1:
        for _ in range(2):
            dist.all_reduce(opt.flat_g)
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(3):
            dist.all_reduce(opt.flat_g)
        e1.record()
        torch.cuda.synchronize()
        tt = torch.tensor([e0.elapsed_time(e1) / 3], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ar_ms = float(tt.item())
        bus = 2.0 * (world - 1) / world * opt.n * 4 / (ar_ms / 1000.0) / 1e9
    fl = 3.0 * pol.net.cfg.forward_flops_per_frame()  # SURVEY 8d: training step ~ 3x forward
    fps = world * B * T / ms * 1000.0
    res = {"workload": f"BC fine-tune step {args.bc_width}, B={B}/GPU T={T}, fwd + bwd + all-reduce(fp32 flat bucket) + Adam, x{world} GPU",
           "ms_per_step": ms, "frames_per_s": fps, "fwd_bwd_ms": fb, "exposed_allreduce_plus_adam_ms": ad,
           "allreduce_alone_ms": ar_ms, "nccl_bus_gb_s": bus, "gradient_bucket_bytes": opt.n * 4,
           "frac_of_flop_roofline": (fps / world) * fl / 1e12 / pk["tflops"], "gflop_per_frame": fl / 1e9,
           "loss_first_last": [float(losses[0]), float(losses[-1])]}
    del pol, tr, opt, img, box
    _free()
    return res

# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist

    import vpt_b200
    from video_pre_training_b200 import _native as nat
    from video_pre_training_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on STDOUT when the communicator is created (eagerly here: device_id is given); the contract is ONE
        # JSON line on stdout, so file descriptor 1 points at stderr for the duration of the initialisation
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    B, T = args.batch, args.timesteps
    kw = vpt_b200.policy_kwargs(args.width)
    torch.manual_seed(0)
    pol = vpt_b200.MinecraftAgentPolicy(vpt_b200.minecraft_action_space(), kw, vpt_b200.PI_HEAD_KWARGS).to(dev)
    pol.net.prepared()
    pol._heads_prepared()
    g = torch.Generator().manual_seed(rank)
    host_img = torch.randint(0, 256, (B, T, 128, 128, 3), dtype=torch.uint8, generator=g).pin_memory()
    host_first = torch.zeros(B, T, dtype=torch.bool).pin_memory()
    img = host_img.to(dev)
    first = host_first.to(dev)
    frames_per_step = B * T

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---------------- device-resident inputs ("value") ----------------
    state = pol.initial_state(B)
    for _ in range(args.warmup):
        (pd, _, _), state = pol({"img": img}, first, state)
        pol.sample(pd)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.GEMM_PROFILE = []
    l0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        (pd, vpred, _), state = pol({"img": img}, first, state)
        ac = pol.sample(pd)  # configs[2]: "forward + action_head sampling"
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = (ops.LAUNCHES - l0) // args.steps
    prof, ops.GEMM_PROFILE = ops.GEMM_PROFILE, None
    clocks = sampler.stop() if rank == 0 else None
    nat.device_check()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pd, vpred, ac, state)
    value = world * frames_per_step * args.steps / (ms / 1000.0)

    # dominant kernel = gemm_tc_kernel (tcgen05 implicit-GEMM conv + linear): live CUDA-event durations of every launch
    g_ms = sum(a.elapsed_time(b) for a, b, _, _, _ in prof)
    g_fl = sum(f for _, _, f, _, _ in prof)
    conv_ms = sum(a.elapsed_time(b) for a, b, _, k, _ in prof if k == "conv")
    conv_fl = sum(f for _, _, f, k, _ in prof if k == "conv")
    pk = peaks()
    by_shape = {}
    for a, b, f, k, shp in prof:
        t, fl_, n = by_shape.get((k, shp), (0.0, 0.0, 0))
        by_shape[(k, shp)] = (t + a.elapsed_time(b), fl_ + f, n + 1)
    shape_rows = [{"kind": k, "mnk": list(shp), "launches_per_step": n // args.steps, "ms_per_step": t / args.steps, "tflops": fl_ / t / 1e9}
                  for (k, shp), (t, fl_, n) in sorted(by_shape.items(), key=lambda kv: -kv[1][0])][:12]
    achieved = g_fl / (g_ms / 1000.0) / 1e12
    flops_frame = pol.net.cfg.forward_flops_per_frame()  # product-side FLOP model (policy.NetConfig), SURVEY 8d
    roofline = {"bound": "tensor", "achieved": achieved, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": achieved / pk["tflops"],
                "traffic": TRAFFIC_NCU, "kernel": "conv3x3_zp_kernel + gemm_tc_kernel (tcgen05 implicit-GEMM conv3x3 / linear)",
                "peak_source": pk["source"],
                "launches_per_step": len(prof) // args.steps, "kernel_ms_per_step": g_ms / args.steps,
                "kernel_share_of_step": g_ms / ms if world == 1 else None,
                "algorithmic_gflop_per_frame": flops_frame / 1e9, "gemm_gflop_per_frame": g_fl / args.steps / frames_per_step / 1e9,
                "conv_only": {"achieved": conv_fl / (conv_ms / 1000.0) / 1e12 if conv_ms else None, "ms_per_step": conv_ms / args.steps},
                "whole_step_frac_of_flop_roofline": (value / world) * flops_frame / 1e12 / pk["tflops"],
                "by_shape": shape_rows}

    # ---------------- end to end through the public API with HOST buffers ("e2e") ----------------
    state2 = state
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d2h = 0
    from video_pre_training_b200.parallel import HostFramePipe
    pipe = HostFramePipe(dev)
    pipe.submit(host_img, host_first)
    for it in range(1 + args.steps):  # first iteration untimed (pinned-path warm-up)
        if it == 1:
            barrier()
            e2.record()
            pipe.submit(host_img, host_first)  # every timed step uploads its own chunk inside the timed region
        d_img, d_first = pipe.take()
        if 1 <= it < args.steps:
            pipe.submit(host_img, host_first)  # upload of the next step's frames overlaps this step's forward
        (pd, vpred, _), state2 = pol({"img": d_img}, d_first, state2)
        ac = pol.sample(pd)
        res = [ac["camera"].cpu(), ac["buttons"].cpu(), vpred.cpu()]  # device -> host read of the step's result (syncs)
        d2h = sum(r.numel() * r.element_size() for r in res)
    e3.record()
    barrier()
    ms2 = max_over_ranks(e2.elapsed_time(e3))
    e2e = {"value": world * frames_per_step * args.steps / (ms2 / 1000.0), "unit": "frames/s",
           "h2d_bytes_per_step": host_img.numel() + host_first.numel(), "d2h_bytes_per_step": d2h,
           "call": "HostFramePipe (pinned host frames -> device, double buffered) + MinecraftAgentPolicy.forward(obs, first, state) + sample(); sampled actions + vpred read back to the host every step"}

    extras = {}
    if not args.no_extras:
        if rank == 0 and world == 1:
            extras["sample_agreement"] = sample_agreement(pol, kw, dev)
        del pol, state, state2, img, host_img, pipe, pd, vpred, ac, res, d_img
        _free()
        if rank == 0 and world == 1:
            extras["gpu_eager_baseline"] = gpu_eager_baseline(args.width, dev)
            extras["configs"] = config_blocks(dev, pk)
        extras["bc"] = bc_block(args, dev, world, rank, pk)  # every rank: the one path with a collective
    cb = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference_fps(args.width, args.cpu_baseline_seconds)
    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
               "data": "synthetic",
               "config": {"workload": f"VPT {args.width} policy (agent.py:16-36 kwargs) forward + action/value heads, B={B} T={T} per GPU "
                                      f"(= BASELINE configs[2] shape), random-init weights, KV memory carried and full",
                          "global_batch": world * B, "seq_len": T, "parallelism": f"batch-sharded x{world}, no collective",
                          "l2_policy": "inputs (805 MB u8 frames/step) exceed the 126 MB L2; no explicit flush"},
               "roofline": roofline, "cpu_baseline": cb, "e2e": e2e, "gpu_launches": launches, "clocks": clocks}
        out.update(extras)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
