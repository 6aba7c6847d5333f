#!/usr/bin/env python
"""RL fine-tuning step (training.RLTrainer) at BASELINE configs[3] shapes: 3x width, bf16, B=16 clips per GPU, T=128, with a frozen 3x
teacher for the KL term, data-parallel under torch.distributed.run.

    python tools/rl_bench.py [--width 3x] [--batch 16] [--steps 4] [--warmup 2]
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/rl_bench.py ...      (weak scaling)

Prints one JSON line: the card and its power limit (read in the same run), RL and BC ms/step of the same policy in the same process
(alternated step by step), the teacher forward, the exposed all-reduce + Adam time, and the loss kernel (vpt_rl_heads_bwd) at
N = 2048 frames timed with CUDA events over 200 launches, against its byte bound (every input byte read once, every output byte
written once) at the data-sheet HBM rate and at a device-to-device copy rate measured in the same run."""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
import vpt_b200
from video_pre_training_b200 import _native as nat, ops
from video_pre_training_b200.parallel import FlatAdamDP
from video_pre_training_b200.training import BCTrainer, RLTrainer

ap = argparse.ArgumentParser()
ap.add_argument("--width", default="3x")
ap.add_argument("--batch", type=int, default=16)
ap.add_argument("--steps", type=int, default=4)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--kernel-rows", type=int, default=2048)
ap.add_argument("--kernel-iters", type=int, default=200)
a = ap.parse_args()
world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ev = lambda: torch.cuda.Event(enable_timing=True)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", str(local)],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return out[0].strip(), float(out[1])
    except Exception:  # no nvidia-smi: the name from the driver, the limit unknown
        return torch.cuda.get_device_name(local), None


# ---- the loss kernel alone -----------------------------------------------------------------------------------------------------
def kernel_bench(N, iters):
    g = torch.Generator(device="cuda").manual_seed(0)
    widths = (121, 8641)
    logp = [torch.log_softmax(torch.randn(N, n, device="cuda", generator=g) * 2, -1) for n in widths]
    logp_t = [torch.log_softmax(torch.randn(N, n, device="cuda", generator=g) * 2, -1) for n in widths]
    idx = [torch.randint(0, n, (N,), device="cuda", generator=g) for n in widths]
    old, adv, ret, vpred = [torch.randn(N, device="cuda", generator=g) for _ in range(4)]
    mu_rsig = torch.tensor([0.0, 1.0], device="cuda")
    ld, ntot = 8768, sum(widths)
    dlog = torch.zeros((N, ld), dtype=torch.bfloat16, device="cuda")
    call = lambda: ops.rl_heads_bwd(logp, logp_t, idx, [0, 121], old, adv, ret, vpred, mu_rsig, 0.2, 0.1, 0.01, 0.5, 0.5, 1.0 / N, dlog, ntot)
    for _ in range(5):
        call()
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    e0.record()
    for _ in range(iters):
        call()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    nbytes = N * ntot * (4 + 4 + 2) + N * (4 * 4 + 2 * 8 + 2 + 5 * 4)  # log-probs in, dlog out; per-row inputs / statistics
    # device-to-device copy of 2 GiB (read + write), the same run's streaming reference
    src = torch.empty(2 ** 29, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    c0, c1 = ev(), ev()
    c0.record()
    for _ in range(10):
        dst.copy_(src)
    c1.record()
    torch.cuda.synchronize()
    copy_tbps = 2 * src.numel() * 4 * 10 / (c0.elapsed_time(c1) * 1e-3) / 1e12
    del src, dst
    return dict(loss_kernel_rows=N, loss_kernel_us=round(us, 2), loss_kernel_bytes=nbytes, loss_kernel_tbps=round(nbytes / (us * 1e-6) / 1e12, 3),
                copy_tbps_measured=round(copy_tbps, 3), loss_kernel_bound_us_at_copy_rate=round(nbytes / (copy_tbps * 1e12) * 1e6, 2),
                loss_kernel_frac_of_copy_rate=round(nbytes / (copy_tbps * 1e12) * 1e6 / us, 3),
                loss_kernel_bound_us_at_7_7_tbps=round(nbytes / 7.7e12 * 1e6, 2), loss_kernel_frac_of_7_7_tbps=round(nbytes / 7.7e12 * 1e6 / us, 3))


res = dict(bench="rl_step", width=a.width, batch_per_gpu=a.batch, T=128, world=world)
res["gpu"], res["power_limit_w"] = card()
res.update(kernel_bench(a.kernel_rows, a.kernel_iters))

# ---- the step ------------------------------------------------------------------------------------------------------------------
torch.manual_seed(0)
mk = lambda: vpt_b200.MinecraftAgentPolicy(vpt_b200.minecraft_action_space(), vpt_b200.policy_kwargs(a.width), vpt_b200.PI_HEAD_KWARGS).cuda()
pol = mk()
teacher = mk()
teacher.load_state_dict(pol.state_dict())
B, T = a.batch, 128
g = torch.Generator(device="cuda").manual_seed(rank)
img = torch.randint(0, 256, (B, T, 128, 128, 3), dtype=torch.uint8, device="cuda", generator=g)
first = torch.zeros(B, T, dtype=torch.bool, device="cuda")
actions = {"camera": torch.randint(0, 121, (B, T, 1), device="cuda", generator=g), "buttons": torch.randint(0, 8641, (B, T, 1), device="cuda", generator=g)}
old = -12.0 + torch.randn(B, T, device="cuda", generator=g)
adv = torch.randn(B, T, device="cuda", generator=g)
ret = torch.randn(B, T, device="cuda", generator=g) * 2 + 1
bc = BCTrainer(pol)
rl = RLTrainer(pol, teacher, clip_eps=0.2, kl_coef=0.1, ent_coef=0.01, vf_coef=0.5)
opt = FlatAdamDP(list(pol.parameters()), lr=1e-5)
split = opt.offset_of(pol.net.img_process.cnn.dense.norm.weight)
hook = lambda: opt.reduce_async(split, opt.n)
state = {"bc": pol.initial_state(B), "rl": pol.initial_state(B), "t": teacher.initial_state(B)}


def step(kind, marks=None):
    opt.zero_grad()
    if marks:
        marks[0].record()
    if kind == "bc":
        _, state["bc"] = bc.loss_and_grad(img, first, state["bc"], actions, upper_grads_ready=hook)
    else:
        _, state["rl"], state["t"] = rl.loss_and_grad(img, first, state["rl"], state["t"], actions, old, adv, ret, upper_grads_ready=hook)
    if marks:
        marks[1].record()
    opt.step()
    if marks:
        marks[2].record()


for _ in range(a.warmup):
    step("bc")
    step("rl")
torch.cuda.synchronize()
nat.device_check()
if world > 1:
    dist.barrier()
marks = {"bc": [], "rl": []}
for i in range(a.steps):
    for kind in (("bc", "rl") if i % 2 == 0 else ("rl", "bc")):
        m = (ev(), ev(), ev())
        step(kind, m)
        marks[kind].append(m)
torch.cuda.synchronize()
for kind, ms in marks.items():
    tot = torch.tensor([sum(m[0].elapsed_time(m[2]) for m in ms) / len(ms)], device="cuda")
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    res[f"{kind}_ms_per_step"] = round(tot.item(), 2)
    res[f"{kind}_reduce_adam_ms"] = round(sum(m[1].elapsed_time(m[2]) for m in ms) / len(ms), 2)
res["rl_over_bc"] = round(res["rl_ms_per_step"] / res["bc_ms_per_step"], 3)
# teacher forward alone (inference, no tape) on the same frames
with torch.no_grad():
    t0, t1 = ev(), ev()
    t0.record()
    for _ in range(3):
        teacher({"img": img}, first, state["t"])
    t1.record()
torch.cuda.synchronize()
res["teacher_fwd_ms"] = round(t0.elapsed_time(t1) / 3, 2)
res["peak_mem_gib"] = round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)
nat.device_check()
if rank == 0:
    print(json.dumps(res))
if world > 1:
    dist.destroy_process_group()
