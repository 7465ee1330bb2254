"""Time the guidance-step kernels alone: python tools/time_guidance.py [scenes] [agents] [--grad-steps 1,2,4]

bf16 mode, one sample per agent.  For every grad_steps value the whole cld_guidance_step (decode + stash, losses, BPTT and
optimizer step, repeated grad_steps times) is timed with CUDA events; the values are interleaved over several rounds and the
median is printed with the card's name and power limit."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cld_b200 import default_algo_config, make_scenes
from cld_b200.dm_model import DmModel
from cld_b200.engine import default_guidance
from cld_b200.vae import VaeModel

ap = argparse.ArgumentParser()
ap.add_argument("scenes", nargs="?", type=int, default=256)
ap.add_argument("agents", nargs="?", type=int, default=16)
ap.add_argument("--grad-steps", default="1", help="comma-separated grad_steps values")
ap.add_argument("--iters", type=int, default=20, help="timed calls per value and round")
ap.add_argument("--rounds", type=int, default=5)
args = ap.parse_args()
ks = [int(v) for v in args.grad_steps.split(",")]
S, A = args.scenes, args.agents
R = S * A
try:
    card = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                                    str(torch.cuda.current_device())], text=True).strip()
except (OSError, subprocess.CalledProcessError):
    card = torch.cuda.get_device_name() + ", power limit unknown"
algo = default_algo_config()
torch.manual_seed(0)
dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=100, precision="bf16", max_rows=R).cuda()
vae = VaeModel(algo).bind(dm)
aux, batch = make_scenes(S, A, seed=123, dense=True)
eng = dm.engine(R)
scene = eng.make_scene(batch, S, A, 1)
z = torch.randn(R, 52, 4).cuda()
cond, curr = aux["cond_feat"].cuda(), aux["curr_states"].cuda()


def t(fn, n):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


print("card: %s" % card)
print("rows %d: decode+rollout %.3f ms" % (R, t(lambda: eng.decode_rollout(z, cond, curr), args.iters)))
times = {k: [] for k in ks}
for _ in range(args.rounds):
    for k in ks:
        g = default_guidance(grad_steps=k)
        times[k].append(t(lambda: eng.guidance_step(z, cond, curr, scene, g), args.iters))
med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
for k in ks:
    line = "guidance step, grad_steps=%d: %.3f ms (median of %d rounds; min %.3f max %.3f)" % (k, med[k], args.rounds, min(times[k]), max(times[k]))
    if k > 1 and 1 in med:
        line += " | per extra iteration %.3f ms" % ((med[k] - med[1]) / (k - 1))
    print(line)
