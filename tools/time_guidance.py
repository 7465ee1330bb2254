"""Time the guidance-step kernels alone:
    python tools/time_guidance.py [scenes] [agents] [--grad-steps 1,2,4] [--horizon 52,104] [--sparse] [--rows 4096]

bf16 mode, one sample per agent.  `agents` and `--horizon` take comma-separated lists; with `--rows` the number of scenes of
each size is rows / agents.  For every (horizon, agents, grad_steps) the whole cld_guidance_step (decode + stash, losses, BPTT
and optimizer step, repeated grad_steps times) is timed with CUDA events; the values are interleaved over several rounds and
the median is printed with the card's name and power limit.  The agent-collision loss kernel (guidance_loss_grad_kernel) is
timed on its own with torch.profiler in a separate pass.  Scenes are dense by default (every agent within +-12 m, the worst
case for the agent-collision term: every pair passes its centre-distance test); --sparse spreads them over +-50 m."""
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
ap.add_argument("agents", nargs="?", default="16", help="agents per scene (comma-separated)")
ap.add_argument("--grad-steps", default="1", help="comma-separated grad_steps values")
ap.add_argument("--horizon", default="52", help="comma-separated horizons")
ap.add_argument("--rows", type=int, default=0, help="rows per call (scenes = rows / agents); 0: scenes x agents")
ap.add_argument("--sparse", action="store_true", help="agents within +-50 m instead of +-12 m")
ap.add_argument("--iters", type=int, default=20, help="timed calls per value and round")
ap.add_argument("--rounds", type=int, default=5)
args = ap.parse_args()
ks = [int(v) for v in args.grad_steps.split(",")]
try:
    card = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                                    str(torch.cuda.current_device())], text=True).strip()
except (OSError, subprocess.CalledProcessError):
    card = torch.cuda.get_device_name() + ", power limit unknown"


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


def loss_kernel_ms(fn, n):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.key_averages() if "guidance_loss_grad_kernel" in e.key]
    return ev[0].device_time / 1000.0 if ev else float("nan")


print("card: %s" % card)
print("scenes: %s" % ("+-50 m (sparse)" if args.sparse else "+-12 m (dense)"))
for T in [int(v) for v in args.horizon.split(",")]:
    for A in [int(v) for v in args.agents.split(",")]:
        S = args.rows // A if args.rows else args.scenes
        R = S * A
        algo = default_algo_config(horizon=T)
        torch.manual_seed(0)
        dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=100, precision="bf16", max_rows=R).cuda()
        VaeModel(algo).bind(dm)
        aux, batch = make_scenes(S, A, horizon=T, seed=123, dense=not args.sparse)
        for k in ("all_other_agents_future_positions", "all_other_agents_future_availability"):
            batch.pop(k)                              # read by the indicators only: [B, A - 1, T, 2] is large for big scenes
        eng = dm.engine(R)
        scene = eng.make_scene(batch, S, A, 1)
        z = torch.randn(R, T, 4).cuda()
        cond, curr = aux["cond_feat"].cuda(), aux["curr_states"].cuda()
        print("T %d, %d scenes x %d agents = %d rows: decode+rollout %.3f ms" % (
            T, S, A, R, t(lambda: eng.decode_rollout(z, cond, curr), args.iters)))
        times = {k: [] for k in ks}
        for _ in range(args.rounds):
            for k in ks:
                g = default_guidance(grad_steps=k)
                times[k].append(t(lambda: eng.guidance_step(z, cond, curr, scene, g), args.iters))
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        for k in ks:
            line = "  guidance step, grad_steps=%d: %.3f ms (median of %d rounds; min %.3f max %.3f)" % (
                k, med[k], args.rounds, min(times[k]), max(times[k]))
            if k > 1 and 1 in med:
                line += " | per extra iteration %.3f ms" % ((med[k] - med[1]) / (k - 1))
            print(line)
        g1 = default_guidance()
        print("  agent-collision loss kernel: %.3f ms" % loss_kernel_ms(lambda: eng.guidance_step(z, cond, curr, scene, g1), args.iters))
        del eng, dm
        torch.cuda.empty_cache()
