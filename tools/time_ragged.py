"""Time a ragged batch in one sampler call against the bucketed sequence it replaces:
    python tools/time_ragged.py [--scenes 256] [--max-agents 64] [--rounds 5] [--seed 2026]

Workload: bf16, 50-step DDIM (n_timesteps 100, stride 2) with the default guidance (agent + map collision), DmModel(lanes=4), one
sample per agent, dense synthetic scenes with bit-packed maps.  The scene sizes are drawn uniformly from 1 .. --max-agents with
torch.Generator().manual_seed(--seed); with the defaults that is 256 scenes of 1 .. 64 agents (the draw is printed).

  one call   DmModel.sample_traj on the whole batch: the scenes go to the kernels with their offsets (CldScene.scene_start).
  bucketed   keys.scene_buckets, then one uniform DmModel call per distinct scene size, results scattered back into batch order
             (what DmModel did for a ragged batch before the kernels took offsets).

Both run on the same model and the same supplied x_init; their outputs are checked to be bit-identical.  The two are alternated
in every round, each timed with CUDA events around the whole call; the median, minimum and maximum over the rounds are printed
with the card's name and power limit."""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cld_b200 import default_algo_config, make_scenes
from cld_b200.dm_model import DmModel
from cld_b200.engine import default_guidance
from cld_b200.keys import scene_buckets
from cld_b200.synthetic import pack_drivable_map
from cld_b200.vae import VaeModel

ap = argparse.ArgumentParser()
ap.add_argument("--scenes", type=int, default=256)
ap.add_argument("--max-agents", type=int, default=64)
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--seed", type=int, default=2026)
args = ap.parse_args()
try:
    card = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                                    str(torch.cuda.current_device())], text=True).strip()
except (OSError, subprocess.CalledProcessError):
    card = torch.cuda.get_device_name() + ", power limit unknown"

sizes = torch.randint(1, args.max_agents + 1, (args.scenes,), generator=torch.Generator().manual_seed(args.seed)).tolist()
S, B = len(sizes), sum(sizes)
algo = default_algo_config(num_samp=1)
torch.manual_seed(0)
dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=100, precision="bf16", lanes=4).cuda()
dm.stride = 2
VaeModel(algo).bind(dm)
aux, batch = make_scenes(1, B, seed=123, dense=True)
batch["drivable_map_bits"] = pack_drivable_map(batch.pop("drivable_map"))
batch["scene_index"] = torch.cat([torch.full((c,), i) for i, c in enumerate(sizes)])
batch = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in batch.items()}
aux = {k: v.cuda() for k, v in aux.items()}
torch.manual_seed(1)
x_init = torch.randn(B, 52, 4).cuda()
kw = dict(sampler="ddim", guidance=default_guidance())
buckets = [(A, idx.cuda()) for A, idx in scene_buckets(sizes)]


def one_call():
    return dm(batch, aux, algo, x_init=x_init, **kw)["pred_traj"]


def bucketed():
    out = torch.empty(B, 52, 4, device="cuda")
    for A, idx in buckets:
        nb = idx.numel()
        sub = {k: (v.index_select(0, idx) if (torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == B) else v) for k, v in batch.items()}
        sub["scene_index"] = torch.arange(nb // A, device="cuda").repeat_interleave(A)
        sa = {k: v.index_select(0, idx) for k, v in aux.items()}
        o = dm(sub, sa, algo, x_init=x_init.index_select(0, idx), agents_per_scene=A, **kw)["pred_traj"]
        out.index_copy_(0, idx, o)
    return out


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


print("card: %s" % card)
print("workload: bf16, 50-step DDIM, default guidance, lanes=4, N=1; %d scenes, %d agents, %d distinct sizes (seed %d): %s" % (
    S, B, len(buckets), args.seed, sizes))
a, b = one_call(), bucketed()                       # warm-up: every engine and bucket shape
print("outputs bit-identical: %s" % torch.equal(a, b))
if not torch.equal(a, b):
    sys.exit("the one-call and the bucketed outputs differ")
ms = {"one call": [], "bucketed": []}
for r in range(args.rounds):
    for name, fn in (("one call", one_call), ("bucketed", bucketed)) if r % 2 == 0 else (("bucketed", bucketed), ("one call", one_call)):
        ms[name].append(timed(fn)[0])
for name, v in ms.items():
    med = statistics.median(v)
    print("%-9s median %8.1f ms (min %8.1f, max %8.1f over %d rounds)  %7.0f scenarios/s" % (
        name, med, min(v), max(v), len(v), S / (med / 1e3)))
print("one call / bucketed, median time: %.3f" % (statistics.median(ms["one call"]) / statistics.median(ms["bucketed"])))
