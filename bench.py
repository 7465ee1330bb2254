#!/usr/bin/env python
"""bench.py -- guided scenarios/s of the CLD sampling hot path on B200 (contract in the task brief).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config cfg1|cfg2|cfg3|cfg4] [--precision bf16|fp32]
                  [--dump-outputs DIR]

A "step" = ONE pass of the hot path over one batch of synthetic nuScenes-shaped scenes:
    S scenes x A agents x N samples  ->  K_d denoising steps (denoiser + posterior update [+ guidance])
    -> LSTM decode + unicycle rollout -> off-road / collision indicators [-> all-gather over ranks].
Workloads = BASELINE.json configs (SURVEY.md sec. 8d):
  cfg1 (default, the configuration the metric is quoted on): 256 scenes x 16 agents, 50-step DDIM, agent + map collision guidance;
        weak scaling (every rank runs its own 256 scenes).
  cfg2: 4096 scenes x 32 agents x 8 samples, 50-step DDIM guided; STRONG scaling: the scenes are sharded over the ranks
        (`shard_scenes`), rows in 65 536-row chunks, one all-gather of 109 MB per rank at N = 8.
  cfg3: horizon 104, 64 scenes x 64 agents, DDPM-100 guided, conditioning from 34 x 224 x 224 rasters (ContextEncoder with the
        fused history rasteriser inside the step).
  cfg4: PPO-mode shape: 8 scenes x 16 agents x 4 samples, 16 DDPM steps with per-step guidance.

Printed JSON (rank 0, one line): metric/value/unit/... per the contract, plus
  roofline      dominant kernel (denoiser forward): algorithmic FLOPs / CUDA-event time vs measured bf16 peak
  roofline_hbm  the HBM-bound kernels (posterior step K3, indicators K6): algorithmic bytes / CUDA-event time vs measured HBM peak
  cpu_baseline  the oracle (CPU port of the reference's PyTorch sampler) on a bounded sample of the workload
  parity        the CUDA path against that oracle run on the same scene (free-running chain)
  e2e           same metric through the public API (cld_b200.DmModel.forward) from pinned HOST buffers
  gpu_launches  kernels launched by libcld_b200.so in the timed region
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_ROW_STEP = {52: 119.23e6, 104: 237.42e6}     # SURVEY.md App. B (hook-counted on the reference module)
WORKLOADS = {
    "cfg1": dict(scenes=256, agents=16, samples=1, horizon=52, n_timesteps=100, stride=2, sampler="ddim", context=False, scaling="weak"),
    "cfg2": dict(scenes=4096, agents=32, samples=8, horizon=52, n_timesteps=100, stride=2, sampler="ddim", context=False, scaling="strong"),
    "cfg3": dict(scenes=64, agents=64, samples=1, horizon=104, n_timesteps=100, stride=1, sampler="ddpm", context=True, scaling="weak"),
    "cfg4": dict(scenes=8, agents=16, samples=4, horizon=52, n_timesteps=16, stride=1, sampler="ddpm", context=False, scaling="weak"),
}
MAX_CHUNK_ROWS = 65536

# dram__bytes_read.sum + dram__bytes_write.sum of ONE denoiser launch from the committed `ncu --set full` capture; only known for
# the captured shape (see profiles/)
NCU_DRAM_BYTES_PER_LAUNCH = {}
_p = os.path.join(ROOT, "profiles", "r02_unet_tc_dram_bytes.json")
if os.path.exists(_p):
    NCU_DRAM_BYTES_PER_LAUNCH = {tuple(k.split(":")): v for k, v in json.load(open(_p)).items()}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg1", choices=sorted(WORKLOADS))
    ap.add_argument("--lanes", type=int, default=0,
                    help="DmModel(lanes=L): whole-scene sub-batches on L engines / CUDA streams (0 = 4 where the workload allows it, else 1)")
    ap.add_argument("--precision", default=os.environ.get("CLD_BENCH_PRECISION", "bf16"), choices=["bf16", "fp32"])
    ap.add_argument("--sampler", default=None, choices=["ddim", "ddpm"])
    ap.add_argument("--no-guidance", action="store_true")
    ap.add_argument("--scenes", type=int, default=None, help="override the number of scenes (total for cfg2, per rank otherwise)")
    ap.add_argument("--cpu-scenes", type=int, default=1, help="scenes in the bounded CPU-baseline sample")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-lanes", action="store_true", help="same as --lanes 1 (one engine / stream; the kernel brackets then come from the timed region)")
    ap.add_argument("--skip-context", action="store_true", help="do not time the context encoder (row a14) after the headline")
    ap.add_argument("--skip-hbm", action="store_true", help="do not time the HBM-bound kernels (K3, K6) alone")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.warmup < 0:
        ap.error("--warmup must not be negative")
    a.w = dict(WORKLOADS[a.config])
    if a.sampler:
        a.w["sampler"] = a.sampler
    if a.scenes:
        a.w["scenes"] = a.scenes
    a.w["guided"] = not a.no_guidance
    return a


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe): ONE `nvidia-smi -lms 200` process,
    started before the warm-up (its NVML start-up stays out of the timed region; a process spawned per sample stalled kernel launches
    for tens of milliseconds), killed after; only the samples that arrived between `mark()` and `stop()` are used."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.t0, self.proc = index, [], None, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.strip().split(",")]
                if len(f) >= 7:
                    self.rows.append((time.perf_counter(), f))
        except Exception:
            pass

    def mark(self):
        self.t0 = time.perf_counter()

    def stop(self):
        t1 = time.perf_counter()
        time.sleep(0.25)                         # let the sample that covers the end of the region arrive
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=3)
        t0 = self.t0 if self.t0 is not None else 0.0
        rows = [f for ts, f in self.rows if t0 <= ts <= t1 + 0.25] or [f for _, f in self.rows[-1:]]
        sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(rows[0][1]) if rows and rows[0][1].replace(".", "").isdigit() else None,
                "reasons": sorted(reasons), "samples": len(rows)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1393.0), d.get("hbm_gbs", 6538.3), "measured"
    return 1590.0, 6650.0, "fallback"


def k_steps(w):
    return len(range(0, w["n_timesteps"], w["stride"]))


def workload_text(a):
    w = a.w
    return ("%s: %d scenes x %d agents x %d sample(s), T=%d, n_timesteps=%d stride %d (%d denoising steps, %s)%s%s, "
            "decode+rollout+indicators; random-init weights" % (
                a.config, w["scenes"], w["agents"], w["samples"], w["horizon"], w["n_timesteps"], w["stride"], k_steps(w),
                w["sampler"], ", agent_collision+map_collision guidance" if w["guided"] else "",
                ", conditioning from 34x224x224 rasters (ContextEncoder + fused history rasteriser in the step)" if w["context"] else ""))


def workload_config(a, world, rows_per_gpu=None):
    w = a.w
    rows = rows_per_gpu if rows_per_gpu is not None else w["scenes"] * w["agents"] * w["samples"] // (world if w["scaling"] == "strong" else 1)
    return {"workload": workload_text(a), "rows_per_gpu": rows, "precision": a.precision,
            "l2": "inputs change every denoising step and the guidance stash (133 KB per row) exceeds L2 beyond ~900 rows; denoiser "
                  "activations are on-chip; no L2 flush needed between steps",
            "parallelism": "scene-sharded (%s scaling), %d rank(s)" % (w["scaling"], world)}


# ---------------------------------------------------------------------------------------------------------------------------
# CPU leg (test infrastructure): the oracle port of the reference's PyTorch sampler on a bounded sample, all host threads.
# The parameter containers are built WITHOUT mapping libcld_b200.so (cld_b200.dm_model / vae import the library lazily).
# ---------------------------------------------------------------------------------------------------------------------------
def cpu_case(a, n_scenes):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import cld_oracle as O
    from cld_b200 import default_algo_config, make_scenes
    from cld_b200.dm_model import DmModel
    from cld_b200.vae import VaeModel
    w = a.w
    A, N, T = w["agents"], w["samples"], w["horizon"]
    algo = default_algo_config(num_samp=N)
    algo.horizon = T
    torch.manual_seed(0)
    dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=w["n_timesteps"])
    vae = VaeModel(algo)
    unet_sd = {k: v.detach() for k, v in dm.model.state_dict().items()}
    dec_sd = {k: v.detach() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}
    aux, batch = make_scenes(n_scenes, A, horizon=T, seed=123, dense=True)
    R = n_scenes * A * N
    torch.manual_seed(7)
    x_init = torch.randn(R, T, 4)
    noises = torch.randn(k_steps(w), R, T, 4) if w["sampler"] == "ddpm" else None
    rep = (lambda v: v.repeat_interleave(N, 0)) if N > 1 else (lambda v: v)
    gd = dict(dec_sd=dec_sd, cond=aux["cond_feat"], curr=aux["curr_states"], batch=batch, A=A, N=N, cfg=O.DEFAULT_GUIDANCE) if w["guided"] else None
    sched = O.make_schedule(w["n_timesteps"])

    def one():
        with torch.no_grad():
            out = O.sample(unet_sd, sched, rep(aux["cond_feat"]), x_init, noises, w["n_timesteps"], w["stride"], w["sampler"], guidance=gd)
            traj, _ = O.decode_rollout(dec_sd, out["pred_traj"], rep(aux["cond_feat"]), rep(aux["curr_states"]))
            off, coll = O.indicators(traj[..., :2], {k: (rep(v) if torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == n_scenes * A else v)
                                                     for k, v in batch.items()})
        return out["pred_traj"], traj, off, coll
    return dict(one=one, aux=aux, batch=batch, x_init=x_init, noises=noises, O=O, unet_sd=unet_sd, A=A, N=N, T=T)


def cpu_oracle_rate(a, n_scenes, steps, warmup):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c = cpu_case(a, n_scenes)
    for _ in range(warmup):
        c["one"]()
    t0 = time.perf_counter()
    res = None
    for _ in range(steps):
        res = c["one"]()
    dt = (time.perf_counter() - t0) / steps
    # the batched denoiser alone (1 024 rows, one step): the CPU's best per-row rate, for scale
    with torch.no_grad():
        xb, cb = torch.randn(1024, c["T"], 4), torch.randn(1024, 256)
        tb = torch.full((1024,), 5, dtype=torch.long)
        c["O"].unet_forward(c["unet_sd"], xb[:64], cb[:64], tb[:64])
        t1 = time.perf_counter()
        c["O"].unet_forward(c["unet_sd"], xb, cb, tb)
        den_rows_s = 1024 / (time.perf_counter() - t1)
    return n_scenes / dt, dt, cores, c, res, den_rows_s


DUMP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """Writes the tensors of `arrays` (name -> tensor; nested dicts as "<outer>.<inner>") to d/<name>.npy, float64 and 32/64-bit
    integer tensors as float64 (float32 cannot hold all their values), everything else as float32, so that the results of two builds
    can be compared output for output.  Above DUMP_BYTES in all, every array keeps the same fraction of its rows (leading dimension),
    chosen by a fixed seed: two runs with the same arguments write the same rows."""
    import numpy as np
    import torch
    flat = {}
    for k, v in arrays.items():
        for k2, v2 in (v.items() if isinstance(v, dict) else [(None, v)]):
            if torch.is_tensor(v2):
                flat[k if k2 is None else "%s.%s" % (k, k2)] = v2
    wide = lambda v: v.dtype in (torch.float64, torch.int32, torch.int64)   # noqa: E731
    total = sum(v.numel() * (8 if wide(v) else 4) for v in flat.values())
    frac = min(1.0, DUMP_BYTES / max(total, 1))
    os.makedirs(d, exist_ok=True)
    for k, v in sorted(flat.items()):
        if frac < 1.0 and v.dim() > 0:
            keep = torch.randperm(v.shape[0], generator=torch.Generator().manual_seed(0))[:max(1, int(v.shape[0] * frac))]
            v = v.index_select(0, keep.sort().values.to(v.device))
        v = v.detach().to("cpu", torch.float64 if wide(v) else torch.float32)
        np.save(os.path.join(d, k + ".npy"), v.numpy())


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = a.steps, a.warmup
    rate, dt, cores, _, res, den = cpu_oracle_rate(a, a.cpu_scenes, steps, warm)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, dict(zip(("pred_traj", "traj", "offroad", "coll"), res)))
    sample = "%d of %d scenes of %s, oracle port of the reference's PyTorch sampler (guidance through autograd as in the reference), %d host threads" % (
        a.cpu_scenes, a.w["scenes"], workload_text(a), cores)
    print(json.dumps({
        "impl": "reference", "metric": "guided scenarios/sec (50-step DDIM)", "value": rate, "unit": "scenarios/s",
        "n_gpus": a.gpus, "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": a.w["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a, a.gpus),
        "cpu_baseline": {"value": rate, "unit": "scenarios/s", "cores": cores, "kind": "port", "sample": sample,
                         "batched_denoiser_rows_per_s": den},
        "e2e": {"value": rate, "unit": "scenarios/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------------------------------
# side measurements (outside the headline's timed region)
# ---------------------------------------------------------------------------------------------------------------------------
def context_encoder_rate(dev, agents=1024, iters=5, warmup=3):
    """SURVEY.md sec. 8 row a14 beside the headline: ContextEncoder.forward (34 x 224 x 224 raster -> cond_feat), inputs resident in HBM."""
    import torch
    from cld_b200 import default_algo_config
    from cld_b200.context import ContextEncoder
    torch.manual_seed(0)
    ce = ContextEncoder(4, default_algo_config(), {"image": (34, 224, 224)}, max_agents=agents).to(dev)
    g = torch.Generator(device=dev).manual_seed(11)
    batch = {"image": (torch.rand(agents, 34, 224, 224, device=dev, generator=g) < 0.05).float(),
             "history_positions": torch.zeros(agents, 31, 2, device=dev), "history_yaws": torch.zeros(agents, 31, 1, device=dev),
             "curr_speed": torch.rand(agents, device=dev, generator=g) * 10}
    for _ in range(warmup):
        ce(batch)
    torch.cuda.synchronize()
    l0 = ce.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        ce(batch)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    tf_peak, _, peak_src = measured_peaks()
    tflops = 6.07e9 * agents / (ms * 1e-3) / 1e12
    out = {"value": agents / ms * 1e3, "unit": "agents/s", "agents": agents, "ms": ms, "iters": iters, "dtype": "bf16 (fp32 accumulate)",
           "algorithmic_gflop_per_agent": 6.07, "executed_gflop_per_agent": ce.conv_flops_per_agent() / 1e9,
           "achieved_tflops": tflops, "frac_of_bf16_peak": tflops / tf_peak, "peak_source": peak_src + " bf16_tflops_sustained",
           "gpu_launches": ce.launch_count() - l0, "bytes_in_per_agent": 34 * 224 * 224 * 4}
    ce.close()
    return out


def ppo_update_rate(dev, skip_cpu, rows=128, iters=20, warmup=3):
    """SURVEY.md sec. 8 f-2 beside the cfg4 line: one minibatch of ppo_update (guide_dm_trainer.py:150-172: denoiser forward,
    log-prob, clipped surrogate, backward, Adam, weight re-pack) on `rows` replay rows (config.yaml:168), inputs resident in HBM;
    CPU: the oracle's autograd restatement of the same minibatch on all host threads (1 warm-up + 1 timed)."""
    import torch
    from cld_b200 import default_algo_config
    from cld_b200.dm_model import DmModel
    from cld_b200.trainer import FusedAdam
    torch.manual_seed(0)
    dm = DmModel(default_algo_config(), {"image": (34, 224, 224)}, n_timesteps=16).to(dev)
    for p in dm.model.parameters():
        p.requires_grad_(True)
    dm.train_precision = "tf32"
    opt = FusedAdam(dm, lr=1e-4, weight_decay=1e-5)
    g = torch.Generator(device=dev).manual_seed(5)
    rn = lambda *sh: torch.randn(*sh, device=dev, generator=g)    # noqa: E731
    x1, x0, cond, lp_old, reward = rn(rows, 52, 4), rn(rows, 52, 4), rn(rows, 256), rn(rows), rn(rows)
    t = torch.full((rows,), 3, dtype=torch.long, device=dev)

    def step():
        loss, _ = dm.ppo_minibatch_grad(x1, x0, cond, t, lp_old, reward, 0.0, 0.2)
        opt.step()
        return loss

    def timed():
        for _ in range(warmup):
            step()
        eng = dm.train_engine(rows)
        torch.cuda.synchronize()
        l0 = eng.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters, (eng.launch_count() - l0) // iters
    ms_eager, launches = timed()
    # the same update captured as a CUDA graph (cld_b200.trainer.GraphedPPOStep: what GuideDMTrainer runs)
    from cld_b200.trainer import GraphedPPOStep
    gs = GraphedPPOStep(dm, opt, rows, 0.2, eager_calls=0)
    for dst, src in zip(gs.buffers(), (x0, x1, lp_old, reward, cond)):
        dst.copy_(src)
    gs.t.copy_(t)
    eager_step = step
    step = lambda: gs(0.0)        # noqa: E731
    ms, _ = timed()
    step = eager_step
    dm.train_precision = "fp32"
    ms32, launches32 = timed()
    out = {"rows": rows, "ms_per_minibatch_update": ms, "updates_per_s": 1e3 / ms, "iters": iters,
           "dtype": "tf32 tensor-core convolutions (tcgen05 kind::tf32, fp32 accumulate), fp32 elsewhere",
           "mode": "one CUDA-graph replay per update (forward, log-prob, surrogate, backward on two streams, Adam, weight re-pack)",
           "gpu_launches_per_update": launches, "ms_per_minibatch_update_without_graph": ms_eager,
           "algorithmic_gflop_per_update": 3 * 119.23e-3 * rows, "achieved_tflops": 3 * 119.23e6 * rows / (ms * 1e-3) / 1e12,
           "ppo_update_s": "%.1f s for the reference's 10 epochs x 300 minibatches" % (3000 * ms * 1e-3),
           "fp32_parity_mode": {"ms_per_minibatch_update": ms32, "gpu_launches_per_update": launches32, "dtype": "fp32 (CUDA cores)"}}
    if not skip_cpu:
        import time
        import cld_oracle as O
        sd = {k: v.detach().cpu() for k, v in dm.model.state_dict().items()}
        args = [v.cpu() for v in (x1, x0, cond, t, lp_old, reward)]
        sched = O.make_schedule(16)
        torch.set_num_threads(os.cpu_count())
        O.ppo_grads(sd, sched, *args, 0.0, 0.2)
        t0 = time.perf_counter()
        O.ppo_grads(sd, sched, *args, 0.0, 0.2)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"ms_per_minibatch_grad": dt * 1e3, "cores": os.cpu_count(), "kind": "port",
                               "sample": "oracle autograd of the same %d-row minibatch (forward + backward, no optimizer step)" % rows}
    return out


def hbm_kernel_rooflines(eng, R, T, A, scene, dev, iters=20):
    """K3 (posterior step) and K6 (indicators) alone at the rows of one launch: algorithmic bytes (SURVEY.md sec. 8d) / CUDA-event time."""
    import torch
    _, hbm_peak, src = measured_peaks()
    x, eps = torch.randn(R, T, 4, device=dev), torch.randn(R, T, 4, device=dev)
    traj = torch.randn(R, T, 6, device=dev)
    res = {}

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters
    n_t = int(eng.cfg.n_timesteps)
    ms = timed(lambda: eng.posterior_step(x, eps, None, n_t - 2, max(n_t - 4, 0), sampler="ddim", want_mean=True))
    by = R * T * 4 * 4 * 4                      # x, eps in; x', mean out (the stand-alone entry point writes both)
    res["posterior_step"] = {"rows": R, "ms": ms, "bytes": by, "achieved": by / ms / 1e6, "peak": hbm_peak, "unit": "GB/s",
                             "frac": by / ms / 1e6 / hbm_peak, "bound": "hbm"}
    ms = timed(lambda: eng.indicators(traj, scene))
    by = R * (T * 6 * 4 + (A - 1) * T * 9 + T + T + 8)
    res["indicators"] = {"rows": R, "ms": ms, "bytes": by, "achieved": by / ms / 1e6, "peak": hbm_peak, "unit": "GB/s",
                         "frac": by / ms / 1e6 / hbm_peak, "bound": "hbm", "note": "traj 6 channels + neighbour futures + map bytes in; flags + counts out"}
    res["peak_source"] = src + " hbm_gbs"
    return res


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from cld_b200 import default_algo_config, make_scenes
    from cld_b200.distributed import gather_results, shard_scenes
    from cld_b200.dm_model import DmModel
    from cld_b200.engine import default_guidance
    from cld_b200.staging import HostStager
    from cld_b200.synthetic import pack_drivable_map
    from cld_b200.vae import VaeModel
    w = a.w
    A, N, T = w["agents"], w["samples"], w["horizon"]
    S_total = w["scenes"]
    if w["scaling"] == "strong":
        s0, s1 = shard_scenes(S_total, world, rank)
        S, row_offset, job_scenes = s1 - s0, s0 * A * N, S_total
    else:
        S, row_offset, job_scenes = S_total, rank * S_total * A * N, world * S_total
    R = S * A * N
    rows_per_launch = min(R, (MAX_CHUNK_ROWS // (A * N)) * A * N)
    algo = default_algo_config(num_samp=N)
    algo.horizon = T
    torch.manual_seed(0)
    dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=w["n_timesteps"], precision=a.precision, max_rows=rows_per_launch).to(dev)
    dm.stride = w["stride"]
    vae = VaeModel(algo).bind(dm)
    # synthetic scenes: at most 256 distinct ones per rank, tiled (identical scenes cost the same as distinct ones)
    S_gen = min(S, 256)
    aux, batch = make_scenes(S_gen, A, horizon=T, seed=123 + rank, dense=True)
    batch["drivable_map_bits"] = pack_drivable_map(batch["drivable_map"])      # the form the data layer ships: 1 bit per pixel
    if S > S_gen:
        rep_n = (S + S_gen - 1) // S_gen
        tile = lambda v: (v.repeat((rep_n,) + (1,) * (v.dim() - 1))[:S * A] if torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == S_gen * A else v)  # noqa: E731
        aux = {k: tile(v) for k, v in aux.items()}
        batch = {k: tile(v) for k, v in batch.items()}
        batch["scene_index"] = torch.arange(S).repeat_interleave(A)
    guidance = default_guidance() if w["guided"] else None
    eng = dm.engine(rows_per_launch)
    # The measured configuration of the product: DmModel(lanes=L) splits the scenes of a call into L whole-scene sub-batches that run
    # concurrently on their own engines / CUDA streams (bit-identical results: scenes never interact, Philox noise is keyed by the
    # global row id).  The sub-batches fill the SMs that the denoiser's last wave (4 096 rows = 3.46 waves of 148 CTAs) and the
    # 128-CTA LSTM kernels leave idle.  The kernel brackets of `roofline` come from a single-lane pass (kernels timed alone).
    n_lanes = 1 if a.skip_lanes else a.lanes if a.lanes > 0 else (4 if (not w["context"] and S >= 8 and 2048 <= R <= MAX_CHUNK_ROWS) else 1)
    dm_run = dm
    if n_lanes > 1:
        torch.manual_seed(0)
        dm_run = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=w["n_timesteps"], precision=a.precision, max_rows=rows_per_launch,
                         lanes=n_lanes).to(dev)
        dm_run.stride = w["stride"]
        VaeModel(algo).bind(dm_run)
    K_d = k_steps(w)
    host_keys = ["extent", "world_from_agent", "raster_from_agent", "curr_speed", "drivable_map_bits", "scene_index",
                 "all_other_agents_future_positions", "all_other_agents_future_availability", "history_positions"]
    aux_d = {k: v.to(dev) for k, v in aux.items()}
    batch_d = {k: batch[k].to(dev) for k in host_keys}
    aux_h = {k: v.pin_memory() for k, v in aux.items()}
    batch_h = {k: batch[k].pin_memory() for k in host_keys}
    # cfg3: conditioning from rasters -- the context encoder with the fused history rasteriser runs inside the step
    ce = hist_d = hist_h = None
    if w["context"]:
        from cld_b200.context import ContextEncoder
        from cld_b200.synthetic import make_history_batch
        torch.manual_seed(0)
        ce = ContextEncoder(4, algo, {"image": (34, 224, 224)}, max_agents=min(S * A, 2048)).to(dev)
        hb = make_history_batch(64, num_neighbors=15, seed=3)
        rep_n = (S * A + 63) // 64
        hist = {"maps": hb["maps"].repeat(rep_n, 1, 1, 1)[:S * A].contiguous(), "hpos": hb["agent_hist_pos"].repeat(rep_n, 1, 1, 1)[:S * A].contiguous(),
                "hmask": hb["agent_hist_mask"].repeat(rep_n, 1, 1)[:S * A].contiguous(),
                "history_yaws": torch.zeros(S * A, 31, 1)}
        hist_d = {k: v.to(dev) for k, v in hist.items()}
        hist_h = {k: v.pin_memory() for k, v in hist.items()}
    gathered = torch.empty(world * R, T * 6 + T + 1, device=dev) if world > 1 else None
    SEED = 20240707

    def hot_path(b, ax, hd=None, model=None):
        model = model if model is not None else dm_run
        if ce is not None:
            cb = {"raster_from_agent": b["raster_from_agent"], "history_positions": b["history_positions"], "history_yaws": hd["history_yaws"],
                  "curr_speed": b["curr_speed"]}
            cx = ce.forward_history(cb, hd["maps"], hd["hpos"], hd["hmask"])
            ax = {"cond_feat": cx["cond_feat"], "curr_states": cx["curr_states"]}
        out = model(b, ax, algo, sampler=w["sampler"], guidance=guidance, want_indicators=True, agents_per_scene=A,
                    use_device_rng=True, seed=SEED, row_offset=row_offset)
        if world > 1:
            # the path's one exchange: trajectories + indicator flags + collision counts of every rank
            out["all_traj"], out["all_offroad"], out["all_coll"] = gather_results(out["traj"], out["offroad"], out["coll"], out=gathered)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler_thread = ClockSampler(local) if rank == 0 else None
    if sampler_thread:
        sampler_thread.start()                  # one long-running nvidia-smi: started before the warm-up, sampled in the timed region
    for _ in range(a.warmup):
        hot_path(batch_d, aux_d, hist_d)
    barrier()
    if sampler_thread:
        sampler_thread.mark()
    def count_launches():
        n = dm_run.launch_count() + (ce.launch_count() if ce is not None else 0)
        return n + (dm.launch_count() if dm_run is not dm else 0)
    l0 = count_launches()
    if n_lanes == 1:
        eng.profile_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        out = hot_path(batch_d, aux_d, hist_d)
    e1.record()
    barrier()
    if n_lanes == 1:
        prof = eng.profile_end()
    launches = count_launches() - l0
    clocks = sampler_thread.stop() if sampler_thread else None
    ms = e0.elapsed_time(e1) / a.steps
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, out)
    single = None
    if n_lanes > 1:
        # the same workload on ONE engine / stream, per-kind CUDA-event brackets around every kernel group: each kernel is timed alone
        hot_path(batch_d, aux_d, hist_d, model=dm)
        barrier()
        eng.profile_begin()
        s0e, s1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0e.record()
        for _ in range(a.steps):
            out1 = hot_path(batch_d, aux_d, hist_d, model=dm)
        s1e.record()
        barrier()
        prof = eng.profile_end()
        ms1 = s0e.elapsed_time(s1e) / a.steps
        single = {"lanes": 1, "value": (job_scenes / world) / (ms1 / 1e3) * world, "unit": "scenarios/s", "ms_per_step": ms1,
                  "equals_lanes_result": bool(torch.equal(out1["traj"], out["traj"]))}
        del out1
    ms_brackets = ms if single is None else single["ms_per_step"]
    tms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = tms.item()
    value = job_scenes / (ms / 1e3)
    gather_ms = None
    if world > 1:
        # share of the one collective: the all-gather alone, device-timed
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        g0.record()
        for _ in range(5):
            gather_results(out["traj"], out["offroad"], out["coll"], out=gathered)
        g1.record()
        barrier()
        gather_ms = g0.elapsed_time(g1) / 5

    # ---- e2e: public API from pinned host buffers; H2D of call i + 1 overlaps call i (HostStager), D2H of the results every call
    host_sets = [batch_h, aux_h] + ([hist_h] if hist_h is not None else [])
    h2d = sum(v.numel() * v.element_size() for d in host_sets for v in d.values() if torch.is_tensor(v))
    d2h = R * T * 6 * 4 + R * T + R * 4
    n_e2e = max(2, min(a.steps, 4))

    def e2e_run(n):
        st = HostStager(dev)
        st.put(*host_sets)
        for i in range(n):
            got = st.get()
            slot = got[-1]
            if i + 1 < n:
                st.put(*host_sets)
            o = hot_path(got[0], got[1], got[2] if hist_h is not None else None)
            st.release(slot)
            st.read_back(o, ("traj", "offroad", "coll"))
        st.finish()
    e2e_run(2)
    barrier()
    t0 = time.perf_counter()
    e2e_run(n_e2e)
    barrier()
    e2e_ms = (time.perf_counter() - t0) / n_e2e * 1e3
    te = torch.tensor([e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = job_scenes / (te.item() / 1e3)

    if rank == 0:
        tf_peak, hbm_peak, peak_src = measured_peaks()
        den_ms, den_n = prof["denoiser"]
        per_launch_ms = den_ms / max(den_n, 1)
        flop = FLOP_PER_ROW_STEP[T] * rows_per_launch
        achieved = flop / (per_launch_ms * 1e-3) / 1e12 if den_n else 0.0
        key = (a.precision, str(rows_per_launch), str(T))
        roof = {"bound": "tensor", "kernel": "denoiser forward (%s)" % ("unet_tc megakernel, CTA pairs" if a.precision == "bf16" else "fp32 SIMT layer kernels"),
                "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
                "traffic": NCU_DRAM_BYTES_PER_LAUNCH.get(key), "traffic_unit": "bytes (dram read + write per launch)",
                "traffic_source": "profiles/r02_unet_tc_ncu_full_4096rows.csv (ncu --set full, one launch)" if key in NCU_DRAM_BYTES_PER_LAUNCH else None,
                "peak_source": peak_src + " bf16_tflops_sustained", "per_launch_ms": per_launch_ms, "launches_timed": den_n,
                "rows_per_launch": rows_per_launch, "algorithmic_flop_per_launch": flop,
                "measured_in": "the timed region" if single is None else "single-lane pass of the same workload and step count (kernels timed alone; "
                               "in the %d-lane timed region kernels of different lanes overlap)" % n_lanes,
                "share_of_step": {k: v[0] / a.steps / ms_brackets for k, v in prof.items()}}
        hbm = None
        if not a.skip_hbm:
            scene = eng.make_scene({k: (v[:rows_per_launch // N] if torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == S * A else v)
                                    for k, v in batch_d.items()}, rows_per_launch // (A * N), A, N)
            hbm = hbm_kernel_rooflines(eng, rows_per_launch, T, A, scene, dev)
        cpu = parity = None
        if not a.skip_cpu and world == 1:
            rate, dt, cores, c, res, den_rows = cpu_oracle_rate(a, a.cpu_scenes, 1, 1)
            cpu = {"value": rate, "unit": "scenarios/s", "cores": cores, "kind": "port",
                   "sample": "%d of %d scenes of %s, oracle port of the reference's PyTorch sampler (guidance through autograd)%s, 1 warm-up + 1 timed pass "
                             "(%.1f s)" % (a.cpu_scenes, S, workload_text(a), " WITHOUT the context encoder" if w["context"] else "", dt),
                   "batched_denoiser_rows_per_s": den_rows}
            # parity of the measured mode on the same scene(s): the CUDA path on the oracle's inputs (free-running chain)
            n = a.cpu_scenes
            sub_b = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in c["batch"].items()}
            sub_a = {k: v.to(dev) for k, v in c["aux"].items()}
            og = dm(sub_b, sub_a, algo, x_init=c["x_init"].to(dev), noise=None if c["noises"] is None else c["noises"].to(dev),
                    sampler=w["sampler"], guidance=guidance, want_indicators=True, agents_per_scene=A)
            o_x0, o_traj, o_off, o_coll = res
            rel = lambda x, y: ((x.double().cpu() - y.double()).norm() / (y.double().norm() + 1e-30)).item()   # noqa: E731
            parity = {"mode": "%s, %s%s, free-running chain vs the oracle (DDIM and the multi-scene composition have no reference "
                              "implementation: the oracle's pieces are pinned one by one, see tests/)" % (a.precision, w["sampler"], " guided" if w["guided"] else ""),
                      "scenes": n, "rows": n * A * N, "denoising_steps": K_d,
                      "rel_pred_traj": rel(og["pred_traj"], o_x0), "rel_traj": rel(og["traj"], o_traj),
                      "latents_off_by_more_than_0.3": ((og["pred_traj"].cpu() - o_x0).abs() > 0.3).float().mean().item(),
                      "offroad_flag_mismatch": (og["offroad"].cpu() != o_off).float().mean().item(),
                      "collision_count_mismatch": (og["coll"].cpu() != o_coll).float().mean().item(),
                      "teacher_forced": "tests/test_gpu_headline.py (16 scenes x 16 agents, every one of the 50 steps)"}
        ctx = None
        if world == 1 and not a.skip_context and a.config == "cfg1":
            del out
            torch.cuda.empty_cache()
            ctx = context_encoder_rate(dev)
        ppo = None
        if world == 1 and a.config == "cfg4":
            ppo = ppo_update_rate(dev, a.skip_cpu)
        line = {
            "metric": "guided scenarios/sec (50-step DDIM)" if a.config in ("cfg1", "cfg2") else "guided scenarios/sec (%s)" % a.config,
            "value": value, "unit": "scenarios/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": a.precision, "data": "synthetic", "config": workload_config(a, world, R),
            "row_steps_per_s": value * A * N * K_d, "roofline": roof, "roofline_hbm": hbm, "cpu_baseline": cpu, "parity": parity,
            "e2e": {"value": e2e_value, "unit": "scenarios/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": te.item(), "staging": "drivable map shipped bit-packed (1 bit per pixel); H2D of call i+1 overlaps call i "
                                                         "(cld_b200.staging.HostStager); results read back to pinned host memory every call"},
            "gpu_launches": launches, "clocks": clocks, "context_encoder": ctx, "lanes": n_lanes, "single_lane": single,
        }
        if ppo is not None:
            line["ppo_update"] = ppo
        if world > 1:
            line["all_gather"] = {"ms": gather_ms, "bytes_per_rank": R * (T * 7 + 1) * 4, "share_of_step": gather_ms / ms}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
