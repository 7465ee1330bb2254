"""GPU (-m gpu): guided sampling of scenes of more than 64 agents.  The agent-collision kernel streams the partners of such a
scene through shared memory in tiles; these tests hold it to the oracle, to the same agents split into small scenes, and to
the sampler's invariances (per-scene calls, ragged batches, chunks, lanes, the policy's sample choice)."""
import pytest
import torch

import cld_oracle as O
from cld_b200.synthetic import make_scenes

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def cu(d):
    return {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in d.items()}


def dec_sd_of(vae):
    return {k: v.detach().cpu() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}


def cpu_sd(m):
    return {k: v.detach().cpu() for k, v in m.state_dict().items()}


def new_model(T=52, precision="fp32", N=1, **kw):
    from cld_b200 import default_algo_config
    from cld_b200.dm_model import DmModel
    from cld_b200.vae import VaeModel
    algo = default_algo_config(horizon=T, num_samp=N)
    torch.manual_seed(0)
    dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=10, precision=precision, **kw).cuda()
    vae = VaeModel(algo).bind(dm)
    return dm, vae, algo


@pytest.fixture(scope="module")
def build():
    cache = {}

    def get(T=52, precision="fp32", N=1, **kw):
        key = (T, precision, N, tuple(sorted(kw.items())))
        if key not in cache:
            cache[key] = new_model(T, precision, N, **kw)
        return cache[key]
    return get


def rows_of(v, N):
    return v.repeat_interleave(N, 0) if N > 1 else v


# --------------------------------------------------------------------------------------------------------------------------
# 1. against the oracle
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("A,T,N", [(65, 52, 1), (128, 52, 1), (256, 52, 1), (100, 104, 2)])
def test_large_scene_guidance_step_vs_oracle(build, A, T, N, precision):
    """Default guidance (agent and map collision), one dense scene: losses and gradient against the oracle's autograd.  The
    bf16 handle decodes with the tensor-core LSTM and takes the suite's bf16 guidance thresholds."""
    from cld_b200.engine import default_guidance
    dm, vae, _ = build(T, precision)
    S = 1
    aux, batch = make_scenes(S, A, horizon=T, seed=7000 + A + T, dense=True)
    torch.manual_seed(7100 + A + T)
    z = torch.randn(S * A * N, T, 4)
    eng = dm.engine(S * A * N)
    scene = eng.make_scene(batch, S, A, N)
    cond, curr = rows_of(aux["cond_feat"], N).cuda(), rows_of(aux["curr_states"], N).cuda()
    _, grad, loss = eng.guidance_step(z.cuda(), cond, curr, scene, default_guidance())
    g_or, per = O.guidance_grad(dec_sd_of(vae), z, aux["cond_feat"], aux["curr_states"], batch, A, N)
    l_ac = torch.cat([p["agent_collision"] for p in per]).reshape(-1)
    l_mc = torch.cat([p["map_collision"] for p in per]).reshape(-1)
    nz = g_or != 0
    sign_agree = (torch.sign(grad.cpu())[nz] == torch.sign(g_or)[nz]).float().mean().item()
    print("A=%d T=%d N=%d %s: rel(l_ac) %.2e rel(l_mc) %.2e rel(grad) %.2e sign %.6f" % (
        A, T, N, precision, rel(loss[0], l_ac), rel(loss[1], l_mc), rel(grad, g_or), sign_agree))
    ltol, gtol, stol = (1e-4, 1e-3, 0.999) if precision == "fp32" else (1e-3, 5e-3, 0.995)
    assert l_ac.abs().sum() > 0
    assert rel(loss[0], l_ac) < ltol and rel(loss[1], l_mc) < ltol
    assert rel(grad, g_or) < gtol and sign_agree > stol
    # the agent-collision term alone moves the latents
    _, g_ac, _ = eng.guidance_step(z.cuda(), cond, curr, scene, default_guidance(map_collision=0.0))
    assert g_ac.abs().sum().item() > 0


# --------------------------------------------------------------------------------------------------------------------------
# 2. a pair that spans the first and the last tile
# --------------------------------------------------------------------------------------------------------------------------
def test_pair_across_first_and_last_tile_vs_oracle(build):
    from cld_b200.engine import default_guidance
    dm, vae, _ = build()
    S, A, N = 1, 200, 1
    aux, batch = make_scenes(S, A, seed=7300)
    wfa = batch["world_from_agent"].clone()
    wfa[:, 0, 2] = torch.arange(A).float() * 300.0              # 300 m apart: no pair but (0, A - 1) is within reach
    wfa[:, 1, 2] = 0.0
    wfa[A - 1] = wfa[0]                                          # agent A - 1 on top of agent 0
    batch["world_from_agent"] = wfa
    speed = batch["curr_speed"].clone()
    speed[0] = speed[A - 1] = 5.0
    batch["curr_speed"] = speed
    curr = aux["curr_states"].clone()
    curr[:, 2] = speed
    aux = dict(aux, curr_states=curr)
    for k in ("all_other_agents_future_positions", "all_other_agents_future_availability"):
        batch.pop(k)
    cfg = default_guidance(map_collision=0.0, optimizer="sgd", lr=1.0)
    torch.manual_seed(7301)
    z = torch.randn(A, 52, 4)
    eng = dm.engine(A)
    _, grad, loss = eng.guidance_step(z.cuda(), aux["cond_feat"].cuda(), curr.cuda(), eng.make_scene(batch, S, A, N), cfg)
    ocfg = dict(O.DEFAULT_GUIDANCE, map_collision=0.0, optimizer="sgd", lr=1.0)
    g_or, per = O.guidance_grad(dec_sd_of(vae), z, aux["cond_feat"], curr, batch, A, N, ocfg)
    l_ac = per[0]["agent_collision"].reshape(-1)
    pair = torch.tensor([0, A - 1])
    assert (l_ac[pair] > 0).all() and l_ac[1:A - 1].abs().sum() == 0
    assert (loss[0].cpu()[pair] > 0).all() and loss[0].cpu()[1:A - 1].abs().sum() == 0
    assert rel(loss[0], l_ac) < 1e-4
    assert grad.cpu()[pair].abs().sum() > 0 and grad.cpu()[1:A - 1].abs().sum() == 0
    assert rel(grad.cpu()[pair], g_or[pair]) < 1e-3


# --------------------------------------------------------------------------------------------------------------------------
# 3. 16 far-apart clusters of 64 agents in one scene equal 16 scenes of 64
# --------------------------------------------------------------------------------------------------------------------------
def test_clusters_of_one_large_scene_equal_small_scenes(build):
    """One scene of 1024 agents made of 16 dense clusters of 64, 1.5 km apart, against the same tensors read as 16 scenes of 64.
    Pairs of different clusters fail the centre-distance test, and the tiles visit the partners in ascending order, so every
    per-agent sum is the small scene's.  The large scene normalises by 1/A and 1/(A N) with A = 1024 instead of 64: powers of
    two, so its loss is exactly 1/16 and its gradient exactly 1/256 of the small scenes'."""
    from cld_b200.engine import default_guidance
    dm, _, _ = build()
    C, A = 16, 64
    B = C * A
    aux, batch = make_scenes(C, A, seed=7400, dense=True)
    wfa = batch["world_from_agent"].clone()
    wfa[:, 0, 2] += torch.arange(C).float().repeat_interleave(A) * 1500.0
    batch["world_from_agent"] = wfa
    for k in ("all_other_agents_future_positions", "all_other_agents_future_availability"):
        batch.pop(k)
    cfg = default_guidance(map_collision=0.0, optimizer="sgd", lr=1.0)
    torch.manual_seed(7401)
    z = torch.randn(B, 52, 4).cuda()
    cond, curr = aux["cond_feat"].cuda(), aux["curr_states"].cuda()
    eng = dm.engine(B)
    _, g_big, l_big = eng.guidance_step(z, cond, curr, eng.make_scene(batch, 1, B, 1), cfg)
    _, g_small, l_small = eng.guidance_step(z, cond, curr, eng.make_scene(batch, C, A, 1), cfg)
    assert l_small[0].abs().sum() > 0 and g_small.abs().sum() > 0
    print("clusters: rel(loss) %.2e rel(grad) %.2e" % (rel(l_big[0] * 16, l_small[0]), rel(g_big * 256, g_small)))
    assert torch.equal(l_big[0] * 16, l_small[0])
    assert torch.equal(g_big * 256, g_small)


# --------------------------------------------------------------------------------------------------------------------------
# 4. the sampler
# --------------------------------------------------------------------------------------------------------------------------
def test_bf16_ddim_two_large_scenes_equal_per_scene_calls(build):
    from cld_b200.engine import default_guidance
    S, A, N = 2, 150, 2
    dm, _, algo = build(52, "bf16", N)
    aux, batch = make_scenes(S, A, seed=7500, dense=True)
    torch.manual_seed(7501)
    x_init = torch.randn(S * A * N, 52, 4)
    kw = dict(sampler="ddim", guidance=default_guidance(), want_indicators=True, agents_per_scene=A)
    full = dm(cu(batch), cu(aux), algo, x_init=x_init.cuda(), **kw)
    assert torch.isfinite(full["pred_traj"]).all()
    for s in range(S):
        sl, rl = slice(s * A, (s + 1) * A), slice(s * A * N, (s + 1) * A * N)
        sb = {k: (v[sl] if torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == S * A else v) for k, v in batch.items()}
        sa = {k: v[sl] for k, v in aux.items()}
        one = dm(cu(sb), cu(sa), algo, x_init=x_init[rl].cuda(), **kw)
        for k in ("pred_traj", "traj", "offroad", "coll"):
            assert torch.equal(full[k][rl], one[k]), (k, s)


def test_ragged_batch_with_large_scenes_equals_per_scene_calls(build):
    from cld_b200.engine import default_guidance
    dm, _, algo = build()
    sizes = [3, 70, 130, 70]
    B = sum(sizes)
    aux, batch = make_scenes(1, B, seed=7600, dense=True)
    batch["scene_index"] = torch.cat([torch.full((c,), 20 + i) for i, c in enumerate(sizes)])
    torch.manual_seed(7601)
    x_init, noises = torch.randn(B, 52, 4), torch.randn(10, B, 52, 4)
    kw = dict(guidance=default_guidance(), want_indicators=True)
    out = dm(cu(batch), cu(aux), algo, noise=noises.cuda(), x_init=x_init.cuda(), **kw)
    pos = 0
    for c in sizes:
        sl = slice(pos, pos + c)
        sb = {k: (v[sl] if (torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == B) else v) for k, v in batch.items()}
        sa = {k: v[sl] for k, v in aux.items()}
        one = dm(cu(sb), cu(sa), algo, noise=noises[:, sl].cuda(), x_init=x_init[sl].cuda(), **kw)
        for k in ("pred_traj", "traj", "offroad", "coll"):
            assert torch.equal(out[k][sl], one[k]), (k, c)
        pos += c


def test_guided_sampler_80_agents_vs_oracle(build):
    """10 guided DDPM steps on supplied noise, one scene of 80 agents: fp32 against the composed oracle (the thresholds of
    test_gpu_parity.py::test_guided_sampler_vs_oracle)."""
    from cld_b200.engine import default_guidance
    dm, vae, algo = build()
    S, A = 1, 80
    aux, batch = make_scenes(S, A, seed=7700, dense=True)
    torch.manual_seed(7701)
    x_init, noises = torch.randn(A, 52, 4), torch.randn(10, A, 52, 4)
    out = dm(cu(batch), cu(aux), algo, noise=noises.cuda(), x_init=x_init.cuda(), guidance=default_guidance(),
             want_indicators=True)
    dec_sd = dec_sd_of(vae)
    gd = dict(dec_sd=dec_sd, cond=aux["cond_feat"], curr=aux["curr_states"], batch=batch, A=A, N=1, cfg=O.DEFAULT_GUIDANCE)
    want = O.sample(cpu_sd(dm.model), O.make_schedule(10), aux["cond_feat"], x_init, noises, 10, 1, "ddpm", guidance=gd)
    frac = ((out["pred_traj"].cpu() - want["pred_traj"]).abs() > 1e-2 * want["pred_traj"].abs().max()).float().mean().item()
    print("A=80 guided sampler: rel %.3e, fraction off by >1%% of max %.5f" % (rel(out["pred_traj"], want["pred_traj"]), frac))
    assert frac < 0.02
    wtraj, _ = O.decode_rollout(dec_sd, out["pred_traj"].cpu(), aux["cond_feat"], aux["curr_states"])
    assert rel(out["traj"], wtraj) < 1e-4
    woff, wcoll = O.indicators(out["traj"].cpu()[..., :2], batch)
    assert torch.equal(out["offroad"].cpu(), woff) and torch.equal(out["coll"].cpu(), wcoll)


# --------------------------------------------------------------------------------------------------------------------------
# 5. chunks and lanes
# --------------------------------------------------------------------------------------------------------------------------
def test_large_scenes_chunks_and_lanes_equal_the_single_call(build):
    """In-kernel Philox noise, 2 scenes of 130 agents x 2 samples: an engine that holds one scene per chunk and two lanes give
    the single-lane, unchunked result bit for bit; an engine smaller than one scene is refused."""
    from cld_b200.engine import default_guidance
    S, A, N = 2, 130, 2
    R = S * A * N
    aux, batch = make_scenes(S, A, seed=7800, dense=True)
    guid = default_guidance()
    kw = dict(sampler="ddpm", guidance=guid, use_device_rng=True, seed=2025, want_indicators=True, agents_per_scene=A)
    dm, _, algo = build(52, "fp32", N, max_rows=R)
    torch.manual_seed(7801)
    x_init = torch.randn(R, 52, 4).cuda()
    full = dm(cu(batch), cu(aux), algo, x_init=x_init, **kw)
    assert torch.isfinite(full["pred_traj"]).all()
    dm_c, _, _ = build(52, "fp32", N, max_rows=A * N)
    eng = dm_c.engine(1)
    assert eng.max_rows == A * N
    cond_rows, curr_rows = aux["cond_feat"].cuda().repeat_interleave(N, 0), aux["curr_states"].cuda().repeat_interleave(N, 0)
    o = eng.sample(x_init, cond_rows, seed=2025, curr_rows=curr_rows, scene=eng.make_scene(batch, S, A, N), guidance=guid,
                   sampler="ddpm", want_indicators=True)
    assert torch.equal(o["x0"], full["pred_traj"]) and torch.equal(o["traj"], full["traj"]) and torch.equal(o["coll"], full["coll"])
    dm_l, _, algo_l = build(52, "fp32", N, max_rows=R, lanes=2)
    lan = dm_l(cu(batch), cu(aux), algo_l, x_init=x_init, **kw)
    for k in ("pred_traj", "traj", "offroad", "coll"):
        assert torch.equal(lan[k], full[k]), k
    dm_s, _, _ = build(52, "fp32", N, max_rows=128)
    e_s = dm_s.engine(1)
    with pytest.raises(RuntimeError, match="smaller than one scene"):
        e_s.sample(x_init, cond_rows, seed=2025, curr_rows=curr_rows, scene=e_s.make_scene(batch, S, A, N), guidance=guid,
                   sampler="ddpm")


# --------------------------------------------------------------------------------------------------------------------------
# 6. the policy
# --------------------------------------------------------------------------------------------------------------------------
def test_policy_get_action_on_large_scenes():
    from cld_b200.engine import default_guidance
    from cld_b200.policy import GuidedDiffusionPolicy
    S, A, N = 2, 96, 3
    dm, vae, algo = new_model(52, "bf16")
    aux, batch = make_scenes(S, A, seed=7900, dense=True)
    pol = GuidedDiffusionPolicy(dm, vae, algo, guidance=default_guidance())
    action, info = pol.get_action(cu(batch), num_action_samples=N, step_index=0, aux_info=cu(aux), use_device_rng=True, seed=5)
    assert action["positions"].shape == (S * A, 52, 2) and torch.isfinite(action["positions"]).all()
    assert torch.isfinite(action["yaws"]).all()
    active = list(info["guide_losses"])
    assert "agent_collision" in active
    stacked = torch.stack([info["guide_losses"][k] for k in active], dim=2).cpu()
    want = O.choose_action_from_guidance(stacked, A, True)
    assert torch.equal(info["act_idx"].cpu(), want)
    ar = torch.arange(S * A)
    assert torch.equal(action["positions"].cpu(), info["action_samples"]["positions"].cpu()[ar, want])
