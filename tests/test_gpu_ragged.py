"""GPU (-m gpu): ragged batches -- scenes of different sizes in ONE call of cld_guidance_step, cld_indicators and cld_sample
(CldScene.scene_start).  Every scene of a ragged call must give what a call on that scene alone gives, bit for bit: the guided
step, the indicators, the samplers with supplied noise and with the in-kernel generator (keyed by the global row), chunks,
lanes and the policy's sample choice.  Malformed offsets are refused before anything runs."""
import pytest
import torch

import cld_oracle as O
from cld_b200.synthetic import make_scenes

pytestmark = pytest.mark.gpu

SIZES = [1, 3, 64, 65, 130, 2]           # single agent, one shared-memory tile, streamed tiles (> 64 agents)
LOSS_MAP = 1                             # loss row of the map-collision term: summed with atomics (last-bit noise)


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def cu(d):
    return {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in d.items()}


def dec_sd_of(vae):
    return {k: v.detach().cpu() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}


def new_model(precision="fp32", N=1, **kw):
    from cld_b200 import default_algo_config
    from cld_b200.dm_model import DmModel
    from cld_b200.vae import VaeModel
    algo = default_algo_config(horizon=52, num_samp=N)
    torch.manual_seed(0)
    dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=10, precision=precision, **kw).cuda()
    vae = VaeModel(algo).bind(dm)
    return dm, vae, algo


@pytest.fixture(scope="module")
def build():
    cache = {}

    def get(precision="fp32", N=1, **kw):
        key = (precision, N, tuple(sorted(kw.items())))
        if key not in cache:
            cache[key] = new_model(precision, N, **kw)
        return cache[key]
    return get


def ragged_case(sizes, seed, waypoints=True):
    """One pool of agents partitioned into scenes of `sizes` agents; target position / speed and (ragged) waypoint entries."""
    from cld_b200.waypoints import TargetPosAtTime
    B = sum(sizes)
    aux, batch = make_scenes(1, B, seed=seed, dense=True)
    batch["scene_index"] = torch.cat([torch.full((c,), 30 + i) for i, c in enumerate(sizes)])
    g = torch.Generator().manual_seed(seed + 1)
    batch["target_pos"] = torch.randn(B, 2, generator=g) * 10
    batch["target_speed"] = (aux["curr_states"][:, 2:3] + torch.randn(B, 1, generator=g)).clamp(min=0).repeat(1, 52)
    if waypoints:
        term = TargetPosAtTime(torch.randn(B, 2, generator=g) * 15, torch.randint(0, 52, (B,), generator=g),
                               agents=torch.rand(B, generator=g) > 0.3)
        batch.update(term.scene_entries(batch, 52, sizes))
    return aux, batch


ALL_TERMS = dict(agent_collision=50.0, map_collision=1.0, target_pos=1.0, target_speed=0.5, acc_limit=1.0, acc_limit_value=1.0,
                 speed_limit=1.0, speed_limit_value=3.0, waypoint=2.0)


def per_scene(batch, aux, sizes):
    """(agent slice, scene batch, scene aux) of every scene."""
    B, pos = sum(sizes), 0
    for c in sizes:
        sl = slice(pos, pos + c)
        sb = {k: (v[sl] if (torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == B) else v) for k, v in batch.items()}
        yield sl, sb, {k: v[sl] for k, v in aux.items()}
        pos += c


def rows(sl, N):
    return slice(sl.start * N, sl.stop * N)


# --------------------------------------------------------------------------------------------------------------------------
# 1. cld_guidance_step and cld_indicators
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("grad_steps", [1, 3])
def test_guidance_step_equals_per_scene_calls(build, precision, grad_steps):
    """All seven terms, N = 2: z_out, the gradient and the losses of every scene equal a call on that scene alone.  The
    map-collision loss row is summed with atomics (its gradient is not), so it is held to the last bits only."""
    from cld_b200.engine import default_guidance
    N = 2
    dm, _, _ = build(precision)
    aux, batch = ragged_case(SIZES, 900)
    R = sum(SIZES) * N
    torch.manual_seed(901)
    z = torch.randn(R, 52, 4).cuda()
    cond, curr = aux["cond_feat"].repeat_interleave(N, 0).cuda(), aux["curr_states"].repeat_interleave(N, 0).cuda()
    g = default_guidance(grad_steps=grad_steps, **ALL_TERMS)
    eng = dm.engine(R)
    scene = eng.make_scene(batch, len(SIZES), 0, N, scene_sizes=SIZES)
    assert scene.scene_start and scene.scene_start_host
    z_out, grad, loss = eng.guidance_step(z, cond, curr, scene, g)
    assert loss[0].abs().sum() > 0 and loss[LOSS_MAP].abs().sum() > 0 and loss[6].abs().sum() > 0     # not vacuous
    for sl, sb, _ in per_scene(batch, aux, SIZES):
        r = rows(sl, N)
        zo, gr, lo = eng.guidance_step(z[r], cond[r], curr[r], eng.make_scene(sb, 1, sl.stop - sl.start, N), g)
        c = sl.stop - sl.start
        assert torch.equal(z_out[r], zo), c
        assert torch.equal(grad[r], gr), c
        keep = [i for i in range(7) if i != LOSS_MAP]
        assert torch.equal(loss[keep][:, r], lo[keep]), c
        assert torch.allclose(loss[LOSS_MAP, r], lo[LOSS_MAP], rtol=1e-6, atol=0.0), c


def test_indicators_equal_per_scene_calls(build):
    from cld_b200.critic import indicators
    N = 2
    dm, _, _ = build()
    aux, batch = ragged_case(SIZES, 910, waypoints=False)
    R = sum(SIZES) * N
    torch.manual_seed(911)
    traj = torch.randn(R, 52, 6).cuda() * 6
    eng = dm.engine(R)
    off, coll, rew = eng.indicators(traj, eng.make_scene(batch, len(SIZES), 0, N, scene_sizes=SIZES))
    assert off.any() and coll.sum() > 0
    for sl, sb, _ in per_scene(batch, aux, SIZES):
        r = rows(sl, N)
        o, c, w = eng.indicators(traj[r], eng.make_scene(sb, 1, sl.stop - sl.start, N))
        assert torch.equal(off[r], o) and torch.equal(coll[r], c) and torch.equal(rew[r], w)
    # the critic drop-in: one call on the ragged batch
    o2, c2, w2 = indicators(dm, traj, cu(batch), N)
    assert torch.equal(o2, off) and torch.equal(c2, coll) and torch.equal(w2, rew)


# --------------------------------------------------------------------------------------------------------------------------
# 2. the samplers
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("sampler", ["ddpm", "ddim"])
def test_sampler_equals_per_scene_calls(build, precision, sampler):
    """Guided, N = 2.  Supplied x_init / noise: every scene equals a call on it alone.  In-kernel generator: every scene equals
    a call on it alone whose row_offset is the scene's first row (the noise of a row is keyed by its row in the batch)."""
    from cld_b200.engine import default_guidance
    N = 2
    dm, _, algo = build(precision, N)
    sizes = [3, 1, 66, 2, 8]
    aux, batch = ragged_case(sizes, 920)
    R = sum(sizes) * N
    torch.manual_seed(921)
    x_init, noises = torch.randn(R, 52, 4).cuda(), torch.randn(10, R, 52, 4).cuda()
    g = default_guidance(**ALL_TERMS)
    kw = dict(sampler=sampler, guidance=g, want_indicators=True)
    sup = dm(cu(batch), cu(aux), algo, x_init=x_init, noise=noises, **kw)
    dev = dm(cu(batch), cu(aux), algo, use_device_rng=True, seed=4242, **kw)
    assert torch.isfinite(sup["pred_traj"]).all() and torch.isfinite(dev["pred_traj"]).all()
    assert not torch.equal(sup["pred_traj"], dev["pred_traj"])
    for sl, sb, sa in per_scene(batch, aux, sizes):
        r = rows(sl, N)
        one = dm(cu(sb), cu(sa), algo, x_init=x_init[r], noise=noises[:, r], **kw)
        two = dm(cu(sb), cu(sa), algo, use_device_rng=True, seed=4242, row_offset=r.start, **kw)
        for k in ("pred_traj", "traj", "offroad", "coll"):
            assert torch.equal(sup[k][r], one[k]), (k, sl)
            assert torch.equal(dev[k][r], two[k]), (k, sl)


def test_launch_count_does_not_grow_with_the_number_of_scene_sizes(build):
    """A batch with three distinct scene sizes launches as many kernels as a uniform batch of as many agents."""
    from cld_b200.engine import default_guidance
    dm, _, algo = build()
    counts = {}
    for tag, sizes in (("warm-up", [4, 4, 4, 4]), ("uniform", [4, 4, 4, 4]), ("ragged", [4, 2, 6, 4])):
        aux, batch = ragged_case(sizes, 930, waypoints=False)
        torch.manual_seed(931)
        x_init, noises = torch.randn(16, 52, 4).cuda(), torch.randn(10, 16, 52, 4).cuda()
        n0 = dm.launch_count()
        dm(cu(batch), cu(aux), algo, x_init=x_init, noise=noises, guidance=default_guidance(), want_indicators=True)
        torch.cuda.synchronize()
        counts[tag] = dm.launch_count() - n0
    print("launches per call:", counts)
    assert counts["ragged"] == counts["uniform"]


def test_chunks_and_lanes_equal_the_single_call(build):
    """In-kernel generator, DDPM, N = 2: an engine whose max_rows packs the scenes into several greedy chunks, and two lanes,
    give the single-lane, unchunked result bit for bit."""
    from cld_b200.engine import default_guidance
    N = 2
    sizes = [3, 7, 66, 1, 5, 2, 6, 4]
    R = sum(sizes) * N
    aux, batch = ragged_case(sizes, 940)
    g = default_guidance(**ALL_TERMS)
    kw = dict(sampler="ddpm", guidance=g, use_device_rng=True, seed=777, want_indicators=True)
    dm, _, algo = build("fp32", N, max_rows=R)
    full = dm(cu(batch), cu(aux), algo, **kw)
    assert torch.isfinite(full["pred_traj"]).all()
    dm_c, _, _ = build("fp32", N, max_rows=134)             # chunks of 20, 134 (a streamed scene + one more) and 34 rows
    eng = dm_c.engine(1)
    assert eng.max_rows == 134
    cond_rows, curr_rows = aux["cond_feat"].cuda().repeat_interleave(N, 0), aux["curr_states"].cuda().repeat_interleave(N, 0)
    o = eng.sample(None, cond_rows, seed=777, curr_rows=curr_rows, scene=eng.make_scene(batch, len(sizes), 0, N, scene_sizes=sizes),
                   guidance=g, sampler="ddpm", want_indicators=True)
    for k, v in (("pred_traj", o["x0"]), ("traj", o["traj"]), ("offroad", o["offroad"]), ("coll", o["coll"])):
        assert torch.equal(v, full[k]), k
    dm_l, _, algo_l = build("fp32", N, max_rows=R, lanes=2)
    lan = dm_l(cu(batch), cu(aux), algo_l, **kw)
    for k in ("pred_traj", "traj", "offroad", "coll"):
        assert torch.equal(lan[k], full[k]), k


# --------------------------------------------------------------------------------------------------------------------------
# 3. refusals
# --------------------------------------------------------------------------------------------------------------------------
def test_malformed_offsets_and_oversized_scenes_are_refused(build):
    """CLD_ERR_ARG (-1) with a message naming the problem, from all three entry points."""
    from cld_b200.engine import default_guidance
    N = 2
    sizes = [3, 5, 2]
    R = sum(sizes) * N
    aux, batch = ragged_case(sizes, 950, waypoints=False)
    eng = build("fp32", N)[0].engine(R)
    g = default_guidance()
    cond, curr = aux["cond_feat"].repeat_interleave(N, 0).cuda(), aux["curr_states"].repeat_interleave(N, 0).cuda()
    torch.manual_seed(951)
    z = torch.randn(R, 52, 4).cuda()
    traj = torch.randn(R, 52, 6).cuda()

    def calls(scene, rows_=R):
        return {
            "cld_guidance_step": lambda: eng.guidance_step(z[:rows_], cond[:rows_], curr[:rows_], scene, g),
            "cld_indicators": lambda: eng.indicators(traj[:rows_], scene),
            "cld_sample": lambda: eng.sample(z[:rows_], cond[:rows_], seed=3, curr_rows=curr[:rows_], scene=scene, guidance=g,
                                             sampler="ddim"),
        }

    def bad(edit):
        sc = eng.make_scene(batch, len(sizes), 0, N, scene_sizes=sizes)
        edit(sc)
        return sc

    cases = {
        "first offset": (lambda sc: sc._keep["scene_start_host"].__setitem__(0, 1), r"scene_start\[0\]=1"),
        "empty scene": (lambda sc: sc._keep["scene_start_host"].__setitem__(2, 3), r"scene 1 holds 0 agents"),
        "not ascending": (lambda sc: sc._keep["scene_start_host"].__setitem__(2, 2), r"scene 1 holds -1 agents"),
        "rows": (lambda sc: sc._keep["scene_start_host"].__setitem__(3, 9), r"scene_start\[S\]\*N = 9\*2 != R=20"),
        "host offsets missing": (lambda sc: setattr(sc, "scene_start_host", None), r"scene_start_host \(host\), one is NULL"),
        "device offsets missing": (lambda sc: setattr(sc, "scene_start", None), r"scene_start_host \(host\), one is NULL"),
    }
    for name, (edit, msg) in cases.items():
        for entry, call in calls(bad(edit)).items():
            with pytest.raises(RuntimeError, match=r"%s failed \(-1\): .*%s" % (entry, msg)):
                call()
    # a scene of 5 agents x 2 samples = 10 rows fits max_rows = 12; 7 agents x 2 do not
    eng = build("fp32", N, max_rows=12)[0].engine(1)
    assert eng.max_rows == 12
    eng_ok = eng.sample(z, cond, seed=3, curr_rows=curr, scene=eng.make_scene(batch, 3, 0, N, scene_sizes=sizes), guidance=g,
                        sampler="ddim")
    assert torch.isfinite(eng_ok["x0"]).all()
    with pytest.raises(RuntimeError, match=r"cld_sample failed \(-1\): max_rows=12 is smaller than one scene \(scene 1: A\*N=14\)"):
        eng.sample(z, cond, seed=3, curr_rows=curr, scene=eng.make_scene(batch, 2, 0, N, scene_sizes=[3, 7]), guidance=g,
                   sampler="ddim")


# --------------------------------------------------------------------------------------------------------------------------
# 4. the policy and the oracle
# --------------------------------------------------------------------------------------------------------------------------
def test_policy_get_action_on_a_ragged_observation(build):
    """Agent collision on (a scene-level choice of the sample): the ragged observation picks, per scene, the sample and the
    actions a call on that scene alone picks."""
    from cld_b200.engine import default_guidance
    from cld_b200.policy import GuidedDiffusionPolicy
    N = 3
    sizes = [5, 1, 70, 3]
    dm, vae, algo = build("bf16")
    aux, batch = ragged_case(sizes, 960, waypoints=False)
    pol = GuidedDiffusionPolicy(dm, vae, algo, guidance=default_guidance())
    kw = dict(num_action_samples=N, step_index=0, use_device_rng=True, seed=11)
    action, info = pol.get_action(cu(batch), aux_info=cu(aux), **kw)
    assert "agent_collision" in info["guide_losses"]
    for sl, sb, sa in per_scene(batch, aux, sizes):
        a1, i1 = pol.get_action(cu(sb), aux_info=cu(sa), row_offset=sl.start * N, **kw)
        assert torch.equal(info["act_idx"][sl], i1["act_idx"]), sl
        assert info["act_idx"][sl].unique().numel() == 1
        assert torch.equal(action["positions"][sl], a1["positions"]) and torch.equal(action["yaws"][sl], a1["yaws"]), sl


def test_ragged_guided_sampler_vs_oracle(build):
    """10 guided DDPM steps on supplied noise, fp32, scenes of 2, 66 and 5 agents in one call, against the oracle run scene by
    scene (the thresholds of test_gpu_large_scenes.py::test_guided_sampler_80_agents_vs_oracle)."""
    from cld_b200.engine import default_guidance
    dm, vae, algo = build()
    sizes = [2, 66, 5]
    aux, batch = ragged_case(sizes, 970, waypoints=False)
    for k in ("target_pos", "target_speed"):
        batch.pop(k)
    B = sum(sizes)
    torch.manual_seed(971)
    x_init, noises = torch.randn(B, 52, 4), torch.randn(10, B, 52, 4)
    out = dm(cu(batch), cu(aux), algo, noise=noises.cuda(), x_init=x_init.cuda(), guidance=default_guidance(), want_indicators=True)
    dec_sd = dec_sd_of(vae)
    unet_sd = {k: v.detach().cpu() for k, v in dm.model.state_dict().items()}
    want = torch.empty(B, 52, 4)
    for sl, sb, sa in per_scene(batch, aux, sizes):
        gd = dict(dec_sd=dec_sd, cond=sa["cond_feat"], curr=sa["curr_states"], batch=sb, A=sl.stop - sl.start, N=1,
                  cfg=O.DEFAULT_GUIDANCE)
        want[sl] = O.sample(unet_sd, O.make_schedule(10), sa["cond_feat"], x_init[sl], noises[:, sl], 10, 1, "ddpm", guidance=gd)["pred_traj"]
    frac = ((out["pred_traj"].cpu() - want).abs() > 1e-2 * want.abs().max()).float().mean().item()
    print("ragged guided sampler: rel %.3e, fraction off by >1%% of max %.5f" % (rel(out["pred_traj"], want), frac))
    assert frac < 0.02
    wtraj, _ = O.decode_rollout(dec_sd, out["pred_traj"].cpu(), aux["cond_feat"], aux["curr_states"])
    assert rel(out["traj"], wtraj) < 1e-4
    woff, wcoll = O.indicators(out["traj"].cpu()[..., :2], batch)
    assert torch.equal(out["offroad"].cpu(), woff) and torch.equal(out["coll"].cpu(), wcoll)
