"""GPU (-m gpu): the bf16 tcgen05 denoiser (unet_tc.cu) against the fp32 oracle / reference goldens.
Tolerance: north_star allows 1e-2 relative under bf16 for denoiser outputs and final trajectories."""
import pytest
import torch

import cld_oracle as O
from cld_b200.synthetic import make_scenes

pytestmark = pytest.mark.gpu
BF16_TOL = 1e-2

STAGES = ["downs.0.0", "downs.0.1", "downs.0.2", "downs.1.0", "downs.1.1", "downs.1.2", "downs.2.0", "downs.2.1",
          "mid_block1", "mid_block2", "ups.0.0", "ups.0.1", "ups.0.2", "ups.1.0", "ups.1.1", "ups.1.2", "final_conv.0"]


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


@pytest.fixture(scope="module")
def bf16_models(models_cpu):
    cache = {}

    def build(n):
        if n not in cache:
            dm, vae, algo = models_cpu(n, precision="bf16")
            dm = dm.cuda()
            vae.bind(dm)
            cache[n] = (dm, vae, algo)
        return cache[n]
    return build


def cpu_sd(m):
    return {k: v.detach().cpu() for k, v in m.state_dict().items()}


def test_unet_bf16_every_stage_vs_oracle(bf16_models, gold):
    g = gold("unet")
    dm, _, _ = bf16_models(10)
    x, cond, t = torch.tensor(g["x"]), torch.tensor(g["cond"]), torch.tensor(g["t"])
    taps = {}
    with torch.no_grad():
        O.unet_forward(cpu_sd(dm.model), x, cond, t, taps=taps)
    eng = dm.engine(x.shape[0])
    worst = 0.0
    for i, nm in enumerate(STAGES):
        _, dbg = eng.unet_forward(x.cuda(), cond.cuda(), t.cuda(), debug_stage=i)
        want = taps[nm].reshape(x.shape[0], -1)
        r = rel(dbg, want)
        worst = max(worst, r)
        print("stage %2d %-14s rel=%.3e" % (i, nm, r))
        assert dbg.shape == want.shape, nm
        assert r < 2e-2, (nm, r)
    eps = eng.unet_forward(x.cuda(), cond.cuda(), t.cuda())
    r = rel(eps, g["eps"])
    print("eps rel=%.3e (worst stage %.3e)" % (r, worst))
    assert r < BF16_TOL


def test_unet_bf16_many_rows_vs_fp32_path(bf16_models, models_cpu):
    """R = 1061 rows (ragged last group, > 148 groups -> every CTA loops) against the fp32 CUDA path."""
    dm, _, _ = bf16_models(10)
    dm32, _, _ = models_cpu(10)
    dm32 = dm32.cuda()
    torch.manual_seed(3)
    R = 1061
    x, cond = torch.randn(R, 52, 4).cuda(), torch.randn(R, 256).cuda()
    t = torch.randint(0, 10, (R,)).cuda()
    a = dm.engine(R).unet_forward(x, cond, t)
    b = dm32.engine(R).unet_forward(x, cond, t)
    assert torch.isfinite(a).all()
    assert rel(a, b) < BF16_TOL
    per_row = ((a - b).flatten(1).norm(dim=1) / b.flatten(1).norm(dim=1)).max().item()
    print("bf16 vs fp32 path: rel %.3e, worst row %.3e" % (rel(a, b), per_row))
    assert per_row < 3e-2
    a2 = dm.engine(R).unet_forward(x, cond, t)
    assert torch.equal(a, a2)                      # deterministic


def test_cfg0_sampler_bf16_vs_reference_golden(bf16_models, gold):
    g = gold("cfg0_sample")
    dm, vae, algo = bf16_models(10)
    out = dm({"history_positions": torch.zeros(16, 31, 2)},
             {"cond_feat": torch.tensor(g["cond"]).cuda(), "curr_states": torch.tensor(g["curr"]).cuda()}, algo,
             noise=torch.tensor(g["noises"]).cuda(), x_init=torch.tensor(g["x_init"]).cuda(), want_traj=True)
    r = rel(out["pred_traj"], g["pred_traj"])
    rt = rel(out["traj"], g["traj"])
    print("bf16 cfg0: rel(pred_traj)=%.3e rel(traj)=%.3e" % (r, rt))
    assert r < BF16_TOL and rt < BF16_TOL


def test_strided_sampler_bf16_vs_reference_golden(bf16_models, gold):
    g = gold("stride2_sample")
    dm, _, algo = bf16_models(100)
    dm.stride = 2
    try:
        out = dm({"history_positions": torch.zeros(4, 31, 2)}, {"cond_feat": torch.tensor(g["cond"]).cuda()}, algo,
                 noise=torch.tensor(g["noises"]).cuda(), x_init=torch.tensor(g["x_init"]).cuda())
    finally:
        dm.stride = 1
    r = rel(out["pred_traj"], g["pred_traj"])
    print("bf16 50-step strided DDPM: rel(pred_traj)=%.3e" % r)
    assert r < BF16_TOL


# ---------------------------------------------------------------------------------------------------
# bf16-precision mode also runs the LSTM decoder (forward + BPTT) on the tensor pipe (kernels_lstm_tc.cu): fp16-rounded
# weights, hi/lo split state operand.  Tolerances: decoder outputs 1e-3 (north_star allows 1e-2 under bf16).
# ---------------------------------------------------------------------------------------------------
def dec_sd_of(vae):
    return {k: v.detach().cpu() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}


def test_decode_rollout_tensor_core_vs_oracle_ragged_rows(bf16_models):
    dm, vae, _ = bf16_models(10)
    torch.manual_seed(11)
    for R in (37, 64, 1):                     # ragged last CTA, exact multiple, single row
        z, cond = torch.randn(R, 52, 4), torch.randn(R, 256)
        curr = torch.cat([torch.zeros(R, 2), torch.rand(R, 1) * 15, torch.zeros(R, 1)], dim=1)
        act, traj = dm.engine(64).decode_rollout(z.cuda(), cond.cuda(), curr.cuda())
        wtraj, wact = O.decode_rollout(dec_sd_of(vae), z, cond, curr)
        ra, rt = rel(act, wact), rel(traj, wtraj)
        print("tensor-core decode R=%d: rel(act)=%.3e rel(traj)=%.3e" % (R, ra, rt))
        assert torch.isfinite(traj).all()
        assert ra < 1e-3 and rt < 1e-3


def test_guidance_step_tensor_core_vs_reference_golden(bf16_models, gold):
    """Same golden as the fp32 test (the reference's own perturb() output); the tensor-core BPTT is held to a
    looser gradient tolerance: 5e-3 relative, >= 99.5 % sign agreement on the non-zero entries."""
    g = gold("guidance")
    dm, vae, _ = bf16_models(10)
    S, A, N = int(g["S"]), int(g["A"]), int(g["N"])
    aux, batch = make_scenes(S, A, seed=int(g["seed"]), dense=True)
    from cld_b200.engine import default_guidance
    eng = dm.engine(S * A * N)
    scene = eng.make_scene(batch, S, A, N)
    z = torch.tensor(g["z"]).cuda()
    cond = aux["cond_feat"].repeat_interleave(N, 0).cuda()
    curr = aux["curr_states"].repeat_interleave(N, 0).cuda()
    z_out, grad, loss = eng.guidance_step(z, cond, curr, scene, default_guidance())
    assert rel(loss[0], g["loss_ac"].reshape(-1)) < 1e-3
    assert rel(loss[1], g["loss_mc"].reshape(-1)) < 1e-3
    g_or, _ = O.guidance_grad(dec_sd_of(vae), torch.tensor(g["z"]), aux["cond_feat"], aux["curr_states"], batch, A, N)
    nz = g_or != 0
    sign_agree = (torch.sign(grad.cpu())[nz] == torch.sign(g_or)[nz]).float().mean().item()
    zero_rows = (g_or.flatten(1) == 0).all(dim=1)
    print("tensor-core guidance: rel(grad)=%.3e sign agreement %.6f" % (rel(grad, g_or), sign_agree))
    assert rel(grad, g_or) < 5e-3
    assert sign_agree > 0.995
    assert (grad.cpu()[zero_rows] == 0).all()              # rows without any active loss get an exactly zero gradient
    frac_bad = ((z_out.cpu() - torch.tensor(g["z_out"])).abs() > 1e-3).float().mean().item()
    print("tensor-core guidance: fraction of z_out entries off by > 1e-3: %.5f" % frac_bad)
    assert frac_bad < 5e-3


def test_guided_sampler_bf16_finite_and_indicators_consistent(bf16_models, models_cpu, monkeypatch):
    """cfg1-shaped guided run in bf16 mode: finite, deterministic, indicators bit-exact on the produced trajectories."""
    dm, vae, algo = bf16_models(100)
    S, A = 4, 16
    aux, batch = make_scenes(S, A, seed=77, dense=True)
    from cld_b200.engine import default_guidance
    torch.manual_seed(78)
    R = S * A
    x_init, noises = torch.randn(R, 52, 4), torch.randn(50, R, 52, 4)
    dm.stride = 2
    try:
        outs = [dm({k: (v.cuda() if torch.is_tensor(v) else v) for k, v in batch.items()}, {k: v.cuda() for k, v in aux.items()},
                   algo, noise=noises.cuda(), x_init=x_init.cuda(), guidance=default_guidance(), want_indicators=True)
                for _ in range(2)]
    finally:
        dm.stride = 1
    a, b = outs
    assert torch.isfinite(a["pred_traj"]).all() and torch.isfinite(a["traj"]).all()
    assert torch.equal(a["pred_traj"], b["pred_traj"]) and torch.equal(a["traj"], b["traj"])
    # the sampler runs the two loss kernels concurrently (auxiliary stream, separate gradient buffers: a + b is rounded once
    # more than the serial fused multiply-add); the serial order must give the same sample up to that rounding
    # (the switch is read when an engine is created: a second model with the same seed-0 weights)
    monkeypatch.setenv("CLD_GUIDANCE_NOFORK", "1")
    dm_s, vae_s, _ = models_cpu(100, precision="bf16")
    dm_s = dm_s.cuda()
    vae_s.bind(dm_s)
    dm_s.stride = 2
    c = dm_s({k: (v.cuda() if torch.is_tensor(v) else v) for k, v in batch.items()}, {k: v.cuda() for k, v in aux.items()},
             algo, noise=noises.cuda(), x_init=x_init.cuda(), guidance=default_guidance(), want_indicators=True)
    monkeypatch.delenv("CLD_GUIDANCE_NOFORK")
    diff = (a["pred_traj"] - c["pred_traj"]).abs()
    frac = (diff > 1e-2 * c["pred_traj"].abs().max()).float().mean().item()
    print("concurrent vs serial loss kernels: rel %.3e, fraction off by > 1%% of max %.5f" % (rel(a["pred_traj"], c["pred_traj"]), frac))
    assert frac < 0.02
    woff, wcoll = O.indicators(a["traj"].cpu()[..., :2], batch)
    assert torch.equal(a["offroad"].cpu(), woff) and torch.equal(a["coll"].cpu(), wcoll)
    wtraj, _ = O.decode_rollout(dec_sd_of(vae), a["pred_traj"].cpu(), aux["cond_feat"], aux["curr_states"])
    assert rel(a["traj"], wtraj) < 1e-3


def test_guidance_step_cfg2_shape_tensor_core_vs_fp32_kernels(bf16_models, models_cpu):
    """cfg2-shaped scenes (32 agents, 8 samples per scene): the bf16-mode guidance step (tensor-core LSTM forward + BPTT)
    against the fp32 SIMT kernels on the same latents."""
    from cld_b200 import default_algo_config
    from cld_b200.dm_model import DmModel
    from cld_b200.engine import default_guidance
    from cld_b200.vae import VaeModel
    S, A, N = 2, 32, 8
    R = S * A * N
    aux, batch = make_scenes(S, A, seed=31, dense=True)
    torch.manual_seed(32)
    z = torch.randn(R, 52, 4).cuda()
    cond = aux["cond_feat"].repeat_interleave(N, 0).cuda()
    curr = aux["curr_states"].repeat_interleave(N, 0).cuda()
    res = {}
    for prec in ("fp32", "bf16"):
        algo = default_algo_config(num_samp=N)
        torch.manual_seed(0)
        dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=10, precision=prec, max_rows=R).cuda()
        VaeModel(algo).bind(dm)
        eng = dm.engine(R)
        res[prec] = eng.guidance_step(z, cond, curr, eng.make_scene(batch, S, A, N), default_guidance())
    (z32, g32, l32), (z16, g16, l16) = res["fp32"], res["bf16"]
    nz = g32 != 0
    sign_agree = (torch.sign(g16)[nz] == torch.sign(g32)[nz]).float().mean().item()
    print("cfg2 shape: rel(loss) %.2e %.2e rel(grad) %.3e sign agreement %.6f" % (rel(l16[0], l32[0]), rel(l16[1], l32[1]), rel(g16, g32), sign_agree))
    assert nz.any()
    assert rel(l16[0], l32[0]) < 1e-3 and rel(l16[1], l32[1]) < 1e-3
    assert rel(g16, g32) < 5e-3 and sign_agree > 0.995
    assert ((g16 == 0) == (g32 == 0)).float().mean().item() > 0.999


def test_ppo_mode_sampler_bf16_outputs(bf16_models, models_cpu):
    """cfg4 (PPO mode): n_timesteps = 16, stride 1, guided, N = 4 samples: pred_traj / x1 / log_prob_final / reward."""
    from cld_b200 import default_algo_config
    from cld_b200.dm_model import DmModel
    from cld_b200.engine import default_guidance
    from cld_b200.vae import VaeModel
    S, A, N = 2, 16, 4
    R = S * A * N
    algo = default_algo_config(num_samp=N)
    torch.manual_seed(0)
    dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=16, precision="bf16", max_rows=R).cuda()
    vae = VaeModel(algo).bind(dm)
    aux, batch = make_scenes(S, A, seed=41, dense=True)
    torch.manual_seed(42)
    x_init, noises = torch.randn(R, 52, 4).cuda(), torch.randn(16, R, 52, 4).cuda()
    out = dm({k: (v.cuda() if torch.is_tensor(v) else v) for k, v in batch.items()}, {k: v.cuda() for k, v in aux.items()}, algo,
             noise=noises, x_init=x_init, guidance=default_guidance(), want_indicators=True, agents_per_scene=A)
    assert out["pred_traj"].shape == (R, 52, 4) and out["x1"] is not None and out["x1"].shape == (R, 52, 4)
    assert torch.isfinite(out["pred_traj"]).all() and torch.isfinite(out["x1"]).all()
    # log_prob_final = Normal(mean_0, sigma_0).log_prob(x_0) with x_0 == mean_0 (dm_model.py:128-132): a constant
    sigma0 = (0.5 * dm.posterior_log_variance_clipped[0]).exp().item()
    import math
    want_lp = -math.log(sigma0) - 0.5 * math.log(2 * math.pi)
    assert out["log_prob_final"].shape == (R,)
    assert torch.allclose(out["log_prob_final"].cpu(), torch.full((R,), want_lp), rtol=1e-5, atol=1e-5)
    # indicators on the produced trajectories are bit-exact against the oracle; the decoded trajectory matches the oracle decoder
    rep = {k: (v.repeat_interleave(N, 0) if torch.is_tensor(v) and v.shape[0] == S * A else v) for k, v in batch.items()}
    woff, wcoll = O.indicators(out["traj"].cpu()[..., :2], rep)
    assert torch.equal(out["offroad"].cpu(), woff) and torch.equal(out["coll"].cpu(), wcoll)
    wtraj, _ = O.decode_rollout(dec_sd_of(vae), out["pred_traj"].cpu(), aux["cond_feat"].repeat_interleave(N, 0),
                                aux["curr_states"].repeat_interleave(N, 0))
    assert rel(out["traj"], wtraj) < 1e-3


def test_lanes_give_the_single_engine_result(models_cpu):
    """DmModel(lanes=2): whole-scene half batches on two engines / CUDA streams.  Scenes never interact and every kernel is
    row-wise deterministic, so the result must equal the single-engine one bit for bit (supplied noise, guided DDPM)."""
    from cld_b200.engine import default_guidance
    S, A = 6, 8
    aux, batch = make_scenes(S, A, seed=31, dense=True)
    torch.manual_seed(32)
    R = S * A
    x_init, noises = torch.randn(R, 52, 4).cuda(), torch.randn(10, R, 52, 4).cuda()
    bd = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in batch.items()}
    ad = {k: v.cuda() for k, v in aux.items()}
    outs = []
    for lanes in (1, 2, 3):
        dm, vae, algo = models_cpu(10, precision="bf16", lanes=lanes)
        dm = dm.cuda()
        vae.bind(dm)
        outs.append(dm(bd, ad, algo, noise=noises, x_init=x_init, guidance=default_guidance(), want_indicators=True, agents_per_scene=A))
        torch.cuda.synchronize()
    for o in outs[1:]:
        for k in ("pred_traj", "traj", "offroad", "coll"):
            assert torch.equal(outs[0][k], o[k]), k


# ----------------------------------------------------------------------------------------------------
# horizon 104 (cfg3): split-time mode of the tensor-core denoiser (4 rows per CTA as two 52-step lanes with halo exchange)
# ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bf16_t104():
    from cld_b200 import default_algo_config
    from cld_b200.dm_model import DmModel
    from cld_b200.vae import VaeModel
    algo = default_algo_config()
    algo.horizon = 104
    torch.manual_seed(0)
    dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=10, precision="bf16", max_rows=1024).cuda()
    vae = VaeModel(algo).bind(dm)
    torch.manual_seed(0)
    dm32 = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=10, max_rows=1024).cuda()
    VaeModel(algo).bind(dm32)
    return dm, vae, dm32, algo


def test_unet_bf16_t104_every_stage_vs_oracle_and_reference_golden(bf16_t104, gold):
    g = gold("unet")
    dm, _, _, _ = bf16_t104
    x, cond, t = torch.tensor(g["x104"]), torch.tensor(g["cond"][:3]), torch.tensor(g["t"][:3])
    taps = {}
    with torch.no_grad():
        O.unet_forward(cpu_sd(dm.model), x, cond, t, taps=taps)
    eng = dm.engine(x.shape[0])
    for i, nm in enumerate(STAGES):
        _, dbg = eng.unet_forward(x.cuda(), cond.cuda(), t.cuda(), debug_stage=i)
        want = taps[nm].reshape(x.shape[0], -1)
        r = rel(dbg, want)
        print("T=104 stage %2d %-14s rel=%.3e" % (i, nm, r))
        assert dbg.shape == want.shape, nm
        assert r < 2e-2, (nm, r)
    eps = eng.unet_forward(x.cuda(), cond.cuda(), t.cuda())
    r = rel(eps, g["eps104"])                                  # the REAL reference's output (oracle/make_golden.py)
    print("T=104 eps rel=%.3e vs the reference golden" % r)
    assert r < BF16_TOL


def test_unet_bf16_t104_many_rows_vs_fp32_path(bf16_t104):
    """R = 611 rows: 153 groups of 4 rows (ragged last group, > 74 CTA pairs -> every pair loops, odd number of groups) vs the fp32 path."""
    dm, _, dm32, _ = bf16_t104
    torch.manual_seed(3)
    R = 611
    x, cond = torch.randn(R, 104, 4).cuda(), torch.randn(R, 256).cuda()
    t = torch.randint(0, 10, (R,)).cuda()
    a = dm.engine(R).unet_forward(x, cond, t)
    b = dm32.engine(R).unet_forward(x, cond, t)
    assert torch.isfinite(a).all()
    per_row = ((a - b).flatten(1).norm(dim=1) / b.flatten(1).norm(dim=1)).max().item()
    print("T=104 bf16 vs fp32 path: rel %.3e, worst row %.3e" % (rel(a, b), per_row))
    assert rel(a, b) < BF16_TOL and per_row < 3e-2
    assert torch.equal(a, dm.engine(R).unet_forward(x, cond, t))      # deterministic
    # a row does not depend on its lane / group / CTA of the pair
    a2 = dm.engine(R).unet_forward(x[5:90].contiguous(), cond[5:90].contiguous(), t[5:90].contiguous())
    assert torch.equal(a[5:90], a2)


def test_sampler_bf16_t104_guided_vs_fp32_path(bf16_t104):
    """cfg3-shaped: horizon 104, one scene of 64 agents, 10 DDPM steps with guidance: the bf16 product path (split-time denoiser +
    tensor-core LSTM decoder / BPTT at T = 104) against the fp32 kernels on the same noise; decode + indicators self-consistent."""
    from cld_b200.engine import default_guidance
    dm, vae, dm32, algo = bf16_t104
    S, A = 1, 64
    aux, batch = make_scenes(S, A, horizon=104, seed=61, dense=True)
    torch.manual_seed(8)
    x_init, noises = torch.randn(S * A, 104, 4).cuda(), torch.randn(10, S * A, 104, 4).cuda()
    cu = lambda d: {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in d.items()}       # noqa: E731
    kw = dict(x_init=x_init, noise=noises, want_indicators=True, agents_per_scene=A)
    a = dm(cu(batch), cu(aux), algo, **kw)
    b = dm32(cu(batch), cu(aux), algo, **kw)
    r = rel(a["pred_traj"], b["pred_traj"])
    print("T=104 unguided bf16 vs fp32: rel(pred_traj) %.3e rel(traj) %.3e" % (r, rel(a["traj"], b["traj"])))
    assert r < BF16_TOL
    dec_sd = {k: v.detach().cpu() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}
    wtraj, _ = O.decode_rollout(dec_sd, a["pred_traj"].cpu(), aux["cond_feat"], aux["curr_states"])
    assert rel(a["traj"], wtraj) < 1e-3
    woff, wcoll = O.indicators(a["traj"].cpu()[..., :2], batch)
    assert torch.equal(a["offroad"].cpu(), woff) and torch.equal(a["coll"].cpu(), wcoll)
    # one guided step: gradient of the bf16-mode kernels vs the fp32 kernels
    z = torch.randn(S * A, 104, 4).cuda()
    e16, e32 = dm.engine(S * A), dm32.engine(S * A)
    _, g16, _ = e16.guidance_step(z, aux["cond_feat"].cuda(), aux["curr_states"].cuda(), e16.make_scene(batch, S, A, 1), default_guidance())
    _, g32, _ = e32.guidance_step(z, aux["cond_feat"].cuda(), aux["curr_states"].cuda(), e32.make_scene(batch, S, A, 1), default_guidance())
    nz = g32 != 0
    agree = (torch.sign(g16)[nz] == torch.sign(g32)[nz]).float().mean().item()
    print("T=104 guidance: rel(grad) %.3e sign agreement %.6f" % (rel(g16, g32), agree))
    assert rel(g16, g32) < 1e-2 and agree > 0.995
    g = dm(cu(batch), cu(aux), algo, guidance=default_guidance(), **kw)
    assert torch.isfinite(g["pred_traj"]).all()


def test_denoiser_pair_kernel_is_race_free_over_many_launches(bf16_models):
    """The CTA-pair megakernel hands activations between the async proxy of two SMs through barriers without a cluster-scope
    release (unet_tc.cu); a missed ordering would show as a rare bit difference.  60 launches at 4 096 rows and 30 at an odd group
    count must reproduce the first result bit for bit, and the single-CTA instance (no pair protocol) must agree with it."""
    import os
    dm, _, _ = bf16_models(10)
    torch.manual_seed(21)
    for R, n in ((4096, 60), (1061, 30)):
        x, cond = torch.randn(R, 52, 4).cuda(), torch.randn(R, 256).cuda()
        t = torch.randint(0, 10, (R,)).cuda()
        eng = dm.engine(4096)
        ref = eng.unet_forward(x, cond, t).clone()
        for _ in range(n):
            assert torch.equal(eng.unet_forward(x, cond, t), ref)
    os.environ["CLD_TC_PAIR"] = "0"
    try:
        from cld_b200 import default_algo_config
        from cld_b200.dm_model import DmModel
        torch.manual_seed(0)
        dm1 = DmModel(default_algo_config(), {"image": (34, 224, 224)}, n_timesteps=10, precision="bf16", max_rows=4096).cuda()
        single = dm1.engine(4096).unet_forward(x, cond, t)
    finally:
        del os.environ["CLD_TC_PAIR"]
    # same arithmetic per row (same MMA shapes per CTA, same epilogue): the two instances agree exactly
    assert torch.equal(single, ref)


def test_bit_packed_drivable_map_equals_byte_map(bf16_models):
    """CldScene.map_packed: indicators and the guided sampler give identical results from the bit-packed map."""
    from cld_b200.engine import default_guidance
    from cld_b200.synthetic import pack_drivable_map
    dm, vae, algo = bf16_models(10)
    S, A = 4, 8
    aux, batch = make_scenes(S, A, seed=91, dense=True)
    packed = dict(batch)
    packed["drivable_map_bits"] = pack_drivable_map(batch["drivable_map"])
    del packed["drivable_map"]
    torch.manual_seed(92)
    x_init, noises = torch.randn(S * A, 52, 4).cuda(), torch.randn(10, S * A, 52, 4).cuda()
    cu = lambda d: {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in d.items()}       # noqa: E731
    kw = dict(x_init=x_init, noise=noises, guidance=default_guidance(), want_indicators=True, agents_per_scene=A)
    a = dm(cu(batch), cu(aux), algo, **kw)
    b = dm(cu(packed), cu(aux), algo, **kw)
    for k in ("pred_traj", "traj", "offroad", "coll"):
        assert torch.equal(a[k], b[k]), k
    assert a["offroad"].any() and not a["offroad"].all()


def test_host_stager_pipeline_equals_direct_calls(bf16_models):
    """cld_b200.staging.HostStager (double-buffered H2D on a copy stream, results read back to pinned memory): three pipelined calls
    with different inputs give what three direct calls give."""
    from cld_b200.staging import HostStager
    dm, vae, algo = bf16_models(10)
    S, A = 3, 8
    cases = [make_scenes(S, A, seed=100 + i, dense=True) for i in range(3)]
    keys = ["extent", "world_from_agent", "raster_from_agent", "curr_speed", "drivable_map", "scene_index",
            "all_other_agents_future_positions", "all_other_agents_future_availability", "history_positions"]
    torch.manual_seed(7)
    x_init = torch.randn(S * A, 52, 4).cuda()
    kw = dict(x_init=x_init, sampler="ddim", want_indicators=True, agents_per_scene=A)
    cu = lambda d: {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in d.items()}       # noqa: E731
    want = [dm(cu({k: b[k] for k in keys}), cu(ax), algo, **kw)["traj"].cpu() for ax, b in cases]
    st = HostStager(torch.device("cuda"))
    host = [({k: b[k].pin_memory() for k in keys}, {k: v.pin_memory() for k, v in ax.items()}) for ax, b in cases]
    st.put(*host[0])
    got = []
    for i in range(3):
        b_d, ax_d, slot = st.get()
        if i + 1 < 3:
            st.put(*host[i + 1])
        o = dm(b_d, ax_d, algo, **kw)
        st.release(slot)
        hb = st.read_back(o, ("traj",))
        torch.cuda.current_stream().synchronize()
        got.append(hb["traj"].clone())
    st.finish()
    for w, g_ in zip(want, got):
        assert torch.equal(w, g_)
