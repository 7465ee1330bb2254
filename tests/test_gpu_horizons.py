"""GPU (-m gpu): every horizon the library accepts, against the oracle (which is fully convolutional in time).

The kernels work out their tiling from the horizon at run time: the 16-slot tiles of the bf16 denoiser and the overlap of a
level's last tile, the half-horizon lanes of its split-time mode, the shared-memory layout and stash indexing of the
tensor-core LSTM, the TMA boxes of the tf32 training step.  Each family is checked at every horizon that reaches a different
case, with the thresholds the suite uses for the same operation at T = 52, and with the worst time slot and the worst row
beside the global relative error: an error confined to one slot of 52 is diluted below the global bound
(tests/test_horizon_metric.py)."""
import os

import pytest
import torch

import cld_oracle as O
from cld_b200 import default_algo_config
from cld_b200.dm_model import DmModel
from cld_b200.synthetic import make_scenes
from cld_b200.vae import VaeModel
from horizon_metric import rel, worst_row_rel, worst_slot_rel
from perturb_oracle import guidance_perturb

pytestmark = pytest.mark.gpu

# bf16: 8 rows per CTA for 16..56; two half-horizon lanes (4 rows per CTA) for 64..104 in multiples of 8
BF16_T = list(range(16, 57, 4)) + list(range(64, 105, 8))
# fp32: both bounds (levels of 8/4/2 and 12/6/3 slots, CLD_MAX_T), odd-length levels, and horizons the bf16 path refuses
FP32_T = [8, 12, 20, 60, 64, 128]
STAGES = ["downs.0.0", "downs.0.1", "downs.0.2", "downs.1.0", "downs.1.1", "downs.1.2", "downs.2.0", "downs.2.1",
          "mid_block1", "mid_block2", "ups.0.0", "ups.0.1", "ups.0.2", "ups.1.0", "ups.1.1", "ups.1.2", "final_conv.0"]
TERMS = ("agent_collision", "map_collision", "target_pos", "target_speed", "acc_limit", "speed_limit")
GRAD_TOL = 1e-4            # fp32 training step: per-tensor relative L2 of every parameter gradient


def cu(d):
    return {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in d.items()}


def cpu_sd(m):
    return {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}


def dec_sd_of(vae):
    return {k: v.detach().cpu() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}


def new_model(T, precision):
    algo = default_algo_config(horizon=T)
    torch.manual_seed(0)
    dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=10, precision=precision, max_rows=64).cuda()
    vae = VaeModel(algo).bind(dm)
    return dm, vae, algo


@pytest.fixture(scope="module")
def build():
    """(T, precision) -> (DmModel, VaeModel, algo) with the seed-0 weights, on the GPU (one per key for the module)."""
    cache = {}

    def get(T, precision="fp32"):
        if (T, precision) not in cache:
            cache[(T, precision)] = new_model(T, precision)
        return cache[(T, precision)]
    return get


def all_terms_case(S, A, T, seed):
    """Scenes of horizon T with every guidance term on; target_speed [B, T] varies over time."""
    aux, batch = make_scenes(S, A, horizon=T, seed=seed, dense=True)
    torch.manual_seed(seed + 1)
    v0 = aux["curr_states"][:, 2:3] + torch.randn(S * A, 1)
    batch["target_speed"] = (v0 + 0.1 * torch.randn(S * A, T).cumsum(1)).clamp(min=0)
    w = dict(agent_collision=50.0, map_collision=1.0, target_pos=1.0, target_speed=0.5, acc_limit=1.0, acc_limit_value=1.0,
             speed_limit=1.0, speed_limit_value=3.0)
    return aux, batch, w


# --------------------------------------------------------------------------------------------------------------------------
# 1. what cld_create accepts is what runs
# --------------------------------------------------------------------------------------------------------------------------
def test_bf16_acceptance_matches_what_runs():
    """Every multiple of 4 in [8, 128]: an fp32 engine is created; a bf16 engine is either refused at creation or loads the
    denoiser and runs it.  A horizon that is accepted but fails later is reported with its error."""
    from cld_b200.engine import Engine
    dm, _, _ = new_model(52, "fp32")
    sd = dm.model.state_dict()
    accepted, late = [], {}
    for T in range(8, 129, 4):
        Engine(horizon=T, precision="fp32", max_rows=8).close()
        try:
            eng = Engine(horizon=T, precision="bf16", max_rows=8)
        except RuntimeError as e:
            assert "bf16 tensor-core path" in str(e), (T, str(e))
            continue
        accepted.append(T)
        try:
            eng.load_unet(sd)
            torch.manual_seed(T)
            eps = eng.unet_forward(torch.randn(5, T, 4).cuda(), torch.randn(5, 256).cuda(), torch.randint(0, 10, (5,)).cuda())
            torch.cuda.synchronize()
            if not torch.isfinite(eps).all():
                late[T] = "non-finite output"
        except RuntimeError as e:
            late[T] = str(e)
        finally:
            eng.close()
    print("bf16 accepts %s; accepted but failing: %s" % (accepted, late))
    assert not late, late
    assert accepted == BF16_T


# --------------------------------------------------------------------------------------------------------------------------
# 2. bf16 denoiser megakernel
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", BF16_T)
def test_unet_bf16_every_stage_vs_oracle(build, T):
    """R = 8k+3 rows (8-row mode) or 4k+1 (split-time mode): a ragged last group and an odd number of groups; t per row."""
    dm, _, _ = build(T, "bf16")
    R = 19 if T <= 56 else 17
    torch.manual_seed(1000 + T)
    x, cond, t = torch.randn(R, T, 4), torch.randn(R, 256), torch.randint(0, 10, (R,))
    taps = {}
    with torch.no_grad():
        want_eps = O.unet_forward(cpu_sd(dm.model), x, cond, t, taps=taps)
    eng = dm.engine(R)
    worst = (0.0, "")
    for i, nm in enumerate(STAGES):
        _, dbg = eng.unet_forward(x.cuda(), cond.cuda(), t.cuda(), debug_stage=i)
        want = taps[nm]
        assert dbg.shape == want.reshape(R, -1).shape, nm
        r = rel(dbg, want.reshape(R, -1))
        print("T=%3d bf16 stage %2d %-13s rel %.3e worst slot %.3e worst row %.3e" % (
            T, i, nm, r, worst_slot_rel(dbg, want, want.shape[1]), worst_row_rel(dbg, want)))
        worst = max(worst, (r, nm))
        assert r < 2e-2, (nm, r)
    eps = eng.unet_forward(x.cuda(), cond.cuda(), t.cuda())
    r, rs, rr = rel(eps, want_eps), worst_slot_rel(eps, want_eps, T), worst_row_rel(eps, want_eps)
    print("T=%3d bf16 eps rel %.3e worst slot %.3e worst row %.3e (worst stage %.3e %s)" % (T, r, rs, rr, *worst))
    assert r < 1e-2 and rr < 3e-2 and rs < 3e-2, (r, rs, rr)
    # deterministic, and a row does not depend on its group, lane or CTA of the pair (shifting by 3 rows moves every row)
    assert torch.equal(eng.unet_forward(x.cuda(), cond.cuda(), t.cuda()), eps)
    sub = eng.unet_forward(x[3:R - 2].cuda(), cond[3:R - 2].cuda(), t[3:R - 2].cuda())
    assert torch.equal(sub, eps[3:R - 2])
    if T in (20, 64):
        # the single-CTA instance (no pair protocol) computes the same bits; the switch is read when the engine is created
        os.environ["CLD_TC_PAIR"] = "0"
        try:
            dm1, _, _ = new_model(T, "bf16")
            single = dm1.engine(R).unet_forward(x.cuda(), cond.cuda(), t.cuda())
        finally:
            del os.environ["CLD_TC_PAIR"]
        assert torch.equal(single, eps)


# --------------------------------------------------------------------------------------------------------------------------
# 3. tensor-core LSTM decoder
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", BF16_T)
def test_decode_rollout_tensor_core_vs_oracle(build, T):
    """R = 37: the second 32-row CTA is partial."""
    dm, vae, _ = build(T, "bf16")
    R = 37
    torch.manual_seed(2000 + T)
    z, cond = torch.randn(R, T, 4), torch.randn(R, 256)
    curr = torch.cat([torch.zeros(R, 2), torch.rand(R, 1) * 15, torch.zeros(R, 1)], dim=1)
    act, traj = dm.engine(R).decode_rollout(z.cuda(), cond.cuda(), curr.cuda())
    wtraj, wact = O.decode_rollout(dec_sd_of(vae), z, cond, curr)
    ra, rt = rel(act, wact), rel(traj, wtraj)
    sa, st = worst_slot_rel(act, wact, T), worst_slot_rel(traj, wtraj, T)
    print("T=%3d tensor-core decode: rel(act) %.3e worst slot %.3e, rel(traj) %.3e worst slot %.3e worst row %.3e" % (
        T, ra, sa, rt, st, worst_row_rel(traj, wtraj)))
    assert torch.isfinite(traj).all()
    assert ra < 1e-3 and rt < 1e-3, (ra, rt)
    assert sa < 3e-3 and st < 3e-3, (sa, st)


# --------------------------------------------------------------------------------------------------------------------------
# 4. guidance step (decode with stash, six losses, BPTT, optimizer step)
# --------------------------------------------------------------------------------------------------------------------------
def _guidance_vs_oracle(dm, vae, T, precision):
    """S = 5 scenes x 4 agents x 2 samples = 40 rows (crosses a 32-row CTA): every term on; -> (losses, gradient, sign and
    zero-set agreement) against the oracle's autograd."""
    from cld_b200.engine import default_guidance
    S, A, N = 5, 4, 2
    aux, batch, w = all_terms_case(S, A, T, 3000 + T)
    torch.manual_seed(3100 + T)
    z = torch.randn(S * A * N, T, 4)
    eng = dm.engine(S * A * N)
    scene = eng.make_scene(batch, S, A, N)
    cond, curr = aux["cond_feat"].repeat_interleave(N, 0), aux["curr_states"].repeat_interleave(N, 0)
    _, grad, loss = eng.guidance_step(z.cuda(), cond.cuda(), curr.cuda(), scene, default_guidance(**w))
    g_or, per = O.guidance_grad(dec_sd_of(vae), z, aux["cond_feat"], aux["curr_states"], batch, A, N, dict(O.DEFAULT_GUIDANCE, **w))
    lrel = {t: rel(loss[i], torch.cat([p[t] for p in per]).reshape(-1)) for i, t in enumerate(TERMS)}
    grad = grad.cpu()
    nz = g_or != 0
    sign_agree = (torch.sign(grad)[nz] == torch.sign(g_or)[nz]).float().mean().item()
    zero_agree = ((grad == 0) == (g_or == 0)).float().mean().item()
    rg = rel(grad, g_or)
    print("T=%3d %s guidance: rel(grad) %.3e worst slot %.3e sign %.6f zero-set %.6f losses %s" % (
        T, precision, rg, worst_slot_rel(grad, g_or, T), sign_agree, zero_agree, " ".join("%s %.1e" % kv for kv in lrel.items())))
    assert nz.any()
    return lrel, rg, sign_agree, zero_agree


@pytest.mark.parametrize("T", BF16_T)
def test_guidance_step_bf16_vs_oracle(build, T):
    dm, vae, _ = build(T, "bf16")
    lrel, rg, sign_agree, zero_agree = _guidance_vs_oracle(dm, vae, T, "bf16")
    assert all(v < 1e-3 for v in lrel.values()), lrel
    assert rg < 5e-3 and sign_agree > 0.995 and zero_agree > 0.999, (rg, sign_agree, zero_agree)


@pytest.mark.parametrize("T", [20, 64])
def test_guidance_two_adam_steps_bf16_vs_oracle_perturb(build, T):
    """grad_steps = 2 with Adam runs the moment-carrying instance of the tensor-core BPTT: the update z' - z against the oracle's
    perturb loop, on its sign and zero set."""
    from cld_b200.engine import default_guidance
    dm, vae, _ = build(T, "bf16")
    S, A, N = 5, 4, 2
    aux, batch, w = all_terms_case(S, A, T, 3200 + T)
    torch.manual_seed(3300 + T)
    z = torch.randn(S * A * N, T, 4)
    eng = dm.engine(S * A * N)
    cond, curr = aux["cond_feat"].repeat_interleave(N, 0), aux["curr_states"].repeat_interleave(N, 0)
    z_out, _, _ = eng.guidance_step(z.cuda(), cond.cuda(), curr.cuda(), eng.make_scene(batch, S, A, N),
                                    default_guidance(grad_steps=2, **w))
    zw, _, _ = guidance_perturb(dec_sd_of(vae), z, aux["cond_feat"], aux["curr_states"], batch, A, N,
                                dict(O.DEFAULT_GUIDANCE, grad_steps=2, **w))
    d16, dw = z_out.cpu() - z, zw - z
    nz = dw != 0
    sign_agree = (torch.sign(d16)[nz] == torch.sign(dw)[nz]).float().mean().item()
    zero_agree = ((d16 == 0) == (dw == 0)).float().mean().item()
    print("T=%3d bf16 two Adam steps: rel(update) %.3e sign %.6f zero-set %.6f" % (T, rel(d16, dw), sign_agree, zero_agree))
    assert nz.any()
    assert sign_agree > 0.995 and zero_agree > 0.999, (sign_agree, zero_agree)


# --------------------------------------------------------------------------------------------------------------------------
# 5. fp32 path
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", FP32_T)
def test_unet_fp32_every_stage_vs_oracle(build, T):
    dm, _, _ = build(T)
    R = 11
    torch.manual_seed(4000 + T)
    x, cond, t = torch.randn(R, T, 4), torch.randn(R, 256), torch.randint(0, 10, (R,))
    taps = {}
    with torch.no_grad():
        want_eps = O.unet_forward(cpu_sd(dm.model), x, cond, t, taps=taps)
    eng = dm.engine(R)
    worst = 0.0
    for i, nm in enumerate(STAGES):
        _, dbg = eng.unet_forward(x.cuda(), cond.cuda(), t.cuda(), debug_stage=i)
        want = taps[nm]
        assert dbg.shape == want.reshape(R, -1).shape, nm
        r = rel(dbg, want.reshape(R, -1))
        worst = max(worst, worst_slot_rel(dbg, want, want.shape[1]))
        assert r < 2e-5, (nm, r)
    eps = eng.unet_forward(x.cuda(), cond.cuda(), t.cuda())
    print("T=%3d fp32 eps rel %.3e worst slot %.3e (worst slot of any stage %.3e)" % (T, rel(eps, want_eps), worst_slot_rel(eps, want_eps, T), worst))
    assert rel(eps, want_eps) < 2e-5


@pytest.mark.parametrize("T", FP32_T)
def test_decode_posterior_and_indicators_fp32_vs_oracle(build, T):
    dm, vae, _ = build(T)
    R = 37
    torch.manual_seed(5000 + T)
    z, cond = torch.randn(R, T, 4), torch.randn(R, 256)
    curr = torch.cat([torch.zeros(R, 2), torch.rand(R, 1) * 15, torch.zeros(R, 1)], dim=1)
    eng = dm.engine(R)
    act, traj = eng.decode_rollout(z.cuda(), cond.cuda(), curr.cuda())
    wtraj, wact = O.decode_rollout(dec_sd_of(vae), z, cond, curr)
    print("T=%3d fp32 decode: rel(act) %.3e rel(traj) %.3e worst slot %.3e" % (T, rel(act, wact), rel(traj, wtraj), worst_slot_rel(traj, wtraj, T)))
    assert rel(act, wact) < 1e-5 and rel(traj, wtraj) < 1e-5
    # posterior step, DDPM (with and without noise) and DDIM
    sch = O.make_schedule(10)
    x, eps, nzs = torch.randn(R, T, 4), torch.randn(R, T, 4), torch.randn(R, T, 4)
    for i in (9, 5, 1, 0):
        mean, sig = O.ddpm_mean_sigma(sch, x, eps, i)
        want = mean + (0.0 if i == 0 else 1.0) * sig * nzs
        got, gmean = eng.posterior_step(x.cuda(), eps.cuda(), nzs.cuda(), i, want_mean=True)
        assert rel(got, want) < 1e-6 and rel(gmean, mean) < 1e-6, i
    for i, nxt in ((9, 7), (2, 0), (0, -1)):
        got = eng.posterior_step(x.cuda(), eps.cuda(), None, i, nxt, sampler="ddim")
        assert rel(got, O.ddim_next(sch, x, eps, i, nxt)) < 1e-6, (i, nxt)
    # indicators of decoded trajectories in dense scenes: 3 scenes x 4 agents x 2 samples
    from cld_b200.critic import indicators
    S, A, N = 3, 4, 2
    aux, batch = make_scenes(S, A, horizon=T, seed=5100 + T, dense=True)
    zs = torch.randn(S * A * N, T, 4)
    _, tr = eng.decode_rollout(zs.cuda(), aux["cond_feat"].repeat_interleave(N, 0).cuda(),
                               aux["curr_states"].repeat_interleave(N, 0).cuda())
    off, coll, _ = indicators(dm, tr, batch, num_samp=N)
    rep = {k: (v.repeat_interleave(N, 0) if torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == S * A else v) for k, v in batch.items()}
    woff, wcoll = O.indicators(tr.cpu()[..., :2], rep)
    print("T=%3d indicators: %d of %d slots off-road, %d collisions" % (T, int(woff.sum()), woff.numel(), int(wcoll.sum())))
    assert torch.equal(off.cpu(), woff) and torch.equal(coll.cpu(), wcoll)


@pytest.mark.parametrize("T", FP32_T)
def test_guidance_step_fp32_vs_oracle(build, T):
    dm, vae, _ = build(T)
    lrel, rg, sign_agree, zero_agree = _guidance_vs_oracle(dm, vae, T, "fp32")
    assert all(v < 1e-4 for v in lrel.values()), lrel
    assert rg < 1e-3 and sign_agree >= 0.999 and zero_agree >= 0.999, (rg, sign_agree, zero_agree)


# --------------------------------------------------------------------------------------------------------------------------
# 6. guided sampler end to end
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [20, 64])
def test_guided_sampler_vs_oracle(build, T):
    """10 guided DDPM steps on supplied noise, 2 scenes x 4 agents: fp32 against the composed oracle; bf16 unguided against fp32,
    bf16 guided self-consistent (its trajectory is the oracle decode of its own latent)."""
    from cld_b200.engine import default_guidance
    dm, vae, algo = build(T)
    dm16, vae16, _ = build(T, "bf16")
    S, A = 2, 4
    aux, batch = make_scenes(S, A, horizon=T, seed=6000 + T, dense=True)
    torch.manual_seed(6100 + T)
    R = S * A
    x_init, noises = torch.randn(R, T, 4), torch.randn(10, R, T, 4)
    kw = dict(noise=noises.cuda(), x_init=x_init.cuda(), want_indicators=True, agents_per_scene=A)
    out = dm(cu(batch), cu(aux), algo, guidance=default_guidance(), **kw)
    dec_sd = dec_sd_of(vae)
    gd = dict(dec_sd=dec_sd, cond=aux["cond_feat"], curr=aux["curr_states"], batch=batch, A=A, N=1, cfg=O.DEFAULT_GUIDANCE)
    want = O.sample(cpu_sd(dm.model), O.make_schedule(10), aux["cond_feat"], x_init, noises, 10, 1, "ddpm", guidance=gd)
    frac = ((out["pred_traj"].cpu() - want["pred_traj"]).abs() > 1e-2 * want["pred_traj"].abs().max()).float().mean().item()
    wtraj, _ = O.decode_rollout(dec_sd, out["pred_traj"].cpu(), aux["cond_feat"], aux["curr_states"])
    print("T=%3d fp32 guided sampler: rel %.3e, fraction off by >1%% of max %.5f, rel(traj) %.3e" % (
        T, rel(out["pred_traj"], want["pred_traj"]), frac, rel(out["traj"], wtraj)))
    assert frac < 0.02
    assert rel(out["traj"], wtraj) < 1e-4
    woff, wcoll = O.indicators(out["traj"].cpu()[..., :2], batch)
    assert torch.equal(out["offroad"].cpu(), woff) and torch.equal(out["coll"].cpu(), wcoll)
    # bf16 mode
    u16, u32 = dm16(cu(batch), cu(aux), algo, **kw), dm(cu(batch), cu(aux), algo, **kw)
    r = rel(u16["pred_traj"], u32["pred_traj"])
    g16 = dm16(cu(batch), cu(aux), algo, guidance=default_guidance(), **kw)
    wtraj16, _ = O.decode_rollout(dec_sd_of(vae16), g16["pred_traj"].cpu(), aux["cond_feat"], aux["curr_states"])
    rt = rel(g16["traj"], wtraj16)
    print("T=%3d bf16 sampler: unguided rel vs fp32 %.3e worst slot %.3e; guided rel(traj) vs oracle decode %.3e" % (
        T, r, worst_slot_rel(u16["pred_traj"], u32["pred_traj"], T), rt))
    assert r < 1e-2
    assert torch.isfinite(g16["pred_traj"]).all() and torch.isfinite(g16["traj"]).all()
    assert rt < 1e-3
    woff, wcoll = O.indicators(g16["traj"].cpu()[..., :2], batch)
    assert torch.equal(g16["offroad"].cpu(), woff) and torch.equal(g16["coll"].cpu(), wcoll)


# --------------------------------------------------------------------------------------------------------------------------
# 7. denoiser training step (forward with stash + analytic backward)
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
@pytest.mark.parametrize("T", [8, 12, 20, 56, 128])
def test_train_backward_vs_oracle_autograd(build, T, mode):
    """R = 37: every parameter gradient and dx against torch autograd on the oracle's U-Net.  tf32 mode runs the stride-1
    convolutions on the tensor pipe with boxes of 128 / T' rows: partial boxes at every level of these horizons."""
    dm, _, _ = build(T)
    tol = GRAD_TOL if mode == "fp32" else 1e-2
    R = 37
    torch.manual_seed(7000 + T)
    x, cond, t, d_eps = torch.randn(R, T, 4), torch.randn(R, 256), torch.randint(0, 10, (R,)), torch.randn(R, T, 4)
    sd = {k: v.requires_grad_(True) for k, v in cpu_sd(dm.model).items()}
    xg = x.clone().requires_grad_(True)
    eps_want = O.unet_forward(sd, xg, cond, t)
    want = torch.autograd.grad((eps_want * d_eps).sum(), list(sd.values()) + [xg])
    dm.train_precision = mode
    try:
        eng = dm.train_engine(R)
        eps = eng.unet_train_forward(x.cuda(), cond.cuda(), t.cuda())
        grads = [torch.empty_like(p) for p in dm.model.parameters()]
        dx = eng.unet_backward(d_eps.cuda(), grads, want_dx=True)
    finally:
        dm.train_precision = "fp32"
    errs = {k: rel(g, w) for k, g, w in zip(sd.keys(), grads, want[:-1])}
    e_eps, e_dx = rel(eps, eps_want.detach()), rel(dx, want[-1])
    print("T=%3d %s training step: rel(eps) %.2e, worst gradient rel %.2e (%s), dx %.2e worst slot %.2e" % (
        T, mode, e_eps, max(errs.values()), max(errs, key=errs.get), e_dx, worst_slot_rel(dx, want[-1], T)))
    assert e_eps < (2e-5 if mode == "fp32" else 1e-2)
    assert max(errs.values()) < tol, {k: v for k, v in errs.items() if v >= tol}
    assert e_dx < tol
