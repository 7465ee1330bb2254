"""GPU (-m gpu): guided steps with several optimizer iterations (`grad_steps` > 1) -- the CUDA loop against the oracle's
perturb loop (tests/perturb_oracle.py), the tensor-core BPTT against the fp32 kernels, the guided samplers, and the invariance
of the result to chunks, lanes and ragged batches."""
import pytest
import torch

import cld_oracle as O
from cld_b200.synthetic import make_scenes
from perturb_oracle import guidance_perturb, sample as perturb_sample

pytestmark = pytest.mark.gpu
TERMS = ("agent_collision", "map_collision", "target_pos", "target_speed", "acc_limit", "speed_limit")


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def cu(d):
    return {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in d.items()}


def dec_sd_of(vae):
    return {k: v.detach().cpu() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}


@pytest.fixture(scope="module")
def build(models_cpu):
    cache = {}

    def get(precision="fp32", n=10, **kw):
        key = (precision, n, tuple(sorted(kw.items())))
        if key not in cache:
            dm, vae, algo = models_cpu(n, precision=precision, **kw)
            dm = dm.cuda()
            vae.bind(dm)
            cache[key] = (dm, vae, algo)
        return cache[key]
    return get


def all_terms_case(S, A, seed):
    aux, batch = make_scenes(S, A, seed=seed, dense=True)
    torch.manual_seed(seed + 1)
    batch["target_speed"] = (aux["curr_states"][:, 2:3] + torch.randn(S * A, 1)).clamp(min=0).repeat(1, 52)
    w = dict(agent_collision=50.0, map_collision=1.0, target_pos=1.0, target_speed=0.5, acc_limit=1.0, acc_limit_value=1.0,
             speed_limit=1.0, speed_limit_value=3.0)
    return aux, batch, w


@pytest.mark.parametrize("S,k,optimizer", [(2, 2, "adam"), (2, 4, "adam"), (2, 2, "sgd"), (2, 4, "sgd"), (5, 3, "adam")])
def test_guidance_steps_vs_oracle_perturb(build, S, k, optimizer):
    """fp32 kernels, every term on: z after k iterations, the last iteration's gradient and losses (S = 5: R = 40 rows, a
    partial CTA)."""
    from cld_b200.engine import default_guidance
    dm, vae, _ = build()
    A, N = 4, 2
    aux, batch, w = all_terms_case(S, A, 301 + S)
    lr = 0.3 if optimizer == "adam" else 1.0
    cfg = default_guidance(optimizer=optimizer, lr=lr, grad_steps=k, **w)
    ocfg = dict(O.DEFAULT_GUIDANCE, optimizer=optimizer, lr=lr, grad_steps=k, **w)
    torch.manual_seed(S * 10 + k)
    z = torch.randn(S * A * N, 52, 4)
    eng = dm.engine(S * A * N)
    scene = eng.make_scene(batch, S, A, N)
    z_out, grad, loss = eng.guidance_step(z.cuda(), aux["cond_feat"].repeat_interleave(N, 0).cuda(),
                                          aux["curr_states"].repeat_interleave(N, 0).cuda(), scene, cfg)
    zw, gw, per = guidance_perturb(dec_sd_of(vae), z, aux["cond_feat"], aux["curr_states"], batch, A, N, ocfg)
    lrel = {t: rel(loss[i], torch.cat([p[t] for p in per]).reshape(-1)) for i, t in enumerate(TERMS)}
    nz = gw != 0
    sign_agree = (torch.sign(grad.cpu())[nz] == torch.sign(gw)[nz]).float().mean().item()
    zero_agree = ((grad.cpu() == 0) == (gw == 0)).float().mean().item()
    frac_bad = ((z_out.cpu() - zw).abs() > 1e-3).float().mean().item()
    print("S=%d k=%d %s: rel(z) %.3e (off by >1e-3: %.5f) rel(grad) %.3e sign %.6f zero-set %.6f losses %s" % (
        S, k, optimizer, rel(z_out, zw), frac_bad, rel(grad, gw), sign_agree, zero_agree,
        " ".join("%s %.1e" % (t, v) for t, v in lrel.items())))
    assert all(v < 1e-4 for v in lrel.values()), lrel
    assert rel(grad, gw) < 1e-3 and sign_agree >= 0.999 and zero_agree >= 0.999
    assert rel(z_out, zw) < 5e-3 and frac_bad < 1e-3
    assert not torch.equal(z_out.cpu(), guidance_perturb(dec_sd_of(vae), z, aux["cond_feat"], aux["curr_states"], batch, A, N,
                                                         dict(ocfg, grad_steps=1))[0])


def test_guidance_steps_tensor_core_vs_fp32_kernels(build):
    """cfg2-shaped scenes (32 agents x 8 samples), k = 3: the bf16-mode step (tensor-core decoder and BPTT) against the fp32
    kernels.  The thresholds are the single-iteration ones; the measured values are printed."""
    from cld_b200.engine import default_guidance
    S, A, N = 2, 32, 8
    R = S * A * N
    aux, batch = make_scenes(S, A, seed=31, dense=True)
    torch.manual_seed(32)
    z = torch.randn(R, 52, 4).cuda()
    cond = aux["cond_feat"].repeat_interleave(N, 0).cuda()
    curr = aux["curr_states"].repeat_interleave(N, 0).cuda()
    res = {}
    for prec in ("fp32", "bf16"):
        dm, _, _ = build(prec, max_rows=R)
        eng = dm.engine(R)
        res[prec] = eng.guidance_step(z, cond, curr, eng.make_scene(batch, S, A, N), default_guidance(grad_steps=3))
    (z32, _, l32), (z16, _, l16) = res["fp32"], res["bf16"]
    d32, d16 = z32 - z, z16 - z
    nz = d32 != 0
    sign_agree = (torch.sign(d16)[nz] == torch.sign(d32)[nz]).float().mean().item()
    zero_agree = ((d16 == 0) == (d32 == 0)).float().mean().item()
    lrel = (rel(l16[0], l32[0]), rel(l16[1], l32[1]))
    print("cfg2 shape, k=3: update sign agreement %.6f zero-set agreement %.6f rel(loss) %.2e %.2e" % (sign_agree, zero_agree, *lrel))
    assert nz.any()
    assert sign_agree >= 0.995 and zero_agree >= 0.999
    assert lrel[0] < 1e-3 and lrel[1] < 1e-3


@pytest.mark.parametrize("sampler", ["ddpm", "ddim"])
def test_guided_sampler_grad_steps_vs_oracle(build, sampler):
    """Strided sampler (10 timesteps, stride 2), guided with k = 3, fp32, against the oracle on identical x_init / noise."""
    from cld_b200.engine import default_guidance
    dm, vae, algo = build("fp32")
    S, A, N = 2, 4, 1
    aux, batch = make_scenes(S, A, seed=55, dense=True)
    torch.manual_seed(57)
    R = S * A * N
    x_init, noises = torch.randn(R, 52, 4), torch.randn(5, R, 52, 4)
    old = dm.stride
    dm.stride = 2
    try:
        out = dm(cu(batch), cu(aux), algo, noise=noises.cuda(), x_init=x_init.cuda(), sampler=sampler,
                 guidance=default_guidance(grad_steps=3), want_indicators=True)
    finally:
        dm.stride = old
    dec_sd = dec_sd_of(vae)
    gd = dict(dec_sd=dec_sd, cond=aux["cond_feat"], curr=aux["curr_states"], batch=batch, A=A, N=N,
              cfg=dict(O.DEFAULT_GUIDANCE, grad_steps=3))
    unet_sd = {k: v.detach().cpu() for k, v in dm.model.state_dict().items()}
    with torch.no_grad():
        want = perturb_sample(unet_sd, O.make_schedule(10), aux["cond_feat"], x_init, noises, 10, 2, sampler, guidance=gd)
    frac = ((out["pred_traj"].cpu() - want["pred_traj"]).abs() > 1e-2 * want["pred_traj"].abs().max()).float().mean().item()
    print("guided %s, k=3: rel %.3e, fraction of elements off by >1%% of max: %.5f" % (sampler, rel(out["pred_traj"], want["pred_traj"]), frac))
    assert frac < 0.02
    wtraj, _ = O.decode_rollout(dec_sd, out["pred_traj"].cpu(), aux["cond_feat"], aux["curr_states"])
    assert rel(out["traj"], wtraj) < 1e-4
    woff, wcoll = O.indicators(out["traj"].cpu()[..., :2], batch)
    assert torch.equal(out["offroad"].cpu(), woff) and torch.equal(out["coll"].cpu(), wcoll)


def test_grad_steps_results_do_not_depend_on_chunks_lanes_or_buckets(build):
    """bf16, k = 3, supplied x_init / noise: an engine whose max_rows forces 3 chunks, DmModel(lanes=2) and a ragged batch (one
    call per scene size inside) are bit-identical to single un-chunked calls."""
    from cld_b200.engine import default_guidance
    g = default_guidance(grad_steps=3)
    S, A, N = 6, 4, 2
    R = S * A * N
    aux, batch = make_scenes(S, A, seed=501, dense=True)
    torch.manual_seed(502)
    x_init, noises = torch.randn(R, 52, 4).cuda(), torch.randn(10, R, 52, 4).cuda()
    dm, _, algo = build("bf16", max_rows=R)
    algo.num_samp = N
    try:
        full = dm(cu(batch), cu(aux), algo, noise=noises, x_init=x_init, guidance=g, want_indicators=True, agents_per_scene=A)
    finally:
        algo.num_samp = 1
    # chunks: 2 scenes per chunk
    dmc, _, _ = build("bf16", max_rows=2 * A * N)
    eng = dmc.engine(1)
    assert eng.max_rows == 2 * A * N
    rep = lambda v: v.cuda().repeat_interleave(N, 0)                            # noqa: E731
    o = eng.sample(x_init, rep(aux["cond_feat"]), noises=noises, curr_rows=rep(aux["curr_states"]), scene=eng.make_scene(batch, S, A, N),
                   guidance=g, sampler="ddpm", want_indicators=True)
    assert torch.equal(o["x0"], full["pred_traj"]) and torch.equal(o["traj"], full["traj"]) and torch.equal(o["coll"], full["coll"])
    # lanes
    dml, _, algol = build("bf16", max_rows=R, lanes=2)
    algol.num_samp = N
    try:
        lan = dml(cu(batch), cu(aux), algol, noise=noises, x_init=x_init, guidance=g, want_indicators=True, agents_per_scene=A)
    finally:
        algol.num_samp = 1
    for key in ("pred_traj", "traj", "offroad", "coll"):
        assert torch.equal(lan[key], full[key]), key
    # ragged: scenes of 4, 2, 6 and 4 agents in one batch vs one call per scene
    dm1, _, algo1 = build("bf16")
    sizes = [4, 2, 6, 4]
    B = sum(sizes)
    aux_r, batch_r = make_scenes(1, B, seed=801, dense=True)
    batch_r["scene_index"] = torch.cat([torch.full((c,), 10 + i) for i, c in enumerate(sizes)])
    torch.manual_seed(802)
    xr, nr = torch.randn(B, 52, 4), torch.randn(10, B, 52, 4)
    out = dm1(cu(batch_r), cu(aux_r), algo1, noise=nr.cuda(), x_init=xr.cuda(), guidance=g, want_indicators=True)
    pos = 0
    for c in sizes:
        sl = slice(pos, pos + c)
        sb = {k: (v[sl].cuda() if (torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == B) else v) for k, v in batch_r.items()}
        one = dm1(sb, {k: v[sl].cuda() for k, v in aux_r.items()}, algo1, noise=nr[:, sl].cuda(), x_init=xr[sl].cuda(), guidance=g,
                  want_indicators=True)
        for k in ("pred_traj", "traj", "offroad", "coll"):
            assert torch.equal(out[k][sl], one[k]), (k, c)
        pos += c


def test_explicit_single_step_equals_the_default(build):
    """grad_steps=1 given explicitly is the guidance dict without the key, bit for bit (guidance_step and the sampler)."""
    from cld_b200.engine import default_guidance
    g1 = default_guidance(grad_steps=1)
    g0 = {k: v for k, v in g1.items() if k != "grad_steps"}
    S, A, N = 2, 4, 2
    aux, batch = make_scenes(S, A, seed=601, dense=True)
    torch.manual_seed(602)
    z = torch.randn(S * A * N, 52, 4).cuda()
    for prec in ("fp32", "bf16"):
        dm, _, algo = build(prec)
        eng = dm.engine(S * A * N)
        scene = eng.make_scene(batch, S, A, N)
        cond, curr = aux["cond_feat"].repeat_interleave(N, 0).cuda(), aux["curr_states"].repeat_interleave(N, 0).cuda()
        a, b = eng.guidance_step(z, cond, curr, scene, g1), eng.guidance_step(z, cond, curr, scene, g0)
        assert all(torch.equal(x, y) for x, y in zip(a, b)), prec
        x_init, noises = torch.randn(S * A, 52, 4).cuda(), torch.randn(10, S * A, 52, 4).cuda()
        oa = dm(cu(batch), cu(aux), algo, noise=noises, x_init=x_init, guidance=g1, want_indicators=True)
        ob = dm(cu(batch), cu(aux), algo, noise=noises, x_init=x_init, guidance=g0, want_indicators=True)
        for k in ("pred_traj", "traj", "offroad", "coll"):
            assert torch.equal(oa[k], ob[k]), (prec, k)


def test_get_action_scores_the_samples_with_one_evaluation(build):
    """GuidedDiffusionPolicy with grad_steps=3: the sampler runs 3 iterations per guided step, but the losses that choose the
    sample are ONE evaluation at the returned x0."""
    from cld_b200.engine import default_guidance
    from cld_b200.policy import GuidedDiffusionPolicy
    dm, vae, algo = build("bf16")
    S, A, N = 2, 4, 3
    aux, batch = make_scenes(S, A, seed=17, dense=True)
    g = default_guidance(grad_steps=3)
    pol = GuidedDiffusionPolicy(dm, vae, algo, guidance=g)
    kw = dict(use_device_rng=True, seed=5)
    _, info = pol.get_action(cu(batch), num_action_samples=N, step_index=0, aux_info=cu(aux), **kw)
    algo.num_samp = N
    try:
        out = dm(cu(batch), cu(aux), algo, guidance=g, want_traj=True, agents_per_scene=A, **kw)
    finally:
        algo.num_samp = 1
    eng = dm.engine(S * A * N)
    scene = eng.make_scene(cu(batch), S, A, N)
    cond, curr = aux["cond_feat"].repeat_interleave(N, 0).cuda(), aux["curr_states"].repeat_interleave(N, 0).cuda()
    _, _, one = eng.guidance_step(out["pred_traj"], cond, curr, scene, default_guidance(grad_steps=1))
    _, _, three = eng.guidance_step(out["pred_traj"], cond, curr, scene, g)
    active = list(info["guide_losses"])
    assert active == ["agent_collision", "map_collision"]
    # the map-collision kernel adds its per-row loss with atomics (the gradient is written without them), so two evaluations of
    # that loss may differ in the last bits; the agent-collision loss is bit-exact
    assert torch.equal(info["guide_losses"]["agent_collision"], one[0].reshape(S * A, N))
    assert torch.allclose(info["guide_losses"]["map_collision"], one[1].reshape(S * A, N), rtol=1e-6, atol=0.0)
    got = torch.stack([info["guide_losses"][k].reshape(-1) for k in active])
    # the last of 3 iterations scores a perturbed latent: its losses move by far more than the atomics' last-bit noise (about 1e-4
    # relative on the largest map-collision loss of this case, against 1e-7)
    assert not torch.allclose(got, three[:2], rtol=1e-5, atol=0.0)
