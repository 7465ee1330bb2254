"""CPU: the oracle (oracle/cld_oracle.py) against the golden vectors produced by the REAL reference
(oracle/make_golden.py).  No GPU, no reference needed."""
import numpy as np
import torch

import cld_oracle as O
from cld_b200.synthetic import make_scenes


def rel(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _sds(models_cpu, n):
    dm, vae, algo = models_cpu(n)
    unet_sd = {k: v.detach() for k, v in dm.model.state_dict().items()}
    dec_sd = {k: v.detach() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}
    return dm, unet_sd, dec_sd


def test_weight_init_matches_reference(models_cpu, gold):
    g = gold("unet")
    dm, unet_sd, dec_sd = _sds(models_cpu, 10)
    assert abs(float(sum(v.double().sum() for v in unet_sd.values())) - float(g["unet_sum"])) < 1e-9
    assert abs(float(sum(v.double().abs().sum() for v in unet_sd.values())) - float(g["unet_abs"])) < 1e-9
    assert abs(float(sum(v.double().sum() for v in dec_sd.values())) - float(g["dec_sum"])) < 1e-9


def test_schedule_known_answers():
    # SURVEY.md Appendix A: betas(n=10) of the reference
    want = [0.027907, 0.075494, 0.124396, 0.17719, 0.237282, 0.309883, 0.404003, 0.536998, 0.743829, 0.999]
    s = O.make_schedule(10)
    assert np.allclose(s["betas"].numpy(), want, atol=1e-6)
    assert len(s) == 14
    assert abs((-torch.log((0.5 * s["posterior_log_variance_clipped"][0]).exp()) - 0.5 * np.log(2 * np.pi)).item() - 22.106915) < 1e-4


def test_unet_oracle_vs_reference_golden(models_cpu, gold):
    g = gold("unet")
    _, unet_sd, _ = _sds(models_cpu, 10)
    with torch.no_grad():
        eps = O.unet_forward(unet_sd, torch.tensor(g["x"]), torch.tensor(g["cond"]), torch.tensor(g["t"]))
        e104 = O.unet_forward(unet_sd, torch.tensor(g["x104"]), torch.tensor(g["cond"][:3]), torch.tensor(g["t"][:3]))
    assert rel(eps, g["eps"]) < 5e-6
    assert rel(e104, g["eps104"]) < 5e-6


def test_sampler_oracle_vs_reference_golden(models_cpu, gold):
    g = gold("cfg0_sample")
    _, unet_sd, dec_sd = _sds(models_cpu, 10)
    with torch.no_grad():
        out = O.sample(unet_sd, O.make_schedule(10), torch.tensor(g["cond"]), torch.tensor(g["x_init"]),
                       torch.tensor(g["noises"]), 10, 1, "ddpm")
        traj, act = O.decode_rollout(dec_sd, torch.tensor(g["pred_traj"]), torch.tensor(g["cond"]), torch.tensor(g["curr"]))
    assert rel(out["pred_traj"], g["pred_traj"]) < 1e-4
    assert rel(out["x1"], g["x1"]) < 1e-4
    assert rel(out["log_prob_final"], g["log_prob_final"]) < 1e-6
    assert rel(act, g["act"]) < 1e-5
    assert rel(traj, g["traj"]) < 1e-5


def test_strided_sampler_oracle_vs_reference_golden(models_cpu, gold):
    g = gold("stride2_sample")
    _, unet_sd, _ = _sds(models_cpu, 100)
    with torch.no_grad():
        out = O.sample(unet_sd, O.make_schedule(100), torch.tensor(g["cond"]), torch.tensor(g["x_init"]),
                       torch.tensor(g["noises"]), 100, 2, "ddpm")
    assert out["x1"] is None            # step index 1 is never visited with stride 2 (dm_model.py:126-127)
    assert rel(out["pred_traj"], g["pred_traj"]) < 1e-4


def test_unicycle_oracle_vs_reference_golden(gold):
    g = gold("unicycle")
    st = O.unicycle_rollout(torch.tensor(g["curr"]), torch.tensor(g["u"]))
    assert rel(st, g["state"]) < 1e-5


def test_unicycle_closed_form_matches_chain_in_bounds():
    # property: inside the bounds the closed form equals the step-by-step integrator
    torch.manual_seed(3)
    u = torch.randn(8, 52, 2) * torch.tensor([0.5, 0.05])
    c0 = torch.cat([torch.zeros(8, 2), 5 + torch.rand(8, 1) * 5, torch.zeros(8, 1)], 1)
    st = O.unicycle_rollout(c0, u)
    x = c0.clone()
    outs = []
    for k in range(52):
        v, th = x[:, 2], x[:, 3]
        vm = v + u[:, k, 0] * 0.1 * 0.5
        x = torch.stack([x[:, 0] + vm * torch.cos(th) * 0.1, x[:, 1] + vm * torch.sin(th) * 0.1,
                         v + u[:, k, 0] * 0.1, th + u[:, k, 1] * 0.1], 1)
        outs.append(x)
    assert rel(st, torch.stack(outs, 1)) < 1e-5


def test_indicators_oracle_vs_reference_golden(gold):
    g = gold("indicators")
    _, batch = make_scenes(2, 8, seed=31, dense=True)
    tr = torch.tensor(g["traj"])
    off, coll = O.indicators(tr[..., :2], batch)
    assert np.array_equal(off.numpy(), g["offroad"])
    assert np.array_equal(coll.numpy(), g["coll"])
    fr = O.failure_rates(tr[..., :2], batch)
    for k in fr:
        assert abs(fr[k] - float(g[k])) < 1e-12
    assert float(g["offroad_failure_rate"]) > 0 and float(g["collision_failure_rate"]) > 0


def test_guidance_oracle_vs_reference_golden(models_cpu, gold):
    g = gold("guidance")
    _, _, dec_sd = _sds(models_cpu, 10)
    S, A, N = int(g["S"]), int(g["A"]), int(g["N"])
    aux, batch = make_scenes(S, A, seed=int(g["seed"]), dense=True)
    z = torch.tensor(g["z"])
    grad, per = O.guidance_grad(dec_sd, z, aux["cond_feat"], aux["curr_states"], batch, A, N)
    z_out = O.apply_guidance_update(z, grad)
    lo_ac = torch.cat([p["agent_collision"] for p in per])
    lo_mc = torch.cat([p["map_collision"] for p in per])
    assert rel(lo_ac.reshape(-1), g["loss_ac"].reshape(-1)) < 1e-5
    assert rel(lo_mc.reshape(-1), g["loss_mc"].reshape(-1)) < 1e-5
    assert rel(z_out, g["z_out"]) < 1e-4
    moved = torch.tensor(g["z_out"]) - z
    assert (torch.sign(grad) == torch.sign(-moved)).float().mean().item() > 0.9999
    assert float(lo_ac.sum()) > 0 and float(lo_mc.sum()) > 0


def test_guidance_terms_oracle_vs_reference_golden(models_cpu, gold):
    """Rows a13 / f-4: TargetPosLoss, TargetSpeedLoss, AccLimitLoss, SpeedLimitLoss alone and all six terms together against
    the outputs of the REAL PerturbationGuidance.perturb (golden written by oracle/make_golden.py --only-guidance-ext)."""
    from conftest import guidance_ext_case
    g = gold("guidance_ext")
    _, _, dec_sd = _sds(models_cpu, 10)
    S, A, N, aux, batch, z, cfgs = guidance_ext_case(g)
    for tag, cfg in cfgs.items():
        grad, per = O.guidance_grad(dec_sd, z, aux["cond_feat"], aux["curr_states"], batch, A, N, cfg)
        for key in ("target_pos", "target_speed", "acc_limit", "speed_limit"):
            if cfg.get(key, 0.0) != 0.0:
                lo = torch.cat([p[key] for p in per]).reshape(-1)
                assert rel(lo, g["%s_loss_%s" % (tag, key)].reshape(-1)) < 2e-5, (tag, key)
        gref = torch.tensor(g[tag + "_grad_sgd"])
        big = gref.abs() > 1e-4 * gref.abs().max()
        assert rel(grad[big], gref[big]) < 1e-3, tag
        assert rel(O.apply_guidance_update(z, grad, cfg), g[tag + "_z_out"]) < 3e-3, tag
        assert float(gref.abs().max()) > 0


def test_guidance_big_shape_oracle_vs_reference_golden(models_cpu, gold):
    """T = 104, 64 agents, 8 samples (cfg2 / cfg3 shapes) against the real reference: per-row gradient sums for all 512 rows,
    full gradients of 96 rows, z' of 64 rows."""
    from conftest import guidance_big_case
    g = gold("guidance_t104")
    _, _, dec_sd = _sds(models_cpu, 10)
    S, A, N, T, aux, batch, z = guidance_big_case(g)
    grad, per = O.guidance_grad(dec_sd, z, aux["cond_feat"], aux["curr_states"], batch, A, N)
    rows = torch.tensor(g["big_rows"]).long()
    assert rel(grad[rows[:96]], g["big_grad_rows"]) < 1e-3
    assert rel(grad.flatten(1).double().abs().sum(1), g["big_grad_rowabs"]) < 1e-3
    nz = (grad.flatten(1).abs().sum(1) > 0).nonzero().flatten()
    assert torch.equal(nz, rows)
    assert rel(O.apply_guidance_update(z, grad)[:64], g["big_z_out_head"]) < 3e-3
    assert rel(torch.cat([p["agent_collision"] for p in per]).reshape(-1), g["big_loss_agent_collision"].reshape(-1)) < 2e-5
    assert rel(torch.cat([p["map_collision"] for p in per]).reshape(-1), g["big_loss_map_collision"].reshape(-1)) < 2e-5


def test_ddim_final_step_is_x0_prediction():
    s = O.make_schedule(100)
    x, eps = torch.randn(2, 52, 4), torch.randn(2, 52, 4)
    x0 = O.ddim_next(s, x, eps, 0, -1)
    assert torch.allclose(x0, s["sqrt_recip_alphas_cumprod"][0] * x - s["sqrt_recipm1_alphas_cumprod"][0] * eps)


# ----------------------------------------------------------------------------------------------------
# a14 context encoder
# ----------------------------------------------------------------------------------------------------
def _context_case(gold):
    import torch
    import cld_oracle as O
    g = gold("context")
    shapes = {str(k): eval(str(s)) for k, s in zip(g["keys"], g["shapes"])}
    sd = O.synth_context_state(shapes)
    batch = {"image": torch.from_numpy(g["image_x2"]).float() / 2, "history_positions": torch.from_numpy(g["history_positions"]),
             "history_yaws": torch.from_numpy(g["history_yaws"]), "curr_speed": torch.from_numpy(g["curr_speed"])}
    return g, sd, batch


def test_context_oracle_vs_reference_golden(gold):
    """oracle.context_encode == the REAL ContextEncoder (models/context_utils.py:40-61) on the golden inputs."""
    import torch
    import cld_oracle as O
    g, sd, batch = _context_case(gold)
    assert abs(float(sum(v.double().sum() for v in sd.values())) - float(g["w_sum"])) < 1e-6 * abs(float(g["w_sum"])) + 1e-6
    with torch.no_grad():
        taps = {}
        out = O.context_encode(sd, batch, taps)
    assert rel(out["cond_feat"], torch.from_numpy(g["cond_feat"])) < 1e-5
    assert torch.equal(out["curr_states"], torch.from_numpy(g["curr_states"]))
    assert rel(taps["map_feat"], torch.from_numpy(g["map_feat"])) < 1e-5
    am = [taps[k].abs().mean().item() for k in ("stem", "layer1", "layer2", "layer3", "layer4")]
    assert max(abs(a - b) / b for a, b in zip(am, g["layer_absmean"])) < 1e-4


def test_context_mirror_state_dict_matches_reference(gold):
    """cld_b200.ContextEncoder exposes the reference's 150 state-dict keys with the reference's shapes, and the C ABI
    gets the 130 floating-point ones."""
    from cld_b200 import default_algo_config
    from cld_b200.context import ContextEncoder
    g = gold("context")
    ce = ContextEncoder(4, default_algo_config(), {"image": (34, 224, 224)})
    sd = ce.state_dict()
    assert list(sd.keys()) == [str(k) for k in g["keys"]]
    assert [str(tuple(v.shape)) for v in sd.values()] == [str(s) for s in g["shapes"]]
    assert len(ce.weight_list()) == 130


def test_rasterize_agents_oracle_vs_reference_golden(gold):
    """oracle.rasterize_agents == the REAL rasterize_agents (src/tbsim/utils/trajdata_utils.py:123-156), bit for bit."""
    import torch
    import cld_oracle as O
    g = gold("raster")
    img = O.rasterize_agents(torch.from_numpy(g["maps_x2"]).float() / 2, torch.from_numpy(g["agent_hist_pos"]),
                             torch.from_numpy(g["agent_hist_mask"]), torch.from_numpy(g["raster_from_agent"]))
    assert torch.equal(img, torch.from_numpy(g["image_x2"]).float() / 2)
    assert int((img[:, :31] == 1).sum()) == int(g["n_ego"]) and int((img[:, :31] == -1).sum()) == int(g["n_oth"])


# ---------------------------------------------------------------------------------------------------- f-2 (PPO update)
def test_ppo_oracle_vs_reference_golden(gold, models_cpu):
    """O.log_prob / O.ppo_loss / autograd gradients against the REAL reference's ppo_update arithmetic (tests/golden/ppo.npz)."""
    g = gold("ppo")
    dm, _, _ = models_cpu(16)
    sd = {k: v.detach() for k, v in dm.model.state_dict().items()}
    names = [str(n) for n in g["names"]]
    assert names == list(sd.keys())
    tt = lambda k: torch.tensor(g[k])
    loss, lp, grads = O.ppo_grads(sd, O.make_schedule(16), tt("x1"), tt("x0"), tt("cond"), tt("t"), tt("log_p_old"), tt("reward"),
                                  float(g["baseline"]), float(g["clip"]))
    assert ((lp - tt("log_p_new")).norm() / tt("log_p_new").norm()).item() < 1e-5
    assert abs(float(loss) - float(g["loss"])) < 1e-5
    for i, k in enumerate(names):
        want = float(g["grad_norm"][i])
        assert abs(grads[k].double().norm().item() - want) <= 1e-4 * want + 1e-12, k
        samp = grads[k].reshape(-1)[torch.tensor(g["grad_idx"][i])]
        assert (samp - torch.tensor(g["grad_samples"][i])).abs().max().item() <= 1e-4 * want, k
    # the clipped surrogate: rows outside the clip range on the side the minimum cuts off carry no gradient
    r, adv = tt("ratios"), tt("reward") - float(g["baseline"])
    cut = ((r > 1.2) & (adv > 0)) | ((r < 0.8) & (adv < 0))
    assert cut.any() and (~cut).any()
    # Adam restatement on one tensor against the reference's sampled update
    k = names[7]
    p = sd[k]
    p1, _, _ = O.adam_update(p, grads[k], torch.zeros_like(p), torch.zeros_like(p), 1, float(g["lr"]), weight_decay=float(g["weight_decay"]))
    idx = torch.tensor(g["grad_idx"][7])
    got = (p1 - p.double()).reshape(-1)[idx]
    big = torch.tensor(g["grad_samples"][7]).abs() > 1e-6
    assert (got[big] - torch.tensor(g["delta_samples"][7]).double()[big]).abs().max().item() < 2e-2 * float(g["lr"])


def test_oracle_runs_in_float64(models_cpu):
    """The float64 oracle is the reference of the large-batch training tests (tests/test_gpu_train_large.py): the U-Net forward
    and the PPO gradients take a float64 state dict, agree with the float32 oracle, and return float64 everywhere."""
    dm, _, _ = models_cpu(16)
    sd32 = {k: v.detach() for k, v in dm.model.state_dict().items()}
    sd64 = {k: v.double() for k, v in sd32.items()}
    torch.manual_seed(11)
    R = 5
    x, cond, t = torch.randn(R, 52, 4), torch.randn(R, 256), torch.randint(0, 16, (R,))
    with torch.no_grad():
        e32 = O.unet_forward(sd32, x, cond, t)
        e64 = O.unet_forward(sd64, x.double(), cond.double(), t)
    assert e32.dtype == torch.float32 and e64.dtype == torch.float64
    assert rel(e32, e64) < 1e-6
    sched64 = {k: v.double() for k, v in O.make_schedule(16).items()}
    t = torch.randint(1, 16, (R,))
    x0 = torch.randn(R, 52, 4, dtype=torch.float64)
    lp_old, reward = -torch.rand(R, dtype=torch.float64), torch.randn(R, dtype=torch.float64)
    loss, lp, grads = O.ppo_grads(sd64, sched64, x.double(), x0, cond.double(), t, lp_old, reward, 0.1, 0.2)
    assert loss.dtype == lp.dtype == torch.float64 and all(g.dtype == torch.float64 for g in grads.values())
    assert list(grads) == list(sd64) and torch.isfinite(lp).all()
    loss32, lp32, grads32 = O.ppo_grads(sd32, O.make_schedule(16), x, x0.float(), cond, t, lp_old.float(), reward.float(), 0.1, 0.2)
    assert rel(lp32, lp) < 1e-5
    assert max(rel(grads32[k], grads[k]) for k in grads) < 1e-3


def test_warmup_cosine_schedule():
    """lr factor of configure_optimizers (guide_dm_trainer.py:67-75)."""
    from cld_b200.trainer import warmup_cosine
    assert warmup_cosine(0, 30) == 0.0 and abs(warmup_cosine(5, 30) - 0.5) < 1e-12 and abs(warmup_cosine(10, 30) - 1.0) < 1e-12
    assert abs(warmup_cosine(20, 30) - 0.5) < 1e-12 and warmup_cosine(30, 30) < 1e-12


# ---------------------------------------------------------------------------------------------------- f-4 (waypoint terms)
def _waypoint_batch(g):
    t = lambda k: torch.tensor(g[k])          # noqa: E731
    return {"agent_from_world": t("agent_from_world"), "world_from_agent": t("world_from_agent"), "agent_hist": t("agent_hist")}


def _waypoint_terms(g):
    from cld_b200.waypoints import GlobalTargetPos, GlobalTargetPosAtTime, TargetPosAtTime
    t = lambda k: torch.tensor(g[k])          # noqa: E731
    tol, an = float(g["target_tolerance"]), int(g["action_num"])
    gat = GlobalTargetPosAtTime(t("target_world"), t("t_gl"), t("urgency"), t("pref_speed"), dt=float(g["dt"]), target_tolerance=tol, action_num=an)
    gat.update(int(g["global_t"]))
    return {"at_time": TargetPosAtTime(t("target_local"), t("t_at")), "global_at_time": gat,
            "global": GlobalTargetPos(t("target_world"), t("urgency"), t("pref_speed"), dt=float(g["dt"]),
                                      min_progress_dist=float(g["min_progress_dist"]), target_tolerance=tol, action_num=an)}


def test_waypoint_terms_vs_reference_golden(gold):
    """Host logic of cld_b200.waypoints (branch per agent, local targets, goal distances, have_reached) and the oracle's four
    formulas against the REAL TargetPosAtTimeLoss / GlobalTargetPosAtTimeLoss / GlobalTargetPosLoss (tests/golden/waypoint.npz)."""
    g = gold("waypoint")
    x = torch.tensor(g["x"])
    B, N, T = x.shape[:3]
    batch = _waypoint_batch(g)
    for tag, term in _waypoint_terms(g).items():
        ent = term.scene_entries(batch, T, B)
        assert torch.equal(ent["wp_mode"], torch.tensor(g[tag + "_mode"])), tag
        act = ent["wp_mode"] != 0
        assert torch.allclose(ent["wp_target"][act], torch.tensor(g[tag + "_target"])[act], atol=1e-5)
        assert torch.equal(ent["wp_time"][ent["wp_mode"] == 1], torch.tensor(g[tag + "_time"])[ent["wp_mode"] == 1])
        assert torch.allclose(ent["wp_dist"], torch.tensor(g[tag + "_dist"]), atol=1e-5)
        assert torch.allclose(ent["wp_weight"], act.float() * (B / act.sum()))
        xo = x.clone().requires_grad_(True)
        wp = {k[3:]: v for k, v in ent.items()}
        l = O.waypoint_loss(xo, wp)
        (gr,) = torch.autograd.grad((l * torch.tensor(g["w_samp"])).sum(), xo)
        assert torch.allclose(l.detach(), torch.tensor(g[tag + "_loss"]), atol=1e-5, rtol=1e-5), tag
        assert torch.allclose(gr, torch.tensor(g[tag + "_grad"]), atol=1e-5, rtol=1e-4), tag
    assert set(g["global_at_time_mode"].tolist()) == {0, 1, 2} and set(g["global_mode"].tolist()) == {0, 3, 4}
