"""GPU (-m gpu): SURVEY.md sec. 8 f-2 -- the PPO inner loop's denoiser update (forward with stash, analytic backward, loss heads,
Adam) through the C ABI, against the REAL reference's autograd (tests/golden/ppo.npz) and the oracle's autograd."""
import numpy as np
import pytest
import torch

import cld_oracle as O

pytestmark = pytest.mark.gpu
GRAD_TOL = 1e-4            # fp32 path: per-tensor relative L2 of every parameter gradient


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def cpu_sd(m):
    return {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}


@pytest.fixture()
def dm16(models_cpu):
    dm, vae, algo = models_cpu(16)
    return dm.cuda(), vae, algo


def _ppo_inputs(g):
    c = lambda k: torch.tensor(g[k]).cuda()
    return c("x1"), c("x0"), c("cond"), c("t"), c("log_p_old"), c("reward"), float(g["baseline"]), float(g["clip"])


def test_train_forward_equals_inference_forward(dm16, gold):
    g = gold("ppo")
    dm, _, _ = dm16
    x1, _, cond, t, *_ = _ppo_inputs(g)
    eng = dm.train_engine(x1.shape[0])
    e_train = eng.unet_train_forward(x1, cond, t)
    e_inf = eng.unet_forward(x1, cond, t)
    assert rel(e_train, e_inf) < 1e-5          # same arithmetic; the training GroupNorm sums a group with several warps (other order)
    with torch.no_grad():
        e_or = O.unet_forward(cpu_sd(dm.model), x1.cpu(), cond.cpu(), t.cpu())
    assert rel(e_train, e_or) < 2e-5


def test_ppo_grad_vs_reference_golden(dm16, gold):
    """cld_ppo_grad (forward + log-prob + clipped surrogate + analytic backward) against the real reference's
    `dm.log_prob(...)` / surrogate / `loss.backward()`: log-probs, loss, the norm and sum of all 148 gradients, 48 sampled
    entries of each."""
    g = gold("ppo")
    dm, _, _ = dm16
    x1, x0, cond, t, lp_old, reward, baseline, clip = _ppo_inputs(g)
    names = [k for k, _ in dm.model.named_parameters()]
    assert names == [str(n) for n in g["names"]]
    loss, logp = dm.ppo_minibatch_grad(x1, x0, cond, t, lp_old, reward, baseline, clip)
    assert rel(logp, g["log_p_new"]) < 1e-5
    assert abs(float(loss) - float(g["loss"])) < 1e-5 * max(1.0, abs(float(g["loss"])))
    grads = dm._flat_views[1]
    worst = 0.0
    for i, (k, gr) in enumerate(zip(names, grads)):
        gn, want = gr.double().norm().item(), float(g["grad_norm"][i])
        assert abs(gn - want) <= 2e-4 * want + 1e-12, (k, gn, want)
        samp = gr.reshape(-1)[torch.tensor(g["grad_idx"][i]).cuda()].cpu().double()
        err = (samp - torch.tensor(g["grad_samples"][i]).double()).abs().max().item()
        assert err <= 2e-4 * want, (k, err, want)                     # a sampled entry against the tensor's own norm
        worst = max(worst, abs(gn - want) / want)
    print("ppo gradients vs reference: worst norm deviation %.2e" % worst)


def test_backward_vs_oracle_autograd_every_tensor(dm16):
    """Random d_eps, per-row t: every parameter gradient and dx against torch autograd on the oracle's U-Net (relative L2)."""
    dm, _, _ = dm16
    torch.manual_seed(5)
    R = 10
    x, cond = torch.randn(R, 52, 4), torch.randn(R, 256)
    t = torch.randint(0, 16, (R,))
    d_eps = torch.randn(R, 52, 4)
    sd = {k: v.requires_grad_(True) for k, v in cpu_sd(dm.model).items()}
    xg = x.clone().requires_grad_(True)
    want = torch.autograd.grad((O.unet_forward(sd, xg, cond, t) * d_eps).sum(), list(sd.values()) + [xg])
    eng = dm.train_engine(R)
    eng.unet_train_forward(x.cuda(), cond.cuda(), t.cuda())
    grads = [torch.empty_like(p) for p in dm.model.parameters()]
    dx = eng.unet_backward(d_eps.cuda(), grads, want_dx=True)
    names = list(sd.keys())
    errs = {k: rel(gr, w) for k, gr, w in zip(names, grads, want[:-1])}
    bad = {k: v for k, v in errs.items() if not v < GRAD_TOL}
    assert not bad, bad
    assert rel(dx, want[-1]) < GRAD_TOL
    print("worst parameter-gradient rel %.2e (%s), dx rel %.2e" % (max(errs.values()), max(errs, key=errs.get), rel(dx, want[-1])))


def test_tf32_tensor_core_mode_vs_oracle(models_cpu):
    """train_precision = "tf32": the stride-1 convolutions of the forward and of the data gradient run as tcgen05 kind::tf32 GEMMs
    fed by 3-D TMA boxes of the fp32 activations (csrc/train_tc.cu).  10-bit mantissa products: 1e-2 budget (measured ~1e-3)."""
    dm, _, _ = models_cpu(16)
    dm = dm.cuda()
    dm.train_precision = "tf32"
    for R in (10, 37):                              # 37 rows: partial last box at every level (2, 4 and 9 rows per box)
        torch.manual_seed(5 + R)
        x, cond = torch.randn(R, 52, 4), torch.randn(R, 256)
        t = torch.randint(0, 16, (R,))
        d_eps = torch.randn(R, 52, 4)
        sd = {k: v.requires_grad_(True) for k, v in cpu_sd(dm.model).items()}
        xg = x.clone().requires_grad_(True)
        eps_want = O.unet_forward(sd, xg, cond, t)
        want = torch.autograd.grad((eps_want * d_eps).sum(), list(sd.values()) + [xg])
        eng = dm.train_engine(R)
        eps = eng.unet_train_forward(x.cuda(), cond.cuda(), t.cuda())
        grads = [torch.empty_like(p) for p in dm.model.parameters()]
        dx = eng.unet_backward(d_eps.cuda(), grads, want_dx=True)
        e_eps = rel(eps, eps_want.detach())
        errs = {k: rel(gr, w) for k, gr, w in zip(sd.keys(), grads, want[:-1])}
        print("tf32 mode R=%d: rel(eps) %.2e, worst gradient rel %.2e (%s), dx %.2e" %
              (R, e_eps, max(errs.values()), max(errs, key=errs.get), rel(dx, want[-1])))
        assert e_eps < 1e-2
        assert max(errs.values()) < 1e-2, {k: v for k, v in errs.items() if v >= 1e-2}
        assert rel(dx, want[-1]) < 1e-2
    # the fp32 mode is untouched by the switch
    dm.train_precision = "fp32"
    eng = dm.train_engine(10)
    e32 = eng.unet_train_forward(x[:10].cuda(), cond[:10].cuda(), t[:10].cuda())
    assert rel(e32, eps_want.detach()[:10]) < 2e-5


def test_backward_single_row_and_tf32_horizon_104(models_cpu):
    """Edge shapes: ONE row in fp32 mode (every GEMM has a single partial tile; the tensor-pipe weight gradient needs whole boxes and
    falls back per layer), and T = 104 on the tensor pipe (boxes of 1 / 2 / 4 rows)."""
    from cld_b200 import default_algo_config
    from cld_b200.dm_model import DmModel
    for T, R, mode, tol in ((52, 1, "fp32", GRAD_TOL), (52, 3, "tf32", 1e-2), (104, 9, "tf32", 1e-2)):
        algo = default_algo_config(horizon=T)
        torch.manual_seed(0)
        dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=16).cuda()
        dm.train_precision = mode
        torch.manual_seed(60 + R)
        x, cond, t, d_eps = torch.randn(R, T, 4), torch.randn(R, 256), torch.randint(0, 16, (R,)), torch.randn(R, T, 4)
        sd = {k: v.requires_grad_(True) for k, v in cpu_sd(dm.model).items()}
        want = torch.autograd.grad((O.unet_forward(sd, x, cond, t) * d_eps).sum(), list(sd.values()))
        eng = dm.train_engine(R)
        eng.unet_train_forward(x.cuda(), cond.cuda(), t.cuda())
        grads = [torch.empty_like(p) for p in dm.model.parameters()]
        eng.unet_backward(d_eps.cuda(), grads)
        worst = max(rel(gr, w) for gr, w in zip(grads, want))
        assert worst < tol, (T, R, mode, worst)


def test_backward_horizon_104(models_cpu):
    """cfg3's horizon: T = 104 (levels of 104 / 52 / 26 slots)."""
    from cld_b200 import default_algo_config
    from cld_b200.dm_model import DmModel
    algo = default_algo_config(horizon=104)
    torch.manual_seed(0)
    dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=16).cuda()
    torch.manual_seed(6)
    R = 5
    x, cond, t, d_eps = torch.randn(R, 104, 4), torch.randn(R, 256), torch.randint(0, 16, (R,)), torch.randn(R, 104, 4)
    sd = {k: v.requires_grad_(True) for k, v in cpu_sd(dm.model).items()}
    want = torch.autograd.grad((O.unet_forward(sd, x, cond, t) * d_eps).sum(), list(sd.values()))
    eng = dm.train_engine(R)
    eng.unet_train_forward(x.cuda(), cond.cuda(), t.cuda())
    grads = [torch.empty_like(p) for p in dm.model.parameters()]
    eng.unet_backward(d_eps.cuda(), grads)
    worst = max(rel(gr, w) for gr, w in zip(grads, want))
    assert worst < GRAD_TOL, worst


def test_backward_is_bit_reproducible_and_guards_stale_stash(dm16, gold):
    g = gold("ppo")
    dm, _, _ = dm16
    x1, x0, cond, t, lp_old, reward, baseline, clip = _ppo_inputs(g)
    dm.ppo_minibatch_grad(x1, x0, cond, t, lp_old, reward, baseline, clip)
    a = dm._flat_grad.clone()
    dm.ppo_minibatch_grad(x1, x0, cond, t, lp_old, reward, baseline, clip)
    assert torch.equal(a, dm._flat_grad)                    # no atomics: fixed reduction order
    eng = dm.train_engine(x1.shape[0])
    eng.unet_train_forward(x1, cond, t)
    eng.unet_forward(x1, cond, t)                           # overwrites the time / cond bias buffers the backward reads
    with pytest.raises(RuntimeError, match="cld_unet_backward"):
        eng.unet_backward(torch.zeros_like(x1), [torch.empty_like(p) for p in dm.model.parameters()])


def test_reference_lines_through_autograd_and_fused_step_agree(models_cpu, gold):
    """(a) the reference's own update lines (log_prob -> surrogate -> loss.backward() -> torch.optim.Adam.step()) with
    DmModel.log_prob as an autograd node, (b) the fused path (cld_ppo_grad + cld_adam_step): both reproduce the parameter
    UPDATE of the real reference's Adam step (48 sampled entries per tensor)."""
    g = gold("ppo")
    from cld_b200.trainer import FusedAdam
    lr, wd = float(g["lr"]), float(g["weight_decay"])
    deltas = []
    for fused in (False, True):
        dm, _, _ = models_cpu(16)
        dm = dm.cuda()
        x1, x0, cond, t, lp_old, reward, baseline, clip = _ppo_inputs(g)
        before = [p.detach().clone() for p in dm.model.parameters()]
        for p in dm.model.parameters():
            p.requires_grad_(True)
        if fused:
            opt = FusedAdam(dm, lr=lr, weight_decay=wd)
            dm.ppo_minibatch_grad(x1, x0, cond, t, lp_old, reward, baseline, clip)
            opt.step()
        else:
            opt = torch.optim.Adam(dm.model.parameters(), lr=lr, weight_decay=wd)
            advantage = reward - baseline
            log_p_new = dm.log_prob(x1, x0, {'cond_feat': cond}, t=t)
            ratios = torch.exp(log_p_new - lp_old)
            loss = -torch.min(ratios * advantage, torch.clamp(ratios, 1 - clip, 1 + clip) * advantage).mean()
            opt.zero_grad()
            loss.backward()
            opt.step()
            assert abs(float(loss.detach()) - float(g["loss"])) < 1e-5
        deltas.append([(p.detach() - b) for p, b in zip(dm.model.parameters(), before)])
        # the first Adam step moves every entry by ~lr * sign(g): compare against the reference where |g| is not at the noise floor
        n_checked = 0
        for i, d in enumerate(deltas[-1]):
            idx = torch.tensor(g["grad_idx"][i]).cuda()
            want = torch.tensor(g["delta_samples"][i]).cuda()
            gs = torch.tensor(g["grad_samples"][i]).cuda().abs()
            ok = gs > 1e-3 * float(g["grad_norm"][i]) / max(1.0, d.numel() ** 0.5)
            got = d.reshape(-1)[idx]
            assert (got[ok] - want[ok]).abs().max().item() <= 2e-2 * lr if ok.any() else True
            n_checked += int(ok.sum())
        assert n_checked > 1000
        # the sampling engine sees the updated weights
        eps_new = dm.denoise(x1, {'cond_feat': cond}, t)
        with torch.no_grad():
            want_eps = O.unet_forward(cpu_sd(dm.model), x1.cpu(), cond.cpu(), t.cpu())
        assert rel(eps_new, want_eps) < 2e-5
        # ... and so does the training engine (re-load of a loaded handle = the fused one-launch re-pack), in both weight layouts
        teng = dm.train_engine(x1.shape[0])
        assert rel(teng.unet_forward(x1, cond, t), want_eps) < 2e-5
        dm.train_precision = "tf32"
        assert rel(dm.train_engine(x1.shape[0]).unet_train_forward(x1, cond, t), want_eps) < 1e-2
        dm.train_precision = "fp32"
    # autograd node + torch Adam  ==  fused kernels.  The first Adam step is -lr g / (|g| + 1e-8): where |g| is near 1e-8 the last bits
    # of g (d_eps from torch's elementwise autograd vs the head kernel) move the update; measured 1.9e-3 of the update's norm
    worst = max(rel(a, b) for a, b in zip(*deltas))
    assert worst < 1e-2, worst


def test_compute_losses_mse_vs_reference_golden(dm16, gold):
    g = gold("ppo")
    dm, _, _ = dm16
    for p in dm.model.parameters():
        p.requires_grad_(True)
    z0, tq, nz, cond = (torch.tensor(g[k]).cuda() for k in ("z0", "tq", "nz", "cond"))
    loss = dm.compute_losses({'cond_feat': cond}, z0, t=tq, noise=nz)
    assert abs(float(loss) - float(g["mse"])) < 1e-5 * float(g["mse"])
    loss.backward()
    for i, p in enumerate(dm.model.parameters()):
        want = float(g["mse_grad_norm"][i])
        assert abs(p.grad.double().norm().item() - want) <= 2e-4 * want + 1e-12
    # the fused head gives the same loss and d_eps
    eng = dm.train_engine(z0.shape[0])
    eps = eng.unet_forward(dm.q_sample(z0, tq, nz), cond, tq)
    l2, d_eps = eng.mse_head(eps, nz)
    assert abs(float(l2) - float(g["mse"])) < 1e-5 * float(g["mse"])
    assert rel(d_eps, 2 * (eps - nz) / eps.numel()) < 1e-6


def test_graph_replay_equals_eager_updates(models_cpu, gold):
    """GraphedPPOStep (the update captured as a CUDA graph: two streams inside, device-side baseline / lr / step) reproduces the
    parameters of the same sequence of un-captured updates bit for bit (tests/ppo_cases.py; six updates of the golden minibatch)."""
    from ppo_cases import assert_graph_replay_equals_eager
    x1, x0, cond, t, lp_old, reward, baseline, clip = _ppo_inputs(gold("ppo"))
    assert_graph_replay_equals_eager(lambda: models_cpu(16)[0].cuda(), x1, x0, cond, t, lp_old, reward, baseline, clip, iters=6)


def test_ppo_minibatch_odd_rows_vs_float64_oracle(dm16):
    """cld_ppo_grad on a training arena carved for 37 rows: a row count that is not a multiple of 4 must leave every arena buffer
    16-byte aligned (the head's d_eps feeds float4 loads of the output convolution's backward).  log_p_new, loss and all 148 gradients
    against O.ppo_grads in float64 (fp32 mode)."""
    from ppo_cases import clip_regions, ppo_case, ppo_oracle
    dm, _, _ = dm16
    R, baseline, clip = 37, 0.05, 0.2
    sd64 = {k: v.detach().cpu().double() for k, v in dm.model.state_dict().items()}
    sched = {k: v.detach().cpu().double() for k, v in dm.named_buffers()}
    case = ppo_case(sched, sd64, R, 37)
    loss_want, lp_want, g_want = ppo_oracle(sd64, sched, *case, baseline, clip)
    inside, cut = clip_regions(lp_want, case[4], case[5], baseline, clip)
    assert inside.any() and cut.any()
    loss, lp = dm.ppo_minibatch_grad(*(v.cuda() for v in case[:4]), case[4].cuda(), case[5].cuda(), baseline, clip)
    assert rel(lp, lp_want) < 1e-5
    assert abs(float(loss) - loss_want) < 1e-5 * max(1.0, abs(loss_want))
    errs = {k: rel(g, w) for k, g, w in zip(dm.model.state_dict(), dm._flat_views[1], g_want)}
    bad = {k: v for k, v in errs.items() if not v < GRAD_TOL}
    assert not bad, bad
    print("R=37 fp32 PPO minibatch: log_p_new rel %.2e, worst gradient %.2e" % (rel(lp, lp_want), max(errs.values())))


def test_adam_kernel_vs_torch(dm16):
    dm, _, _ = dm16
    eng = dm.train_engine(1)
    torch.manual_seed(3)
    n = 100_003
    p = torch.randn(n, device="cuda")
    ref = p.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=3e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    for step in range(1, 6):
        gr = torch.randn(n, device="cuda") * (10.0 ** float(torch.randint(-3, 2, (1,))))
        ref.grad = gr.clone()
        opt.step()
        eng.adam_step(p, gr, m, v, step, 3e-4, (0.9, 0.999), 1e-8, 1e-2)
        assert (p - ref.detach()).abs().max().item() < 1e-6          # a few ulp of |p| <= 4
    st = opt.state[ref]
    assert rel(m, st['exp_avg']) < 1e-6 and rel(v, st['exp_avg_sq']) < 1e-6


def test_trainer_ppo_update_loop(models_cpu):
    """GuideDMTrainer (mirror of guide_dm_trainer.py:85-183): sampling steps fill the device replay buffer, ppo_update runs its
    minibatches in both modes.  PPO evaluates log_prob at t = 0 where sigma = 1e-10 (oracle/make_golden.py:ppo_golden): an fp32
    rounding difference of the posterior mean (fused multiply-add or not) moves log_p_new by 1e5, so ratios are 0, 1 or inf
    depending on the last bit -- in the reference as well.  Values of the two modes are therefore NOT comparable here (their
    agreement is asserted at well-conditioned steps in test_reference_lines_through_autograd_and_fused_step_agree); this test
    checks the loop itself: buffer contents, update cadence, finite parameters, engine refresh."""
    from cld_b200 import default_algo_config, make_scenes
    from cld_b200.dm_model import DmModel
    from cld_b200.trainer import GuideDMTrainer
    from cld_b200.vae import VaeModel
    results = []
    for fused in (True, False):
        algo = default_algo_config(num_samp=2, ppo_mini_batch=16, ppo_update_times=2, update_interval=2)
        torch.manual_seed(0)
        dm = DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=16).cuda()
        vae = VaeModel(algo).cuda().bind(dm)
        aux, batch = make_scenes(2, 4, seed=3, dense=True)
        batch = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in batch.items()}
        aux = {k: v.cuda() for k, v in aux.items()}
        gen = torch.Generator(device="cuda").manual_seed(11)
        tr = GuideDMTrainer(dm, vae, algo, batch_size=8, learning_rate=1e-4, weight_decay=1e-5, fused=fused, ppo_epochs=2,
                            sample_kw=dict(use_device_rng=True, seed=77), generator=gen)
        for _ in range(2):
            out = tr.training_step(batch, aux)
        assert out['traj'].shape == (8, 2, 52, 2) and len(tr.replay_buffer) == 32
        assert 'train/ppo_loss' in tr.log and tr.steps_since_update == 0
        tr.on_epoch_end()
        results.append((tr.log['train/ppo_loss'], torch.cat([p.detach().reshape(-1) for p in dm.model.parameters()]).clone()))
        p_now = results[-1][1]
        assert torch.isfinite(p_now).all()
        torch.manual_seed(0)
        p_init = torch.cat([p.detach().reshape(-1) for p in DmModel(algo, {"image": (34, 224, 224)}, n_timesteps=16).model.parameters()])
        moved = (p_now.cpu() - p_init).abs().max().item()
        assert 0 < moved <= 4 * 3.2e-4                     # 2 epochs x 2 minibatches; an Adam step moves an entry by <= lr (1 - b1) / sqrt(1 - b2)
        # the sampler picks up the updated weights (engine re-packed from the changed parameters)
        out2 = dm(batch, aux, algo, use_device_rng=True, seed=77)
        assert torch.isfinite(out2['pred_traj']).all()
