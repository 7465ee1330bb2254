"""GPU (-m gpu): cld_load_unet -- a re-load equals a fresh load, an fp32 load is one launch, a rejected load changes nothing."""
import pytest
import torch

from cld_b200.engine import Engine, default_guidance
from cld_b200.synthetic import make_scenes

pytestmark = pytest.mark.gpu
S, A = 2, 4
R = S * A


def perturbed(sd, seed):
    g = torch.Generator().manual_seed(seed)
    return {k: v + 0.02 * torch.randn(v.shape, generator=g).to(v.device) for k, v in sd.items()}


def wrong_numel(sd, i):
    """`sd` with one element appended to its i-th tensor."""
    k = list(sd)[i]
    return dict(sd, **{k: torch.cat([sd[k].flatten(), sd[k].new_zeros(1)])})


def inputs():
    torch.manual_seed(3)
    x, cond, t = torch.randn(R, 52, 4).cuda(), torch.randn(R, 256).cuda(), torch.randint(0, 10, (R,)).cuda()
    aux, batch = make_scenes(S, A, seed=12, dense=True)
    return x, cond, t, aux, batch


def outputs(eng, x, cond, t, aux, batch):
    eps = eng.unet_forward(x, cond, t)
    out = eng.sample(x, aux["cond_feat"].cuda(), curr_rows=aux["curr_states"].cuda(), scene=eng.make_scene(batch, S, A, 1),
                     guidance=default_guidance(), sampler="ddim", stride=5, want_traj=True)
    return eps, out["x0"], out["traj"]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_reload_equals_fresh_load(models_cpu, precision):
    """W1 then W2 on one handle (a guided sample in between fills the time-bias table with W1) and W2 on a fresh handle: the
    denoiser and a guided sample agree bit for bit."""
    dm, vae, _ = models_cpu(10, precision=precision)
    dm = dm.cuda()
    vae.bind(dm)
    args = inputs()
    eng = dm._build_engine(R, dm.betas.device)                  # W1
    w1 = outputs(eng, *args)
    w2 = perturbed(dm.model.state_dict(), 1)
    eng.load_unet(w2)
    dm.model.load_state_dict(w2)
    fresh = dm._build_engine(R, dm.betas.device)                # W2 only
    reloaded, want = outputs(eng, *args), outputs(fresh, *args)
    assert not torch.equal(w1[0], want[0])
    for a, b in zip(reloaded, want):
        assert torch.equal(a, b)


def test_fp32_load_is_one_launch(models_cpu):
    dm, _, _ = models_cpu(10)
    eng = Engine(n_timesteps=10, max_rows=R)
    for sd in (dm.model.state_dict(), perturbed(dm.model.state_dict(), 2)):      # first load, re-load
        n0 = eng.launch_count()
        eng.load_unet(sd)
        assert eng.launch_count() == n0 + 1


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_rejected_reload_keeps_weights(models_cpu, precision):
    dm, _, _ = models_cpu(10, precision=precision)
    dm = dm.cuda()
    x, cond, t, _, _ = inputs()
    eng = dm.engine(R)
    before = eng.unet_forward(x, cond, t)
    with pytest.raises(RuntimeError, match="tensor 37 has"):
        eng.load_unet(wrong_numel(perturbed(dm.model.state_dict(), 3), 37))
    assert torch.equal(eng.unet_forward(x, cond, t), before)


def test_rejected_first_load_leaves_handle_usable(models_cpu):
    """A first load that fails its argument check, then the decoder load and a guidance step: as on a clean handle."""
    dm, vae, _ = models_cpu(10)
    z, cond, t, aux, batch = inputs()
    dec = {k: v.detach().cuda() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}
    sd = dm.model.state_dict()
    res = []
    for bad_first in (True, False):
        eng = Engine(n_timesteps=10, max_rows=R)
        if bad_first:
            with pytest.raises(RuntimeError, match="tensor 60 has"):
                eng.load_unet(wrong_numel(sd, 60))
        eng.load_decoder(dec)
        out = eng.guidance_step(z, cond, aux["curr_states"].cuda(), eng.make_scene(batch, S, A, 1), default_guidance())
        eng.load_unet(sd)
        res.append(out + (eng.unet_forward(z, cond, t),))
    for a, b in zip(*res):
        assert torch.equal(a, b)


def test_bf16_reload_invalidates_training_stash(models_cpu):
    """unet_train_forward, then a weight load, then unet_backward: refused (the stash belongs to the old weights)."""
    dm, _, _ = models_cpu(10, precision="bf16")
    dm = dm.cuda()
    x, cond, t, _, _ = inputs()
    eng = dm.engine(R)
    eng.unet_train_forward(x, cond, t)
    eng.load_unet(perturbed(dm.model.state_dict(), 4))
    with pytest.raises(RuntimeError, match="cld_unet_backward"):
        eng.unet_backward(torch.zeros_like(x), [torch.empty_like(p) for p in dm.model.parameters()])
