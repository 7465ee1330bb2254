"""CPU: guidance with several optimizer iterations per guided step (`grad_steps`): the oracle's loop, the guidance-dict
validation and the C struct layout of `CldGuidanceConfig.grad_steps`."""
import ctypes
import os
import subprocess

import pytest
import torch

import cld_oracle as O
from cld_b200.synthetic import make_scenes
from perturb_oracle import guidance_perturb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _case(models_cpu, S=3, A=4, N=2, seed=71):
    _, vae, _ = models_cpu(10)
    dec_sd = {k: v.detach().clone() for k, v in vae.lstmvae.lstm_dec.state_dict().items()}
    aux, batch = make_scenes(S, A, seed=seed, dense=True)
    torch.manual_seed(seed + 1)
    batch["target_speed"] = (aux["curr_states"][:, 2:3] + torch.randn(S * A, 1)).clamp(min=0).repeat(1, 52)
    z = torch.randn(S * A * N, 52, 4)
    return dec_sd, aux, batch, z


def _cfg(**kw):
    return dict(O.DEFAULT_GUIDANCE, target_pos=1.0, target_speed=0.5, acc_limit=1.0, acc_limit_value=1.0, speed_limit=1.0,
                speed_limit_value=3.0, **kw)


@pytest.mark.parametrize("optimizer", ["adam", "sgd"])
def test_one_iteration_is_the_pinned_single_update(models_cpu, optimizer):
    dec_sd, aux, batch, z = _case(models_cpu)
    g = _cfg(optimizer=optimizer, lr=0.3 if optimizer == "adam" else 1.0, grad_steps=1)
    zp, gp, lp = guidance_perturb(dec_sd, z, aux["cond_feat"], aux["curr_states"], batch, 4, 2, g)
    g1, l1 = O.guidance_grad(dec_sd, z, aux["cond_feat"], aux["curr_states"], batch, 4, 2, g)
    assert torch.equal(gp, g1)
    assert torch.equal(zp, O.apply_guidance_update(z, g1, g))
    for a, b in zip(lp, l1):
        assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)


@pytest.mark.parametrize("optimizer", ["adam", "sgd"])
def test_three_iterations_equal_a_hand_unrolled_loop(models_cpu, optimizer):
    dec_sd, aux, batch, z = _case(models_cpu)
    lr = 0.3 if optimizer == "adam" else 1.0
    g = _cfg(optimizer=optimizer, lr=lr, grad_steps=3)
    zp, gp, lp = guidance_perturb(dec_sd, z, aux["cond_feat"], aux["curr_states"], batch, 4, 2, g)
    zh, m, v = z.clone(), torch.zeros_like(z, dtype=torch.float64), torch.zeros_like(z, dtype=torch.float64)
    for step in range(1, 4):
        grad, per = O.guidance_grad(dec_sd, zh, aux["cond_feat"], aux["curr_states"], batch, 4, 2, g)
        if optimizer == "adam":
            zd, m, v = O.adam_update(zh, grad, m, v, step, lr)
        else:
            zd = zh.double() - lr * grad.double()
        zh = zd.float()               # the loop's z is fp32: the next gradient is evaluated where perturb evaluates it
    # Adam normalises every element: a one-ulp difference of z after iteration 1 (fp32 optimizer vs float64 restatement) moves
    # an element's tiny fp32 gradient by its rounding noise (~1e-5 relative), and the next step turns that into ~lr * 1e-5.
    # So the whole tensor is compared to 1e-6 relative, each element to 1e-5.
    d = (zp - zh).abs().max().item()
    r = ((zp - zh).double().norm() / zh.double().norm()).item()
    print("grad_steps=3 %s: max |dz| %.3e, rel %.3e" % (optimizer, d, r))
    assert r < 1e-6 and d < 1e-5
    assert ((gp - grad).double().norm() / grad.double().norm()).item() < 1e-6
    for a, b in zip(lp, per):
        assert all((a[k] - b[k]).abs().max().item() < 1e-6 for k in a)
    assert not torch.equal(zp, O.apply_guidance_update(z, O.guidance_grad(dec_sd, z, aux["cond_feat"], aux["curr_states"],
                                                                            batch, 4, 2, g)[0], g))


def test_make_guidance_grad_steps():
    from cld_b200.engine import Engine, default_guidance
    assert default_guidance()["grad_steps"] == 1
    assert Engine.make_guidance(default_guidance()).grad_steps == 1
    assert Engine.make_guidance({}).grad_steps == 1
    assert Engine.make_guidance(default_guidance(grad_steps=4)).grad_steps == 4
    for bad in (0, -1, 2.5, True, "3", None):
        with pytest.raises(ValueError, match="grad_steps"):
            Engine.make_guidance(default_guidance(grad_steps=bad))


def test_guidance_config_struct_matches_the_header(tmp_path):
    from cld_b200._lib import CldGuidanceConfig
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "cld_b200.h"\n'
                   'int main(void) { printf("%zu %zu\\n", sizeof(CldGuidanceConfig), offsetof(CldGuidanceConfig, grad_steps)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    size, off = (int(v) for v in subprocess.check_output([str(exe)]).split())
    assert size == ctypes.sizeof(CldGuidanceConfig)
    assert off == CldGuidanceConfig.grad_steps.offset
    assert off == size - 4                     # appended as the last field: older callers' prefix is unchanged
