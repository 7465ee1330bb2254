"""Oracle of the multi-iteration guidance update: PerturbationGuidance.perturb (guidance_loss.py:2221-2282) with
`grad_steps` > 1, and the guided sampler on top of it.

    opt = Adam([z], lr)            # or SGD; a fresh optimizer for each perturb call
    for _ in range(grad_steps):
        L = losses(transform(decoder(z)))
        L.backward(); opt.step()
    return z, guide_losses         # the losses of the last iteration

The single iteration is `cld_oracle.guidance_grad` + `apply_guidance_update`, pinned to the reference's outputs by the
goldens; the loop around it is restated here (there is no reference run with grad_steps > 1 to pin it to).  Scenes are
independent and Adam is elementwise, so one optimizer per scene equals the reference's one perturb call per scene."""
import torch

import cld_oracle as O


def guidance_perturb(dec_sd, z, cond, curr, batch, agents_per_scene, num_samp, g=O.DEFAULT_GUIDANCE):
    """z [R,T,4] (R = S*A*N), cond / curr per agent -> (z' [R,T,4], gradient of the last iteration [R,T,4], per-scene dicts of
    the last iteration's per-term losses, as `cld_oracle.guidance_grad` returns them)."""
    A, N = agents_per_scene, num_samp
    R = z.shape[0]
    S = R // (A * N)
    steps = max(1, int(g.get("grad_steps", 1)))
    rep = lambda v: v.repeat_interleave(N, dim=0)                             # noqa: E731
    outs, grads, losses = [], [], []
    for s in range(S):
        r0, r1 = s * A * N, (s + 1) * A * N
        scene = O.slice_scene(batch, s * A, (s + 1) * A)
        c, cu = rep(cond[s * A:(s + 1) * A]), rep(curr[s * A:(s + 1) * A])
        p = z[r0:r1].detach().clone().requires_grad_()
        opt = torch.optim.Adam([p], lr=g["lr"]) if g["optimizer"] == "adam" else torch.optim.SGD([p], lr=g["lr"])
        for _ in range(steps):
            with torch.enable_grad():
                x6, _ = O.decode_rollout(dec_sd, p, c, cu)
                tot, per = O.guidance_loss_scene(x6.reshape(A, N, x6.shape[1], 6), scene, g)
                grad = None
                if tot.requires_grad:
                    grad = torch.autograd.grad(tot, p, allow_unused=True)[0]
                if grad is None:
                    grad = torch.zeros_like(p)
            # a zero gradient still counts as a step (the optimizer's step counter and the moments advance)
            p.grad = grad.clone()
            opt.step()
        outs.append(p.detach())
        grads.append(grad.detach())
        losses.append(per)
    return torch.cat(outs, 0), torch.cat(grads, 0), losses


def sample(unet_sd, sched, cond_rows, x_init, noises, n_timesteps, stride=1, sampler="ddpm", guidance=None):
    """`cld_oracle.sample` whose guided steps run `guidance_perturb` (guidance['cfg']['grad_steps'] iterations).  With one
    iteration it is `cld_oracle.sample` itself."""
    if guidance is None or int(guidance["cfg"].get("grad_steps", 1)) <= 1:
        return O.sample(unet_sd, sched, cond_rows, x_init, noises, n_timesteps, stride, sampler, guidance=guidance)
    steps = O.step_indices(n_timesteps, stride)
    x = x_init.clone()
    R = x.shape[0]
    gd = guidance
    x0 = None
    for k, i in enumerate(steps):
        t = torch.full((R,), i, dtype=torch.long)
        eps = O.unet_forward(unet_sd, x, cond_rows, t)
        i_next = steps[k + 1] if k + 1 < len(steps) else -1
        if sampler == "ddpm":
            mean, sigma = O.ddpm_mean_sigma(sched, x, eps, i)
        else:
            mean = O.ddim_next(sched, x, eps, i, i_next)
        if i != 0:
            mean, _, _ = guidance_perturb(gd["dec_sd"], mean, gd["cond"], gd["curr"], gd["batch"], gd["A"], gd["N"], gd["cfg"])
        x = mean + sigma * noises[k] if (sampler == "ddpm" and i != 0) else mean
        if i == 0:
            x0 = x.clone()
    return {"pred_traj": x0}
