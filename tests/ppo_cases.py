"""PPO minibatch inputs with a float64 reference, and the graph-replay-versus-eager comparison of the PPO update, shared by the
training tests (test_gpu_train.py at minibatch sizes, test_gpu_train_large.py at large batches)."""
import torch

import cld_oracle as O

CHUNK = 256                     # rows per float64 autograd graph (~1.4 GB of host memory)


def ppo_case(sched, sd64, R, seed, T=52, n_t=16, clip=0.2):
    """Inputs of one PPO minibatch -> (x1, x0, cond, t, log_p_old, reward), all float32 on the CPU.  t runs over 1 .. n_t - 1 (at t = 0
    sigma is 1e-10 and the ratios are 0 / 1 / inf).  x0 is drawn from the model's own posterior, so log-probabilities are O(1); log_p_old
    puts every third row inside the clip range (ratio 0.9 .. 1.1), above it (1.5) and below it (0.6); rewards take both signs.
    sched: the model's schedule buffers in float64."""
    g = torch.Generator().manual_seed(seed)
    x1, cond = torch.randn(R, T, 4, generator=g), torch.randn(R, 256, generator=g)
    t = torch.randint(1, n_t, (R,), generator=g)
    with torch.no_grad():
        eps = torch.cat([O.unet_forward(sd64, x1[s].double(), cond[s].double(), t[s]) for s in _chunks(R)])
    c = lambda k: sched[k][t].view(-1, 1, 1)                                      # noqa: E731
    x0 = (c("x_t_cof") * x1.double() - c("noise_cof") * eps
          + (0.5 * c("posterior_log_variance_clipped")).exp() * torch.randn(R, T, 4, generator=g, dtype=torch.float64)).float()
    with torch.no_grad():
        lp_new = torch.cat([O.log_prob(sd64, sched, x1[s].double(), x0[s].double(), cond[s].double(), t[s]) for s in _chunks(R)])
    kind = torch.arange(R) % 3
    ratio = torch.where(kind == 0, 0.9 + 0.2 * torch.rand(R, generator=g, dtype=torch.float64),
                        torch.where(kind == 1, torch.full((R,), 1.5, dtype=torch.float64), torch.full((R,), 0.6, dtype=torch.float64)))
    lp_old = (lp_new - ratio.log()).float()
    reward = torch.randn(R, generator=g)
    return x1, x0, cond, t, lp_old, reward


def ppo_oracle(sd64, sched, x1, x0, cond, t, lp_old, reward, baseline, clip=0.2):
    """O.ppo_grads in float64, in row chunks -> (loss, log_p_new [R], [gradients]).  The loss is a mean over rows, so chunk c
    contributes n_c / R of its own mean and of its own gradients."""
    R = x1.shape[0]
    loss, lps, grads = 0.0, [], None
    for s in _chunks(R):
        n = x1[s].shape[0]
        l, lp, gr = O.ppo_grads(sd64, sched, x1[s].double(), x0[s].double(), cond[s].double(), t[s], lp_old[s].double(),
                                reward[s].double(), baseline, clip)
        loss += float(l) * n / R
        lps.append(lp)
        gr = [v * (n / R) for v in gr.values()]
        grads = gr if grads is None else [a + b for a, b in zip(grads, gr)]
    return loss, torch.cat(lps), grads


def clip_regions(lp_want, lp_old, reward, baseline, clip=0.2):
    """-> (inside, cut): rows whose ratio lies in the clip range, and rows that the clipped minimum cuts off (no gradient)."""
    ratio, adv = (lp_want - lp_old.double()).exp(), reward.double() - baseline
    inside = (ratio >= 1 - clip) & (ratio <= 1 + clip)
    cut = ((ratio > 1 + clip) & (adv > 0)) | ((ratio < 1 - clip) & (adv < 0))
    return inside, cut


def assert_graph_replay_equals_eager(make_dm, x1, x0, cond, t, lp_old, reward, baseline, clip, iters):
    """GraphedPPOStep (the update captured as a CUDA graph: two streams inside, device-side baseline / lr / step) reproduces the
    losses and parameters of the same sequence of un-captured updates bit for bit.  `make_dm()` -> a fresh CUDA DmModel (same seed
    every call).  Every iteration sees a different minibatch; the baseline changes after three updates, the learning rate after
    four.  The first two calls of GraphedPPOStep run eagerly, the rest are graph replays."""
    from cld_b200.trainer import FusedAdam, GraphedPPOStep
    x1, x0, cond, t, lp_old, reward = (v.cuda() for v in (x1, x0, cond, t, lp_old, reward))
    finals = []
    for use_graph in (False, True):
        dm = make_dm()
        try:
            dm.train_precision = "tf32"
            for p in dm.model.parameters():
                p.requires_grad_(True)
            opt = FusedAdam(dm, lr=1e-4, weight_decay=1e-5)
            gs = GraphedPPOStep(dm, opt, x1.shape[0], clip) if use_graph else None
            losses = []
            for it in range(iters):
                xs = x1 + 0.01 * it
                base = baseline + 0.1 * (it // 3)
                opt.lr = 1e-4 * (1.0 if it < 4 else 0.5)
                if use_graph:
                    for dst, src in zip(gs.buffers(), (x0, xs, lp_old, reward, cond)):
                        dst.copy_(src)
                    losses.append(float(gs(base, t)))
                else:
                    loss, _ = dm.ppo_minibatch_grad(xs, x0, cond, t, lp_old, reward, base, clip)
                    opt.step()
                    losses.append(float(loss))
            assert opt.step_count == iters
            if use_graph:
                assert gs.graph is not None                                       # the updates after the first two were replays
            finals.append((losses, dm._flat.clone()))
        finally:
            if dm._train_eng is not None:
                dm._train_eng.close()
                dm._train_eng = None
            del dm
            torch.cuda.empty_cache()
    assert finals[0][0] == finals[1][0], (finals[0][0], finals[1][0])
    assert torch.equal(finals[0][1], finals[1][1])


def _chunks(R):
    return [slice(lo, lo + CHUNK) for lo in range(0, R, CHUNK)]
