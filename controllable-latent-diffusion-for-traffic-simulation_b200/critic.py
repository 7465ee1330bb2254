"""Drop-ins for models/rl/criticmodel.py on the sampling path: failure_rate_compute, compute_reward."""
import torch


@torch.no_grad()
def indicators(dm, state_action, batch, num_samp=1):
    """Per-row indicators: offroad [R,T] bool, collision counts [R], reward [R].  Scenes may differ in size (`scene_index`): the
    batch is evaluated in one call either way."""
    from .keys import scene_sizes
    R = state_action.shape[0]
    x = state_action
    if x.shape[-1] < 6:
        x = torch.cat([x, x.new_zeros(*x.shape[:-1], 6 - x.shape[-1])], dim=-1)
    B = R // num_samp
    sizes = scene_sizes(batch.get('scene_index'), B)
    eng = dm.engine(R)
    return eng.indicators(x, eng.make_scene(batch, len(sizes), sizes[0], num_samp, scene_sizes=sizes))


@torch.no_grad()
def failure_rate_compute(dm, state_action, batch):
    """criticmodel.py:114-145."""
    off, coll, _ = indicators(dm, state_action, batch, 1)
    no_off = (~off).all(dim=-1).float().mean().item()
    no_col = (coll <= 0).float().mean().item()
    o, c = 1.0 - no_off, 1.0 - no_col
    return {'offroad_failure_rate': o, 'collision_failure_rate': c, 'overall_failure_rate': (o + c) / 2.0}


@torch.no_grad()
def compute_reward(dm, state_act, batch, state_act_scaled=None):
    """criticmodel.py:7-40 with its evident [B,N,T,6] intent; returns [B*N]."""
    B, N, T, _ = state_act.shape
    _, _, rew = indicators(dm, state_act.reshape(B * N, T, -1), batch, N)
    return rew
