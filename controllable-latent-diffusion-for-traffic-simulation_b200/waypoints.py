"""Waypoint guidance (SURVEY.md sec. 8 f-4): host side of `TargetPosAtTimeLoss` (src/tbsim/utils/guidance_loss.py:630-670),
`GlobalTargetPosAtTimeLoss` (:930-1031) and `GlobalTargetPosLoss` (:1033-1135, with `compute_progress_loss` :876-927).

The reference's `forward()` is two things: host logic that turns WORLD targets into a per-agent (local target, branch) -- exact vs
progress, target time passed, `have_reached_mask` -- and one of four per-agent formulas.  The formulas and their analytic gradients are
in the guidance kernel (`CldScene.wp_*`, `CldGuidanceConfig.w_waypoint`); the classes here reproduce the host logic on device tensors and
hand the kernel its five per-agent arrays through `scene_entries()`, which is merged into the `data_batch` (`agents_per_scene`: an int, or the scene sizes of a ragged batch):

    term = GlobalTargetPosAtTime(target_pos_world, target_time, urgency, pref_speed, dt=0.1, target_tolerance=2, action_num=5)
    term.update(global_t)                                  # GuidanceLoss.update (guidance_loss.py:196-202)
    batch.update(term.scene_entries(batch, horizon=52, agents_per_scene=A))
    dm(batch, aux, algo, guidance=dict(waypoint=1.0, ...))

`have_reached` is kept per agent across calls like the reference's `have_reached_mask`.  The reference averages a term over the guided
agents only (`agt_mask`, guidance_loss.py:2159-2172): `wp_weight` = A / (guided agents of the scene) restores that under the kernel's 1 / (A N).
"""
import numbers

import torch

from .keys import scene_size_list


def _tf_points(pts, mat):
    """transform_points_tensor (geometry_utils.py:98-141) for pts [B,K,2], mat [B,3,3]."""
    return torch.einsum('bij,bkj->bki', mat[:, :2, :2], pts) + mat[:, None, :2, 2]


def _weights(mode, agents_per_scene):
    """A / (guided agents of the scene) for the guided agents, 0 for the others; agents_per_scene: an int or the scene sizes of a
    ragged batch."""
    if isinstance(agents_per_scene, numbers.Integral):
        act = (mode != 0).float().view(-1, agents_per_scene)
        k = act.sum(dim=1, keepdim=True).clamp(min=1.0)
        return (act * (agents_per_scene / k)).reshape(-1)
    sizes = torch.tensor(scene_size_list(agents_per_scene, mode.shape[0]), device=mode.device)
    seg = torch.repeat_interleave(torch.arange(sizes.numel(), device=mode.device), sizes)
    act = (mode != 0).float()
    k = torch.zeros(sizes.numel(), device=mode.device).index_add_(0, seg, act).clamp(min=1.0)   # counts: exact in any order
    return act * (k.reciprocal() * sizes.float())[seg]          # how torch evaluates the int form's `A / k`


class TargetPosAtTime:
    """guidance_loss.py:630-670: || p[target_time] - target_pos || with the target in the AGENT frame."""

    def __init__(self, target_pos, target_time, agents=None):
        self.target_pos, self.target_time = torch.as_tensor(target_pos, dtype=torch.float32), torch.as_tensor(target_time).long()
        self.agents = agents                     # optional bool mask [B] of the guided agents (the reference's `agents` list)

    def update(self, global_t=None):
        pass

    def scene_entries(self, data_batch, horizon, agents_per_scene):
        B = self.target_pos.shape[0]
        dev = self.target_pos.device
        mode = torch.ones(B, dtype=torch.long, device=dev)
        if self.agents is not None:
            mode = mode * torch.as_tensor(self.agents, device=dev).long()
        return {"wp_target": self.target_pos, "wp_mode": mode, "wp_time": self.target_time.clamp(0, horizon - 1),
                "wp_dist": torch.zeros(B, device=dev), "wp_weight": _weights(mode, agents_per_scene)}


class _GlobalTarget:
    def __init__(self, target_pos, urgency, pref_speed, dt, target_tolerance, action_num, agents):
        f = lambda v: torch.as_tensor(v, dtype=torch.float32)      # noqa: E731
        self.target_pos, self.urgency, self.pref_speed = f(target_pos), f(urgency), f(pref_speed)
        self.dt, self.target_tolerance, self.action_num, self.agents = float(dt), target_tolerance, int(action_num), agents
        self.global_t = 0
        self.have_reached = None

    def update(self, global_t=None):
        if global_t is not None:
            self.global_t = int(global_t)

    def _local(self, data_batch):
        dev = data_batch["agent_from_world"].device
        self.target_pos, self.urgency, self.pref_speed = (v.to(dev) for v in (self.target_pos, self.urgency, self.pref_speed))
        return _tf_points(self.target_pos[:, None], data_batch["agent_from_world"].float())[:, 0]

    def _finish(self, data_batch, local, mode, time, dist, agents_per_scene):
        B = mode.shape[0]
        if self.have_reached is None:
            self.have_reached = torch.zeros(B, dtype=torch.bool, device=mode.device)
        if self.target_tolerance is not None:
            # guidance_loss.py:1019-1026 / 1122-1131 as written: the OLDEST of the last `action_num` history points of every agent, and
            # the minimum over ALL agents' points (the [B,2] - [B,1,2] broadcast): an agent j near agent b's target marks b as arrived
            hist_w = _tf_points(data_batch["agent_hist"][:, -self.action_num:, :2].float(), data_batch["world_from_agent"].float())[:, 0]
            d = (hist_w[None, :, :] - self.target_pos[:, None, :]).norm(dim=-1).min(dim=-1)[0]
            self.have_reached |= d < self.target_tolerance
            mode = torch.where(self.have_reached, torch.zeros_like(mode), mode)
        if self.agents is not None:
            mode = mode * torch.as_tensor(self.agents, device=mode.device).long()
        return {"wp_target": local, "wp_mode": mode, "wp_time": time, "wp_dist": dist, "wp_weight": _weights(mode, agents_per_scene)}


class GlobalTargetPosAtTime(_GlobalTarget):
    """guidance_loss.py:930-1031: hit a WORLD waypoint at a global time step.  Within the planning horizon: the at-time distance;
    further away: relu(|| p[T-1] - g || - time_left dt pref_speed (1 - urgency)); time passed: nothing."""

    def __init__(self, target_pos, target_time, urgency, pref_speed=1.42, dt=0.1, target_tolerance=2, action_num=5, agents=None):
        super().__init__(target_pos, urgency, pref_speed, dt, target_tolerance, action_num, agents)
        self.target_time = torch.as_tensor(target_time).long()

    def scene_entries(self, data_batch, horizon, agents_per_scene):
        local = self._local(data_batch)
        ltt = self.target_time.to(local.device) - self.global_t
        exact = (ltt < horizon) & (ltt >= 0)
        prog = (~exact) & (ltt >= 0)
        zl = torch.zeros_like(ltt)
        mode = torch.where(exact, torch.ones_like(ltt), torch.where(prog, torch.full_like(ltt, 2), zl))
        dist = torch.where(prog, ltt.float() * self.dt * self.pref_speed * (1.0 - self.urgency), torch.zeros_like(local[:, 0]))
        return self._finish(data_batch, local, mode, torch.where(exact, ltt, zl), dist, agents_per_scene)


class GlobalTargetPos(_GlobalTarget):
    """guidance_loss.py:1033-1135: reach a WORLD waypoint some time.  Within one horizon at the preferred speed: TargetPosLoss on the
    local target; else relu(goal - progress towards it), goal = max(urgency T dt pref_speed, min_progress_dist)."""

    def __init__(self, target_pos, urgency, pref_speed=1.42, dt=0.1, min_progress_dist=0.5, target_tolerance=None, action_num=5,
                 agents=None):
        super().__init__(target_pos, urgency, pref_speed, dt, target_tolerance, action_num, agents)
        self.min_progress_dist = float(min_progress_dist)

    def scene_entries(self, data_batch, horizon, agents_per_scene):
        local = self._local(data_batch)
        reach = horizon * self.dt * self.pref_speed
        exact = local.norm(dim=-1) < reach
        goal = torch.maximum(self.urgency * reach, torch.full_like(reach, self.min_progress_dist))
        mode = torch.where(exact, torch.full_like(exact, 4, dtype=torch.long), torch.full_like(exact, 3, dtype=torch.long))
        dist = torch.where(exact, torch.zeros_like(goal), goal)
        return self._finish(data_batch, local, mode, torch.zeros_like(mode), dist, agents_per_scene)
