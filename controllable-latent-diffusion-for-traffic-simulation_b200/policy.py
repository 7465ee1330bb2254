"""`get_action` on top of the B200 sampler (SURVEY.md sec. 8 f-3): the part of the reference's closed-loop policy wrapper that sits
directly on the sampling path -- `DiffuserTrafficModel.get_action` (src/tbsim/algos/algos.py:2024-2099) with
`choose_action_from_guidance` (src/tbsim/utils/guidance_loss.py:22-65).  N samples per agent are drawn with guidance, the sample
with the smallest (unweighted, summed) guidance loss is chosen -- per SCENE when a scene-level term (agent_collision) is active,
per agent otherwise -- and stationary agents are zeroed.  The simulator / trajdata environment around it is out of scope.
"""
import numbers

import torch

from .keys import default_guidance, scene_size_list, scene_sizes

SCENE_LEVEL_TERMS = ("agent_collision",)      # + social_group / gpt* in the reference, which are not built
LOSS_ROWS = ("agent_collision", "map_collision", "target_pos", "target_speed", "acc_limit", "speed_limit", "waypoint")


def choose_action_from_guidance(guide_losses, agents_per_scene, scene_level):
    """guide_losses [B, N, G] (B agents, N samples, G active terms, NaN = not applicable) -> act_idx [B].  agents_per_scene: an
    int (B = S * A) or the list of scene sizes of a ragged batch.
    scene_level: argmin over samples of the loss summed over the agents of the scene (guidance_loss.py:50-56), else per agent."""
    B, N, _ = guide_losses.shape
    tot = torch.nansum(guide_losses, dim=-1)                                  # [B, N]
    if not scene_level:
        return torch.argmin(tot, dim=-1)
    if not isinstance(agents_per_scene, numbers.Integral):
        # segment sums: the scenes of one size are summed as one uniform batch, so every scene's sum is the one a call on that
        # scene alone computes
        sizes = scene_size_list(agents_per_scene, B)
        starts = torch.tensor([0] + sizes[:-1]).cumsum(0)
        idx = torch.empty(B, dtype=torch.long, device=tot.device)
        for A in sorted(set(sizes)):
            first = starts[torch.tensor(sizes) == A]
            rows = (first[:, None] + torch.arange(A)[None, :]).reshape(-1).to(tot.device)
            pick = torch.argmin(tot.index_select(0, rows).reshape(-1, A, N).sum(dim=1), dim=1)
            idx[rows] = pick.repeat_interleave(A)
        return idx
    S = B // agents_per_scene
    idx = torch.argmin(tot.reshape(S, agents_per_scene, N).sum(dim=1), dim=1)   # [S]
    return idx.repeat_interleave(agents_per_scene)


class GuidedDiffusionPolicy:
    def __init__(self, dm, vae, algo_config, context_encoder=None, guidance=None, disable_control_on_stationary=True,
                 moving_speed_th=0.5):
        self.dm, self.vae, self.algo = dm, vae, algo_config
        self.context_encoder = context_encoder
        self.guidance = guidance
        self.disable_control_on_stationary = disable_control_on_stationary
        self.moving_speed_th = moving_speed_th

    @torch.no_grad()
    def get_action(self, obs_dict, num_action_samples=1, step_index=0, sampler="ddpm", aux_info=None, **kw):
        """-> (action {positions [B,T,2], yaws [B,T,1]}, info {action_samples {positions [B,N,T,2], yaws [B,N,T,1]}, act_idx [B],
        guide_losses {term: [B,N]}})."""
        B = obs_dict["history_positions"].shape[0]
        N = int(num_action_samples)
        sizes = scene_sizes(obs_dict.get("scene_index"), B)
        # a uniform batch keeps the integer form (its scene-level choice is one reshape)
        A = sizes[0] if len(set(sizes)) == 1 else sizes
        if aux_info is None:
            if self.context_encoder is None:
                raise ValueError("get_action needs aux_info (cond_feat, curr_states) or a context encoder")
            aux_info = self.context_encoder(obs_dict)
        algo = self.algo
        old = algo.num_samp
        algo.num_samp = N
        try:
            out = self.dm(obs_dict, aux_info, algo, sampler=sampler, guidance=self.guidance, want_traj=True, agents_per_scene=A, **kw)
        finally:
            algo.num_samp = old
        T = out["traj"].shape[1]
        traj = out["traj"].reshape(B, N, T, 6)
        positions, yaws = traj[..., :2].clone(), traj[..., 3:4].clone()
        act_idx = torch.zeros(B, dtype=torch.long, device=traj.device)
        losses = {}
        if self.guidance is not None:
            # the samples are scored by ONE loss evaluation at their x0: more optimizer iterations would score a perturbed latent
            g = dict(default_guidance(), **self.guidance)
            g["grad_steps"] = 1
            eng = self.dm.engine(B * N)
            scene = eng.make_scene(obs_dict, len(sizes), sizes[0], N, scene_sizes=sizes)
            rep = (lambda v: v.repeat_interleave(N, dim=0)) if N > 1 else (lambda v: v)
            _, _, per = eng.guidance_step(out["pred_traj"], rep(aux_info["cond_feat"]), rep(aux_info["curr_states"]), scene, g)
            active = [k for k in LOSS_ROWS if float(g.get(k, 0.0)) != 0.0]
            losses = {k: per[LOSS_ROWS.index(k)].reshape(B, N) for k in active}
            if active:
                stacked = torch.stack([losses[k] for k in active], dim=2)
                act_idx = choose_action_from_guidance(stacked, A, any(k in SCENE_LEVEL_TERMS for k in active))
        ar = torch.arange(B, device=traj.device)
        a_pos, a_yaw = positions[ar, act_idx], yaws[ar, act_idx]
        if self.disable_control_on_stationary and "curr_speed" in obs_dict:
            stat = obs_dict["curr_speed"].to(traj.device).abs() < self.moving_speed_th
            positions[stat] = 0
            yaws[stat] = 0
            a_pos[stat] = 0
            a_yaw[stat] = 0
        info = {"action_samples": {"positions": positions, "yaws": yaws}, "act_idx": act_idx, "guide_losses": losses}
        return {"positions": a_pos, "yaws": a_yaw}, info
