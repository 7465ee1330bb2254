"""Constants shared by the parameter containers and the engine.  No shared-library import here, so the containers
(`DmModel`, `VaeModel`) can be constructed -- e.g. to draw the reference's random initialisation -- without mapping
libcld_b200.so; anything that computes goes through `engine.Engine` and fails loudly when the library is missing."""

NORM_MEAN = (13.162, -0.13891, 5.0223, -0.0046415, -0.0080072, -0.0013546)
NORM_STD = (13.0717, 2.2462, 3.6187, 0.2210, 2.5770, 0.0840)

DECODER_KEYS = [
    "lstm.weight_ih_l0", "lstm.weight_hh_l0", "lstm.bias_ih_l0", "lstm.bias_hh_l0",
    "lstm.weight_ih_l1", "lstm.weight_hh_l1", "lstm.bias_ih_l1", "lstm.bias_hh_l1",
    "cond2hidden.weight", "cond2hidden.bias", "hid2act.weight", "hid2act.bias",
]


def default_guidance(**over):
    """Defaults of the reference's SceneEditingConfig (src/tbsim/configs/scene_edit_config.py:73-92,302-325)."""
    g = dict(agent_collision=50.0, map_collision=1.0, target_pos=0.0, num_disks=2, buffer_dist=0.2, decay=0.9,
             num_points=(10, 10), speed_th=0.5, min_target_time=0.0, optimizer="adam", lr=0.3,
             # SURVEY.md sec. 8 f-4 (off by default): weights and limits of TargetSpeedLoss / AccLimitLoss / SpeedLimitLoss
             target_speed=0.0, acc_limit=0.0, acc_limit_value=0.0, speed_limit=0.0, speed_limit_value=0.0,
             # waypoint terms (cld_b200.waypoints: target_pos_at_time / global_target_pos_at_time / global_target_pos)
             waypoint=0.0,
             # optimizer iterations per guided denoising step (PerturbationGuidance.perturb's grad_steps)
             grad_steps=1)
    g.update(over)
    return g


def scene_sizes(scene_index, B):
    """Agents per scene, in batch order, checked for contiguity (the agents of a scene must be adjacent rows)."""
    import torch
    if scene_index is None:
        return [int(B)]
    sidx = torch.as_tensor(scene_index).reshape(-1)
    if sidx.numel() != B:
        raise ValueError("scene_index has %d entries for %d agents" % (sidx.numel(), B))
    _, counts = torch.unique_consecutive(sidx, return_counts=True)
    if torch.unique(sidx).numel() != counts.numel():
        raise ValueError("scene_index is not contiguous: the agents of a scene must be adjacent rows")
    return [int(c) for c in counts.tolist()]


def scene_buckets(sizes):
    """Ragged batches (the reference builds a block-diagonal scene mask from `scene_index`, guidance_loss.py:493-503, and accepts
    scenes of different sizes): the kernels index rows as (scene * A + agent) * N + sample with ONE A per call, so a ragged batch is
    sampled as one uniform sub-batch per distinct scene size.  Returns [(A, agent_index LongTensor)], sizes ascending; the agent
    indices of a bucket are scene-major in batch order."""
    import torch
    starts, pos = [], 0
    for c in sizes:
        starts.append(pos)
        pos += c
    out = []
    for A in sorted(set(sizes)):
        idx = torch.cat([torch.arange(st, st + A) for st, c in zip(starts, sizes) if c == A])
        out.append((A, idx))
    return out


def agents_per_scene(scene_index, B):
    """Number of agents A of every scene of a UNIFORM batch, checked (ragged batches: `scene_buckets`)."""
    import torch
    if scene_index is None:
        return int(B)
    sidx = torch.as_tensor(scene_index).reshape(-1)
    if sidx.numel() != B:
        raise ValueError("scene_index has %d entries for %d agents" % (sidx.numel(), B))
    _, counts = torch.unique_consecutive(sidx, return_counts=True)
    ids = torch.unique(sidx)
    if ids.numel() != counts.numel():
        raise ValueError("scene_index is not contiguous: the agents of a scene must be adjacent rows")
    A = int(counts[0].item())
    if not bool((counts == A).all().item()):
        raise ValueError("cld_b200 needs the same number of agents in every scene of a call (got sizes %s); pad the "
                         "scenes to a common size or call once per scene size" % sorted(set(counts.tolist())))
    return A
