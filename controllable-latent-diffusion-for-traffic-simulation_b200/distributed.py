"""Scene sharding across ranks and the path's single exchange (SURVEY.md section 8e).

The sampling path shards by scene: rows of different scenes never interact (the agent-collision mask is
block-diagonal per scene, reference src/tbsim/utils/guidance_loss.py:493-503), so rank r owns scenes
[r*S/G, (r+1)*S/G) with replicated weights and there is NO collective inside the denoising loop.  The
only exchange is one all-gather of (trajectories, off-road flags, collision counts) at the end.

One process per GPU (torchrun); the backend is whatever the default process group uses (NCCL on the
B200 box, gloo in the CPU tests).  Nothing here computes: it slices, packs and gathers.
"""
import torch
import torch.distributed as dist

from .keys import scene_size_list, scene_sizes

# data_batch / aux_info entries indexed by agent row (B = S*A, scene-major)
PER_AGENT_KEYS = (
    "extent", "world_from_agent", "raster_from_agent", "curr_speed", "drivable_map", "drivable_map_bits", "scene_index", "target_pos", "target_speed",
    "wp_target", "wp_mode", "wp_time", "wp_dist", "wp_weight",
    "all_other_agents_future_positions", "all_other_agents_future_availability", "history_positions",
    "history_yaws", "cond_feat", "curr_states", "image",
)


def shard_scenes(num_scenes, world_size, rank):
    """Contiguous scene range of `rank`; the first `num_scenes % world_size` ranks get one extra scene."""
    if world_size < 1 or not 0 <= rank < world_size:
        raise ValueError("bad rank %d / world %d" % (rank, world_size))
    base, extra = divmod(int(num_scenes), int(world_size))
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def shard_batch(batch, agents_per_scene, world_size, rank):
    """Slice every per-agent tensor of a data_batch / aux_info dict to this rank's scenes (whole scenes, `shard_scenes`).
    agents_per_scene: an int, the list of scene sizes of a ragged batch, or None to read the sizes from batch["scene_index"]."""
    some = next(v for k, v in batch.items() if k in PER_AGENT_KEYS and torch.is_tensor(v))
    B = some.shape[0]
    sizes = scene_sizes(batch.get("scene_index"), B) if agents_per_scene is None else scene_size_list(agents_per_scene, B)
    s0, s1 = shard_scenes(len(sizes), world_size, rank)
    a0 = sum(sizes[:s0])
    a1 = a0 + sum(sizes[s0:s1])
    out = {}
    for k, v in batch.items():
        out[k] = v[a0:a1] if (k in PER_AGENT_KEYS and torch.is_tensor(v) and v.shape[0] == B) else v
    return out


def pack_results(traj, offroad, coll):
    """[R,T,6] fp32, [R,T] bool, [R] fp32 -> one [R, 6T + T + 1] fp32 payload."""
    R = traj.shape[0]
    return torch.cat([traj.reshape(R, -1), offroad.to(traj.dtype), coll.reshape(R, 1)], dim=1).contiguous()


def unpack_results(payload, horizon):
    R, T = payload.shape[0], int(horizon)
    traj = payload[:, :6 * T].reshape(R, T, 6)
    offroad = payload[:, 6 * T:7 * T] != 0
    coll = payload[:, 7 * T]
    return traj, offroad, coll


def gather_results(traj, offroad, coll, rows_per_rank=None, group=None, out=None):
    """The path's one collective: every rank ends with all ranks' trajectories and indicators.

    Equal shards use a single all_gather_into_tensor (ncclAllGather over NVLink); ragged shards
    (`rows_per_rank` given and not all equal) pad to the largest shard and trim afterwards.
    Returns (traj [Rtot,T,6], offroad [Rtot,T] bool, coll [Rtot]).
    """
    T = traj.shape[1]
    payload = pack_results(traj, offroad, coll)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return unpack_results(payload, T)
    world = dist.get_world_size(group)
    R = payload.shape[0]
    if rows_per_rank is None:
        rows_per_rank = [R] * world
    rmax = max(rows_per_rank)
    if R < rmax:
        payload = torch.cat([payload, payload.new_zeros(rmax - R, payload.shape[1])], dim=0)
    if out is None:
        out = payload.new_empty(world * rmax, payload.shape[1])
    dist.all_gather_into_tensor(out, payload, group=group)
    if any(r != rmax for r in rows_per_rank):
        out = torch.cat([out[i * rmax:i * rmax + r] for i, r in enumerate(rows_per_rank)], dim=0)
    return unpack_results(out, T)
