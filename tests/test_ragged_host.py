"""Host logic of ragged batches (scenes of different sizes in one call), on CPU: the waypoint weights, the policy's scene-level
sample choice, scene sharding over ranks and the ctypes layout of CldScene."""
import os
import shutil
import socket
import subprocess

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from cld_b200 import make_scenes
from cld_b200.distributed import gather_results, shard_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [1, 3, 64, 65, 130, 2]


def _split(v, sizes):
    out, pos = [], 0
    for c in sizes:
        out.append(v[pos:pos + c])
        pos += c
    return out


def test_ragged_waypoint_weights_equal_per_scene_weights():
    from cld_b200.waypoints import TargetPosAtTime
    torch.manual_seed(0)
    B = sum(SIZES)
    agents = torch.rand(B) > 0.4
    agents[3:67] = False                                         # a scene without guided agents: weight 0, not a division by 0
    term = TargetPosAtTime(torch.randn(B, 2), torch.randint(0, 52, (B,)), agents=agents)
    got = term.scene_entries({}, 52, SIZES)["wp_weight"]
    want = torch.cat([TargetPosAtTime(p, t, agents=a).scene_entries({}, 52, c)["wp_weight"]
                      for p, t, a, c in zip(_split(term.target_pos, SIZES), _split(term.target_time, SIZES), _split(agents, SIZES), SIZES)])
    assert torch.equal(got, want)
    assert got[3:67].abs().sum() == 0 and got.sum() > 0
    # on a uniform batch a list of equal sizes gives the weights of the int form
    uni = TargetPosAtTime(term.target_pos[:60], term.target_time[:60], agents=agents[:60])
    assert torch.equal(uni.scene_entries({}, 52, [4] * 15)["wp_weight"], uni.scene_entries({}, 52, 4)["wp_weight"])


def test_choose_action_with_scene_sizes_equals_per_scene_calls():
    from cld_b200.policy import choose_action_from_guidance
    torch.manual_seed(1)
    B, N = sum(SIZES), 5
    losses = torch.rand(B, N, 2) * 10
    losses[::7, :, 1] = float("nan")
    for scene_level in (True, False):
        got = choose_action_from_guidance(losses, SIZES, scene_level)
        want = torch.cat([choose_action_from_guidance(l, c, scene_level) for l, c in zip(_split(losses, SIZES), SIZES)])
        assert torch.equal(got, want), scene_level
    # a scene-level choice is one index per scene
    got = choose_action_from_guidance(losses, SIZES, True)
    assert all(p.unique().numel() == 1 for p in _split(got, SIZES))
    # uniform sizes as a list equal the int form
    assert torch.equal(choose_action_from_guidance(losses[:60], [4] * 15, True), choose_action_from_guidance(losses[:60], 4, True))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, sizes, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        B = sum(sizes)
        aux, batch = make_scenes(1, B, seed=5, dense=True)
        batch["scene_index"] = torch.cat([torch.full((c,), 100 + i) for i, c in enumerate(sizes)])
        full = dict(batch, **aux)
        mine = shard_batch(full, None, world, rank)
        same = shard_batch(full, sizes, world, rank)
        ok = all(torch.equal(mine[k], same[k]) for k in mine if torch.is_tensor(mine[k]))
        # whole scenes: every scene id of the shard has all its agents in it, and they start at a scene boundary
        ids, counts = torch.unique_consecutive(mine["scene_index"], return_counts=True)
        ok = ok and all(int(c) == sizes[int(i) - 100] for i, c in zip(ids, counts))
        a0 = sum(sizes[:int(ids[0]) - 100])
        ok = ok and torch.equal(mine["extent"], full["extent"][a0:a0 + mine["extent"].shape[0]])
        # stand-in for the sampler's outputs: a deterministic function of the global row index
        rows = torch.arange(a0, a0 + mine["extent"].shape[0], dtype=torch.float32)
        traj = rows[:, None, None] + torch.arange(52 * 6, dtype=torch.float32).reshape(1, 52, 6) / 1000
        off = (rows[:, None].long() + torch.arange(52)[None]) % 3 == 0
        counts = [torch.zeros(1, dtype=torch.long) for _ in range(world)]
        dist.all_gather(counts, torch.tensor([rows.numel()]))
        gt, go, gc = gather_results(traj, off, rows % 5, rows_per_rank=[int(c) for c in counts])
        all_rows = torch.arange(B, dtype=torch.float32)
        ok = (ok and gt.shape == (B, 52, 6) and torch.equal(gt[:, 0, 0], all_rows) and torch.equal(gc, all_rows % 5)
              and torch.equal(go, (all_rows[:, None].long() + torch.arange(52)[None]) % 3 == 0))
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_shard_ragged_batch_world2_gloo_keeps_scenes_whole():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, SIZES, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = [q.get(timeout=120) for _ in ps]
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(res) == [(0, True), (1, True)]


def test_shard_batch_refuses_sizes_that_do_not_cover_the_batch():
    aux, batch = make_scenes(2, 3, seed=5)
    with pytest.raises(ValueError, match="sum to B=6"):
        shard_batch(batch, [2, 2], 2, 0)


CHECK_LAYOUT = r"""
#include <stddef.h>
#include <stdio.h>
#include "cld_b200.h"
#define F(name) printf(#name " %zu\n", offsetof(CldScene, name));
int main(void) {
  F(num_scenes) F(agents_per_scene) F(num_samp) F(extent) F(world_from_agent) F(raster_from_agent) F(curr_speed) F(drivable_map)
  F(map_h) F(map_w) F(target_pos) F(others_pos) F(others_avail) F(num_others) F(map_packed) F(target_speed) F(wp_target) F(wp_mode)
  F(wp_time) F(wp_dist) F(wp_weight) F(scene_start) F(scene_start_host)
  printf("sizeof %zu\n", sizeof(CldScene));
  return 0;
}
"""


def test_ctypes_scene_layout_matches_the_header(tmp_path):
    """The Python mirror of CldScene against the offsets the host C compiler gives the header's struct."""
    import ctypes
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no host C compiler")
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text(CHECK_LAYOUT)
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    want = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    from cld_b200._lib import CldScene
    names = [f[0] for f in CldScene._fields_]
    assert names == [k for k in want if k != "sizeof"]
    for name in names:
        assert getattr(CldScene, name).offset == int(want[name]), name
    assert ctypes.sizeof(CldScene) == int(want["sizeof"])
    # a zero-initialised struct is the uniform layout
    sc = CldScene()
    assert not sc.scene_start and not sc.scene_start_host
