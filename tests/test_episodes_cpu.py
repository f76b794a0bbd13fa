"""Episode statistics (extension) without a GPU: the config key, the all-or-none pointer check of the C ABI, the torch
restatement on a hand-made sequence, and the job-wide sums and means through a world-size-2 gloo all-reduce."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from episode_reference import EpisodeTracker, episode_statistics
from leibnizgym_b200 import _native as nat
from leibnizgym_b200.config import default_trifinger_config, resolve_config
from leibnizgym_b200.distributed import all_reduce_stats, stats_to_info

EPISODE_FIELDS = ("episode_return", "last_episode_return", "last_episode_length", "last_episode_success", "episode_stats")


def test_config_key_defaults_off():
    assert default_trifinger_config()["episode_statistics"] == {"activate": False}
    assert resolve_config({"command_mode": "torque"})["episode_statistics"]["activate"] is False
    assert resolve_config({"episode_statistics": {"activate": True}})["episode_statistics"]["activate"] is True


def _abi_args():
    p, s, b = nat.LgParams(), nat.LgSimState(), nat.LgBuffers()
    p.num_envs, p.action_dim = 64, 9
    s.dof_state, s.root_state, s.rigid_body = 0x10000, 0x20000, 0x30000
    for i, name in enumerate(("obs", "action", "reward", "reset", "goal_reset", "successes", "steps_count", "goal_pose",
                              "goal_movement", "history", "control")):
        setattr(b, name, 0x100000 * (i + 1))
    return p, s, b


def test_pointers_all_or_none_through_the_abi():
    """Validation runs before any CUDA call: lg_reset_envs with an empty id list returns right after it."""
    lib = nat.load()
    p, s, b = _abi_args()
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0
    for k in range(len(EPISODE_FIELDS)):
        for i, name in enumerate(EPISODE_FIELDS):
            setattr(b, name, 0x4000000 * (i + 1) if i <= k else None)
        rc = lib.lg_reset_envs(p, s, b, None, 0, None)
        if k < len(EPISODE_FIELDS) - 1:
            assert rc == -1, k
            assert b"episode_stats go together" in lib.lg_last_error()
            assert lib.lg_post_physics(p, s, b, 0.0, None) == -1
            assert lib.lg_pre_physics(p, s, b, 0x5000000, None) == -1
        else:
            assert rc == 0
    b.episode_return = None   # one missing of five
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == -1


def test_restatement_on_a_hand_made_sequence():
    f = lambda *v: torch.tensor(v, dtype=torch.float32)  # noqa: E731
    b = lambda *v: torch.tensor(v, dtype=torch.bool)  # noqa: E731
    rewards = [f(1, 2, 3), f(10, 20, 30), f(100, 200, 300), f(0.5, 0.25, 0.125), f(4, 4, 4)]
    succ = [b(0, 0, 0), b(1, 0, 0), b(1, 0, 1), b(0, 0, 0), b(0, 0, 0)]
    # step 0: fresh env (everything reset, nothing ended); step 2: envs 0, 1 reset; step 3: env 0 again, env 2
    resets = [[0, 1, 2], [], [0, 1], [0, 2], []]
    tr, stats = episode_statistics(rewards, resets, succ)
    assert stats[0].tolist() == [0, 0, 0, 0] and stats[1].tolist() == [0, 0, 0, 0]
    # env 0 ended with 11 after 2 steps (success set at step 1), env 1 with 22 after 2 steps
    assert stats[2].tolist() == [2, 33, 4, 1]
    # env 0 ended with 100 after 1 step (success from step 2), env 2 with 333 after 3 steps (success from step 2)
    assert stats[3].tolist() == [2, 433, 4, 2]
    assert stats[4].tolist() == [0, 0, 0, 0]
    assert tr.episode_return.tolist() == [4.5, 204.25, 4.125]
    assert tr.last_episode_return.tolist() == [100, 22, 333]
    assert tr.last_episode_length.tolist() == [1, 2, 3]
    assert tr.last_episode_success.tolist() == [True, False, True]
    # a second reset before any step leaves the record alone and reports it once
    tr.reset([1])
    tr.reset([1])
    assert tr.last_episode_length.tolist() == [1, 3, 3] and tr.last_episode_return[1] == 204.25
    assert tr.post(f(0, 0, 0), b(0, 0, 0)).tolist() == [1, 204.25, 3, 0]
    assert tr.post(f(0, 0, 0), b(0, 0, 0)).tolist() == [0, 0, 0, 0]


def test_restatement_adds_in_fp32():
    tr = EpisodeTracker(1)
    for _ in range(3):
        tr.post(torch.tensor([0.1], dtype=torch.float32), torch.zeros(1, dtype=torch.bool))
    want = np.float32(np.float32(np.float32(0.1) + np.float32(0.1)) + np.float32(0.1))
    assert tr.episode_return.numpy()[0] == want


def test_info_helpers_without_episodes_are_unchanged():
    v = torch.arange(nat.LG_NUM_STATS, dtype=torch.float64)
    plain = stats_to_info(all_reduce_stats(v, 4, 4), ["object_dist"])
    assert not any(k.startswith("env/episodes/") for k in plain)
    stats, ep = all_reduce_stats(v, 4, 4, episode_stats=torch.zeros(nat.LG_NUM_EPISODE_STATS, dtype=torch.float64))
    assert torch.equal(stats, all_reduce_stats(v, 4, 4))
    info = stats_to_info(stats, ["object_dist"], episode_stats=ep)
    assert {k: info[k] for k in plain} == plain
    assert info["env/episodes/count"] == 0 and "env/episodes/mean_return" not in info


SHARD_STATS = [torch.tensor([3.0, -7.5, 21.0, 1.0], dtype=torch.float64),
               torch.tensor([1.0, 2.25, 5.0, 1.0], dtype=torch.float64)]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    step = torch.full((nat.LG_NUM_STATS,), float(rank + 1), dtype=torch.float64)
    stats, ep = all_reduce_stats(step, 8, 16, episode_stats=SHARD_STATS[rank])
    if rank == 0:
        q.put((stats.numpy(), ep.numpy(), stats_to_info(stats, ["object_dist"], episode_stats=ep)))
    dist.barrier()
    dist.destroy_process_group()


def test_all_reduce_and_means_through_gloo():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    stats, ep, info = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    # the step statistics are what the one-vector all-reduce gives: means (1 and 2 over 8 envs each -> 1.5), counts 3
    expect = np.full(nat.LG_NUM_STATS, 3.0)
    expect[[0, 1, 2, 3, 4, 5, 6, nat.STAT_SUCCESSES, nat.STAT_REWARD]] = 1.5
    np.testing.assert_array_equal(stats, expect)
    np.testing.assert_array_equal(ep, [4.0, -5.25, 26.0, 2.0])
    assert info["env/episodes/count"] == 4.0 and info["env/episodes/return_sum"] == -5.25
    assert info["env/episodes/mean_return"] == pytest.approx(-5.25 / 4, abs=0)
    assert info["env/episodes/mean_length"] == 6.5 and info["env/episodes/success_rate"] == 0.5
