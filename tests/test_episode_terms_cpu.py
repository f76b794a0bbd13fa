"""Per-term episode returns (extension) without a GPU: the config key and its dependency, the pointer rules of the C
ABI, the ctypes layout, the torch restatement on a hand-made sequence, and the job-wide sums and means through a
world-size-2 gloo all-reduce."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from episode_term_reference import EpisodeTermTracker, slot_sum_bound
from leibnizgym_b200 import _native as nat
from leibnizgym_b200.config import default_trifinger_config, difficulty_config, resolve_config
from leibnizgym_b200.distributed import all_reduce_stats, stats_to_info

EPISODE_FIELDS = ("episode_return", "last_episode_return", "last_episode_length", "last_episode_success", "episode_stats")
TERM_FIELDS = ("episode_term_return", "last_episode_term_return", "episode_term_stats")


def test_config_key_defaults_off():
    assert default_trifinger_config()["episode_term_returns"] == {"activate": False}
    assert resolve_config({"command_mode": "torque"})["episode_term_returns"]["activate"] is False
    on = resolve_config({"episode_term_returns": {"activate": True}, "episode_statistics": {"activate": True}})
    assert on["episode_term_returns"]["activate"] is True and on["episode_statistics"]["activate"] is True


def test_on_without_episode_statistics_is_refused_at_construction():
    """Checked before anything touches a device, so the error is the same on a machine without a GPU."""
    from leibnizgym_b200.env import TrifingerEnv
    cfg = difficulty_config(4, 64)
    cfg["episode_term_returns"] = {"activate": True}
    with pytest.raises(ValueError, match="episode_term_returns.*episode_statistics"):
        TrifingerEnv(cfg, device="cpu", verbose=False)


def test_slot_names():
    assert nat.LG_NUM_EPISODE_TERMS == 8 and nat.LG_EPISODE_TERM_BONUS == 7
    assert nat.EPISODE_TERM_NAMES == nat.TERM_NAMES + ("success_bonus",)
    assert nat.EPISODE_TERM_NAMES[nat.LG_EPISODE_TERM_BONUS] == "success_bonus"


def test_ctypes_layout():
    names = [f[0] for f in nat.LgBuffers._fields_]
    assert names[-1] == "torch_rng"
    i = names.index("episode_stats")
    assert names[i + 1:i + 4] == list(TERM_FIELDS)
    lib = nat.load()
    assert lib.lg_struct_size(2) == C.sizeof(nat.LgBuffers)


def _abi_args():
    p, s, b = nat.LgParams(), nat.LgSimState(), nat.LgBuffers()
    p.num_envs, p.action_dim = 64, 9
    s.dof_state, s.root_state, s.rigid_body = 0x10000, 0x20000, 0x30000
    for i, name in enumerate(("obs", "action", "reward", "reset", "goal_reset", "successes", "steps_count", "goal_pose",
                              "goal_movement", "history", "control")):
        setattr(b, name, 0x100000 * (i + 1))
    return p, s, b


def _refused(lib, p, s, b, text):
    """lg_reset_envs with an empty id list returns right after validation: the rule is checked before any CUDA call."""
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == -1
    assert text in lib.lg_last_error()
    assert lib.lg_post_physics(p, s, b, 0.0, None) == -1
    assert lib.lg_pre_physics(p, s, b, 0x5000000, None) == -1


def test_pointers_all_or_none_through_the_abi():
    lib = nat.load()
    p, s, b = _abi_args()
    for i, name in enumerate(EPISODE_FIELDS):
        setattr(b, name, 0x4000000 * (i + 1))
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0
    for k in range(len(TERM_FIELDS)):
        for i, name in enumerate(TERM_FIELDS):
            setattr(b, name, 0x8000000 * (i + 1) if i <= k else None)
        if k < len(TERM_FIELDS) - 1:
            _refused(lib, p, s, b, b"episode_term_stats go together")
        else:
            assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0
    b.episode_term_return = None   # one missing of three
    _refused(lib, p, s, b, b"episode_term_stats go together")


def test_needs_the_episode_pointers_through_the_abi():
    lib = nat.load()
    p, s, b = _abi_args()
    for i, name in enumerate(TERM_FIELDS):
        setattr(b, name, 0x8000000 * (i + 1))
    _refused(lib, p, s, b, b"needs the episode statistics buffers")
    for i, name in enumerate(EPISODE_FIELDS):
        setattr(b, name, 0x4000000 * (i + 1))
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0


@pytest.mark.parametrize("field", ["episode_term_return", "last_episode_term_return"])
def test_rows_must_be_16_byte_aligned_through_the_abi(field):
    lib = nat.load()
    p, s, b = _abi_args()
    for i, name in enumerate(EPISODE_FIELDS):
        setattr(b, name, 0x4000000 * (i + 1))
    for i, name in enumerate(TERM_FIELDS):
        setattr(b, name, 0x8000000 * (i + 1))
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0
    setattr(b, field, getattr(b, field) + 8)
    _refused(lib, p, s, b, b"must be 16-byte aligned")
    b.episode_term_stats += 8   # the fp64 statistics vector only needs its natural alignment
    setattr(b, field, getattr(b, field) - 8)
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0


def test_restatement_on_a_hand_made_sequence():
    active = [True, True, False, True, False, False, True]   # terms 2, 4, 5 inactive
    tr = EpisodeTermTracker(3, active, 5000.0)
    f = lambda *rows: torch.tensor(rows, dtype=torch.float32)  # noqa: E731   [7, 3]
    b = lambda *v: torch.tensor(v, dtype=torch.bool)  # noqa: E731
    terms = [f(*[[k + 1.0, 10.0 * (k + 1), 100.0 * (k + 1)] for k in range(7)]) for _ in range(4)]
    paid = [b(0, 0, 0), b(1, 0, 0), b(0, 0, 1), b(0, 0, 0)]
    resets = [[0, 1, 2], [], [0, 1], [0, 2]]
    out = []
    for t in range(4):
        tr.reset(resets[t])
        out.append(tr.post(terms[t], paid[t]))
    # steps 0, 1: nothing ended
    assert out[0][0] == 0 and out[1][0] == 0 and out[1][1].abs().sum() == 0
    # step 2: envs 0, 1 end after 2 steps; env 0 was paid the bonus once
    n, st = out[2]
    row0 = [2.0, 4.0, 0.0, 8.0, 0.0, 0.0, 14.0, 5000.0]
    row1 = [20.0, 40.0, 0.0, 80.0, 0.0, 0.0, 140.0, 0.0]
    assert n == 2 and st.tolist() == [a + c for a, c in zip(row0, row1)]
    # step 3: env 0 ends after 1 step, env 2 after 3 steps (bonus at step 2)
    n, st = out[3]
    row2 = [300.0, 600.0, 0.0, 1200.0, 0.0, 0.0, 2100.0, 5000.0]
    assert n == 2 and st.tolist() == [a + c for a, c in zip([1.0, 2.0, 0.0, 4.0, 0.0, 0.0, 7.0, 0.0], row2)]
    assert tr.last_episode_term_return[2].tolist() == row2
    # inactive slots stay 0 everywhere; a second reset before any step leaves the record and reports it once
    assert tr.episode_term_return[:, [2, 4, 5]].abs().sum() == 0
    tr.reset([1])
    tr.reset([1])
    assert tr.last_episode_term_return[1].tolist() == row1
    zero = torch.zeros(7, 3)
    assert tr.post(zero, b(0, 0, 0))[0] == 1 and tr.post(zero, b(0, 0, 0))[0] == 0


def test_restatement_adds_in_fp32_in_step_order():
    tr = EpisodeTermTracker(1, [True] * 7, 0.1)
    for _ in range(3):
        tr.post(torch.full((7, 1), 0.1), torch.ones(1, dtype=torch.bool))
    want = np.float32(np.float32(np.float32(0.1) + np.float32(0.1)) + np.float32(0.1))
    assert (tr.episode_term_return.numpy()[0] == want).all()


def test_slot_sum_bound_covers_a_reordered_sum():
    g = torch.Generator().manual_seed(5)
    L = 40
    x = (torch.randn(L, 8, generator=g) * torch.tensor([1e3, 1e-2, 5.0, 1e2, 1.0, 3.0, 2e3, 0.0])).float()
    by_step = torch.zeros((), dtype=torch.float32)
    for t in range(L):
        r = torch.zeros((), dtype=torch.float32)
        for k in range(8):
            r = r + x[t, k]
        by_step = by_step + r
    by_term = torch.zeros(8, dtype=torch.float32)
    for t in range(L):
        by_term = by_term + x[t]
    diff = abs(float(by_term.double().sum()) - float(by_step))
    assert diff <= float(slot_sum_bound(x.abs().double().sum(), torch.tensor(L)))


def test_info_helpers_old_calls_are_unchanged():
    v = torch.arange(nat.LG_NUM_STATS, dtype=torch.float64)
    ep = torch.tensor([2.0, 10.0, 8.0, 1.0], dtype=torch.float64)
    plain = stats_to_info(all_reduce_stats(v, 4, 4), ["object_dist"])
    stats, ep_only = all_reduce_stats(v, 4, 4, episode_stats=ep)
    with_ep = stats_to_info(stats, ["object_dist"], episode_stats=ep_only)
    ts = torch.arange(nat.LG_NUM_EPISODE_TERMS, dtype=torch.float64)
    s3, e3, t3 = all_reduce_stats(v, 4, 4, episode_stats=ep, episode_term_stats=ts)
    assert torch.equal(s3, all_reduce_stats(v, 4, 4)) and torch.equal(e3, ep_only) and torch.equal(t3, ts)
    info = stats_to_info(s3, ["object_dist"], episode_stats=e3, episode_term_stats=t3,
                         episode_terms=["object_dist", "success_bonus"])
    assert {k: info[k] for k in with_ep} == with_ep
    assert not any("/return_sum/" in k or "/mean_return/" in k for k in with_ep) and "env/episodes/return_sum" not in plain
    extra = sorted(set(info) - set(with_ep))
    assert extra == ["env/episodes/mean_return/object_dist", "env/episodes/mean_return/success_bonus",
                     "env/episodes/return_sum/object_dist", "env/episodes/return_sum/success_bonus"]
    assert info["env/episodes/return_sum/object_dist"] == 2.0 and info["env/episodes/mean_return/success_bonus"] == 3.5
    every = stats_to_info(s3, [], episode_stats=e3, episode_term_stats=t3)
    assert sum(k.startswith("env/episodes/return_sum/") for k in every) == 8
    none = stats_to_info(s3, [], episode_stats=torch.zeros(4, dtype=torch.float64), episode_term_stats=t3)
    assert not any(k.startswith("env/episodes/mean_return") for k in none)
    with pytest.raises(ValueError):
        all_reduce_stats(v, 4, 4, episode_term_stats=ts)


SHARD_EP = [torch.tensor([3.0, -7.5, 21.0, 1.0], dtype=torch.float64),
            torch.tensor([1.0, 2.25, 5.0, 1.0], dtype=torch.float64)]
SHARD_TERMS = [torch.arange(8, dtype=torch.float64) * 0.5, torch.arange(8, dtype=torch.float64) - 3.0]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    step = torch.full((nat.LG_NUM_STATS,), float(rank + 1), dtype=torch.float64)
    stats, ep, terms = all_reduce_stats(step, 8, 16, episode_stats=SHARD_EP[rank], episode_term_stats=SHARD_TERMS[rank])
    plain = all_reduce_stats(step, 8, 16)
    if rank == 0:
        q.put((stats.numpy(), plain.numpy(), ep.numpy(), terms.numpy(),
               stats_to_info(stats, ["object_dist"], episode_stats=ep, episode_term_stats=terms,
                             episode_terms=["object_dist", "keypoint"])))
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
    stats, plain, ep, terms, info = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    np.testing.assert_array_equal(stats, plain)
    np.testing.assert_array_equal(ep, [4.0, -5.25, 26.0, 2.0])
    np.testing.assert_array_equal(terms, np.arange(8) * 1.5 - 3.0)
    assert info["env/episodes/return_sum/object_dist"] == 0.0
    assert info["env/episodes/return_sum/keypoint"] == 6.0 and info["env/episodes/mean_return/keypoint"] == 1.5
    assert "env/episodes/return_sum/success_bonus" not in info
