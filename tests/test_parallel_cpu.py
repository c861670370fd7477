"""world_size-2 gloo tests (CPU) of the multi-GPU host logic: env sharding, the episode-stat all-gather in global env
order, and the max-over-ranks timing reduction."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, n_total, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from rl4mm_b200 import parallel

    r, w, _ = parallel.init_from_env("gloo")
    assert (r, w) == (rank, world)
    ids = parallel.shard_env_ids(n_total, rank, world)
    # a statistic that encodes the global env id, so the gathered order can be checked
    local = torch.stack([torch.tensor(ids, dtype=torch.float32), torch.tensor(ids * 10.0 + rank, dtype=torch.float32)], dim=1)
    full = parallel.gather_episode_stats(local, n_total)
    t = parallel.max_over_ranks(1.0 + rank)
    if rank == 0:
        np.save(os.path.join(out_dir, "full.npy"), full.numpy())
        np.save(os.path.join(out_dir, "t.npy"), np.array([t]))
    dist.barrier()
    dist.destroy_process_group()


def test_shard_and_gather_world2(tmp_path):
    world, n_total = 2, 12
    mp.spawn(_worker, args=(world, _free_port(), n_total, str(tmp_path)), nprocs=world, join=True)
    full = np.load(tmp_path / "full.npy")
    assert full.shape == (n_total, 2)
    assert np.array_equal(full[:, 0], np.arange(n_total))               # global env order restored
    assert np.array_equal(full[:, 1], np.arange(n_total) * 10 + np.arange(n_total) % world)
    assert np.load(tmp_path / "t.npy")[0] == 2.0                        # max over ranks


def test_shard_env_ids_partition():
    from rl4mm_b200.parallel import shard_env_ids

    for world in (1, 2, 4, 8):
        parts = [shard_env_ids(1000, r, world) for r in range(world)]
        assert sorted(np.concatenate(parts).tolist()) == list(range(1000))
        assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


def test_episode_stats_shapes():
    from rl4mm_b200 import abi
    from rl4mm_b200.parallel import STAT_FIELDS, episode_stats

    T, N = 5, 3
    rew = torch.arange(T * N, dtype=torch.float64).view(T, N)
    done = torch.zeros((T, N), dtype=torch.uint8)
    done[-1] = 1
    st = np.zeros(N, abi.ENV_STATE_DTYPE)
    st["inventory"], st["cash"], st["price"] = [1, -2, 3], [10.0, 20.0, 30.0], [2.0, 2.0, 2.0]
    out = episode_stats(rew, done, st)
    assert out.shape == (N, len(STAT_FIELDS)) and out.dtype == torch.float32
    assert out[:, 0].tolist() == rew.sum(0).tolist() and out[:, 6].tolist() == [1, 1, 1]
    assert out[:, 4].tolist() == [12.0, 16.0, 36.0]


def test_episode_stats_dev_decodes_state_records_like_episode_stats():
    """episode_stats_dev reads lobsim_env_state_t records by byte offset (the device path of the collect workload): on hand-built
    records with every field distinct, it must give what episode_stats computes from the named fields."""
    from rl4mm_b200 import abi
    from rl4mm_b200.parallel import episode_stats, episode_stats_dev

    T, N = 4, 5
    rng = np.random.default_rng(0)
    rew = torch.tensor(rng.normal(size=(T, N)))
    done = torch.tensor(rng.integers(0, 2, size=(T, N)), dtype=torch.uint8)
    st = np.zeros(N, abi.ENV_STATE_DTYPE)
    for i, name in enumerate(abi.ENV_STATE_DTYPE.names):     # a distinct non-zero value in every field, so a wrong offset shows
        st[name] = (np.arange(N) + 1 + 10 * i).reshape((N,) + (1,) * (st[name].ndim - 1))
    st["inventory"] = [-7, 0, 3, 120, -40]
    st["cash"] = [1e6, -2.5e3, 0.0, 7.25, 1e9]
    st["price"] = [101.5, 99.0, np.nan, 1e4, 0.5]
    st["err"] = [0, abi.ERR_EMPTY_BOOK, abi.ERR_AGENT_OVERFLOW | abi.ERR_FILL_LOG_FULL, 0, abi.ERR_BAD_ACTION]
    spread = torch.tensor(rng.uniform(1, 5, size=(T, N)))
    state_dev = torch.from_numpy(st.view(np.uint8).reshape(N, abi.ENV_STATE_DTYPE.itemsize).copy())
    want = episode_stats(rew, done, st, spread)
    got = episode_stats_dev(rew, done, state_dev, spread)
    assert torch.equal(torch.isnan(want), torch.isnan(got))
    assert torch.equal(torch.nan_to_num(want), torch.nan_to_num(got)), (want, got)
