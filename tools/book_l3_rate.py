#!/usr/bin/env python
"""Cost of the batched L3 read and write (LobSim.book_l3 = lobsim_get_book_dev, kernel k_get_book; LobSim.set_books =
lobsim_set_book_dev, kernel k_set_book).  Writes one JSON file.

    python tools/book_l3_rate.py --out DIR/book_l3_rate.json [--calls 200]

Cases (CUDA events around --calls back-to-back calls into preallocated tensors, after 20 warm-up calls; max_entries =
max_orders_per_side, so every order is read):
  a  book_l3 of 4 096 books of the headline replay config (10 levels, 64/256/32) after one hour of replay: flat blobs
  b  book_l3 and set_books of 65 536 envs of the rollout config after a reset and 20 env steps (set_books writes back the books
     book_l3 read, so every call does the same work)
  c  book_l3 and set_books of 8 192 books of the multiticker capacities (128/1024/64, 50 levels) after a replay
  d  the host alternative: dump_book x 2 sides and set_book, per env over 256 envs, extrapolated to 65 536 envs
Bytes per call are the bytes each call needs, computed from the books: book_l3 reads the header and the occupied book (a flat
blob's pool, or a sorted blob's level prices and ends and its orders) and writes the entries and counts; set_books reads the
entries in use and the counts and writes the occupied book, the agent tables, the header words and the status.  They are set
against a device-to-device copy measured in the same run."""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import bench  # noqa: E402
from book_depth_rate import card, copy_bandwidth  # noqa: E402
from rl4mm_b200 import abi, synthetic  # noqa: E402
from rl4mm_b200.device import LobSim  # noqa: E402


def time_calls(fn, calls, launches, sim):
    for _ in range(20):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = sim.launch_count
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    e1.synchronize()
    assert sim.launch_count - l0 == calls * launches
    return e0.elapsed_time(e1) * 1e3 / calls


def book_sizes(sim, count, entries):
    """Per env and side: orders, levels, agent entries (from a full read), and whether the blob is flat."""
    st = sim.state()
    flat = (st["reserved"] & 1).astype(bool)
    n = count.cpu().numpy().astype(np.int64)
    e = entries.cpu().numpy()
    levels = np.where(n > 0, e[..., 3].max(axis=2) + 1, 0).astype(np.int64)
    agents = ((e[..., 2].view(np.uint32) & abi.REF_AGENT) != 0).sum(axis=2).astype(np.int64)
    return flat, n, levels, agents


def record(sim, calls, note, with_set):
    E = sim.cfg.max_orders_per_side
    N = sim.n_envs
    out = sim.book_l3(E)
    flat, n, levels, agents = book_sizes(sim, *out)
    read = 128 + np.where(flat, 16 * n.sum(axis=1), (6 * levels + 2 + 8 * n).sum(axis=1))
    get_b = {"read_bytes": int(read.sum()), "written_bytes": N * (8 + 2 * E * 16)}
    res = {"envs": N, "max_entries": E, "calls": calls, "note": note, "kernel_path": sim.kernel_path, "blob_bytes": sim.state_bytes,
           "blob_total_mb": sim.state_bytes * N / 1e6, "flat_books": int(flat.sum()), "mean_orders_per_side": float(n.mean()),
           "mean_levels_per_side": float(levels.mean()), "mean_agent_orders_per_side": float(agents.mean())}
    us = time_calls(lambda: sim.book_l3(E, out=out), calls, 1, sim)
    res["book_l3"] = dict(get_b, us_per_call=us, bytes_per_s=(get_b["read_bytes"] + get_b["written_bytes"]) / (us * 1e-6))
    if with_set:
        count, entries = (t.clone() for t in out)
        status = sim.set_books(entries, count)
        assert bool((status == abi.SETBOOK_OK).all())
        set_b = {"read_bytes": int(8 * N + 16 * n.sum()),
                 "written_bytes": int((6 * levels + 8 * n + 12 * agents).sum() + N * (32 + 4))}
        us = time_calls(lambda: sim.set_books(entries, count, out=status), calls, 1, sim)
        assert bool((status == abi.SETBOOK_OK).all())
        res["set_books"] = dict(set_b, us_per_call=us, bytes_per_s=(set_b["read_bytes"] + set_b["written_bytes"]) / (us * 1e-6))
        after = sim.book_l3(E)
        assert torch.equal(after[0], count) and torch.equal(after[1], entries), "set_books(book_l3()) changed a book"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--n-msgs", type=int, default=10_000_000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the L3 read and write run on the GPU only"
    res = {"card": card(), "copy_bandwidth_bytes_per_s": copy_bandwidth()}
    stream = bench.make_stream(argparse.Namespace(n_msgs=args.n_msgs))

    # (a) headline replay config, one hour of replay: the books stay in the flat form between launches
    cfg = abi.default_cfg(n_envs=4096, n_levels=stream.n_levels, outer_levels=20, max_levels_per_side=64, max_orders_per_side=256,
                          max_agent_orders=32)
    sim = LobSim(cfg, 0)
    sim.load_stream(0, stream)
    sim.reset_book(0, 0)
    for _ in range(36000 // 2340 + 1):
        sim.replay(2340)
    res["a_flat_4096"] = record(sim, args.calls, "4 096 headline-config books after 16 launches of 2 340 grid steps; the blobs "
                                                 "(20 MB) fit in L2, so repeated calls read them from there", with_set=False)
    sim.close()

    # (b) + (d) rollout config, 65 536 envs
    rcfg = bench.rollout_cfg(65_536, stream)
    sim = LobSim(rcfg, 0)
    sim.load_stream(0, stream)
    rng = np.random.default_rng(1234)
    starts = ((1800 + rng.integers(0, 5 * 3600, size=65_536)) * stream.steps_per_second).astype(np.int32)
    sim.reset(0, starts)
    act = torch.full((65_536, sim.action_dim), 2.0, dtype=torch.float64, device="cuda")
    for _ in range(20):
        sim.step(act)
    res["b_rollout_65536"] = record(sim, args.calls, "65 536 rollout-config envs after a reset and 20 env steps (agent ladders "
                                                     "resting); blobs and entries larger than L2", with_set=True)
    t0 = time.perf_counter()
    books = []
    for env in range(256):
        books.append((sim.dump_book(env, 0), sim.dump_book(env, 1)))
    t_dump = (time.perf_counter() - t0) / 256
    t0 = time.perf_counter()
    for env, (buy, sell) in enumerate(books):
        sim.set_book(env, buy, sell)
    t_set = (time.perf_counter() - t0) / 256
    res["d_host_per_env"] = {"dump_book_x2_s_per_env_measured_over_256": t_dump, "set_book_s_per_env_measured_over_256": t_set,
                             "dump_book_x2_s_for_65536_envs_extrapolated": t_dump * 65_536,
                             "set_book_s_for_65536_envs_extrapolated": t_set * 65_536,
                             "note": "host round trips per env on the 65 536-env rollout handle; the 65 536-env figures are "
                                     "extrapolated, not measured"}
    sim.close()

    # (c) multiticker capacities
    streams = [synthetic.generate(synthetic.heavy_cancel_ticker(seed=k, n_msgs=1_000_000)) for k in range(8)]
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100000, 0, 5000)]
    ccfg = abi.default_cfg(n_envs=8192, n_levels=50, outer_levels=20, max_levels_per_side=128, max_orders_per_side=1024,
                           max_agent_orders=64, features=feats, episode_steps=18000, warmup_steps=0)
    sim = LobSim(ccfg, 0)
    for k, s in enumerate(streams):
        sim.load_stream(k, s)
    sid = (np.arange(8192) % 8).astype(np.int32)
    span = min(s.n_seconds for s in streams) - 200
    cst = (np.random.default_rng(555).integers(0, span, size=8192) * streams[0].steps_per_second).astype(np.int32)
    sim.reset_book(sid, cst)
    sim.replay(1170)
    assert np.all(sim.state()["err"] == 0)
    res["c_multiticker_8192"] = record(sim, args.calls, "8 192 books, 128/1024/64 capacities, 8 heavy-cancel streams of 1e6 "
                                                        "messages, after 1 170 grid steps of replay", with_set=True)
    sim.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
