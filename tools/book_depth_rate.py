#!/usr/bin/env python
"""Cost of the batched L2 depth read (LobSim.book_depth = lobsim_get_depth_dev, kernel k_book_depth).  Writes one JSON file.

    python tools/book_depth_rate.py --out DIR/book_depth_rate.json [--calls 1000]

Cases (CUDA events around --calls back-to-back calls into preallocated tensors, after 50 warm-up calls):
  a  4 096 books of the headline replay config (10 levels, 64/256/32) after one hour of replay: flat blobs, depth 10
  b  65 536 envs of the rollout config after a reset and 20 env steps: sorted blobs, depth 10
  c  8 192 books of the multiticker capacities (128/1024/64, 50 levels, heavy-cancel streams) after a replay: depth 50
  d  65 536 rollout envs: step_torch alone against step_torch + book_depth(10), alternated in one run, per step
  e  the host alternative: dump_book x 2 sides, per env over 256 envs, extrapolated to 65 536 envs
Bytes per call are the bytes the read needs, computed from the books it read (header, level prices and ends, the orders of the
top `depth` levels or the whole flat pool, the outputs), against a device-to-device copy measured in the same run."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench  # noqa: E402
from rl4mm_b200 import abi, synthetic  # noqa: E402
from rl4mm_b200.device import LobSim  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except OSError:
        out = ""
    return {"nvidia_smi": {k: v.strip() for k, v in zip(q.split(","), out.split(","))} if out else None,
            "torch_name": torch.cuda.get_device_name(0)}


def copy_bandwidth():
    """Device-to-device copy of 2 GiB (read + write bytes over time), best of 5."""
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    best = 0.0
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * a.numel() / (e0.elapsed_time(e1) * 1e-3))
    del a, b
    return best


def time_calls(sim, depth, calls, orders=True, agent=True):
    out = sim.book_depth(depth, orders=orders, agent=agent)
    for _ in range(50):
        sim.book_depth(depth, orders=orders, agent=agent, out=out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = sim.launch_count
    e0.record()
    for _ in range(calls):
        sim.book_depth(depth, orders=orders, agent=agent, out=out)
    e1.record()
    e1.synchronize()
    assert sim.launch_count - l0 == calls
    return e0.elapsed_time(e1) * 1e3 / calls, out


def bytes_per_call(sim, depth, out):
    """Bytes the read needs: per env the 128-byte header; per side of a flat blob the pool (16 B per order), of a sorted blob
    the top levels' prices (4 B) and ends (2 B, one more for the start) and their orders (8 B); the four outputs (24 B per level)."""
    st = sim.state()
    flat = (st["reserved"] & 1).astype(bool)
    n_side = np.stack([(st["reserved"] >> 8) & 0xFFF, (st["reserved"] >> 20) & 0xFFF], 1).astype(np.int64)
    orders = out[2].cpu().numpy().astype(np.int64)
    levels = (out[0].cpu().numpy() != abi.NO_PRICE).sum(axis=2)
    sorted_bytes = (6 * levels + 2 + 8 * orders.sum(axis=2)).sum(axis=1)
    read = 128 + np.where(flat, 16 * n_side.sum(axis=1), sorted_bytes)
    written = 24 * 2 * depth
    return {"read_bytes": int(read.sum()), "written_bytes": int(written * sim.n_envs), "flat_books": int(flat.sum()),
            "mean_orders_read_per_env": float(np.where(flat, n_side.sum(axis=1), orders.sum(axis=(1, 2))).mean()),
            "mean_levels_per_side": float(levels.mean())}


def record(sim, depth, calls, note):
    us, out = time_calls(sim, depth, calls)
    b = bytes_per_call(sim, depth, out)
    return dict(b, envs=sim.n_envs, depth=depth, calls=calls, us_per_call=us, note=note,
                bytes_per_s=(b["read_bytes"] + b["written_bytes"]) / (us * 1e-6),
                blob_bytes=sim.state_bytes, blob_total_mb=sim.state_bytes * sim.n_envs / 1e6, kernel_path=sim.kernel_path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=1000)
    ap.add_argument("--n-msgs", type=int, default=10_000_000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the depth read runs on the GPU only"
    res = {"card": card(), "copy_bandwidth_bytes_per_s": copy_bandwidth()}
    ns = argparse.Namespace(n_msgs=args.n_msgs)
    stream = bench.make_stream(ns)

    # (a) headline replay config, one hour of replay: the books stay in the flat form between launches
    cfg = abi.default_cfg(n_envs=4096, n_levels=stream.n_levels, outer_levels=20, max_levels_per_side=64, max_orders_per_side=256,
                          max_agent_orders=32)
    sim = LobSim(cfg, 0)
    sim.load_stream(0, stream)
    sim.reset_book(0, 0)
    for _ in range(36000 // 2340 + 1):
        sim.replay(2340)
    res["a_flat_4096_depth10"] = record(sim, 10, args.calls, "4 096 headline-config books after 16 launches of 2 340 grid steps (37 440 steps, ~1 h of the day); "
                                                              "the blobs (20 MB) fit in L2, so repeated calls read them from there")
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
    res["b_sorted_65536_depth10"] = record(sim, 10, args.calls, "65 536 rollout-config envs after a reset and 20 env steps; "
                                                                "blobs larger than L2")
    out = sim.book_depth(10, orders=True, agent=True)
    alone, both = [], []
    for rnd in range(40):
        for with_depth in ((False, True) if rnd % 2 == 0 else (True, False)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                sim.step(act)
                if with_depth:
                    sim.book_depth(10, orders=True, agent=True, out=out)
            e1.record()
            e1.synchronize()
            if rnd >= 4:
                (both if with_depth else alone).append(e0.elapsed_time(e1) / 10)
    a_ms, b_ms = float(np.median(alone)), float(np.median(both))
    res["d_step_overhead_65536_depth10"] = {
        "step_ms_median": a_ms, "step_plus_depth_ms_median": b_ms, "overhead_ms_per_step": b_ms - a_ms,
        "overhead_fraction": (b_ms - a_ms) / a_ms, "rounds": len(alone), "steps_per_round": 10,
        "step_ms_spread": [float(np.min(alone)), float(np.max(alone))], "step_plus_depth_ms_spread": [float(np.min(both)), float(np.max(both))],
        "note": "rounds of 10 env steps with and without a book_depth(10, orders, agent) after each step, alternated; medians"}

    # (e) host alternative: lobsim_dump_book of both sides, per env
    t0 = time.perf_counter()
    for env in range(256):
        sim.dump_book(env, 0)
        sim.dump_book(env, 1)
    per_env = (time.perf_counter() - t0) / 256
    res["e_host_dump_book"] = {"s_per_env_measured_over_256": per_env, "s_for_65536_envs_extrapolated": per_env * 65_536,
                               "note": "dump_book x 2 sides per env (host round trips); the 65 536-env figure is extrapolated, "
                                       "not measured"}
    sim.close()

    # (c) multiticker capacities, depth 50
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
    res["c_multiticker_8192_depth50"] = record(sim, 50, args.calls, "8 192 books, 128/1024/64 capacities, 8 heavy-cancel streams "
                                                                   "of 1e6 messages, after 1 170 grid steps of replay")
    sim.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
