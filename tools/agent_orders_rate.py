#!/usr/bin/env python
"""Cost of the batched agent-order read (LobSim.agent_orders = lobsim_get_agent_orders_dev, kernel k_agent_orders).  Writes one
JSON file.

    python tools/agent_orders_rate.py --out DIR/agent_orders_rate.json [--calls 1000]

Cases (CUDA events around --calls back-to-back calls into preallocated tensors, after 50 warm-up calls):
  a  65 536 envs of the rollout config after a reset and a 20-step FixedAction rollout (agent ladders resting):
     max_orders = max_agent_orders (64), with queue positions and without
  b  8 192 books of the multiticker capacities (128/1024/64, 50 levels, heavy-cancel streams) after a reset and a 20-step
     FixedAction rollout, with queue positions
  c  65 536 rollout envs: step alone against step + agent_orders(), alternated in one run, per step
  d  the host alternative: dump_agent_orders x 2 sides, per env over 256 envs, extrapolated to 65 536 envs
Bytes per call are a lower bound of what the read needs, computed from what it returned: the 128-byte header, 12 B per agent
order read from the agent table, with queue positions 8 B per FIFO entry up to the last agent order of each level walked
(the binary searches over the level prices are not counted), and the outputs; against a device-to-device copy measured in the
same run."""
import argparse
import ctypes
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench  # noqa: E402
from rl4mm_b200 import abi, synthetic  # noqa: E402
from rl4mm_b200.device import LobSim  # noqa: E402
from tools.book_depth_rate import card, copy_bandwidth  # noqa: E402

FIXED = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 2, 1, 2, 0))


def time_calls(sim, calls, queue):
    out = sim.agent_orders(queue=queue)
    for _ in range(50):
        sim.agent_orders(queue=queue, out=out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = sim.launch_count
    e0.record()
    for _ in range(calls):
        sim.agent_orders(queue=queue, out=out)
    e1.record()
    e1.synchronize()
    assert sim.launch_count - l0 == calls
    return e0.elapsed_time(e1) * 1e3 / calls, out


def bytes_per_call(out, queue):
    count = out[0].cpu().numpy().astype(np.int64)
    A = out[1].shape[2]
    m = np.minimum(count, A)
    read = 128 * len(count) + 12 * int(m.sum())
    walked = 0
    if queue:
        level, ahead = out[4].cpu().numpy(), out[5].cpu().numpy().astype(np.int64)
        for env in range(len(count)):
            for side in (0, 1):
                lv, ah = level[env, side], ahead[env, side]
                for j in np.unique(lv[lv >= 0]):
                    walked += int(ah[lv == j].max()) + 1
        read += 8 * walked
    written = 8 * len(count) + (24 if queue else 12) * 2 * A * len(count)
    return {"read_bytes": read, "written_bytes": written, "mean_agent_orders_per_env": float(count.sum(axis=1).mean()),
            "max_agent_orders_per_side": int(count.max()), "fifo_entries_walked_per_env": walked / len(count)}


def record(sim, calls, queue, note):
    us, out = time_calls(sim, calls, queue)
    b = bytes_per_call(out, queue)
    return dict(b, envs=sim.n_envs, max_orders=sim.cfg.max_agent_orders, queue=queue, calls=calls, us_per_call=us, note=note,
                bytes_per_s=(b["read_bytes"] + b["written_bytes"]) / (us * 1e-6), kernel_path=sim.kernel_path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=1000)
    ap.add_argument("--n-msgs", type=int, default=10_000_000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the agent-order read runs on the GPU only"
    res = {"card": card(), "copy_bandwidth_bytes_per_s": copy_bandwidth()}
    stream = bench.make_stream(argparse.Namespace(n_msgs=args.n_msgs))

    # (a) + (c) rollout config, 65 536 envs, agent ladders resting after a fused FixedAction rollout
    rcfg = bench.rollout_cfg(65_536, stream)
    sim = LobSim(rcfg, 0)
    sim.load_stream(0, stream)
    rng = np.random.default_rng(1234)
    starts = ((1800 + rng.integers(0, 5 * 3600, size=65_536)) * stream.steps_per_second).astype(np.int32)
    sim.reset(0, starts)
    sim.rollout(20, FIXED, want_obs=False)
    note = "65 536 rollout-config envs after a reset and a 20-step FixedAction rollout; blobs larger than L2"
    res["a_rollout_65536_queue"] = record(sim, args.calls, True, note)
    res["a_rollout_65536_no_queue"] = record(sim, args.calls, False, note)
    act = torch.full((65_536, sim.action_dim), 2.0, dtype=torch.float64, device="cuda")
    out = sim.agent_orders()
    alone, both = [], []
    for rnd in range(40):
        for with_read in ((False, True) if rnd % 2 == 0 else (True, False)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                sim.step(act)
                if with_read:
                    sim.agent_orders(out=out)
            e1.record()
            e1.synchronize()
            if rnd >= 4:
                (both if with_read else alone).append(e0.elapsed_time(e1) / 10)
    a_ms, b_ms = float(np.median(alone)), float(np.median(both))
    res["c_step_overhead_65536"] = {
        "step_ms_median": a_ms, "step_plus_read_ms_median": b_ms, "overhead_ms_per_step": b_ms - a_ms,
        "overhead_fraction": (b_ms - a_ms) / a_ms, "rounds": len(alone), "steps_per_round": 10,
        "step_ms_spread": [float(np.min(alone)), float(np.max(alone))], "step_plus_read_ms_spread": [float(np.min(both)), float(np.max(both))],
        "note": "rounds of 10 env steps with and without an agent_orders() (queue positions, max_orders 64) after each step, "
                "alternated; medians"}

    # (d) host alternative: lobsim_dump_agent_orders of both sides, per env
    t0 = time.perf_counter()
    for env in range(256):
        sim.dump_agent_orders(env, 0)
        sim.dump_agent_orders(env, 1)
    per_env = (time.perf_counter() - t0) / 256
    res["d_host_dump_agent_orders"] = {"s_per_env_measured_over_256": per_env, "s_for_65536_envs_extrapolated": per_env * 65_536,
                                       "note": "dump_agent_orders x 2 sides per env (host round trips, no queue positions); the "
                                               "65 536-env figure is extrapolated, not measured"}
    sim.close()

    # (b) multiticker capacities
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
    sim.reset(sid, cst)
    sim.rollout(20, FIXED, want_obs=False)
    res["b_multiticker_8192_queue"] = record(sim, args.calls, True, "8 192 books, 128/1024/64 capacities, 8 heavy-cancel streams "
                                                                    "of 1e6 messages, after a reset and a 20-step FixedAction rollout")
    res["b_multiticker_8192_queue"]["errors"] = int(np.count_nonzero(sim.state()["err"]))
    sim.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
