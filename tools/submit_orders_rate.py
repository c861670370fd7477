#!/usr/bin/env python
"""Cost of the batched order submission (LobSim.submit_orders = lobsim_submit_orders_dev): the straight-line kernel
k_submit_orders<LT> of the compiled layouts against the runtime-layout k_submit_orders_general (LOBSIM_FORCE_GENERAL=1).  Writes
one JSON file.

    python tools/submit_orders_rate.py --out DIR/submit_orders_rate.json [--calls 40]

The workload is a ladder refresh: each submitting env cancels every resting agent order by id (DELETE with volume None), then
places K/2 limit orders of 10 shares at the quote levels (best price and up to 3 ticks behind, both sides), 1 in 8 of them
(counted over the whole batch) at the opposite best price (crossing).  The rows are built on the device from agent_orders() and book_depth() before each call
(untimed); before each timed call L2 is flushed by writing a 256 MiB buffer, and the call is timed alone with CUDA events.  The
straight-line and general handles run the same history and are timed alternately, call by call.
  a  65 536 envs of the rollout config (64/256/64) after a reset and a 20-step FixedAction rollout: K = 8 and 32, all envs
     submitting, and 1 % of the envs submitting (count 0 elsewhere)
  b  8 192 books of the multiticker capacities (128/1024/64, heavy-cancel streams) after a reset and a 20-step FixedAction
     rollout: K = 32
  c  context: one lobsim_step of the (a) handle (CUDA events), and lobsim_process_orders with the same orders on 1 024 envs
     (host wall clock including its synchronise), extrapolated to 65 536 envs and labelled as such
After timing, sampled envs of each handle are checked against a twin handle that applies the same rows through
process_orders: the twin gets the envs' books by set_book, both apply one more refresh, and the books, the agent orders, the
rest pattern of the refs, the fills and the error bits must agree."""
import argparse
import ctypes
import json
import os
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench  # noqa: E402
from rl4mm_b200 import abi, synthetic  # noqa: E402
from rl4mm_b200.device import LobSim  # noqa: E402
from tools.book_depth_rate import card  # noqa: E402

FIXED = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 2, 1, 2, 0))
TICK = 100


def make_handle(cfg, streams, general):
    os.environ["LOBSIM_FORCE_GENERAL"] = "1" if general else "0"
    sim = LobSim(cfg, 0)
    os.environ.pop("LOBSIM_FORCE_GENERAL")
    for k, s in enumerate(streams):
        sim.load_stream(k, s)
    return sim


def refresh_orders(sim, K, active):
    """The ladder refresh rows [N, K, 8] on the device: up to K/2 cancels of the env's resting agent orders (by id, volume None),
    then K/2 limits; rows of inactive envs get count 0."""
    N, H = sim.n_envs, K // 2
    count, price, _, ids = sim.agent_orders(H, queue=False)
    best = sim.book_depth(1)[0][:, :, 0].to(torch.int64)                         # [N, 2]
    dev = price.device
    slot = torch.arange(H, device=dev)
    # the first H resting orders over both sides (buy side first), as cancels
    nb = count[:, 0].clamp(max=H)[:, None]
    from_buy = slot[None, :] < nb
    j = torch.where(from_buy, slot[None, :], slot[None, :] - nb).clamp(max=H - 1)
    live = torch.where(from_buy, True, (slot[None, :] - nb) < count[:, 1].clamp(max=H)[:, None])
    c_side = (~from_buy).to(torch.int64)
    c_price = torch.where(from_buy, price[:, 0].gather(1, j), price[:, 1].gather(1, j)).to(torch.int64)
    c_id = torch.where(from_buy, ids[:, 0].gather(1, j), ids[:, 1].gather(1, j)).to(torch.int64)
    c_type = torch.where(live, abi.MSG_DELETE, 0)
    q = torch.arange(H, device=dev)
    l_side = (q % 2)[None, :].expand(N, H)
    behind = ((q // 2) % 4)[None, :].expand(N, H)
    cross = (torch.arange(N, device=dev)[:, None] * H + q[None, :]) % 8 == 7   # 1 in 8 limits over the whole batch
    own = best.gather(1, l_side)
    opp = best.gather(1, 1 - l_side)
    away = torch.where(l_side == 0, -TICK, TICK) * behind
    l_price = torch.where(cross, opp, own + away)
    orders = abi.pack_orders(torch.cat([c_type, torch.full((N, H), abi.MSG_LIMIT, device=dev)], 1),
                             torch.cat([c_side, l_side], 1), torch.cat([c_price, l_price], 1),
                             torch.cat([torch.zeros((N, H), dtype=torch.int64, device=dev), torch.full((N, H), 10, device=dev)], 1),
                             0, torch.cat([c_id, torch.zeros((N, H), dtype=torch.int64, device=dev)], 1))
    cnt = torch.where(active, K, 0).to(torch.int32)
    return orders, cnt


def cleanup(sim):
    """Cancel every resting agent order (so that the refresh rows hold them all from the first timed call on)."""
    A = sim.cfg.max_agent_orders
    count, price, _, ids = sim.agent_orders(A, queue=False)
    N = sim.n_envs
    live = torch.arange(A, device=price.device)[None, None, :] < count[:, :, None]
    side = torch.arange(2, device=price.device)[None, :, None].expand(N, 2, A)
    o = abi.pack_orders(torch.where(live, abi.MSG_DELETE, 0).reshape(N, 2 * A), side.reshape(N, 2 * A), price.reshape(N, 2 * A),
                        0, 0, ids.reshape(N, 2 * A))
    sim.submit_orders(o, refs=False)


def time_alternating(handles, K, active, calls, flush):
    """Per handle: `calls` timed refreshes (CUDA events around the one launch, L2 flushed before it), alternated call by call."""
    times = {name: [] for name in handles}
    outs = {}
    for i in range(calls + 5):
        for name, sim in (handles.items() if i % 2 == 0 else reversed(handles.items())):
            orders, cnt = refresh_orders(sim, K, active)
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = sim.launch_count
            e0.record()
            outs[name] = sim.submit_orders(orders, cnt, max_fills=64)
            e1.record()
            e1.synchronize()
            assert sim.launch_count == l0 + 1
            if i >= 5:                                     # warm-up calls
                times[name].append(e0.elapsed_time(e1) * 1e3)
    return times, outs


def summary(times, n_active, K, outs, sim):
    t = np.array(times)
    refs, _, nf = outs
    return {"us_median": float(np.median(t)), "us_min": float(t.min()), "us_max": float(t.max()), "calls": len(t),
            "submitting_envs": int(n_active), "orders_per_submitting_env": K,
            "orders_per_s": n_active * K / (np.median(t) * 1e-6), "kernel_path": sim.kernel_path,
            "rested_per_call": int((refs.view(torch.int32) != 0).sum()), "fills_per_call": int(nf.sum())}


def check_twin(sim, K, active, n_sample, rng):
    """Sampled envs of `sim` against a twin that gets their books by set_book and the same rows through process_orders."""
    cand = np.flatnonzero(active.cpu().numpy() & (sim.errors() == 0))      # (set_book would revive a dead env)
    envs = np.sort(rng.choice(cand, size=min(n_sample, len(cand)), replace=False))
    cfg = abi.default_cfg(n_envs=len(envs), n_levels=sim.cfg.n_levels, max_levels_per_side=sim.cfg.max_levels_per_side,
                          max_orders_per_side=sim.cfg.max_orders_per_side, max_agent_orders=sim.cfg.max_agent_orders)
    twin = LobSim(cfg, 0)
    for i, e in enumerate(envs):
        twin.set_book(i, sim.dump_book(int(e), 0), sim.dump_book(int(e), 1))
    err0 = sim.errors()[envs]
    orders, cnt = refresh_orders(sim, K, active)
    refs, fills, nf = sim.submit_orders(orders, cnt, max_fills=256)
    rows = orders.cpu().numpy().view(abi.ORDER_DTYPE).reshape(sim.n_envs, K)[envs].copy()
    rows["env"] = np.arange(len(envs))[:, None]
    flat = rows.reshape(-1)
    flat = flat[(flat["type"] >= 1) & (flat["type"] <= 4)]
    tf, trefs = twin.process_orders(flat, max_fills=1 << 16)
    refs = refs.view(torch.int32).cpu().numpy().view(np.uint32)[envs]
    nf = nf.cpu().numpy()[envs]
    fl = fills.cpu().numpy()[envs]
    live = (rows["type"] >= 1) & (rows["type"] <= 4)
    dref = refs[live]
    assert np.array_equal(dref == 0, trefs == 0) and np.array_equal(dref == 0xFFFFFFFF, trefs == 0xFFFFFFFF)
    got = np.concatenate([fl[i].copy().view(abi.FILL_DTYPE).reshape(-1)[: nf[i]] for i in range(len(envs))])
    key = ["list", "direction", "price", "volume", "is_market"]
    assert np.array_equal(got[key], tf[key]), "fills"
    assert np.array_equal(sim.errors()[envs] & ~err0, twin.errors() & ~np.uint32(0)), "error bits"
    for i, e in enumerate(envs):
        for side in (0, 1):
            a, b = sim.dump_book(int(e), side), twin.dump_book(i, side)
            assert np.array_equal(a[["price", "volume", "level"]], b[["price", "volume", "level"]]), (e, side)
            assert np.array_equal(a["ref"] & abi.REF_AGENT, b["ref"] & abi.REF_AGENT), (e, side)
            x, y = sim.dump_agent_orders(int(e), side), twin.dump_agent_orders(i, side)
            assert np.array_equal(x[["price", "volume"]], y[["price", "volume"]]), (e, side)
    twin.close()
    return {"envs_checked": int(len(envs)), "orders_checked": int(len(flat)), "fills_checked": int(len(tf)), "ok": True}


def run_case(res, tag, handles, K, active, calls, flush, rng):
    times, outs = time_alternating(handles, K, active, calls, flush)
    n_active = int(active.sum())
    for name, sim in handles.items():
        res[f"{tag}_{name}"] = summary(times[name], n_active, K, outs[name], sim)
    f, g = (np.median(times[n]) for n in handles)
    res[f"{tag}_general_over_straight_line"] = float(g / f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=40)
    ap.add_argument("--n-msgs", type=int, default=10_000_000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the order submission runs on the GPU only"
    res = {"card": card(), "l2": "flushed before every timed call by writing a 256 MiB buffer",
           "workload": "ladder refresh: cancel every resting agent order by id (volume None), then K/2 limits of 10 shares at "
                       "the quote levels (best and up to 3 ticks behind, both sides), 1 in 8 at the opposite best (crossing)"}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rng = np.random.default_rng(99)
    stream = bench.make_stream(argparse.Namespace(n_msgs=args.n_msgs))

    # (a) rollout config, 65 536 envs
    N = 65_536
    rcfg = bench.rollout_cfg(N, stream)
    starts = ((1800 + np.random.default_rng(1234).integers(0, 5 * 3600, size=N)) * stream.steps_per_second).astype(np.int32)
    handles = {"straight_line": make_handle(rcfg, [stream], False), "general": make_handle(rcfg, [stream], True)}
    assert handles["straight_line"].kernel_path == "fast" and handles["general"].kernel_path == "general"
    for sim in handles.values():
        sim.reset(0, starts)
        sim.rollout(20, FIXED, want_obs=False)
        cleanup(sim)
    a, b = handles.values()
    assert torch.equal(a.state_dev(), b.state_dev()), "the two handles start from the same state"
    all_on = torch.ones(N, dtype=torch.bool, device="cuda")
    one_pct = torch.zeros(N, dtype=torch.bool, device="cuda")
    one_pct[torch.from_numpy(rng.choice(N, size=N // 100, replace=False)).cuda()] = True
    for K in (8, 32):
        run_case(res, f"a_rollout_65536_K{K}", handles, K, all_on, args.calls, flush, rng)
        run_case(res, f"a_rollout_65536_K{K}_1pct", handles, K, one_pct, args.calls, flush, rng)
    assert torch.equal(a.state_dev(), b.state_dev()), "both kernels computed the same books"
    res["a_check_straight_line"] = check_twin(a, 32, all_on, 256, rng)
    res["a_check_general"] = check_twin(b, 32, all_on, 256, rng)

    # (c) context: one env step of the same handle; process_orders on 1 024 envs
    sim = a
    act = torch.full((N, sim.action_dim), 2.0, dtype=torch.float64, device="cuda")
    steps = []
    for i in range(25):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sim.step(act)
        e1.record()
        e1.synchronize()
        if i >= 5:
            steps.append(e0.elapsed_time(e1) * 1e3)
    res["c_step_65536"] = {"us_median": float(np.median(steps)), "us_min": float(np.min(steps)), "steps": len(steps),
                           "note": "one lobsim_step of the (a) straight-line handle, CUDA events, L2 flushed before each"}
    orders, _ = refresh_orders(sim, 32, all_on)
    rows = orders.cpu().numpy().view(abi.ORDER_DTYPE).reshape(N, 32)[:1024].reshape(-1)
    rows = rows[(rows["type"] >= 1) & (rows["type"] <= 4)].copy()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sim.process_orders(rows, max_fills=1 << 16)
    dt = time.perf_counter() - t0
    res["c_process_orders_1024"] = {"s_measured_1024_envs": dt, "orders": int(len(rows)), "s_for_65536_envs_extrapolated": dt * 64,
                                    "note": "lobsim_process_orders with the K = 32 refresh rows of the first 1 024 envs: host wall "
                                            "clock including its H2D copy and synchronise; the 65 536-env figure is extrapolated "
                                            "(x 64), not measured"}
    for sim in handles.values():
        sim.close()

    # (b) multiticker capacities, 8 192 books
    streams = [synthetic.generate(synthetic.heavy_cancel_ticker(seed=k, n_msgs=1_000_000)) for k in range(8)]
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100000, 0, 5000)]
    ccfg = abi.default_cfg(n_envs=8192, n_levels=50, outer_levels=20, max_levels_per_side=128, max_orders_per_side=1024,
                           max_agent_orders=64, features=feats, episode_steps=18000, warmup_steps=0)
    sid = (np.arange(8192) % 8).astype(np.int32)
    span = min(s.n_seconds for s in streams) - 200
    cst = (np.random.default_rng(555).integers(0, span, size=8192) * streams[0].steps_per_second).astype(np.int32)
    handles = {"straight_line": make_handle(ccfg, streams, False), "general": make_handle(ccfg, streams, True)}
    for sim in handles.values():
        sim.reset(sid, cst)
        sim.rollout(20, FIXED, want_obs=False)
        cleanup(sim)
    all_on = torch.ones(8192, dtype=torch.bool, device="cuda")
    run_case(res, "b_multiticker_8192_K32", handles, 32, all_on, args.calls, flush, rng)
    a, b = handles.values()
    assert torch.equal(a.state_dev(), b.state_dev()), "both kernels computed the same books"
    res["b_check_straight_line"] = check_twin(a, 32, all_on, 256, rng)
    res["b_errors"] = int(np.count_nonzero(a.state()["err"]))
    for sim in handles.values():
        sim.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
