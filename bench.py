#!/usr/bin/env python
"""Benchmark of the LOB simulation step (BASELINE.json metric: LOB messages/s and env steps/s, whole box).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload all|replay|rollout|collect|multiticker]
                    [--dump-outputs DIR]

ONE JSON line.  The headline (`value`, `e2e`, `roofline`, `cpu_baseline`) is BASELINE.json configs[1]: a synthetic
SPY-shaped day (10 levels, 1e7 messages, seed 0) replayed through 4096 batched books per GPU (weak scaling); one bench
"step" = every book advances `--segment-steps` simulation steps (default 2340 x 0.1 s = 1 % of the day, ~1e5 messages per
book).  The same line carries one sub-record per other BASELINE config, each with its own value / roofline / e2e:

  "rollout"      configs[2]: HistoricalOrderbookEnvironment rollouts, 65 536 envs per GPU, a torch MLP Beta policy between
                 steps (one lobsim_step launch per env step), PnL reward, default full_state features -> env steps/s
  "collect"      configs[3]: PPO-style collection, 131 072 envs per GPU (1 048 576 on 8 GPUs), T = 128 fused Teradactyl
                 rollout + episode statistics + NCCL all-gather of the [N, 8] f32 stats INSIDE the timed region; the
                 collective's own time is reported next to it
  "multiticker"  configs[4]: 8 synthetic tickers, 50 levels, heavy cancel / modify flow, deep queues, 8 192 books per GPU:
                 replay (messages/s) and a fused FixedActionAgent([1,2,1,2]) rollout (env steps/s)
  "replay_varied_starts", "books_curve"   the headline replay with per-book random start seconds, and at 4096 / 8192 /
                 16384 books per GPU (N = 1 only)

Timing: CUDA events on the launching stream around the timed calls, inputs resident in HBM (`value`); the same work
through the host-buffer C-ABI calls (`lobsim_replay_host` / `lobsim_step_host`, pinned host memory, H2D + D2H inside the
timed region) gives `e2e`.  L2 is flushed (256 MiB write) between timed iterations.  Multi-GPU: one process per GPU
(torchrun), books sharded by rank; times are the max over ranks.

`--dump-outputs DIR` writes what the timed calls returned in their last step, one DIR/<name>.npy per array (float64, or
float32 where the call returns float32): the book states after the replays, the books of 16 sampled envs, and the rollout
tensors of a fixed sample of 1024 envs.  Every input is generated from fixed seeds, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import traceback
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

ALGO_BYTES_PER_MSG = 16          # packed record (SURVEY.md section 8d)
ALGO_BYTES_PER_STEP_REPLAY = 4   # CSR step offset
ALGO_BYTES_PER_STEP_ENV = 65     # action 4x4 B + obs 10x4 B + reward 4 B + done 1 B + CSR offset 4 B
S_STATE_L10 = 1216               # SURVEY.md section 8d book-state size for L=10 (round trip per launch)
S_STATE_L50 = 10816              # ... for L=50, mean queue 12
CPU_SAMPLE_SECONDS = 10.0        # bounded cpu_baseline sample (the contract asks for about 10-30 s of CPU work)
PY_REFERENCE_MSGS_PER_CORE = 4.9e4   # BASELINE.md section 2: the CPython reference's Exchange.process_order loop (survey container)
PY_REFERENCE_ENV_STEPS_PER_CORE = (42, 72)
HBM_PEAK_GBS = 7700.0            # HBM3e bandwidth of one B200 (NVIDIA HGX B200 data sheet): the roofline's denominator
HBM_PEAK_SOURCE = "NVIDIA HGX B200 data sheet, one GPU (not measured)"
DUMP_SAMPLE_ENVS = 1024          # --dump-outputs: envs kept of the large per-env rollout outputs (fixed seeded sample)
DUMP_MAX_BYTES = 64 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "replay", "rollout", "collect", "multiticker"])
    ap.add_argument("--envs-per-gpu", type=int, default=4096, help="books per GPU of the headline replay")
    ap.add_argument("--rollout-envs", type=int, default=65_536)
    ap.add_argument("--collect-envs", type=int, default=131_072)
    ap.add_argument("--multiticker-envs", type=int, default=8192)
    ap.add_argument("--multiticker-msgs", type=int, default=5_000_000)
    ap.add_argument("--n-msgs", type=int, default=10_000_000)
    ap.add_argument("--segment-steps", type=int, default=2340)
    ap.add_argument("--sub-steps", type=int, default=4, help="timed steps of each sub-record (warm-up: 3)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed calls returned in their last step as "
                                                           "DIR/<name>.npy (float64 / float32), to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def sub_schedule(args):
    """(timed steps, warm-up steps) of the rollout / collect / multiticker records: --steps / --warmup when that workload
    was asked for alone, else --sub-steps after 3 warm-up steps."""
    return (args.steps, args.warmup) if args.workload != "all" else (args.sub_steps, 3)


def ncu_traffic(key: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of the same
    command (profiles/traffic.json), or None."""
    p = ROOT / "profiles" / "traffic.json"
    try:
        return json.loads(p.read_text())[key]["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        return None


def roofline(algo_bytes_per_launch: float, launch_ms: float, kernel: str, traffic_key: str = None, **extra):
    achieved = algo_bytes_per_launch / (launch_ms / 1e3) / 1e9
    r = {"bound": "hbm", "achieved": achieved, "peak": HBM_PEAK_GBS, "unit": "GB/s", "frac": achieved / HBM_PEAK_GBS,
         "traffic": ncu_traffic(traffic_key) if traffic_key else None, "peak_source": HBM_PEAK_SOURCE, "kernel": kernel,
         "algorithmic_bytes_per_launch": algo_bytes_per_launch, "launch_ms": launch_ms}
    r.update(extra)
    return r


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_stream(args):
    from rl4mm_b200 import synthetic

    return synthetic.generate(synthetic.spy_day(seed=0, n_msgs=args.n_msgs, duration_s=23_400))


# ======================================================================================================================
#  CPU arm: the oracle (C port of the reference algorithm) on the host cores
# ======================================================================================================================
def _pinned_pool(threads: int):
    """Thread pool with worker i pinned to host CPU i: freshly created threads otherwise start on their parent's CPU
    and this VM's scheduler takes about a second to spread them, which made 8 threads measure like 1."""
    import itertools
    from concurrent.futures import ThreadPoolExecutor

    cpus = sorted(os.sched_getaffinity(0))
    counter, lock = itertools.count(), threading.Lock()

    def pin():
        with lock:
            i = next(counter)
        try:
            os.sched_setaffinity(0, {cpus[i % len(cpus)]})       # pid 0 = the calling thread
        except OSError:
            pass

    return ThreadPoolExecutor(threads, initializer=pin)


def cpu_oracle_throughput(stream, sample_steps: int, threads: int, reps: int = 1):
    """`threads` books replay the first `sample_steps` grid steps of the stream concurrently (ctypes releases the GIL)."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import abi

    cfg = abi.default_cfg(n_levels=stream.n_levels, outer_levels=20)
    oracles = [Oracle(cfg, stream) for _ in range(threads)]
    msgs = int(stream.step_off[sample_steps])

    def work(o):
        for _ in range(reps):
            o.reset_book(0)
            o.replay(sample_steps)
        return int(o.state()["err"])

    with _pinned_pool(threads) as ex:
        list(ex.map(work, oracles[:1]))  # warm the caches / page in
        t0 = time.perf_counter()
        errs = list(ex.map(work, oracles))
        dt = time.perf_counter() - t0
    assert not any(errs), errs
    return threads * reps * msgs / dt, threads * reps * sample_steps / dt, dt, msgs


def cpu_oracle_env_throughput(stream, cfg, threads: int, n_steps: int, seconds: float = CPU_SAMPLE_SECONDS):
    """Env steps/s of the oracle (C port of the reference env step) on `threads` host threads: one env per task,
    same features / rewards as the GPU run, random Beta actions; enough tasks for about `seconds` of work."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import abi

    c1 = abi.Cfg.from_buffer_copy(bytes(cfg))
    c1.n_envs = 1
    sps = stream.steps_per_second
    agent = abi.Agent(kind=abi.AGENT_EXTERNAL)
    acts = np.random.default_rng(0).uniform(0.0, 10.0, size=(n_steps, abi.action_dim(c1)))
    last = stream.n_seconds - (n_steps + c1.warmup_steps) // sps - 60

    def make(i):
        o = Oracle(c1, stream)
        o.reset(int((600 + (i * 97) % max(last - 600, 1)) * sps))
        return o

    def work(o):
        o.rollout(n_steps, agent, acts)
        return int(o.state()["err"])

    with _pinned_pool(threads) as ex:
        oracles = list(ex.map(make, range(threads)))
        t0 = time.perf_counter()
        errs = list(ex.map(work, oracles))                                          # calibrate (and warm the caches)
        dt1 = time.perf_counter() - t0
        k = int(min(max(round(seconds / dt1), 1), 256))
        oracles = list(ex.map(make, range(threads, threads * (k + 1))))
        t0 = time.perf_counter()
        errs += list(ex.map(work, oracles))
        dt = time.perf_counter() - t0
    assert not any(errs), errs
    return len(oracles) * n_steps / dt, dt, len(oracles)


def rollout_cfg(n_envs: int, stream):
    """BASELINE.json configs[2] / [3]: default full_state features (F = 10), PnL reward, 30-minute episodes."""
    from datetime import timedelta

    from rl4mm_b200 import abi
    from rl4mm_b200.gym import HistoricalOrderbookEnvironment

    feats = HistoricalOrderbookEnvironment.get_default_features(timedelta(seconds=0.1), timedelta(minutes=30))
    warm = int(max(f.window_size for f in feats) / timedelta(seconds=0.1))
    return abi.default_cfg(n_envs=n_envs, n_levels=stream.n_levels, episode_steps=18000, warmup_steps=warm,
                           features=[f.to_abi() for f in feats], step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
                           terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), initial_cash=1000.0,
                           max_levels_per_side=int(os.environ.get("LOBSIM_BENCH_NL", "64")), max_orders_per_side=256, max_agent_orders=64,
                           outer_levels=20)


def run_reference(args):
    """--impl reference: the reference's algorithm on the host cores (the reference itself is pure Python and cannot
    be compiled; oracle/lob_oracle.c is its C restatement, pinned against the reference by tests/golden/)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    stream = make_stream(args)
    threads = os.cpu_count() or 1
    sample_steps = min(stream.n_grid_steps, args.segment_steps * 20)
    _, _, dt1, _ = cpu_oracle_throughput(stream, sample_steps, threads)                     # calibrate: ~4 s per step
    reps = int(min(max(round(4.0 / max(dt1, 1e-3)), 1), 200))
    for _ in range(max(args.warmup, 1)):
        cpu_oracle_throughput(stream, sample_steps, threads, reps=max(reps // 4, 1))
    vals, steps_s, t_all = [], [], 0.0
    for _ in range(args.steps):
        v, s, dt, msgs = cpu_oracle_throughput(stream, sample_steps, threads, reps=reps)
        vals.append(v); steps_s.append(s); t_all += dt
    value = float(np.mean(vals))
    sample = (f"{threads} books x {reps} replays of the first {sample_steps} grid steps ({msgs} messages each) per step, "
              f"C port of the reference algorithm on {threads} host threads")
    line = {
        "impl": "reference", "metric": "lob_messages_per_sec", "value": value, "unit": "messages/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": workload_config(args, stream),
        "grid_steps_per_sec": float(np.mean(steps_s)),
        "cpu_baseline": {"value": value, "unit": "messages/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "messages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "python_reference_context": python_reference_context(threads),
    }
    try:   # the env-steps/s half of the metric on the same host threads (configs[2] features / reward)
        v, dt, n_cpu = cpu_oracle_env_throughput(stream, rollout_cfg(1, stream), threads, 8000)
        line["rollout"] = {"metric": "env_steps_per_sec", "value": v, "unit": "env steps/s",
                           "cpu_baseline": {"value": v, "unit": "env steps/s", "cores": threads, "kind": "port",
                                            "sample": f"{n_cpu} envs x 8000 env steps (random Beta actions, default full_state "
                                                      f"features, PnL) on {threads} host threads, {dt:.2f} s wall"}}
    except Exception as e:  # noqa: BLE001
        line["rollout"] = {"error": repr(e)}
    print(json.dumps(line))


def python_reference_context(threads: int):
    """BASELINE.md section 2: the CPython reference itself (measured in the survey container, NOT on this box)."""
    return {"not_measured_on_this_box": True, "source": "BASELINE.md section 2 (survey container, 1 core, MSFT fixture)",
            "msgs_per_sec_per_core": PY_REFERENCE_MSGS_PER_CORE, "env_steps_per_sec_per_core": list(PY_REFERENCE_ENV_STEPS_PER_CORE),
            "extrapolated_msgs_per_sec_on_this_host": PY_REFERENCE_MSGS_PER_CORE * threads, "host_threads": threads}


def workload_config(args, stream):
    return {
        "workload": "configs[1]: synthetic SPY-shaped day (10 levels, %d messages, seed 0) replayed through %d "
                    "batched books per GPU" % (stream.n_msgs, args.envs_per_gpu),
        "envs_per_gpu": args.envs_per_gpu, "n_levels": stream.n_levels, "segment_steps": args.segment_steps,
        "step_us": stream.step_us, "mode": "replay", "l2": "flushed between timed iterations (256 MiB write)",
        "starts": "every book starts at step 0 of the stream (identical replicas; `replay_varied_starts` has per-book random starts)",
        "parallelism": f"books sharded over {args.gpus} GPU(s), no data-path collective",
    }


# ======================================================================================================================
#  GPU arm
# ======================================================================================================================
class Ctx:
    def __init__(self, args):
        import torch
        import torch.distributed as dist

        from rl4mm_b200 import parallel

        self.args, self.torch, self.dist = args, torch, dist
        assert torch.cuda.is_available(), "bench.py needs a GPU (the hot path has no CPU fallback)"
        self.rank, self.world, self.local_rank = parallel.init_from_env()
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.cur = torch.cuda.current_stream(self.dev)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
        self.launches = 0
        self.outputs = {} if args.dump_outputs else None

    def keep(self, name: str, arr, envs=None, env_axis: int = 0):
        """--dump-outputs: hold `arr` (numpy or torch), restricted to `envs` along `env_axis`, as <name>.npy."""
        if self.outputs is None:
            return
        a = arr.detach().cpu().numpy() if hasattr(arr, "detach") else np.asarray(arr)
        if envs is not None:
            a = np.take(a, envs, axis=env_axis)
        self.outputs[name] = a.astype(np.float32 if a.dtype == np.float32 else np.float64)

    def keep_state(self, prefix: str, state):
        for f in state.dtype.names:
            self.keep(f"{prefix}_{f}", state[f])

    @staticmethod
    def env_sample(n_envs: int):
        return np.sort(np.random.default_rng(0).choice(n_envs, min(n_envs, DUMP_SAMPLE_ENVS), replace=False))

    def write_outputs(self, out_dir: str):
        total = sum(a.nbytes for a in self.outputs.values())
        assert total <= DUMP_MAX_BYTES, f"--dump-outputs: {total} bytes"
        d = Path(out_dir)
        d.mkdir(parents=True, exist_ok=True)
        for name, a in self.outputs.items():
            np.save(d / f"{name}.npy", a)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        out = [float(x) for x in t.cpu()]
        return out if len(out) > 1 else out[0]

    def timed(self, fn, steps: int, warmup: int, before=None):
        """`warmup` untimed + `steps` timed calls of fn(i); L2 flushed before each timed call; per-step device ms."""
        torch = self.torch
        for i in range(warmup):
            if before:
                before(i)
            fn(i)
        self.barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            if before:
                before(warmup + i)
            self.flush.zero_()
            ev[i][0].record(self.cur)
            fn(warmup + i)
            ev[i][1].record(self.cur)
        self.barrier()
        return [a.elapsed_time(b) for a, b in ev]


def run_replay(ctx: Ctx, stream, line):
    """BASELINE.json configs[1] -- the headline."""
    args, torch = ctx.args, ctx.torch
    from rl4mm_b200 import abi
    from rl4mm_b200.device import LobSim

    n_envs, seg = args.envs_per_gpu, args.segment_steps
    cfg = abi.default_cfg(n_envs=n_envs, n_levels=stream.n_levels, outer_levels=20, max_levels_per_side=64,
                          max_orders_per_side=256, max_agent_orders=32)
    sim = LobSim(cfg, ctx.local_rank)
    assert sim.kernel_path == "fast"
    sim.load_stream(0, stream)
    total = args.warmup + args.steps
    # bench step i replays segment i mod n_seg of the day; when the day is used up every book starts over from its first
    # snapshot (untimed), so --steps is not bounded by the length of the stream
    n_seg = stream.n_grid_steps // seg
    assert n_seg >= 1, "the stream is shorter than one segment"
    end = ((total - 1) % n_seg + 1) * seg                       # grid step every book stands at after the last step
    off = stream.step_off.astype(np.int64)
    msgs_per_env = int(sum(off[(i % n_seg + 1) * seg] - off[i % n_seg * seg] for i in range(args.warmup, total)))

    # ---- device-resident arm -----------------------------------------------------------------------------------------
    sim.reset_book(0, 0)
    sampler = ClockSampler(ctx.local_rank).start()
    l0, rewind_launches = sim.launch_count, 0

    def rewind(i):
        nonlocal rewind_launches
        if i and i % n_seg == 0:
            c = sim.launch_count
            sim.reset_book(0, 0)
            rewind_launches += sim.launch_count - c

    ms = ctx.timed(lambda i: sim.replay(seg), args.steps, args.warmup, before=rewind)
    launches = sim.launch_count - l0 - args.warmup - rewind_launches
    clocks = sampler.stop()
    t_dev = sum(ms) / 1e3
    state = sim.state()
    assert np.all(state["err"] == 0), "error flags raised during the bench: %s" % np.unique(state["err"])
    assert np.all(state["now_step"] == end)
    # every book replayed the same stream: they must be identical, and equal to the historical book
    assert len(np.unique(state[["best_buy", "best_sell", "best_buy_volume", "best_sell_volume"]])) == 1
    snap = stream.snapshots[end // stream.steps_per_second]
    assert state["best_buy"][0] == snap[0, 0, 0] and state["best_sell"][0] == snap[1, 0, 0]
    ctx.keep_state("replay_state", state)
    if ctx.outputs is not None:     # every entry of both sides of 16 sampled books; rows: env, side, price, volume, ref, level
        books = [np.column_stack([np.full(len(b), env), np.full(len(b), side)] + [b[f] for f in b.dtype.names])
                 for env in ctx.env_sample(n_envs)[:16] for side in (0, 1) for b in [sim.dump_book(int(env), side)]]
        ctx.keep("replay_books", np.concatenate(books))

    # ---- end-to-end arm: host buffers through lobsim_replay_host ---------------------------------------------------
    pinned = torch.from_numpy(stream.msgs.view(np.uint8).reshape(-1, 16)).pin_memory()
    host_msgs = pinned.numpy().view(abi.MSG_DTYPE).reshape(-1)
    state_out_t = torch.empty((n_envs, abi.ENV_STATE_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
    state_out = state_out_t.numpy().view(abi.ENV_STATE_DTYPE).reshape(-1)
    sim.reset_book(0, 0)
    h2d = d2h = 0
    t_e2e = 0.0
    for i in range(total):
        s = i % n_seg
        a, b = int(stream.step_off[s * seg]), int(stream.step_off[(s + 1) * seg])
        if i and s == 0:
            sim.reset_book(0, 0)
        if i == args.warmup:
            ctx.barrier()
        ctx.flush.zero_()
        torch.cuda.synchronize(ctx.dev)
        t0 = time.perf_counter()
        sim.replay_host(0, host_msgs[a:b], a, seg, state_out)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            t_e2e += dt
            h2d += (b - a) * 16
            d2h += state_out.nbytes
    assert np.all(state_out["err"] == 0) and np.all(state_out["now_step"] == end)

    t_dev, t_e2e = ctx.max_over_ranks(t_dev, t_e2e)
    world = ctx.world
    env_msgs = msgs_per_env * n_envs * world
    algo = (ALGO_BYTES_PER_MSG * msgs_per_env / args.steps + ALGO_BYTES_PER_STEP_REPLAY * seg + 2 * S_STATE_L10) * n_envs
    line.update({
        "metric": "lob_messages_per_sec", "value": env_msgs / t_dev, "unit": "messages/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": workload_config(args, stream),
        "grid_steps_per_sec": args.steps * seg * n_envs * world / t_dev,
        "e2e": {"value": env_msgs / t_e2e, "unit": "messages/s", "h2d_bytes_per_step": h2d // args.steps,
                "d2h_bytes_per_step": d2h // args.steps, "api": "lobsim_replay_host (C ABI, pinned host buffers)"},
        "gpu_launches": int(launches), "clocks": clocks,
        "roofline": roofline(algo, 1e3 * t_dev / args.steps, ("k_replay_flat" if os.environ.get("LOBSIM_REPLAY_FLAT", "1") != "0" else "k_replay_fast") + "<StaticLayout<64,256,32>>",
                             "k_replay_fast" if (n_envs, seg) == (4096, 2340) else None,
                             note="16 B per env-message + 4 B per env-step + 2 x 1216 B book state per book per launch; all books "
                                  "of a GPU replay the same stream, so DRAM traffic (ncu) is far BELOW the algorithmic bytes (L2 "
                                  "serves the other readers); per-book processing is serially dependent, so the kernel is "
                                  "instruction-issue bound, not HBM bound (DESIGN.md section 3)"),
    })
    ctx.launches += launches

    # ---- the same replay with per-book random start seconds (no two books walk the stream in lockstep) -------------
    sub_steps, warm = args.sub_steps, 3
    rng = np.random.default_rng(99 + ctx.rank)
    sps = stream.steps_per_second
    starts = (rng.integers(0, stream.n_seconds - (sub_steps + warm) * seg // sps - 2, size=n_envs) * sps).astype(np.int32)
    sim.reset_book(0, starts)
    ms = ctx.timed(lambda i: sim.replay(seg), sub_steps, warm)
    st = sim.state()
    assert np.all(st["err"] == 0), np.unique(st["err"])
    off = stream.step_off.astype(np.int64)
    msgs = int((off[starts + (sub_steps + warm) * seg] - off[starts + warm * seg]).sum())
    t = ctx.max_over_ranks(sum(ms) / 1e3)
    line["replay_varied_starts"] = {"metric": "lob_messages_per_sec", "value": msgs * world / t, "unit": "messages/s",
                                    "steps": sub_steps, "warmup": warm, "ms_per_step": 1e3 * t / sub_steps,
                                    "config": {"workload": "configs[1] with a random start second per book", "envs_per_gpu": n_envs}}

    # ---- books-per-GPU curve (N = 1): separates the config's occupancy limit (4096 books = 28 warps per SM) from the kernel's
    if world == 1:
        curve = []
        for nb in (4096, 8192, 16384):
            c2 = abi.default_cfg(n_envs=nb, n_levels=stream.n_levels, outer_levels=20, max_levels_per_side=64,
                                 max_orders_per_side=256, max_agent_orders=32)
            s2 = LobSim(c2, ctx.local_rank)
            s2.load_stream(0, stream)
            s2.reset_book(0, 0)
            ms = ctx.timed(lambda i: s2.replay(seg), sub_steps, warm)
            m = int(stream.step_off[(warm + sub_steps) * seg]) - int(stream.step_off[warm * seg])
            assert np.all(s2.state()["err"] == 0)
            curve.append({"books": nb, "value": m * nb / (sum(ms) / 1e3), "ms_per_step": sum(ms) / sub_steps})
            s2.close()
        line["books_curve"] = curve
    if ctx.rank == 0 and not args.no_cpu_baseline and world == 1:
        threads = os.cpu_count() or 1
        sample_steps = min(stream.n_grid_steps, seg * 20)
        _, _, dt1, _ = cpu_oracle_throughput(stream, sample_steps, threads, reps=1)       # calibrate
        reps = int(min(max(round(CPU_SAMPLE_SECONDS / max(dt1, 1e-3)), 2), 400))
        v, s, dt, m = cpu_oracle_throughput(stream, sample_steps, threads, reps=reps)
        line["cpu_baseline"] = {"value": v, "unit": "messages/s", "cores": threads, "kind": "port",
                                "sample": f"{threads} books x {reps} replays of the first {sample_steps} grid steps "
                                          f"({m} messages) on {threads} host threads, {dt:.2f} s wall",
                                "python_reference_context": python_reference_context(threads)}
    sim.close()


def run_rollout(ctx: Ctx, stream):
    """BASELINE.json configs[2]: HistoricalOrderbookEnvironment rollouts with a Beta policy (torch MLP 2x64 tanh ->
    sigmoid x 10) between steps, PnL reward, default full_state features.  One bench step = T = 128 env steps of every
    env: policy forward (torch) + lobsim_step (one launch) per env step."""
    args, torch = ctx.args, ctx.torch
    from rl4mm_b200.device import LobSim

    dev, world = ctx.dev, ctx.world
    n_envs, T = args.rollout_envs, 128
    cfg = rollout_cfg(n_envs, stream)
    sim = LobSim(cfg, ctx.local_rank)
    assert sim.kernel_path == "fast"
    sim.load_stream(0, stream)
    rng = np.random.default_rng(1234 + ctx.rank)
    sps = stream.steps_per_second
    starts = ((1800 + rng.integers(0, 5 * 3600, size=n_envs)) * sps).astype(np.int32)   # whole seconds in [10:00, 15:00]
    obs = sim.reset(0, starts)
    torch.manual_seed(0)
    policy = torch.nn.Sequential(torch.nn.Linear(obs.shape[1], 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                                 torch.nn.Linear(64, 4)).to(dev)          # fp32, like the reference's RLlib torch policy
    scale = torch.tensor([1e-2, 1e-2, 1e-2, 1e3, 1e3, 1e-2, 1.0, 0.1, 1.0, 1.0], device=dev, dtype=torch.float64)
    box = {"obs": obs}
    kev = []      # CUDA events around every lobsim_step launch of the timed region (the kernel's own duration)

    def act(o):
        with torch.no_grad():
            return (torch.sigmoid(policy((o * scale).float())) * 10.0).double()   # env actions are fp64 (Python floats in the reference)

    def rollout(i, timed=False):
        o = box["obs"]
        for _ in range(T):
            a = act(o)
            if timed:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(ctx.cur)
            o, r, d = sim.step(a)
            if timed:
                e1.record(ctx.cur)
                kev.append((e0, e1))
        box.update(obs=o, rew=r, done=d)

    steps, warm = sub_schedule(args)
    sampler = ClockSampler(ctx.local_rank).start()
    l0 = sim.launch_count
    now0 = None

    def before(i):
        nonlocal now0
        if i == warm:
            now0 = sim.state()["now_step"].astype(np.int64)

    ms = ctx.timed(lambda i: rollout(i, timed=i >= warm), steps, warm, before=before)
    launches = sim.launch_count - l0 - warm * T
    clocks = sampler.stop()
    st = sim.state()
    assert np.all(st["err"] == 0), np.unique(st["err"])
    off = stream.step_off.astype(np.int64)
    msgs = int((off[st["now_step"]] - off[now0]).sum())
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    envs = ctx.env_sample(n_envs)           # the last env step of the last bench step
    for k in ("obs", "rew", "done"):
        ctx.keep(f"rollout_{k}", box[k], envs)
    # end-to-end: host actions in, host obs/reward/done out through lobsim_step_host (pinned buffers)
    a_host = torch.empty((n_envs, 4), dtype=torch.float64).pin_memory()
    o_host = torch.empty((n_envs, obs.shape[1]), dtype=torch.float64).pin_memory()
    r_host = torch.empty(n_envs, dtype=torch.float64).pin_memory()
    d_host = torch.empty(n_envs, dtype=torch.uint8).pin_memory()
    a_host.copy_(act(box["obs"]))
    torch.cuda.synchronize(dev)
    n_e2e = 32
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        sim.step_host(a_host.numpy(), o_host.numpy(), r_host.numpy(), d_host.numpy())
    t_e2e = time.perf_counter() - t0
    t_dev, t_e2e, kernel_ms = ctx.max_over_ranks(sum(ms) / 1e3, t_e2e, kernel_ms)
    env_steps = steps * T * n_envs * world
    algo = ALGO_BYTES_PER_MSG * msgs / (steps * T) + (ALGO_BYTES_PER_STEP_ENV + 2 * S_STATE_L10) * n_envs
    rec = {
        "metric": "env_steps_per_sec", "value": env_steps / t_dev, "unit": "env steps/s", "n_gpus": world,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * t_dev / steps, "higher_is_better": True,
        "scaling": "weak", "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[2]: HistoricalOrderbookEnvironment rollouts, torch MLP Beta policy (2 x 64 tanh, fp32) between steps, "
                               "PnL reward, default full_state features (F=10), %d envs per GPU, T=128 env steps per bench step" % n_envs,
                   "envs_per_gpu": n_envs, "n_levels": stream.n_levels, "T": T, "l2": "flushed between timed iterations (256 MiB write)"},
        "lob_messages_per_sec": msgs * world / t_dev,
        "env_step_kernel_only_steps_per_sec": n_envs * world / (kernel_ms / 1e3),
        "e2e": {"value": n_e2e * n_envs * world / t_e2e, "unit": "env steps/s", "h2d_bytes_per_step": a_host.numel() * 8,
                "d2h_bytes_per_step": o_host.numel() * 8 + r_host.numel() * 8 + d_host.numel(),
                "api": "lobsim_step_host (C ABI, pinned host buffers), policy excluded"},
        "gpu_launches": int(launches), "clocks": clocks,
        "roofline": roofline(algo, kernel_ms, "k_env_fast<StaticLayout<64,256,64>> (one launch per env step; CUDA events around the "
                                              "lobsim_step launches only, the torch policy is outside)",
                             "k_env_fast" if n_envs == 65536 else None),
    }
    ctx.launches += launches
    form = sim.state()["reserved"]                      # lobsim_env_state_t.reserved: bit 0 flat form, bits 8-19 / 20-31 orders per side
    n_side = np.maximum((form >> 8) & 0xfff, (form >> 20) & 0xfff)
    rec["book_forms"] = {"flat_fraction": float((form & 1).mean()), "orders_per_side_p50": float(np.median(n_side)),
                         "orders_per_side_p99": float(np.percentile(n_side, 99)), "orders_per_side_max": int(n_side.max())}
    if ctx.rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, dt, n_cpu = cpu_oracle_env_throughput(stream, cfg, threads, 8000)
        rec["cpu_baseline"] = {"value": v, "unit": "env steps/s", "cores": threads, "kind": "port",
                               "sample": f"{n_cpu} envs x 8000 env steps (random Beta actions, same features / reward) on "
                                         f"{threads} host threads after the feature warm-up, {dt:.2f} s wall"}
    sim.close()
    return rec


def run_collect(ctx: Ctx, stream):
    """BASELINE.json configs[3]: PPO-style rollout collection -- `collect_envs` envs per GPU (1 048 576 on 8 GPUs), a fused
    T = 128 Teradactyl rollout, the [N_local, 8] f32 episode statistics computed on the device and all-gathered over NCCL
    (`parallel.gather_episode_stats`), all inside the timed region; the collective is timed on its own as well."""
    args, torch = ctx.args, ctx.torch
    from rl4mm_b200 import abi, parallel
    from rl4mm_b200.device import LobSim

    world = ctx.world
    n_envs, T = args.collect_envs, 128
    cfg = rollout_cfg(n_envs, stream)
    sim = LobSim(cfg, ctx.local_rank)
    assert sim.kernel_path == "fast"
    sim.load_stream(0, stream)
    rng = np.random.default_rng(4321 + ctx.rank)
    sps = stream.steps_per_second
    starts = ((1800 + rng.integers(0, 5 * 3600, size=n_envs)) * sps).astype(np.int32)
    sim.reset(0, starts)
    agent = abi.Agent(kind=abi.AGENT_TERADACTYL, inventory_index=5, max_inventory=10000.0, default_kappa=10.0, default_omega=0.5,
                      max_kappa=50.0, exponent=1.0)
    steps, warm = sub_schedule(args)
    gev, res, last = [], {}, {}

    def step(i):
        obs, act, rew, done = sim.rollout(T, agent)
        stats = parallel.episode_stats_dev(rew, done, sim.state_dev(), obs[:, :, 0])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ctx.cur)
        allstats = parallel.gather_episode_stats(stats)
        e1.record(ctx.cur)
        gev.append((e0, e1))
        if ctx.outputs is not None:
            last.update(obs=obs, act=act, rew=rew, done=done, stats=allstats)
        res["mean_return"] = float(allstats[:, 0].mean().item())          # D2H read of the result: the step's sync point
        res["shape"] = list(allstats.shape)
        res["errs"] = int((allstats[:, 7] != 0).sum().item())

    sampler = ClockSampler(ctx.local_rank).start()
    l0 = sim.launch_count
    now0 = None

    def before(i):
        nonlocal now0
        if i == warm:
            now0 = sim.state()["now_step"].astype(np.int64)

    ms = ctx.timed(step, steps, warm, before=before)
    launches = sim.launch_count - l0
    clocks = sampler.stop()
    st = sim.state()
    assert np.all(st["err"] == 0), np.unique(st["err"])
    assert res["errs"] == 0 and res["shape"] == [n_envs * world, 8], res
    envs = ctx.env_sample(n_envs)           # [T, N, ...] rollout tensors and the gathered [N, 8] stats of the last bench step
    for k, v in last.items():
        ctx.keep(f"collect_{k}", v, envs, env_axis=0 if k == "stats" else 1)
    off = stream.step_off.astype(np.int64)
    msgs = int((off[st["now_step"]] - off[now0]).sum())
    gather_ms = float(np.mean([a.elapsed_time(b) for a, b in gev[warm:]]))
    t_dev, gather_ms = ctx.max_over_ranks(sum(ms) / 1e3, gather_ms)
    env_steps = steps * T * n_envs * world
    algo = ALGO_BYTES_PER_MSG * msgs / steps + (ALGO_BYTES_PER_STEP_ENV * T + 2 * S_STATE_L10) * n_envs
    rec = {
        "metric": "env_steps_per_sec", "value": env_steps / t_dev, "unit": "env steps/s", "n_gpus": world, "steps": steps,
        "warmup": warm, "ms_per_step": 1e3 * t_dev / steps, "higher_is_better": True, "scaling": "weak", "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "configs[3]: PPO-style rollout collection, %d envs per GPU (%d in total), fused T=128 Teradactyl "
                               "rollout + device-side episode stats + NCCL all-gather of the [N, 8] f32 stats inside the timed region"
                               % (n_envs, n_envs * world), "envs_per_gpu": n_envs, "envs_total": n_envs * world, "T": T,
                   "n_levels": stream.n_levels},
        "lob_messages_per_sec": msgs * world / t_dev,
        "all_gather_ms": gather_ms, "all_gather_bytes_total": n_envs * world * 8 * 4,
        "all_gather_share_of_step": gather_ms / (1e3 * t_dev / steps),
        "gathered_shape": res["shape"], "mean_return": res["mean_return"],
        "gpu_launches": int(launches), "clocks": clocks,
        "roofline": roofline(algo, 1e3 * t_dev / steps, "k_env_fast<StaticLayout<64,256,64>> (one launch = 128 env steps of every env; "
                                                         "the step time includes the stats kernels and the all-gather)"),
    }
    ctx.launches += launches
    sim.close()
    return rec


def run_multiticker(ctx: Ctx):
    """BASELINE.json configs[4]: 8 synthetic tickers (seeds 0-7, mids $30-$500), 50 levels, heavy cancel / modify flow,
    deep queues; `multiticker_envs` books per GPU, ticker = book index mod 8, a random start second per book.  Replay
    (messages/s, k_replay_hyb<128,1024,64>: hot order pool near the touch + cold level arrays) and a fused FixedActionAgent([1,2,1,2]) rollout (env steps/s)."""
    args, torch = ctx.args, ctx.torch
    import ctypes

    from rl4mm_b200 import abi, synthetic
    from rl4mm_b200.device import LobSim

    world = ctx.world
    n_envs, seg, n_streams = args.multiticker_envs, 1170, 8
    streams = [synthetic.generate(synthetic.heavy_cancel_ticker(seed=k, n_msgs=args.multiticker_msgs)) for k in range(n_streams)]
    steps, warm = sub_schedule(args)
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100000, 0, 5000), abi.feature(abi.FEAT_BOOK_IMBALANCE, 0, 100000, -1, 1),
             abi.feature(abi.FEAT_INVENTORY, 0, 100000, -1e6, 1e6)]
    # capacities: a side of these streams holds at most ~620 orders over the whole day (oracle replay) + ~45 agent orders: 1 024
    # per side (compiled layout 128/1024/64) leaves 1.5x headroom and fits 12 books per SM instead of 8 with 1 536
    cfg = abi.default_cfg(n_envs=n_envs, n_levels=50, outer_levels=20, max_levels_per_side=128, max_orders_per_side=1024,
                          max_agent_orders=64, features=feats, episode_steps=18000, warmup_steps=0,
                          step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0))
    sim = LobSim(cfg, ctx.local_rank)
    path = sim.kernel_path
    for k, s in enumerate(streams):
        sim.load_stream(k, s)
    rng = np.random.default_rng(555 + ctx.rank)
    sps = streams[0].steps_per_second
    sid = (np.arange(n_envs) % n_streams).astype(np.int32)
    span = (steps + warm) * seg // sps + 2
    starts = (rng.integers(0, streams[0].n_seconds - span, size=n_envs) * sps).astype(np.int32)
    offs = [s.step_off.astype(np.int64) for s in streams]

    def count_msgs(a, b):
        return int(sum((offs[k][b[sid == k]] - offs[k][a[sid == k]]).sum() for k in range(n_streams)))

    # ---- replay ------------------------------------------------------------------------------------------------------
    sim.reset_book(sid, starts)
    sampler = ClockSampler(ctx.local_rank).start()
    l0 = sim.launch_count
    ms = ctx.timed(lambda i: sim.replay(seg), steps, warm)
    launches = sim.launch_count - l0 - warm
    clocks = sampler.stop()
    st = sim.state()
    assert np.all(st["err"] == 0), np.unique(st["err"])
    ctx.keep_state("multiticker_state", st)
    msgs = count_msgs(starts.astype(np.int64) + warm * seg, starts.astype(np.int64) + (warm + steps) * seg)
    t_dev = ctx.max_over_ranks(sum(ms) / 1e3)
    algo = ALGO_BYTES_PER_MSG * msgs / steps + (ALGO_BYTES_PER_STEP_REPLAY * seg + 2 * S_STATE_L50) * n_envs
    rec = {
        "metric": "lob_messages_per_sec", "value": msgs * world / t_dev, "unit": "messages/s", "n_gpus": world, "steps": steps,
        "warmup": warm, "ms_per_step": 1e3 * t_dev / steps, "higher_is_better": True, "scaling": "weak", "dtype": "int32",
        "data": "synthetic", "kernel_path": path,
        "config": {"workload": "configs[4]: %d synthetic tickers (50 levels, %d messages each, 25%% partial cancels, mean queue 12), "
                               "%d books per GPU, ticker = book mod %d, random start second per book, %d grid steps per bench step"
                               % (n_streams, args.multiticker_msgs, n_envs, n_streams, seg),
                   "envs_per_gpu": n_envs, "n_levels": 50, "n_streams": n_streams, "segment_steps": seg,
                   "capacities": [128, 1024, 64]},
        "gpu_launches": int(launches), "clocks": clocks,
        "roofline": roofline(algo, 1e3 * t_dev / steps,
                             "k_replay_hyb<StaticLayout<128,1024,64>> (hot order pool + cold level arrays, book_hybrid.cuh)"
                             if os.environ.get("LOBSIM_REPLAY_HYBRID", "1") != "0" and os.environ.get("LOBSIM_REPLAY_FLAT", "1") != "0"
                             else "k_replay_flat<StaticLayout<128,1024,64>> (deep books: its sorted-array path)",
                             "k_replay_hyb_L50" if n_envs == 8192 else None),
    }
    ctx.launches += launches
    # ---- fused FixedActionAgent rollout --------------------------------------------------------------------------------
    T = 128
    starts2 = (rng.integers(600, streams[0].n_seconds - (steps + warm) * T // sps - 2, size=n_envs) * sps).astype(np.int32)
    sim.reset(sid, starts2)
    agent = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 2, 1, 2, 0))
    l0, last = sim.launch_count, []

    def roll(i):
        out = sim.rollout(T, agent, want_obs=True)
        if ctx.outputs is not None:
            last[:] = out

    ms = ctx.timed(roll, steps, warm)
    launches = sim.launch_count - l0 - warm
    st = sim.state()
    bad = st["err"] & ~np.uint32(abi.ERR_AGENT_OVERFLOW)
    assert np.all(bad == 0), np.unique(st["err"])
    envs = ctx.env_sample(n_envs)           # [T, N, ...] obs, act, rew, done of the last bench step
    for k, v in zip(("obs", "act", "rew", "done"), last):
        ctx.keep(f"multiticker_env_{k}", v, envs, env_axis=1)
    msgs = count_msgs(starts2.astype(np.int64) + warm * T, starts2.astype(np.int64) + (warm + steps) * T)
    t_env = ctx.max_over_ranks(sum(ms) / 1e3)
    algo = ALGO_BYTES_PER_MSG * msgs / steps + (ALGO_BYTES_PER_STEP_ENV * T + 2 * S_STATE_L50) * n_envs
    rec["env"] = {"metric": "env_steps_per_sec", "value": steps * T * n_envs * world / t_env, "unit": "env steps/s",
                  "ms_per_step": 1e3 * t_env / steps, "lob_messages_per_sec": msgs * world / t_env, "T": T,
                  "agent": "FixedActionAgent([1,2,1,2]) fused on the device", "features": "Spread, BookImbalance, Inventory; PnL",
                  "agent_overflow_envs": int((st["err"] & abi.ERR_AGENT_OVERFLOW != 0).sum()), "gpu_launches": int(launches),
                  "roofline": roofline(algo, 1e3 * t_env / steps, "k_env_fast<StaticLayout<128,1024,64>> (one launch = 128 env steps)")}
    ctx.launches += launches
    if ctx.rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        sample_steps = 20_000
        _, _, dt1, _ = cpu_oracle_throughput(streams[0], sample_steps, threads, reps=1)
        reps = int(min(max(round(5.0 / max(dt1, 1e-3)), 1), 400))
        v, s, dt, m = cpu_oracle_throughput(streams[0], sample_steps, threads, reps=reps)
        rec["cpu_baseline"] = {"value": v, "unit": "messages/s", "cores": threads, "kind": "port",
                               "sample": f"{threads} books x {reps} replays of the first {sample_steps} grid steps of ticker 0 "
                                         f"({m} messages) on {threads} host threads, {dt:.2f} s wall"}
    sim.close()
    return rec


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    ctx = Ctx(args)
    stream = make_stream(args)
    line = {}
    want = (lambda w: args.workload in ("all", w))
    if want("replay"):
        run_replay(ctx, stream, line)

    def sub(name, fn):
        try:
            line[name] = fn()
        except Exception as e:  # noqa: BLE001 -- a failing sub-record must not take the headline with it
            line[name] = {"error": repr(e), "trace": traceback.format_exc()[-800:]}
        ctx.barrier()

    if want("rollout"):
        sub("rollout", lambda: run_rollout(ctx, stream))
    if want("collect"):
        sub("collect", lambda: run_collect(ctx, stream))
    if want("multiticker"):
        sub("multiticker", lambda: run_multiticker(ctx))
    if "metric" not in line:       # a single sub-workload was asked for: promote it to the top level
        name = args.workload
        rec = line.pop(name)
        line.update(rec)
        line.setdefault("vs_baseline", None)
    line["gpu_launches_total"] = int(ctx.launches)
    if ctx.rank == 0 and ctx.outputs is not None:
        ctx.write_outputs(args.dump_outputs)
    if ctx.rank == 0:
        print(json.dumps(line))
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
