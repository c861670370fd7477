"""CPU-side checks of the C-ABI library and the host logic (no compute calls: there is no GPU here)."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from rl4mm_b200 import abi

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def lobsim_lib():
    from rl4mm_b200.build import build_all

    build_all()
    from rl4mm_b200._lib import lib

    return lib()


def test_header_symbols_are_exported(lobsim_lib):
    header = (ROOT / "include" / "lobsim.h").read_text()
    declared = sorted(set(re.findall(r"\b(lobsim_[a-z_]+)\s*\(", header)))
    assert len(declared) >= 20
    from rl4mm_b200._lib import EXPORTED_SYMBOLS

    assert sorted(EXPORTED_SYMBOLS) == declared
    for name in declared:
        assert hasattr(lobsim_lib, name), f"{name} declared in include/lobsim.h but not exported by liblobsim.so"


def test_ingest_header_symbols_are_exported():
    """include/lobingest.h <-> libingest.so (the LOBSTER packer's C ABI)."""
    import ctypes

    from rl4mm_b200.build import build_ingest

    header = (ROOT / "include" / "lobingest.h").read_text()
    declared = sorted(set(re.findall(r"\b(lobingest_[a-z_]+)\s*\(", header)))
    assert declared == ["lobingest_count_lines", "lobingest_count_rows", "lobingest_pack_close", "lobingest_pack_copy", "lobingest_pack_open",
                        "lobingest_pack_sizes", "lobingest_parse_book_rows", "lobingest_parse_messages"]
    lib = ctypes.CDLL(str(build_ingest()))
    for name in declared:
        assert hasattr(lib, name), name


def test_abi_version_and_dims(lobsim_lib):
    assert lobsim_lib.lobsim_abi_version() == abi.ABI_VERSION
    cfg = abi.default_cfg(features=[abi.feature(abi.FEAT_SPREAD, 0, 100000, 0, 5000)] * 3, inc_prev_action_in_obs=1)
    assert lobsim_lib.lobsim_action_dim(C.byref(cfg)) == abi.action_dim(cfg) == 4
    assert lobsim_lib.lobsim_obs_dim(C.byref(cfg)) == abi.obs_dim(cfg) == 7
    cfg2 = abi.default_cfg(concentration=10.0, market_order_clearing=1)
    assert lobsim_lib.lobsim_action_dim(C.byref(cfg2)) == 3
    assert lobsim_lib.lobsim_state_bytes(C.byref(cfg)) % 16 == 0


def test_struct_sizes_match_header():
    """ctypes mirrors must have the C layout: compile a tiny probe with gcc and compare sizeof()."""
    import subprocess
    import tempfile

    src = '#include <stdio.h>\n#include "lobsim.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",' \
          "sizeof(lobsim_msg_t),sizeof(lobsim_feature_t),sizeof(lobsim_reward_t),sizeof(lobsim_agent_t)," \
          "sizeof(lobsim_cfg_t),sizeof(lobsim_stream_t),sizeof(lobsim_order_t),sizeof(lobsim_fill_t)," \
          "sizeof(lobsim_book_entry_t),sizeof(lobsim_env_state_t));return 0;}\n"
    with tempfile.TemporaryDirectory() as d:
        (Path(d) / "p.c").write_text(src)
        subprocess.run(["gcc", "-I", str(ROOT / "include"), "-o", f"{d}/p", f"{d}/p.c"], check=True)
        out = subprocess.run([f"{d}/p"], capture_output=True, text=True, check=True).stdout.split()
    got = [int(x) for x in out]
    want = [abi.MSG_DTYPE.itemsize, C.sizeof(abi.Feature), C.sizeof(abi.Reward), C.sizeof(abi.Agent), C.sizeof(abi.Cfg),
            C.sizeof(abi.Stream), abi.ORDER_DTYPE.itemsize, abi.FILL_DTYPE.itemsize, abi.BOOK_ENTRY_DTYPE.itemsize,
            abi.ENV_STATE_DTYPE.itemsize]
    assert got == want
    assert C.sizeof(abi.Order) == abi.ORDER_DTYPE.itemsize


def test_no_cpu_fallback(lobsim_lib):
    """Without a CUDA device the product must fail loudly, not fall back to the oracle or any CPU path."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    cfg = abi.default_cfg()
    rc = lobsim_lib.lobsim_create(C.byref(cfg), 0, C.byref(h))
    assert rc == abi.E_CUDA and b"no CUDA device" in lobsim_lib.lobsim_last_error()
    from rl4mm_b200.device import LobSim
    from rl4mm_b200._lib import LobsimError

    with pytest.raises(LobsimError):
        LobSim(cfg)


def test_invalid_cfg_rejected(lobsim_lib):
    cfg = abi.default_cfg(max_quote_level=40)
    assert lobsim_lib.lobsim_state_bytes(C.byref(cfg)) == abi.E_INVALID


def test_product_never_imports_oracle():
    for py in (ROOT / "rl4mm_b200").rglob("*.py"):
        text = py.read_text()
        assert "import oracle" not in text and "from oracle" not in text, py
    for src in (ROOT / "rl4mm_b200" / "csrc").iterdir():
        assert not re.search(r'#include\s*[<"][^>"]*oracle', src.read_text()), src


def test_packer_matches_committed_fixture():
    """pack_arrays semantics on a hand-made LOBSTER snippet: type map, direction flip, hidden executions dropped,
    lexicographic tie order, CSR step offsets, per-second snapshots."""
    from rl4mm_b200.packing import pack_arrays

    L = 2
    t = np.array([34200_100_000_000, 34200_100_000_500, 34200_100_000_900, 34200_950_000_000, 34201_000_000_000,
                  34201_050_000_000, 34201_050_000_000, 34201_050_000_000, 34201_050_000_000, 34201_050_000_000,
                  34201_050_000_000, 34201_050_000_000, 34201_050_000_000, 34201_050_000_000, 34201_050_000_000,
                  34201_050_000_000], np.int64)
    n = len(t)
    ty = np.array([1, 4, 5, 3, 2] + [1] * 11)
    oid = np.arange(100, 100 + n)
    size = np.full(n, 10)
    price = np.full(n, 1000)
    direction = np.array([1, 1, 1, -1, -1] + [1] * 11)
    books = np.tile(np.array([1100, 5, 1000, 7, 9999999999, 0, -9999999999, 0], np.int64), (n, 1))
    books[:, 1] = np.arange(n)  # ask size encodes the row, to check snapshot alignment
    s = pack_arrays(t, ty, oid, size, price, direction, books, L, step_us=100_000)
    assert s.t0_us == 34200_000_000 and s.n_grid_steps == 20 and s.n_seconds == 2
    assert s.n_msgs == n - 1  # the hidden execution is dropped
    m = s.msgs
    assert (m["meta"][0] & 7, (m["meta"][0] >> 3) & 1) == (abi.MSG_LIMIT, abi.BUY)
    assert (m["meta"][1] & 7, (m["meta"][1] >> 3) & 1) == (abi.MSG_MARKET, abi.SELL)   # execution of a buy => sell aggressor
    assert (m["meta"][2] & 7, (m["meta"][2] >> 3) & 1) == (abi.MSG_DELETE, abi.SELL)
    assert (m["meta"][3] & 7, (m["meta"][3] >> 3) & 1) == (abi.MSG_CANCEL, abi.SELL)
    # rows 5..15 share one microsecond: the reference orders them by the STRING row id: "10" < "11" < ... < "15" < "5" ...
    tied = [int(s.ext_ids[r]) - 100 for r in m["ref"][4:]]
    assert tied == sorted(range(5, 16), key=str)
    # 0.1 s (+ sub-microsecond digits) truncates to exactly 0.1 s => step 0 = (0, 0.1 s] holds the first two kept messages, 0.95 s is step 9, 1.0 s exactly is step 9 too
    assert list(s.step_off[:3]) == [0, 2, 2] and s.step_off[9] == 2 and s.step_off[10] == 4
    assert s.step_off[11] == n - 1
    # snapshots: second 0 has no data, second 1 = row 4 (ts == boundary), second 2 = last row
    assert list(s.snap_valid) == [0, 1, 1]
    assert s.snapshots[1, abi.SELL, 0, 1] == 4 and s.snapshots[2, abi.SELL, 0, 1] == n - 1
    assert s.snapshots[1, abi.SELL, 1, 0] == abi.NO_PRICE and s.snapshots[1, abi.BUY, 1, 0] == abi.NO_PRICE
    assert tuple(s.snapshots[1, abi.BUY, 0]) == (1000, 7)
    # file order keeps the rows as they are
    s2 = pack_arrays(t, ty, oid, size, price, direction, books, L, step_us=100_000, tie_order="file")
    assert [int(s2.ext_ids[r]) - 100 for r in s2.msgs["ref"][4:]] == list(range(5, 16))
    with pytest.raises(ValueError):
        pack_arrays(t, np.where(ty == 2, 6, ty), oid, size, price, direction, books, L)


def test_synthetic_stream_is_self_consistent():
    """Replaying a synthetic stream through the oracle from the initial snapshot reproduces every later snapshot's
    top of book (the generator's own book and the simulator agree), with no error flags."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic

    sc = synthetic.spy_day(seed=1, n_msgs=100_000, duration_s=234)
    s = synthetic.generate(sc)
    s2 = synthetic.generate(sc)
    assert np.array_equal(s.msgs, s2.msgs) and np.array_equal(s.step_off, s2.step_off)  # seeded => reproducible
    ty = s.msgs["meta"] & 7
    frac = np.bincount(ty, minlength=5)[1:] / len(ty)
    assert abs(frac[0] - 0.48) < 0.03 and abs(frac[2] - 0.42) < 0.03 and 0.05 < frac[3] < 0.12
    o = Oracle(abi.default_cfg(n_levels=10, outer_levels=20), s)
    o.reset_book(0)
    for sec in range(1, 235):
        o.replay(10)
        st = o.state()
        assert st["err"] == 0
        snap = s.snapshots[sec]
        assert st["best_buy"] == snap[0, 0, 0] and st["best_sell"] == snap[1, 0, 0], sec
        if sec > 120:  # the initial aggregates near the touch are gone by now: volumes agree too
            assert st["best_buy_volume"] == snap[0, 0, 1] and st["best_sell_volume"] == snap[1, 0, 1], sec


def test_host_beta_distributor_matches_reference_lots():
    """rl4mm_b200.gym.BetaOrderDistributor (the host twin of the kernel's ladder) against scipy's lot sizes."""
    import parity_helpers as H
    from rl4mm_b200.gym import BetaOrderDistributor

    n = 0
    for grp in H.load_golden("beta_ladders.json.gz"):
        d = BetaOrderDistributor(grp["quote_levels"], grp["active_volume"], grp["concentration"])
        acts = np.array([c["action"] for c in grp["cases"]])
        out = d.convert_action(acts)
        for i, c in enumerate(grp["cases"]):
            assert list(out["buy"][i]) == c["buy"] and list(out["sell"][i]) == c["sell"], (grp["quote_levels"], c["action"])
            n += 1
    assert n > 900


def test_fast_lobster_reader_matches_python_packer(tmp_path):
    """csrc/lobster_ingest.cpp (mmap CSV reader, only the needed orderbook rows) == the pure-Python path, on a
    generated LOBSTER-format file pair with odd rows: sub-microsecond digits, no fraction, hidden executions, dummy
    levels, duplicate timestamps."""
    from rl4mm_b200.packing import pack_lobster, read_lobster_book_rows, read_lobster_messages

    rng = np.random.default_rng(5)
    n, L = 600, 3
    t = rng.integers(34_200_000_000_000, 34_206_000_000_000, size=n)
    t[0] = 34_203_000_000_000      # a whole second: written without a fractional part
    t = np.sort(t)
    t[100:104] = t[100]            # duplicate timestamps
    ty = rng.choice([1, 2, 3, 4, 5], size=n, p=[0.45, 0.1, 0.3, 0.1, 0.05])
    oid = rng.integers(1, 10**9, size=n)
    sz = rng.integers(1, 5000, size=n)
    pr = rng.integers(3_000_000, 3_100_000, size=n) // 100 * 100
    di = rng.choice([-1, 1], size=n)
    msg = tmp_path / "X_2020-01-02_34200000_57600000_message_3.csv"
    book = tmp_path / "X_2020-01-02_34200000_57600000_orderbook_3.csv"
    with open(msg, "w") as f:
        for i in range(n):
            sec, ns = divmod(int(t[i]), 10**9)
            ts = f"{sec}" if ns == 0 else f"{sec}.{ns:09d}"
            f.write(f"{ts},{ty[i]},{oid[i]},{sz[i]},{pr[i]},{di[i]}\n")
    rows = np.zeros((n, 4 * L), np.int64)
    for i in range(n):
        for lv in range(L):
            dummy = lv == 2 and i % 7 == 0
            rows[i, 4 * lv: 4 * lv + 4] = (9999999999, 0, -9999999999, 0) if dummy else \
                (3_050_100 + 100 * lv, 10 + i + lv, 3_050_000 - 100 * lv, 20 + i + lv)
    np.savetxt(book, rows, fmt="%d", delimiter=",")
    rt, rty, roid, rsz, rpr, rdi = read_lobster_messages(msg)
    assert np.array_equal(rt, t) and np.array_equal(rty, ty) and np.array_equal(roid, oid)
    assert np.array_equal(rsz, sz) and np.array_equal(rpr, pr) and np.array_equal(rdi, di)
    idx = np.array([0, 0, 5, 17, 17, 599])
    assert np.array_equal(read_lobster_book_rows(book, idx, L), rows[idx])
    for tie in ("reference", "file"):
        a = pack_lobster(msg, book, L, fast=True, tie_order=tie)          # the native packer (lobingest_pack_open)
        r = pack_lobster(msg, book, L, fast="reader", tie_order=tie)      # C++ reader + numpy packer
        b = pack_lobster(msg, book, L, fast=False, tie_order=tie)         # pure Python
        for f_ in ("msgs", "step_off", "snapshots", "snap_valid", "ext_ids"):
            assert np.array_equal(getattr(a, f_), getattr(b, f_)), (tie, f_)
            assert np.array_equal(getattr(r, f_), getattr(b, f_)), (tie, f_)
        assert a.t0_us == r.t0_us == b.t0_us == 34_200_000_000
    for kw in (dict(max_rows=250), dict(step_us=50_000), dict(t0_us=34_199_000_000), dict(db_batch_size=100)):
        a, b = pack_lobster(msg, book, L, fast=True, **kw), pack_lobster(msg, book, L, fast=False, **kw)
        for f_ in ("msgs", "step_off", "snapshots", "snap_valid", "ext_ids"):
            assert np.array_equal(getattr(a, f_), getattr(b, f_)), (kw, f_)
    assert np.array_equal(read_lobster_messages(msg, max_rows=10)[0], t[:10])

    # ADVICE r1: blank / "\r"-only lines are not data rows in EITHER file (the readers used to count them differently, which
    # silently shifted the snapshots against the messages); an empty field is malformed; unequal row counts are an error
    msg2, book2 = tmp_path / "blank_message_3.csv", tmp_path / "blank_orderbook_3.csv"
    ml, bl = open(msg).read().splitlines(), open(book).read().splitlines()
    with open(msg2, "w") as f:
        f.write("\n".join(ml[:50] + ["", "\r"] + ml[50:]) + "\n\n")
    with open(book2, "w") as f:
        f.write("\n".join(bl[:300] + [""] + bl[300:]) + "\n")
    ref = pack_lobster(msg, book, L, fast=True)
    for fast in (True, "reader"):
        got = pack_lobster(msg2, book2, L, fast=fast)
        for f_ in ("msgs", "step_off", "snapshots", "snap_valid", "ext_ids"):
            assert np.array_equal(getattr(got, f_), getattr(ref, f_)), (fast, f_)
    with open(book2, "w") as f:
        f.write("\n".join(bl[:-1]) + "\n")
    for fast in (True, "reader"):
        with pytest.raises(ValueError, match="different row counts"):
            pack_lobster(msg, book2, L, fast=fast)
    with open(msg2, "w") as f:
        f.write("\n".join(ml[:10] + ["34203.5,1,,100,3000000,1"] + ml[10:]) + "\n")
    with pytest.raises(ValueError, match="malformed"):
        pack_lobster(msg2, book, L, fast=True)
    with pytest.raises(ValueError, match="malformed"):
        read_lobster_messages(msg2)


def test_native_packer_on_the_msft_fixture_and_a_1e6_row_day(tmp_path):
    """SURVEY 8f.1: the native packer == the numpy packer on the reference's own MSFT fixture, and on a 1e6-row synthetic
    LOBSTER file pair (written from a packed synthetic stream), where it also has to be much faster."""
    import os
    import time

    from pathlib import Path

    from parity_helpers import load_fixture_stream
    from rl4mm_b200 import synthetic
    from rl4mm_b200.packing import pack_lobster

    # the CSV pair ships with the original rl4mm project (RL4MM_REFERENCE), not with this repository; its packed form is committed
    ref_dir = Path(os.environ.get("RL4MM_REFERENCE", "")) / "test_data"
    m = ref_dir / "MSFT_2012-06-21_34200000_37800000_message_50.csv"
    b = ref_dir / "MSFT_2012-06-21_34200000_37800000_orderbook_50.csv"
    if os.environ.get("RL4MM_REFERENCE"):
        for tie in ("reference", "file"):
            x, y = pack_lobster(m, b, 50, max_rows=1000, fast=True, tie_order=tie), load_fixture_stream(tie)
            for f_ in ("msgs", "step_off", "snapshots", "snap_valid", "ext_ids"):
                assert np.array_equal(getattr(x, f_), getattr(y, f_)), (tie, f_)
    n, L = 1_000_000, 10
    s = synthetic.generate(synthetic.spy_day(seed=3, n_msgs=n, duration_s=2340))
    # a LOBSTER file pair carrying that stream: time inside the step, LOBSTER's resting-order direction for executions
    step = np.repeat(np.arange(s.n_grid_steps), np.diff(s.step_off.astype(np.int64)))
    us = s.t0_us + step * s.step_us + 1 + (np.arange(n) - s.step_off.astype(np.int64)[step])   # strictly increasing inside (k*step, (k+1)*step]
    assert np.all(np.diff(us) > 0) and np.all(us <= s.t0_us + (step + 1) * s.step_us)
    ty = (s.msgs["meta"] & 7).astype(np.int64)
    side = ((s.msgs["meta"] >> 3) & 1).astype(np.int64)
    lob_dir = np.where(ty == 4, 1 - side, side)
    di = np.where(lob_dir == 0, 1, -1)
    msg, book = tmp_path / "SYN_message_10.csv", tmp_path / "SYN_orderbook_10.csv"
    sec_of = (us - s.t0_us) // 1_000_000
    with open(msg, "w") as f:
        f.write("".join(f"{u // 1_000_000}.{u % 1_000_000:06d}000,{t},{r},{v},{p},{d}\n" for u, t, r, v, p, d in
                        zip(us.tolist(), ty.tolist(), s.msgs["ref"].tolist(), s.msgs["volume"].tolist(), s.msgs["price"].tolist(), di.tolist())))
    snap = s.snapshots.astype(np.int64)
    snap_rows = np.zeros((snap.shape[0], 4 * L), np.int64)
    for lv in range(L):
        ap, av, bp, bv = snap[:, 1, lv, 0], snap[:, 1, lv, 1], snap[:, 0, lv, 0], snap[:, 0, lv, 1]
        snap_rows[:, 4 * lv + 0] = np.where(ap == abi.NO_PRICE, 9999999999, ap)
        snap_rows[:, 4 * lv + 1] = av
        snap_rows[:, 4 * lv + 2] = np.where(bp == abi.NO_PRICE, -9999999999, bp)
        snap_rows[:, 4 * lv + 3] = bv
    lines = [",".join(map(str, r)) for r in snap_rows.tolist()]
    with open(book, "w") as f:
        f.write("".join(lines[k] + "\n" for k in sec_of.tolist()))
    t0 = time.perf_counter()
    a = pack_lobster(msg, book, L, fast=True, t0_us=s.t0_us)
    t_native = time.perf_counter() - t0
    t0 = time.perf_counter()
    r = pack_lobster(msg, book, L, fast="reader", t0_us=s.t0_us)
    t_numpy = time.perf_counter() - t0
    for f_ in ("msgs", "step_off", "snapshots", "snap_valid", "ext_ids"):
        assert np.array_equal(getattr(a, f_), getattr(r, f_)), f_
    # round trip: the packed stream is the one the files were written from (refs are re-ranked densely: same order)
    assert np.array_equal(a.step_off, s.step_off)
    for f_ in ("price", "volume", "meta"):
        assert np.array_equal(a.msgs[f_], s.msgs[f_]), f_
    assert np.array_equal(a.ext_ids[a.msgs["ref"]], s.msgs["ref"].astype(np.int64))
    print(f"native packer: {n / t_native:.3g} rows/s, C++ reader + numpy packer: {n / t_numpy:.3g} rows/s")


def test_gae_matches_naive_sum():
    import torch

    from rl4mm_b200.ppo import gae

    torch.manual_seed(0)
    T, N = 7, 3
    rew, val, last = torch.randn(T, N), torch.randn(T, N), torch.randn(N)
    done = torch.zeros(T, N, dtype=torch.bool)
    done[3, 1] = True
    adv, ret = gae(rew, val, last, done, 0.9, 0.8)
    for n in range(N):
        for t in range(T):
            a, coef = 0.0, 1.0
            for k in range(t, T):
                nv = last[n] if k == T - 1 else val[k + 1, n]
                a += coef * (rew[k, n] + 0.9 * nv * (0.0 if done[k, n] else 1.0) - val[k, n])
                if done[k, n]:
                    break
                coef *= 0.9 * 0.8
            assert abs(float(a) - float(adv[t, n])) < 1e-5
    assert torch.allclose(ret, adv + val)


def test_get_sharpe_matches_reference_formula():
    """rl4mm/rewards/RewardFunctions.py:10-22 (ddof=1, + float_min), batched over the leading axis."""
    import sys

    from rl4mm_b200.evaluation import get_sharpe

    rng = np.random.default_rng(0)
    aum = 1000.0 + np.cumsum(rng.normal(0, 1, size=(4, 50)), axis=1)
    got = get_sharpe(aum)
    for i in range(4):
        r = np.exp(np.diff(np.log(aum[i]))) - 1
        assert abs(got[i] - np.mean(r) / (np.std(r, ddof=1) + sys.float_info.min)) < 1e-12
    with pytest.raises(Exception):
        get_sharpe(np.array([1.0, 0.0, 2.0]))


def test_weighted_midprice_offsets_match_info_calculator():
    """evaluation.weighted_midprice_offsets (batched over [T, N, A]) == SimpleInfoCalculator's weighted_midprice_offset
    (InfoCalculators.py:44-50) evaluated action by action."""
    from rl4mm_b200 import evaluation
    from rl4mm_b200.gym import BetaOrderDistributor, SimpleInfoCalculator

    rng = np.random.default_rng(5)
    acts = rng.uniform(0.0, 10.0, size=(6, 3, 4))
    dist = BetaOrderDistributor(10)
    got = evaluation.weighted_midprice_offsets(acts, dist)
    st = np.zeros(3, dtype=abi.ENV_STATE_DTYPE)
    st["best_buy"], st["best_sell"], st["price"], st["cash"] = 999900, 1000100, 1e6, 1e3
    calc = SimpleInfoCalculator(order_distributor=dist)
    for t in range(6):
        info = calc.calculate(st, acts[t])
        assert np.allclose(info["weighted_midprice_offset"], got[t], rtol=0, atol=1e-12)


def test_episode_summary_shapes_and_reference_quirks():
    """append_to_episode_summary_dict quirks (utils.py:146-190): mean action drops its LAST component, one entry per env."""
    from rl4mm_b200 import evaluation
    from rl4mm_b200.gym import BetaOrderDistributor

    T, N = 5, 3
    rng = np.random.default_rng(1)
    act, rew = rng.uniform(0, 10, size=(T, N, 4)), rng.normal(size=(T, N))
    info = np.zeros((T, N, abi.INFO_DIM))
    info[..., abi.INFO_FIELDS.index("aum")] = 1000.0 + np.arange(T)[:, None]
    info[..., abi.INFO_FIELDS.index("inventory")] = np.arange(N)[None, :]
    esd = evaluation.episode_summary_from_rollout(act, rew, info, BetaOrderDistributor(10))
    assert set(esd) == set(evaluation.SUMMARY_KEYS) and all(len(v) == N for v in esd.values())
    assert esd["actions"][1].shape == (3,) and np.allclose(esd["actions"][1], act[:, 1, :].mean(axis=0)[:-1])
    assert esd["inventory"][2] == 2.0 and np.allclose(esd["rewards"][0], rew[:, 0].mean())
    assert np.isfinite(evaluation.get_sharpe(np.stack(esd["equity_curves"]))).all()


def test_compress_order_dict_reference_test():
    """rl4mm/simulation/tests/testOrderbookSimulator.py:110-114 (test_compare_order_dict), on the façade's Order classes."""
    from collections import deque
    from datetime import datetime

    from rl4mm_b200.orderbook import Cancellation, LimitOrder
    from rl4mm_b200.simulation import OrderbookSimulator

    limit_1 = LimitOrder(datetime(2012, 6, 21, 12, 0), "buy", "MSFT", None, 50, True, int(30.1 * 10000), 1000)
    limit_2 = LimitOrder(datetime(2012, 6, 21, 12, 1), "buy", "MSFT", None, 100, True, int(30.1 * 10000), 200)
    cancellation_1 = Cancellation(datetime(2012, 6, 21, 12, 1), "buy", "MSFT", None, 50, True, int(30.1 * 10000), 200)
    cancellation_2 = Cancellation(datetime(2012, 6, 21, 12, 2), "buy", "MSFT", None, 50, False, int(30.1 * 10000), 1100)
    order_dict = {"gen_1": deque([limit_1, cancellation_1]), "gen_2": deque([limit_2, cancellation_2])}
    assert OrderbookSimulator._compress_order_dict(order_dict) == [limit_1, cancellation_1, limit_2, cancellation_2]
    assert OrderbookSimulator._compress_order_dict({"only": deque([limit_2, limit_1])}) == [limit_2, limit_1]   # one generator: as is


def test_generator_merge_matches_reference_golden():
    """The pack-time merge (packing.compress_order_sources) == the reference's ``_compress_order_dict`` on 200 random 2- / 3-generator
    step windows with colliding timestamps and cross-generator duplicate orders (tests/golden/generator_merge.json.gz, generated
    by oracle/gen_golden.py::golden_generator_merge from the unmodified reference)."""
    import gzip
    import json
    from pathlib import Path

    from rl4mm_b200.packing import RawMessages, compress_order_sources

    cases = json.loads(gzip.open(Path(__file__).parent / "golden" / "generator_merge.json.gz").read())
    assert len(cases) == 200
    t0_us, step_us = 36_000_000_000, 100_000
    n_multi = 0
    for c in cases:
        sources = {}
        for g, rows in enumerate(c["generators"]):
            col = lambda k: np.array([r[k] for r in rows], np.int64)        # noqa: E731
            sources[f"gen_{g}"] = RawMessages((t0_us + col("us")) * 1000, col("type"), col("ext_id"), col("size"), col("price"), col("direction"))
        merged = compress_order_sources(sources, t0_us, step_us)
        exp = [c["generators"][g][i] for g, i in c["merged"]]
        assert len(merged) == len(exp)
        for k, r in enumerate(exp):
            got = (int(merged.time_ns[k] // 1000 - t0_us), int(merged.msg_type[k]), int(merged.direction[k]), int(merged.ext_id[k]),
                   int(merged.size[k]), int(merged.price[k]))
            assert got == (r["us"], r["type"], r["direction"], r["ext_id"], r["size"], r["price"]), (c, k)
        n_multi += len(c["generators"]) > 1
    assert n_multi == 200


def test_pack_merged_two_generators():
    """Two generators end to end: per-source generator order (hidden dropped, lexicographic ties), step-wise merge, one packed
    stream whose snapshots follow the historical source."""
    from rl4mm_b200.packing import RawMessages, pack_arrays, pack_merged

    L = 2
    t0 = 34_200_000_000
    hist = RawMessages(np.array([t0 + 50_000, t0 + 50_000, t0 + 150_000, t0 + 1_250_000], np.int64) * 1000, np.array([1, 5, 3, 4]),
                       np.array([7, 8, 7, 9]), np.array([10, 10, 10, 5]), np.array([1000, 1000, 1000, 1100]), np.array([1, 1, 1, -1]))
    synth = RawMessages(np.array([t0 + 40_000, t0 + 50_000, t0 + 1_250_000], np.int64) * 1000, np.array([1, 1, 1]),
                        np.array([100, 101, 102]), np.array([3, 4, 5]), np.array([900, 1000, 1200]), np.array([1, 1, -1]))
    books = np.tile(np.array([1100, 5, 1000, 7, 9999999999, 0, -9999999999, 0], np.int64), (4, 1))
    books[:, 1] = np.arange(4)
    s = pack_merged({"historical": hist, "synthetic": synth}, books, L, t0_us=t0)
    assert s.generators == ("historical", "synthetic")
    # step 0: synth@40ms, then the two 50 ms orders -- equal timestamps keep the first generator (historical) first; the hidden
    # execution is gone; step 1: the deletion; step 12: equal timestamps again: historical first
    assert [int(x) for x in s.ext_ids[s.msgs["ref"]]] == [100, 7, 101, 7, 9, 102]
    assert list(s.step_off[:3]) == [0, 3, 4] and s.step_off[13] == 6 and s.step_off[12] == 4
    alone = pack_arrays(hist.time_ns, hist.msg_type, hist.ext_id, hist.size, hist.price, hist.direction, books, L, t0_us=t0)
    assert np.array_equal(s.snapshots, alone.snapshots) and np.array_equal(s.snap_valid, alone.snap_valid)
    one = pack_merged({"historical": hist}, books, L, t0_us=t0)
    assert np.array_equal(one.msgs, alone.msgs) and np.array_equal(one.step_off, alone.step_off)


def test_correctly_rounded_log_and_exp(tmp_path):
    """csrc/crmath.cuh (the RollingSharpe log / exp of the device path) compiled for the host: correctly rounded against
    60-digit decimal arithmetic on 2e4 arguments (AUM-like values around 1e12, the whole double range, values near 1; log-return
    sized exp arguments).  glibc's log -- what numpy calls -- is the same value except for a few arguments in 1e4."""
    import ctypes
    import math
    import subprocess
    from decimal import Decimal, getcontext
    from pathlib import Path

    src = tmp_path / "cr.cpp"
    src.write_text('#include "crmath.cuh"\nextern "C" double t_log(double x) { return cr_log(x); }\n'
                   'extern "C" double t_exp(double x) { return cr_exp(x); }\n')
    so = tmp_path / "libcr.so"
    csrc = Path(__file__).resolve().parent.parent / "rl4mm_b200" / "csrc"
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-I", str(csrc), "-o", str(so), str(src)], check=True)
    L = ctypes.CDLL(str(so))
    for f in (L.t_log, L.t_exp):
        f.restype, f.argtypes = ctypes.c_double, [ctypes.c_double]
    getcontext().prec = 60
    rng = np.random.default_rng(0)
    xs = np.concatenate([rng.uniform(0.5, 2, 3000), 10 ** rng.uniform(-300, 300, 3000), 1e12 + rng.uniform(-1e6, 1e6, 6000),
                         rng.uniform(0.99, 1.01, 2000), [1.0, 2.0, 0.5, 1e12, 1.4142135623730951, 1.414213562373095, 5e-324 * 2 ** 60]])
    glibc_differs = 0
    for x in xs.tolist():
        cr = float(Decimal(x).ln())
        assert L.t_log(x) == cr, x
        glibc_differs += math.log(x) != cr
    assert glibc_differs < len(xs) // 500
    for x in np.concatenate([rng.uniform(-0.015625, 0.015625, 3000), rng.uniform(-1e-8, 1e-8, 3000), [0.0, 0.015625, -0.015625]]).tolist():
        assert L.t_exp(x) == float(Decimal(x).exp()), x
    assert L.t_exp(0.5) == math.exp(0.5) and math.isnan(L.t_log(-1.0)) and L.t_log(float("inf")) == float("inf")


def test_reference_seeded_episode_starts():
    """VERDICT r1: with start_rng="numpy_global" the env draws its episode starts from numpy's global state with the reference's own
    call sequence (HOE.py:196,333-351), so np.random.seed(k) reproduces the reference's starts -- golden from the unmodified
    reference (oracle/gen_golden.py::golden_episode_starts): single day, a two-week range, and an empty offset range."""
    import gzip
    import json
    from datetime import datetime, timedelta
    from pathlib import Path

    import pandas as pd

    from rl4mm_b200.gym import reference_random_start_time

    cases = json.loads(gzip.open(Path(__file__).parent / "golden" / "episode_starts.json.gz").read())
    assert len(cases) == 18
    for c in cases:
        lo, hi = datetime.fromisoformat(c["min_date"]), datetime.fromisoformat(c["max_date"])
        days = [d.to_pydatetime() for d in pd.bdate_range(lo, hi)]           # every business day has packed data
        np.random.seed(c["seed"])
        got = [reference_random_start_time(lo, hi, timedelta(seconds=c["min_start_s"]), timedelta(seconds=c["max_end_s"]),
                                           timedelta(seconds=c["episode_s"]), timedelta(seconds=0.1), days).isoformat() for _ in range(4)]
        assert got == c["starts"], c


def test_month_archives_are_ingested_in_date_order(tmp_path, monkeypatch):
    """run_populate_database_from_zipped.py:50-109: archives ordered by the dates behind `__` (not the download number), ticker /
    dates / levels from the file name, one stream per trading day inside, extracted CSVs removed afterwards, days that are
    already loaded skipped, and a loud error when there is no 7z executable."""
    import shutil
    from datetime import datetime

    from rl4mm_b200 import archives
    from rl4mm_b200.simulation import DeviceDatabase

    # the reference's own example (its comment lists this folder): sorting whole names would put May first
    names = ["_data_dwn_50_385__KO_2018-04-01_2018-04-30_3.7z", "_data_dwn_50_389__KO_2018-02-01_2018-02-28_3.7z",
             "_data_dwn_50_386__KO_2018-03-01_2018-03-31_3.7z", "_data_dwn_50_384__KO_2018-05-01_2018-05-31_3.7z"]
    assert [n.split("_")[-3] for n in archives.archive_order(names)] == ["2018-02-01", "2018-03-01", "2018-04-01", "2018-05-01"]
    tk, d0, d1, L = archives.parse_archive_name("/data/KO/" + names[0])
    assert (tk, d0, d1, L) == ("KO", datetime(2018, 4, 1), datetime(2018, 4, 30), 3)
    with pytest.raises(ValueError):
        archives.parse_archive_name("/data/readme.7z")

    def write_day(folder, ticker, day, n=200, L=3, seed=0):
        rng = np.random.default_rng(seed)
        t = np.sort(rng.integers(34_200_000_000_000, 34_206_000_000_000, size=n))
        with open(folder / f"{ticker}_{day}_34200000_57600000_message_{L}.csv", "w") as f:
            for i in range(n):
                sec, ns = divmod(int(t[i]), 10**9)
                f.write(f"{sec}.{ns:09d},{rng.choice([1, 3, 4])},{rng.integers(1, 10**6)},{rng.integers(1, 500)},"
                        f"{3_000_000 + 100 * int(rng.integers(0, 50))},{rng.choice([-1, 1])}\n")
        rows = np.zeros((n, 4 * L), np.int64)
        for lv in range(L):
            rows[:, 4 * lv: 4 * lv + 4] = (3_050_100 + 100 * lv, 10 + lv, 3_050_000 - 100 * lv, 20 + lv)
        np.savetxt(folder / f"{ticker}_{day}_34200000_57600000_orderbook_{L}.csv", rows, fmt="%d", delimiter=",")

    content = {names[0]: ["2018-04-02", "2018-04-03"], names[1]: ["2018-02-01"], names[2]: ["2018-03-01", "2018-03-02"], names[3]: []}
    folder = tmp_path / "KO"
    folder.mkdir()
    for n_ in names:
        (folder / n_).write_bytes(b"7z\xbc\xaf\x27\x1c")          # only the name matters to the fake extractor below
    (folder / "notes.csv").write_text("keep me\n")                 # not created by an extraction: must survive
    seen = []

    def fake_extract(fpath, out_dir):
        seen.append(Path(fpath).name)
        for k, day in enumerate(content[Path(fpath).name]):
            write_day(Path(out_dir), "KO", day, seed=len(seen) * 10 + k)

    db = DeviceDatabase()
    ids = db.populate_from_archives(folder, extractor=fake_extract)
    assert seen == [names[1], names[2], names[0], names[3]]
    assert ids == [0, 1, 2, 3, 4]
    assert [d.strftime("%Y-%m-%d") for d in db.dates] == ["2018-02-01", "2018-03-01", "2018-03-02", "2018-04-02", "2018-04-03"]
    assert set(db.tickers) == {"KO"} and all(s.n_levels == 3 and len(s.msgs) > 0 for s in db.streams)
    assert sorted(p.name for p in folder.glob("*.csv")) == ["notes.csv"]
    assert db.stream_id("KO", datetime(2018, 3, 2)) == 2
    # a second pass adds nothing: every day is already there
    assert db.populate_from_archives(folder, extractor=fake_extract) == []
    # the default extractor is the reference's `7z x`: without the executable it must fail loudly, not skip
    monkeypatch.setattr(shutil, "which", lambda exe: None)
    with pytest.raises(RuntimeError, match="7z"):
        DeviceDatabase().populate_from_archives(folder)


def test_extract_7z_calls_the_tool_like_the_reference(tmp_path, monkeypatch):
    """run_populate_database_from_zipped.py:99 runs `7z x <archive> -o<folder>`: the default extractor builds the same command line
    (plus -y so that a re-run does not prompt) and fails loudly when the tool fails."""
    import os
    import stat
    import subprocess

    from rl4mm_b200 import archives

    bindir = tmp_path / "bin"
    bindir.mkdir()
    log = tmp_path / "args.txt"
    tool = bindir / "7z"
    tool.write_text(f"#!/bin/sh\necho \"$@\" > {log}\ncase \"$2\" in *broken*) exit 2;; esac\nexit 0\n")
    tool.chmod(tool.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", f"{bindir}{os.pathsep}{os.environ['PATH']}")
    archives.extract_7z(tmp_path / "a__KO_2018-02-01_2018-02-28_10.7z", tmp_path / "out")
    assert log.read_text().split() == ["x", str(tmp_path / "a__KO_2018-02-01_2018-02-28_10.7z"), "-o" + str(tmp_path / "out"), "-y"]
    with pytest.raises(subprocess.CalledProcessError):
        archives.extract_7z(tmp_path / "broken__KO_2018-02-01_2018-02-28_10.7z", tmp_path / "out")
