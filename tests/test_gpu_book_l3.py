"""lobsim_get_book_dev / lobsim_set_book_dev and LobSim.book_l3 / set_books: every env's L3 book read and replaced on the device
in one launch each.  book_l3 must equal lobsim_dump_book of every env and side bit for bit (price, volume, ref, level), on flat
blobs (read first: dump_book converts them), sorted, hybrid-replayed and deep-mode blobs and the books of dead envs, and must
change nothing.  set_books must do exactly what lobsim_set_book does per env, on the same entries, and report the env it
rejects or skips without touching it."""
import ctypes

import numpy as np
import pytest

import adversarial_streams as A
import parity_helpers as H
import random_cases as R
from rl4mm_b200 import abi

pytestmark = pytest.mark.gpu

EMPTY_SLOT = np.array([abi.NO_PRICE, 0, 0, -1], np.int32)


def rows_of(buy, sell, E):
    """dump_book-format arrays of one env -> (entries int32 [2, E, 4], count [2])."""
    ent = np.zeros((2, E, 4), np.int32)
    cnt = np.zeros(2, np.int32)
    for side, e in enumerate((buy, sell)):
        e = np.ascontiguousarray(e, abi.BOOK_ENTRY_DTYPE)
        ent[side, : len(e)] = e.view(np.int32).reshape(-1, 4)
        cnt[side] = len(e)
    return ent, cnt


def to_dev(books, E):
    """[(buy, sell)] per env -> entries [N, 2, E, 4] and count [N, 2] on the GPU."""
    import torch

    ents, cnts = zip(*(rows_of(b, s, E) for b, s in books))
    return torch.tensor(np.stack(ents), device="cuda"), torch.tensor(np.stack(cnts), device="cuda")


def assert_l3_is_dump(sim, what, E=None):
    """book_l3(E) == dump_book of every env and side.  The read comes first: dump_book converts flat blobs."""
    E = sim.cfg.max_orders_per_side if E is None else E
    count, entries = (t.cpu().numpy() for t in sim.book_l3(E))
    st = sim.state()
    for env in range(sim.n_envs):
        for side in (0, 1):
            d = sim.dump_book(env, side).view(np.int32).reshape(-1, 4)
            assert count[env, side] == len(d), (what, env, side, count[env, side], len(d))
            m = min(len(d), E)
            assert np.array_equal(entries[env, side, :m], d[:m]), (what, env, side)
            assert np.all(entries[env, side, m:] == EMPTY_SLOT), (what, env, side)
    return st


def same(x, y):
    """Bit-identical tensors (NaN observations of a dead book included)."""
    import torch

    if x.dtype.is_floating_point:
        return x.dtype == y.dtype and torch.equal(x.view(torch.int64), y.view(torch.int64))
    return torch.equal(x, y)


def canon(entries):
    """dump_book entries with the agent's ids dropped (the oracle numbers the agent's orders its own way)."""
    e = np.ascontiguousarray(entries, abi.BOOK_ENTRY_DTYPE)
    refs = np.where(e["ref"] & abi.REF_AGENT, abi.REF_AGENT, e["ref"])
    return [(int(p), int(v), int(r), int(k)) for p, v, r, k in zip(e["price"], e["volume"], refs, e["level"])]


# ---- 1. the read equals dump_book ------------------------------------------------------------------------------------------
@pytest.mark.replay_path
@pytest.mark.parametrize("seed", [2, 13, 15, 20])
def test_read_after_ragged_replays_equals_dump(seed, kernel_family):
    """Random replay cases (thin books in the flat pools, books around the pool capacity, deep books): book_l3 after every launch
    of a ragged replay, with room for every order and with max_entries 7 (count beyond max_entries)."""
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    c = R.random_replay_case(seed)
    s = synthetic.generate(c["synth"])
    cfg = abi.default_cfg(n_envs=c["n_envs"], **c["cfg_kw"])
    sim = make_sim(cfg, [s])
    sim.reset_book(0, c["starts"])
    flat_seen = False
    for chunk in c["chunks"]:
        for E in (cfg.max_orders_per_side, 7):
            sim.replay(chunk)
            flat_seen |= bool(np.any(sim.state()["reserved"] & 1))
            assert_l3_is_dump(sim, (seed, chunk, E), E)
    if kernel_family == "fast" and sim.kernel_path == "fast" and c["synth"].target_orders <= 30:
        assert flat_seen, "thin books are read in the flat form"
    sim.close()


STREAMS = [(shape, seed) for shape, sh in A.SHAPES.items() for seed in sh["seeds"]]


@pytest.mark.replay_path
@pytest.mark.parametrize("shape,seed", STREAMS)
def test_read_on_adversarial_streams(shape, seed, kernel_family):
    """Sides emptied by sweeps, dead books (read as they are), full flat pools and an uncompiled layout: book_l3 after every
    ragged replay launch."""
    from rl4mm_b200.device import LobSim

    s = A.build(shape, seed)
    starts = [10 * t for t in A.STARTS]
    cfg = A.cfg_for(shape, n_envs=len(starts), resync=0, outer_levels=2)
    sim = LobSim(cfg, 0)
    sim.load_stream(0, s)
    sim.reset_book(0, np.array(starts, np.int32))
    done, k, flat_reads = 0, 0, 0
    while done < s.n_grid_steps:
        chunk = (1, 3, 7, 10, 23, 57)[k % 6]
        k += 1
        sim.replay(chunk)
        done += chunk
        flat_reads += int(np.sum(sim.state()["reserved"] & 1))
        st = assert_l3_is_dump(sim, (shape, seed, done))
    assert np.any(st["err"] & abi.ERR_EMPTY_BOOK), "the stream kills at least one of its books"
    if shape == "thin" and kernel_family in ("fast", "hybrid"):
        assert flat_reads > 0, "flat blobs were read"
    sim.close()


def _agent_bed(n=4, seed=3):
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    s = synthetic.generate(synthetic.spy_day(seed=seed, n_msgs=60_000, duration_s=200))
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6)]
    kw = dict(n_levels=10, episode_steps=60, warmup_steps=10, features=feats, step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
              terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), initial_cash=1e7, max_levels_per_side=64, max_orders_per_side=256,
              max_agent_orders=64)
    return s, kw, (lambda m=n: make_sim(abi.default_cfg(n_envs=m, **kw), [s]))


TERADACTYL = abi.Agent(kind=abi.AGENT_TERADACTYL, inventory_index=1, max_inventory=300.0, default_kappa=6.0, default_omega=0.5,
                       max_kappa=12.0, exponent=1.5, market_clearing=0)


def test_read_with_agent_orders(kernel_family):
    """The agent's ladders from rollouts, then process_orders and submit_orders with agent limits: book_l3 == dump_book, with
    agent refs in the books."""
    import torch

    _, _, make = _agent_bed()
    sim = make()
    n = sim.n_envs
    sim.reset(0, np.array([200, 500, 900, 1400], np.int32))
    fixed = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 3, 2, 1, 0))
    agents = 0
    for t, agent in enumerate((fixed, TERADACTYL, fixed)):
        sim.rollout(4, agent)
        count, entries = sim.book_l3()
        agents += int(((entries[..., 2].cpu().numpy().view(np.uint32) & abi.REF_AGENT) != 0).sum())
        assert_l3_is_dump(sim, ("rollout", t))
    assert agents > 0, "the agent's orders rest in the books"
    st = sim.state()
    orders = []
    for env in range(n):
        bb, bs = int(st["best_buy"][env]), int(st["best_sell"][env])
        orders += [(env, abi.MSG_LIMIT, 0, bb, 37, 0, 0, 0), (env, abi.MSG_LIMIT, 1, bs + 1300, 3, 0, 0, 0),
                   (env, abi.MSG_LIMIT, 0, bb - 4100, 8, 0, 0, 0)]
    sim.process_orders(np.array(orders, abi.ORDER_DTYPE))
    assert_l3_is_dump(sim, "process_orders", 16)
    st = sim.state()
    bb = torch.tensor(st["best_buy"].astype(np.int64))
    typ = torch.full((n, 2), abi.MSG_LIMIT)
    sim.submit_orders(abi.pack_orders(typ, torch.tensor([0, 1]).expand(n, 2), torch.stack([bb - 200, bb + 5000], 1), 9).cuda())
    assert_l3_is_dump(sim, "submit_orders")
    assert_l3_is_dump(sim, "submit_orders, 1 entry", 1)
    sim.close()


@pytest.mark.fast_only        # deep-book capacities always run the general kernel on the blobs in HBM
def test_read_deep_books_in_hbm():
    """256 levels x 16 384 orders per side (deep-book mode, blobs in HBM): book_l3 == dump_book with every order."""
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    sc = synthetic.SynthConfig(seed=11, n_msgs=300_000, duration_s=600, n_levels=50, mid0=2_000_000, p_limit=0.40, p_cancel=0.15,
                               p_delete=0.37, p_exec=0.08, geom_p=0.10, init_levels=70, mean_queue=80, target_orders=6000,
                               max_offset_ticks=80)
    s = synthetic.generate(sc)
    sim = make_sim(abi.default_cfg(n_envs=3, n_levels=50, outer_levels=20, max_levels_per_side=256, max_orders_per_side=16384,
                                   max_agent_orders=64), [s])
    assert sim.kernel_path == "deep"
    sim.reset_book(0, np.array([0, 500, 1500], np.int32))
    for chunk in (1, 99, 1900):
        sim.replay(chunk)
        assert_l3_is_dump(sim, ("deep", chunk))
    count = sim.book_l3(100)[0].cpu().numpy()
    assert count.max() > 1600, count
    sim.close()


# ---- 2. the read changes nothing -------------------------------------------------------------------------------------------
def test_read_has_no_side_effects(kernel_family):
    """Handles a and b run the same program; a reads book_l3 before and after every call, b never does.  State (book form bit
    included), errors, outputs and the final books are identical, and every read is exactly one launch."""
    import torch

    s, kw, make = _agent_bed(n=6, seed=5)
    a, b = make(), make()
    n = 6
    starts = np.array([100, 300, 500, 700, 900, 1100], np.int32)
    rng = np.random.default_rng(2)
    acts = [torch.tensor(rng.uniform(0.5, 6.0, size=(n, abi.action_dim(a.cfg))), device="cuda") for _ in range(3)]
    program = [lambda h: h.reset_book(0, starts), lambda h: h.replay(7), lambda h: h.replay(23), lambda h: h.reset(0, starts + 100)]
    program += [lambda h, x=x: h.step(x) for x in acts]
    program += [lambda h: h.rollout(5, TERADACTYL), lambda h: h.reset_book(0, starts + 50), lambda h: h.replay(31)]
    flat_reads = 0
    for i, call in enumerate(program):
        for E in (a.cfg.max_orders_per_side, 5):
            c = a.launch_count
            a.book_l3(E)
            assert a.launch_count == c + 1, (i, E)
        flat_reads += int(np.sum(a.state()["reserved"] & 1))
        ra, rb = call(a), call(b)
        if isinstance(ra, tuple):
            for x, y in zip(ra, rb):
                assert same(x, y), i
        elif isinstance(ra, torch.Tensor):
            assert torch.equal(ra, rb), i
        a.book_l3()
        assert torch.equal(a.state_dev(), b.state_dev()), i
        assert np.array_equal(a.errors(), b.errors()), i
    if kernel_family == "fast":
        assert flat_reads > 0, "some reads found flat blobs pending"
    for env in range(n):
        for side in (0, 1):
            assert np.array_equal(a.dump_book(env, side), b.dump_book(env, side)), (env, side)
            assert np.array_equal(a.dump_agent_orders(env, side), b.dump_agent_orders(env, side)), (env, side)
    a.close()
    b.close()


# ---- 3. set_books == set_book per env ---------------------------------------------------------------------------------------
def _hand_books(rng, mid, caps):
    """Books with agent orders (duplicate ids within and across sides), an empty and a one-sided book, and one at exactly
    max_levels_per_side levels and max_orders_per_side orders."""
    NL, NO, _ = caps
    E = abi.BOOK_ENTRY_DTYPE
    dup = [np.array([(mid - 100, 5, 0, 0), (mid - 100, 7, abi.REF_AGENT | 9, 0), (mid - 200, 3, 1 << 28, 0),
                     (mid - 200, 4, abi.REF_AGENT | 9, 0), (mid - 400, 2, abi.REF_AGENT | 3, 0), (mid - 400, 6, (1 << 28) + 1, 0)], E),
           np.array([(mid + 100, 8, abi.REF_AGENT | 3, 0), (mid + 100, 1, (1 << 28) + 2, 0), (mid + 300, 2, abi.REF_AGENT | 40, 0),
                     (mid + 300, 5, abi.REF_AGENT | 3, 0)], E)]
    empty = [np.zeros(0, E), np.zeros(0, E)]
    one_sided = [np.array([(mid - 100 * (k + 1), int(rng.integers(1, 50)), (1 << 28) + 10 + k, 0) for k in range(5)], E), np.zeros(0, E)]
    per = NO // NL
    full_buy = np.array([(mid - 100 * (k // per + 1), 1 + k % 13, (1 << 28) + 100 + k, 0) for k in range(NO)], E)
    full = [full_buy, np.array([(mid + 100, 4, 0, 0)], E)]
    return [dup, empty, one_sided, full]


def test_set_books_equals_set_book_and_oracle(kernel_family):
    """Oracle dumps of replayed books, hand-built books (duplicate agent ids, empty, one-sided, exactly NL levels and NO orders)
    and random books: set_books on one handle, set_book per env on a twin, Oracle.set_book.  Books, agent tables and state
    agree; then a Teradactyl rollout, replay and forward_step on all three give identical books and outputs (the oracle: books
    and obs / rewards within the parity tolerance)."""
    import torch

    from oracle.oracle import Oracle
    from test_gpu_call_sequences import _random_book

    s, kw, make = _agent_bed(n=10, seed=7)
    a, b = make(10), make(10)
    cfg = a.cfg
    caps = (cfg.max_levels_per_side, cfg.max_orders_per_side, cfg.max_agent_orders)
    starts = np.array([300, 400, 500, 600, 700, 800, 900, 1000, 1100, 1200], np.int32)
    oracles = [Oracle(abi.default_cfg(**kw), s, env_index=i) for i in range(10)]
    a.reset(0, starts)
    b.reset(0, starts)
    for o, st in zip(oracles, starts):
        o.reset(int(st))
    rng = np.random.default_rng(17)
    mids = [(int(o.state()["best_buy"]) + int(o.state()["best_sell"])) // 200 * 100 for o in oracles]
    books = []
    for env in range(10):
        if env in (0, 1, 2):            # the book of the same stream at an earlier clock, replayed
            src = Oracle(abi.default_cfg(**kw), s)
            src.reset_book(int(starts[env]) - 100)
            src.replay(37)
            books.append([src.dump_book(0), src.dump_book(1)])
        elif env in (3, 4, 5, 6):
            books.append(_hand_books(rng, mids[env], caps)[env - 3])
        else:
            books.append(_random_book(rng, mids[env], caps, (1 << 29) + 1000 * env)[0])
    E = max(cfg.max_orders_per_side, max(len(x) for bk in books for x in bk))
    ent, cnt = to_dev(books, E)
    status = a.set_books(ent, cnt)
    assert status.cpu().tolist() == [abi.SETBOOK_OK] * 10
    no_oracle = {3}                     # agent ids that do not rise along their queues: a book the reference cannot hold
    for env, (buy, sell) in enumerate(books):
        b.set_book(env, buy, sell)
        if env not in no_oracle:
            oracles[env].set_book(buy, sell)
    sa = a.state()
    assert torch.equal(a.state_dev(), b.state_dev())
    assert not sa["err"].any()
    for env, (buy, sell) in enumerate(books):
        for side, want in enumerate((buy, sell)):
            d = a.dump_book(env, side)
            assert np.array_equal(d, b.dump_book(env, side)), (env, side)
            assert np.array_equal(d[["price", "volume", "ref"]], np.ascontiguousarray(want, abi.BOOK_ENTRY_DTYPE)[["price", "volume", "ref"]])
            assert np.array_equal(a.dump_agent_orders(env, side), b.dump_agent_orders(env, side)), (env, side)
            assert env in no_oracle or canon(d) == canon(oracles[env].dump_book(side)), (env, side)
            assert len(a.dump_agent_orders(env, side)) == sa["n_agent_orders"][env][side]
        ids = [int(e["ref"]) & 0x7FFFFFFF for x in (buy, sell) for e in x if e["ref"] & abi.REF_AGENT]
        if ids:
            assert sa["next_agent_id"][env] >= max(ids) + 1
    ag = a.dump_agent_orders(3, 0)
    assert list(ag["ref"] & 0x7FFFFFFF) == [3, 9, 9] and list(ag["price"]) == [mids[3] - 400, mids[3] - 100, mids[3] - 200]
    # then the same program on the three
    ra, rb = a.rollout(20, TERADACTYL), b.rollout(20, TERADACTYL)
    for x, y in zip(ra, rb):
        assert same(x, y)
    obs, _, rew, _ = (x.cpu().numpy() for x in ra)
    orc = [o.rollout(20, TERADACTYL) for o in oracles]
    a.replay(7)
    b.replay(7)
    a.forward_step(13)
    b.forward_step(13)
    for o in oracles:
        o.replay(7)
        o.forward_step(13)
    st = a.state()
    assert torch.equal(a.state_dev(), b.state_dev())
    compared = 0
    for env, o in enumerate(oracles):
        for side in (0, 1):
            assert np.array_equal(a.dump_book(env, side), b.dump_book(env, side)), (env, side)
            assert np.array_equal(a.dump_agent_orders(env, side), b.dump_agent_orders(env, side)), (env, side)
        if env in no_oracle or H.capacity_excluded(st["err"][env], o, cfg, env) or int(o.state()["err"]) & abi.ERR_EMPTY_BOOK:
            continue
        compared += 1
        for t in range(20):
            H.assert_close_vec(obs[t, env], orc[env][0][t], (env, t))
            assert H.close(rew[t, env], orc[env][2][t]), (env, t)
        for side in (0, 1):
            d = a.dump_book(env, side)
            assert np.array_equal(d, b.dump_book(env, side)), (env, side)
            assert canon(d) == canon(o.dump_book(side)), (env, side)
    assert compared >= 5, compared
    a.close()
    b.close()


# ---- 4. flat blobs ----------------------------------------------------------------------------------------------------------
@pytest.mark.replay_path
def test_set_books_between_flat_replays(kernel_family):
    """Thin books left flat by a replay: set_books replaces every other env (count -1 skips the rest).  The set envs read back
    what was set and then stay bit-identical to a twin handle that got the same books from set_book per env; the others stay
    flat and unchanged, and equal to the oracle, through the next replays."""
    import torch

    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim

    s = A.build("thin", 0)
    starts = [10 * t for t in A.STARTS]
    n = len(starts)
    cfg = A.cfg_for("thin", n_envs=n, resync=0, outer_levels=2)
    sim, twin = LobSim(cfg, 0), LobSim(cfg, 0)
    for h in (sim, twin):
        h.load_stream(0, s)
        h.reset_book(0, np.array(starts, np.int32))
    oracles = [Oracle(A.cfg_for("thin", resync=0, outer_levels=2), s) for _ in starts]
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    for _ in range(40):              # until an env that will be skipped holds a flat blob (fast family)
        for h in (sim, twin, *oracles):
            h.replay(3)
        before = sim.state()
        if kernel_family != "fast" or np.any(before["reserved"][1::2] & 1):
            break
    if kernel_family == "fast":
        assert np.any(before["reserved"][1::2] & 1), "the replay left blobs flat"
    # a set env gets the (oracle) book of the env before it, from an earlier clock of the same stream
    E = cfg.max_orders_per_side
    books = [[oracles[max(e - 1, 0)].dump_book(0), oracles[max(e - 1, 0)].dump_book(1)] for e in range(n)]
    ent, cnt = to_dev(books, E)
    cnt[1::2] = -1
    status = sim.set_books(ent, cnt).cpu().numpy()
    assert list(status) == [abi.SETBOOK_OK if e % 2 == 0 else abi.SETBOOK_SKIPPED for e in range(n)]
    after = sim.state()
    for e in range(n):
        if e % 2 == 0:
            assert not after["reserved"][e] & 1
            twin.set_book(e, *books[e])
        else:
            assert after[e].tobytes() == before[e].tobytes(), e
    assert_l3_is_dump(sim, "after set_books")
    for e, o in enumerate(oracles):
        for side in (0, 1):
            assert canon(sim.dump_book(e, side)) == canon(o.dump_book(side) if e % 2 else books[e][side]), (e, side)
    for chunk in (3, 10, 57):
        sim.replay(chunk)
        twin.replay(chunk)
        for o in oracles:
            o.replay(chunk)
        assert_l3_is_dump(sim, ("replay", chunk))
        assert torch.equal(sim.state_dev(), twin.state_dev()), chunk
        for e, o in enumerate(oracles):
            for side in (0, 1):
                d = sim.dump_book(e, side)
                assert np.array_equal(d, twin.dump_book(e, side)), (chunk, e, side)
                if e % 2 and not int(o.state()["err"]) & abi.ERR_EMPTY_BOOK:
                    assert canon(d) == canon(o.dump_book(side)), (chunk, e, side)
    sim.close()
    twin.close()


# ---- 5. skip and reject ------------------------------------------------------------------------------------------------------
def test_skip_and_reject_in_one_call(kernel_family):
    """Every LOBSIM_SETBOOK_E_* condition, two conditions at once (the first in check order is reported) and the skip, next to
    valid envs in one call.  Rejected and skipped envs are unchanged, their error bits included; valid envs are set and their
    error bits cleared."""
    import torch

    from rl4mm_b200.device import LobSim

    kw = dict(n_levels=10, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32)
    n = 11
    sim = LobSim(abi.default_cfg(n_envs=n, **kw), 0)
    mid = 1_000_000
    base = [np.array([(mid - 100, 5, 1, 0), (mid - 200, 6, 2, 0)], abi.BOOK_ENTRY_DTYPE),
            np.array([(mid + 100, 7, 3, 0), (mid + 100, 8, abi.REF_AGENT | 4, 0)], abi.BOOK_ENTRY_DTYPE)]
    for env in range(n):
        sim.set_book(env, *base)
    # BAD_VOLUME on every env: a limit order of volume 0
    sim.process_orders(np.array([(e, abi.MSG_LIMIT, 0, mid - 100, 0, 0, 0, 0) for e in range(n)], abi.ORDER_DTYPE))
    assert np.all(sim.errors() & abi.ERR_BAD_VOLUME)
    E = 320
    ent = np.zeros((n, 2, E, 4), np.int32)
    cnt = np.zeros((n, 2), np.int32)

    def put(env, side, rows):
        rows = np.array(rows, np.int64).astype(np.uint32).view(np.int32)
        ent[env, side, : len(rows)] = rows
        cnt[env, side] = len(rows)

    def ladder(side, n_levels, per, start=0, agent=False):
        sgn = -1 if side == 0 else 1
        return [(mid + sgn * 100 * (k // per + 1), 1 + k % 5, (abi.REF_AGENT | (k + 1)) if agent else 1000 + k + start, 0)
                for k in range(n_levels * per)]

    want = {}
    put(0, 0, ladder(0, 3, 2)), put(0, 1, ladder(1, 2, 1)); want[0] = abi.SETBOOK_OK
    put(1, 0, ladder(0, 2, 2)); cnt[1, 1] = -1; want[1] = abi.SETBOOK_SKIPPED
    put(2, 0, ladder(0, 2, 2)); cnt[2, 1] = E + 1; want[2] = abi.SETBOOK_E_COUNT
    put(3, 0, ladder(0, 2, 2)), put(3, 1, [(mid + 100, -1, 5, 0)]); want[3] = abi.SETBOOK_E_VOLUME
    put(4, 0, [(mid - 100, 1, 1, 0), (mid - 200, 1, 2, 0), (mid - 100, 1, 3, 0)]); want[4] = abi.SETBOOK_E_UNSORTED
    put(5, 1, [(mid + 200, 1, 1, 0), (mid + 100, 1, 2, 0)]); want[5] = abi.SETBOOK_E_UNSORTED
    put(6, 0, ladder(0, 65, 1)); want[6] = abi.SETBOOK_E_LEVELS
    put(7, 1, ladder(1, 64, 5)); want[7] = abi.SETBOOK_E_ORDERS
    put(8, 0, ladder(0, 33, 1, agent=True)); want[8] = abi.SETBOOK_E_AGENTS
    put(9, 0, [(mid - 100, -4, 1, 0), (mid, 1, 2, 0)]); want[9] = abi.SETBOOK_E_VOLUME      # negative and unsorted: the first
    put(10, 0, ladder(0, 64, 4)), put(10, 1, ladder(1, 1, 32, agent=True)); want[10] = abi.SETBOOK_OK   # exactly at every capacity
    before = sim.state()
    books = [[sim.dump_book(e, s) for s in (0, 1)] for e in range(n)]
    agents = [[sim.dump_agent_orders(e, s) for s in (0, 1)] for e in range(n)]
    status = sim.set_books(torch.tensor(ent, device="cuda"), torch.tensor(cnt, device="cuda")).cpu().numpy()
    assert list(status) == [want[e] for e in range(n)]
    after = sim.state()
    for e in range(n):
        if want[e] == abi.SETBOOK_OK:
            assert after["err"][e] == 0
            for s in (0, 1):
                got = sim.dump_book(e, s).view(np.int32).reshape(-1, 4)
                assert np.array_equal(got[:, :3], ent[e, s, : cnt[e, s], :3]), (e, s)
        else:
            assert after[e].tobytes() == before[e].tobytes(), e
            assert after["err"][e] & abi.ERR_BAD_VOLUME
            for s in (0, 1):
                assert np.array_equal(sim.dump_book(e, s), books[e][s]), (e, s)
                assert np.array_equal(sim.dump_agent_orders(e, s), agents[e][s]), (e, s)
    assert len(sim.dump_agent_orders(10, 1)) == 32 and after["n_agent_orders"][10][1] == 32
    sim.close()


# ---- 6. round trip and tiling ------------------------------------------------------------------------------------------------
def test_round_trip_and_tiling(kernel_family):
    """set_books(*book_l3()) on a fresh handle reproduces every book (agent orders included); 8 source books tiled over 4 096
    envs give the same books and state as set_book per env on a twin."""
    import torch

    _, _, make = _agent_bed(n=8, seed=9)
    src = make(8)
    src.reset(0, np.array([200, 350, 500, 650, 800, 950, 1100, 1250], np.int32))
    src.rollout(12, TERADACTYL)
    src.replay(4)
    count, entries = src.book_l3()
    dst = make(8)
    assert dst.set_books(entries, count).cpu().tolist() == [abi.SETBOOK_OK] * 8
    c2, e2 = dst.book_l3()
    assert torch.equal(c2, count) and torch.equal(e2, entries)
    for env in range(8):
        for side in (0, 1):
            assert np.array_equal(dst.dump_book(env, side), src.dump_book(env, side)), (env, side)
            assert np.array_equal(dst.dump_agent_orders(env, side), src.dump_agent_orders(env, side)), (env, side)
    N = 4096
    tiled, twin = make(N), make(N)
    idx = torch.arange(N, device="cuda") % 8
    assert bool((tiled.set_books(entries[idx].contiguous(), count[idx].contiguous()) == abi.SETBOOK_OK).all())
    host = [[src.dump_book(e, s) for s in (0, 1)] for e in range(8)]
    for env in range(N):
        twin.set_book(env, *host[env % 8])
    assert torch.equal(tiled.state_dev(), twin.state_dev())
    ct, et = tiled.book_l3()
    cw, ew = twin.book_l3()
    assert torch.equal(ct, cw) and torch.equal(et, ew)
    assert torch.equal(et, entries[idx])
    for h in (src, dst, tiled, twin):
        h.close()


# ---- 7. CUDA graph -----------------------------------------------------------------------------------------------------------
def test_cuda_graph_capture(kernel_family):
    """set_books(out=) + forward_step + book_l3(out=) captured once in a CUDA graph on a side stream and replayed == an eager twin."""
    import torch

    s, kw, make = _agent_bed(n=12, seed=21)
    g, e_ = make(12), make(12)
    starts = np.arange(12, dtype=np.int32) * 100 + 200
    for h in (g, e_):
        h.reset_book(0, starts)
        h.replay(5)
    count, entries = g.book_l3()
    count = count.flip(0).contiguous()            # each env gets another env's book
    entries = entries.flip(0).contiguous()
    count[3] = -1
    E = g.cfg.max_orders_per_side
    out_s = torch.empty(12, dtype=torch.int32, device="cuda")
    out_l3 = (torch.empty((12, 2), dtype=torch.int32, device="cuda"), torch.empty((12, 2, E, 4), dtype=torch.int32, device="cuda"))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g.set_books(entries, count, out=out_s, stream=side)
        g.forward_step(2, stream=side)
        g.book_l3(out=out_l3, stream=side)
    torch.cuda.current_stream().wait_stream(side)
    e_.set_books(entries, count)
    e_.forward_step(2)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        g.set_books(entries, count, out=out_s, stream=side)
        g.forward_step(2, stream=side)
        g.book_l3(out=out_l3, stream=side)
    for k in range(4):
        graph.replay()
        st = e_.set_books(entries, count)
        e_.forward_step(2)
        want = e_.book_l3()
        torch.cuda.synchronize()
        assert torch.equal(out_s, st), k
        assert torch.equal(out_l3[0], want[0]) and torch.equal(out_l3[1], want[1]), k
        assert torch.equal(g.state_dev(), e_.state_dev()), k
    assert out_s.cpu().tolist() == [abi.SETBOOK_SKIPPED if i == 3 else abi.SETBOOK_OK for i in range(12)]
    g.close()
    e_.close()


# ---- 8. argument errors ------------------------------------------------------------------------------------------------------
def test_argument_errors(kernel_family):
    """NULL pointers, max_entries out of range and misaligned pointers are LOBSIM_E_INVALID and launch nothing; the façade rejects
    wrong shapes, dtypes, devices and non-contiguous tensors.  A fresh handle reads empty books."""
    import torch

    from rl4mm_b200._lib import LobsimError, lib
    from rl4mm_b200.device import LobSim

    sim = LobSim(abi.default_cfg(n_envs=5, n_levels=10, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32), 0)
    count, entries = sim.book_l3()
    assert count.shape == (5, 2) and entries.shape == (5, 2, 256, 4) and entries.dtype == torch.int32
    assert not count.any() and bool((entries == torch.tensor(EMPTY_SLOT, device="cuda")).all())
    L = lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    cp, ep = ctypes.c_void_p(count.data_ptr()), ctypes.c_void_p(entries.data_ptr())
    status = torch.empty(5, dtype=torch.int32, device="cuda")
    sp = ctypes.c_void_p(status.data_ptr())
    assert L.lobsim_get_book_dev(sim._h, 3, cp, ep, st) == abi.OK
    assert L.lobsim_set_book_dev(sim._h, 3, ep, cp, sp, st) == abi.OK
    mis = ctypes.c_void_p(entries.data_ptr() + 4)
    for args in ((0, cp, ep), (257, cp, ep), (-1, cp, ep), (3, None, ep), (3, cp, None), (3, cp, mis)):
        c = sim.launch_count
        assert L.lobsim_get_book_dev(sim._h, *args, st) == abi.E_INVALID, args
        assert sim.launch_count == c
    for args in ((0, ep, cp, sp), (3, None, cp, sp), (3, ep, None, sp), (3, ep, cp, None), (3, mis, cp, sp),
                 (3, ep, ctypes.c_void_p(count.data_ptr() + 2), sp)):
        c = sim.launch_count
        assert L.lobsim_set_book_dev(sim._h, *args, st) == abi.E_INVALID, args
        assert sim.launch_count == c
    assert L.lobsim_get_book_dev(None, 3, cp, ep, st) == abi.E_INVALID
    assert L.lobsim_set_book_dev(None, 3, ep, cp, sp, st) == abi.E_INVALID
    for bad in (0, -1, 257):
        with pytest.raises(LobsimError):
            sim.book_l3(bad)
    with pytest.raises(ValueError):
        sim.book_l3(out=(count, entries[:, :, :8]))
    with pytest.raises(ValueError):
        sim.book_l3(out=(count.to(torch.int64), entries))
    ent = torch.zeros((5, 2, 4, 4), dtype=torch.int32, device="cuda")
    for bad in (ent[:4], ent.to(torch.int64), ent.cpu(), ent[:, :1], ent.transpose(0, 1).contiguous().transpose(0, 1),
                torch.zeros((5, 2, 0, 4), dtype=torch.int32, device="cuda"), torch.zeros((5, 2, 4, 3), dtype=torch.int32, device="cuda")):
        with pytest.raises(ValueError):
            sim.set_books(bad)
    with pytest.raises(ValueError):
        sim.set_books(ent, torch.zeros(5, dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        sim.set_books(ent, out=torch.zeros(5, dtype=torch.int64, device="cuda"))
    assert sim.set_books(ent).cpu().tolist() == [abi.SETBOOK_OK] * 5       # E = 4 zero entries: price 0, volume 0 on each side
    sim.close()
