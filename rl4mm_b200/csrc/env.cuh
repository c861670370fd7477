// env.cuh -- simulator / gym-environment layer on top of book.cuh: outer-level resync, the agent's action ->
// orders conversion, features and rewards.  Everything is warp-collective (uniform control flow) except the feature
// updates, which run one feature per lane.
#pragma once
#include <math.h>

#include "book.cuh"
#include "book_fast.cuh"
#include "crmath.cuh"

struct __align__(16) FeatState {
  double cur;        // Feature.current_value
  long long total;   // total_trades / total_volume
  long long diff;    // trade_diff / volume_imbalance
  int32_t len;       // deque length (bit 30: running sums valid)
  int32_t head;      // circular write position
};
static_assert(sizeof(FeatState) == 32, "FeatState layout");
// rolling z-score (Feature.normalise): shifted running sums over the history ring.  A separate array that exists only for
// configurations with normalisation_on features: the per-step feature phase of every other configuration moves 32 B per feature.
struct __align__(16) NormState {
  double nK, nS1, nS2; // shift K (first history value), sum (x-K), sum (x-K)^2
  int32_t nlen, nhead; // history length, next write position (= oldest entry once full)
  int32_t nrun;        // number of equal trailing history values (constant window)
  int32_t pad;
  double nS2max;       // largest nS2 since the sums were last recomputed exactly (bounds their accumulated rounding error)
};
static_assert(sizeof(NormState) == 48, "NormState layout");
#define FEAT_SUMS_VALID (1 << 30)

struct EnvConst { // what the device needs of lobsim_cfg_t, by value in the kernel parameters
  lobsim_cfg_t cfg;
  int32_t ring_off[LOBSIM_MAX_FEATURES]; // slot offset of each feature's ring inside an env's ring block
  int32_t hist_off[LOBSIM_MAX_FEATURES]; // slot offset of each feature's normalisation history (norm_len slots)
  int32_t ring_stride;                   // slots per env
  int32_t action_dim, obs_dim;
  int32_t steps_per_sec;                 // 1000000 / step_us        } precomputed on the host: 64-bit and fp64 divisions are
  double outer_prop;                     // outer_levels / n_levels  } subroutine calls on the device, unwanted in the hot kernels
  int32_t steps_per_min;                 // 60000000 / step_us
  int32_t pad0;
  long long feat_aux[LOBSIM_MAX_FEATURES]; // TIME_OF_DAY: the bucket width in microseconds (Features.py:526-536), else 0
};

__device__ __forceinline__ long long now_us_of(const lobsim_stream_t& st, const lobsim_cfg_t& c, int now_step) {
  return st.t0_us + (long long)now_step * c.step_us;
}

// a[i] for a register-resident 5-vector and a runtime index (keeps the array out of local memory)
__device__ __forceinline__ double pick5(const double* a, int i) {
  double r = a[0];
#pragma unroll
  for (int k = 1; k < 5; k++) r = (i == k) ? a[k] : r;
  return r;
}

// ---- OrderbookSimulator._near_exiting_initial_price_range, OrderbookSimulator.py:177-183 -------------------------
__device__ __forceinline__ bool near_exiting(const Book& b, const WarpState& w, const lobsim_cfg_t& c) {
  const BookHdr* h = b.hdr();
  double prop = (double)c.outer_levels / (double)c.n_levels;
  double bb = w.nlv0 ? (double)b.lvp(0)[w.nlv0 - 1] : 0.0;
  double bs = w.nlv1 ? (double)b.lvp(1)[w.nlv1 - 1] : (double)INFINITY;
  return bb < (double)h->min_buy + prop * (double)h->init_buy_range || bs > (double)h->max_sell - prop * (double)h->init_sell_range;
}

// ---- OrderbookSimulator.update_outer_levels, OrderbookSimulator.py:105-135 ---------------------------------------
// scratch: per-warp shared int2[2*NA] for the agent orders that are cancelled and re-queued behind the aggregates.
__device__ __forceinline__ void update_outer_levels_impl(const Book& b, WarpState& w, const lobsim_cfg_t& c, const int32_t* __restrict__ row, int2* scratch) {
  BookHdr* h = b.hdr();
  const int L = c.n_levels;
  const int min_buy = h->min_buy, max_sell = h->max_sell;
  int nrepl = 0, nrepl_buy = 0;
  for (int side = 0; side < 2; side++) {
    for (int lvl = 0; lvl < L; lvl++) {
      int price = __ldg(&row[(side * L + lvl) * 2]), vol = __ldg(&row[(side * L + lvl) * 2 + 1]);
      if (price == LOBSIM_NO_PRICE) continue;
      if (!(side == 0 ? price < min_buy : price > max_sell)) continue; // _initial_prices_filter_function :99-103
      for (int i = 0; i < NAG(w, side);) { // internal orders at this price: cancel now, re-queue later (:116-129)
        int ap = b.aprice(side)[i], av = b.avol(side)[i];
        uint32_t id = b.aid(side)[i];
        __syncwarp();
        if (ap != price) { i++; continue; }
        if (b.lane == 0) scratch[nrepl] = make_int2(price, av);
        nrepl++;
        int before = NAG(w, side);
        remove_order(b, w, side, price, av, true, LOBSIM_REF_AGENT | id, true);
        if (NAG(w, side) == before) agent_remove_at(b, w, side, i); // keep internal and central consistent
      }
      bool found;
      int j = find_level(b, side, NLV(w, side), price, found); // central[dir][price] = deque([aggregate]) :130
      if (found) {
        int start = level_start(b, side, j), end = b.lvend(side)[j];
        __syncwarp();
        if (end - start > 1) remove_entries(b, w, side, j, start + 1, end - start - 1);
        if (b.lane == 0) b.ord(side)[start] = make_uint2((unsigned)vol, LOBSIM_REF_AGGREGATE);
        __syncwarp();
      } else if (NORD(w, side) >= b.L.NO) {
        w.err |= LOBSIM_ERR_ORDER_OVERFLOW;
      } else if (insert_level(b, w, side, j, price)) {   // (a full side: insert_level flags LEVEL_OVERFLOW)
        add_order(b, w, side, j, vol, LOBSIM_REF_AGGREGATE);
      }
    }
    if (side == 0) nrepl_buy = nrepl;
  }
  __syncwarp();
  for (int i = 0; i < nrepl; i++) { // :132-133
    int2 r = scratch[i];
    submit_or_execute(b, w, i < nrepl_buy ? 0 : 1, r.x, r.y, 0, true, true);
  }
  if (b.lane == 0) { // :134-135 (Exchange.orderbook_price_range, Exchange.py:160-170)
    if (w.nlv0 && b.lvp(0)[0] < h->min_buy) h->min_buy = b.lvp(0)[0];
    if (w.nlv1 && b.lvp(1)[0] > h->max_sell) h->max_sell = b.lvp(1)[0];
  }
  __syncwarp();
}

// cold wrapper: a real function call keeps the second copy of the book routines out of the kernel's hot code
static __device__ __noinline__ WarpState update_outer_levels(const Book b, WarpState w, const lobsim_cfg_t* c, const int32_t* row, int2* scratch) {
  update_outer_levels_impl(b, w, *c, row, scratch);
  return w;
}

// ---- OrderbookSimulator.reset_episode, OrderbookSimulator.py:55-68,156-188 + Exchange.py:172-178 ---------------
__device__ __forceinline__ void init_book_from_snapshot(const Book& b, WarpState& w, const lobsim_cfg_t& c, const lobsim_stream_t& st, int stream_id, int start_step) {
  BookHdr* h = b.hdr();
  const int L = c.n_levels;
  w.nlv0 = w.nlv1 = w.nord0 = w.nord1 = w.nag0 = w.nag1 = 0;
  w.err = 0; w.dead = 0;
  reset_flow(w);
  long long rel_us = (long long)start_step * c.step_us;
  long long sec = rel_us / 1000000;
  bool ok = start_step >= 0 && rel_us % 1000000 == 0 && sec <= (long long)st.n_seconds && st.snap_valid[sec] != 0;
  if (!ok) { w.err |= LOBSIM_ERR_NO_SNAPSHOT; w.dead = 1; }
  else {
    const int32_t* row = st.snapshots + (size_t)sec * 2 * L * 2;
    for (int side = 0; side < 2; side++) {
      int nvalid = 0;
      for (int base = 0; base < L; base += 32) nvalid += __popc(__ballot_sync(FULL_MASK, base + b.lane < L && __ldg(&row[(side * L + base + b.lane) * 2]) != LOBSIM_NO_PRICE));
      if (nvalid > b.L.NL || nvalid > b.L.NO) { w.err |= LOBSIM_ERR_LEVEL_OVERFLOW; w.dead = 1; nvalid = 0; }
      int seen = 0;
      for (int base = 0; base < L; base += 32) {
        int lvl = base + b.lane;
        int price = lvl < L ? __ldg(&row[(side * L + lvl) * 2]) : LOBSIM_NO_PRICE;
        int vol = lvl < L ? __ldg(&row[(side * L + lvl) * 2 + 1]) : 0;
        unsigned m = __ballot_sync(FULL_MASK, price != LOBSIM_NO_PRICE);
        if (price != LOBSIM_NO_PRICE && nvalid) {
          int k = seen + __popc(m & ((1u << b.lane) - 1)); // rank from the best
          int j = nvalid - 1 - k;                          // worst -> best storage
          b.lvp(side)[j] = price;
          b.lvend(side)[j] = (uint16_t)(j + 1);
          b.ord(side)[j] = make_uint2((unsigned)vol, LOBSIM_REF_AGGREGATE);
        }
        seen += __popc(m);
      }
      SET_NLV(w, side, nvalid);
      SET_NORD(w, side, nvalid);
    }
  }
  __syncwarp();
  if (b.lane == 0) {
    h->now_step = start_step;
    h->stream_id = stream_id;
    // _reset_initial_price_ranges :185-188
    int bb = w.nlv0 ? b.lvp(0)[w.nlv0 - 1] : 0, wb = w.nlv0 ? b.lvp(0)[0] : 0;
    int bs = w.nlv1 ? b.lvp(1)[w.nlv1 - 1] : 0, ws = w.nlv1 ? b.lvp(1)[0] : 0;
    h->min_buy = wb; h->max_sell = ws;
    h->init_buy_range = bb - wb; h->init_sell_range = ws - bs;
  }
  __syncwarp();
}

static __device__ __noinline__ WarpState init_book_cold(const Book b, WarpState w, const lobsim_cfg_t* c, const lobsim_stream_t* st, int stream_id, int start_step) {
  init_book_from_snapshot(b, w, *c, *st, stream_id, start_step);
  return w;
}

// ---- BetaOrderDistributor, rl4mm/gym/action_interpretation/OrderDistributors.py:23-56 ----------------------------
// lane k < Q returns the lot size of quote level k.  The sum follows numpy's pairwise summation order.
// log_x / log1m_x: ln(x_k) and ln(1 - x_k) = log1p(-x_k) of this lane's level midpoint x_k = (k + 0.5) / Q -- constants of the
// configuration, tabulated once by lobsim_create (the reference evaluates the Beta pdf at the same fixed midpoints every step,
// OrderDistributors.py:37); what is left per step is one exp per level.
static __device__ __noinline__ int beta_ladder_lane(double a, double bpar, int Q, int active_volume, int lane, double log_x, double log1m_x) {
  double A = -INFINITY;
  if (lane < Q) {
    double lx = (a - 1.0) == 0.0 ? 0.0 : (a - 1.0) * log_x;
    double l1 = (bpar - 1.0) == 0.0 ? 0.0 : (bpar - 1.0) * log1m_x;
    A = lx + l1;
  }
  double amax = A;
  for (int d = 16; d; d >>= 1) amax = fmax(amax, __shfl_xor_sync(FULL_MASK, amax, d));
  double e = lane < Q ? exp(A - amax) : 0.0;
  double s;
  if (Q >= 8) {
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = __shfl_sync(FULL_MASK, e, j);
    int i = 8;
    for (; i + 8 <= Q; i += 8) {
#pragma unroll
      for (int j = 0; j < 8; j++) r[j] += __shfl_sync(FULL_MASK, e, i + j);
    }
    s = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < Q; i++) s += __shfl_sync(FULL_MASK, e, i);
  } else {
    s = 0.0;
    for (int i = 0; i < Q; i++) s += __shfl_sync(FULL_MASK, e, i);
  }
  const double lots = rint(e / s * (double)active_volume);
  if (lane >= Q) return 0;
  return isfinite(lots) ? (int)lots : INT32_MIN;   // np.round(nan).astype(int): the reference then raises (agent_prepare)
}

// ---- HistoricalOrderbookEnvironment.convert_action_to_orders (HOE.py:206-258) as a GENERATOR -----------------------
// agent_prepare() computes the desired ladders and the per-level volume differences (one quote level per lane);
// agent_next() then yields the agent's orders one at a time, in the reference's order -- per side: ladder level
// k = 0..Q-1 (one limit order, or cancellations from the back of the agent's queue at that price, :231-249), then
// the off-ladder ("wide") orders cancelled in full (:250-257); finally the inventory-clearing market order
// (:213-215,260-266).  The kernel feeds them through the same process_order call site as the historical messages
// (agent orders first: OrderbookSimulator.py:76-77).  Cancellations are resolved against the agent table when
// they are yielded; this equals the reference's up-front list because orders yielded earlier in the same batch never
// touch the agent's orders at other prices of the same side.
struct AgentGen {
  int side, k, need, wide_i;   // cursor: side 0/1 (2 = market order stage, 3 = done)
  int diff0, diff1, price0, price1; // this lane's quote level
  int Q, clearing, clear_vol, clear_side;
  uint32_t pending_id;         // last wide cancel yielded (forces progress if it could not be applied)
  uint32_t err_out; int dead_out; // error bits raised while preparing
};

// Cold (noinline, everything by value): the fp64 ladder math must not inflate the register budget of the hot loop.
// beta_tab: [2][32] doubles (ln x_k, ln(1 - x_k)) in global memory; vol_scratch: per-warp int[64] in shared memory.
// best_buy / best_sell: the best prices of the central book (INT32_MIN / INT32_MAX: that side is empty) -- passed in, because the
// caller's book may be in the flat form (book_flat.cuh), which has no level arrays to read them from.
static __device__ __noinline__ AgentGen agent_prepare(const Book b, int best_buy, int best_sell, int nag0, int nag1, long long inventory, const EnvConst* ecp,
                                               double a0, double a1, double a2, double a3, double a4, const double* __restrict__ beta_tab, int* vol_scratch) {
  const EnvConst& ec = *ecp;
  const lobsim_cfg_t& c = ec.cfg;
  const double action[5] = {a0, a1, a2, a3, a4};
  AgentGen g;
  g.side = 3; g.err_out = 0; g.dead_out = 0;
  g.k = g.need = g.wide_i = g.diff0 = g.diff1 = g.price0 = g.price1 = g.Q = g.clearing = g.clear_vol = g.clear_side = 0; g.pending_id = 0;
  const int Q = c.max_quote_level - c.min_quote_level;
  const double EPS = 0.000001;
  double ab, bbp, as, bsp;
  if (c.concentration >= 0) {
    ab = action[0] + EPS; bbp = c.concentration - ab + EPS; as = action[1] + EPS; bsp = c.concentration - as + EPS;
  } else { ab = action[0] + EPS; bbp = action[1] + EPS; as = action[2] + EPS; bsp = action[3] + EPS; }
  const double log_x = __ldg(&beta_tab[b.lane]), log1m_x = __ldg(&beta_tab[32 + b.lane]);
  int desired0 = beta_ladder_lane(ab, bbp, Q, c.active_volume, b.lane, log_x, log1m_x);
  int desired1 = beta_ladder_lane(as, bsp, Q, c.active_volume, b.lane, log_x, log1m_x);
  long long absinv = inventory < 0 ? -inventory : inventory;
  const bool clearing = c.market_order_clearing && (double)absinv > pick5(action, ec.action_dim - 1);
  if (clearing) desired0 = desired1 = 0;
  if (__any_sync(FULL_MASK, desired0 == INT32_MIN || desired1 == INT32_MIN)) { g.err_out = LOBSIM_ERR_BAD_ACTION; g.dead_out = 1; return g; }
  if (best_buy == INT32_MIN || best_sell == INT32_MAX) { g.err_out = LOBSIM_ERR_EMPTY_BOOK; g.dead_out = 1; return g; }
  int bb = best_buy, bs = best_sell;
  const int tick = c.tick_size;
  if (c.enter_spread) { // _get_best_prices :298-309
    double mid = (double)(bs + bb) / 2.0;
    bb = (int)(floor(mid / (double)tick) * (double)tick);
    bs = (int)(ceil(mid / (double)tick) * (double)tick);
  }
  g.price0 = bb - (c.min_quote_level + b.lane) * tick; // ladder price of this lane's quote level
  g.price1 = bs + (c.min_quote_level + b.lane) * tick;
  { // _get_current_internal_order_volumes :291-296 -- one agent order per lane: its ladder index k = distance from the ladder's
    // first price in ticks; the resting volume per ladder level is accumulated with shared-memory atomics (integers: order-free)
    __syncwarp();
    vol_scratch[b.lane] = 0; vol_scratch[32 + b.lane] = 0;
    __syncwarp();
    const int base0 = bb - c.min_quote_level * tick, base1 = bs + c.min_quote_level * tick;
    for (int i = b.lane; i < nag0; i += 32) {
      const int d = base0 - b.aprice(0)[i];
      if (d >= 0) { const int q = d / tick; if (q * tick == d && q < Q) atomicAdd(&vol_scratch[q], b.avol(0)[i]); }
    }
    for (int i = b.lane; i < nag1; i += 32) {
      const int d = b.aprice(1)[i] - base1;
      if (d >= 0) { const int q = d / tick; if (q * tick == d && q < Q) atomicAdd(&vol_scratch[32 + q], b.avol(1)[i]); }
    }
    __syncwarp();
    if (b.lane < Q) { g.diff0 = desired0 - vol_scratch[b.lane]; g.diff1 = desired1 - vol_scratch[32 + b.lane]; }
    __syncwarp();
  }
  g.side = 0; g.Q = Q;
  g.clearing = clearing;
  g.clear_vol = clearing ? (int)rint((double)absinv * c.market_order_fraction_of_inventory) : 0;
  g.clear_side = inventory < 0 ? 0 : 1;
  return g;
}

// yields the next agent order; false when the batch is exhausted
__device__ __forceinline__ bool agent_next(const Book& b, WarpState& w, AgentGen& g, int& type, int& side, int& price, int& vol, uint32_t& ref) {
  for (;;) {
    if (w.dead || g.side >= 3) return false;
    if (g.side == 2) { // _get_inventory_clearing_market_order :260-266
      g.side = 3;
      if (!g.clearing) return false;
      if (g.clear_vol <= 0) { w.err |= LOBSIM_ERR_BAD_VOLUME; return false; } // assert volume > 0, Exchange.py:59-60
      type = LOBSIM_MSG_MARKET; side = g.clear_side; price = 0; vol = g.clear_vol; ref = 0;
      return true;
    }
    const int s = g.side;
    const int myprice = s ? g.price1 : g.price0;
    if (g.k < g.Q) {
      const int p = __shfl_sync(FULL_MASK, myprice, g.k);
      if (g.need == 0) {
        const int d = __shfl_sync(FULL_MASK, s ? g.diff1 : g.diff0, g.k);
        if (d > 0) { type = LOBSIM_MSG_LIMIT; side = s; price = p; vol = d; ref = 0; g.k++; return true; }
        if (d == 0) { g.k++; continue; }
        g.need = -d;
      }
      // cancel from the back of the agent's queue at this price, :239-249
      const int nag = NAG(w, s);
      int hit = -1;
      for (int base = (nag - 1) & ~31; base >= 0; base -= 32) {
        const int i = base + b.lane;
        const unsigned m = __ballot_sync(FULL_MASK, i < nag && b.aprice(s)[i] == p);
        if (m) { hit = base + 31 - __clz(m); break; }
      }
      if (hit < 0) { g.need = 0; g.k++; continue; }
      const int av = b.avol(s)[hit];
      const uint32_t id = b.aid(s)[hit];
      const int v = av < g.need ? av : g.need;
      g.need -= v;
      if (g.need == 0) g.k++;
      type = LOBSIM_MSG_CANCEL; side = s; price = p; vol = v; ref = LOBSIM_REF_AGENT | id;
      return true;
    }
    // agent orders off the ladder are cancelled in full, :250-257
    if (g.wide_i >= NAG(w, s)) { g.side = s + 1; g.k = 0; g.need = 0; g.wide_i = 0; g.pending_id = 0; continue; }
    const int ap = b.aprice(s)[g.wide_i], av = b.avol(s)[g.wide_i];
    const uint32_t id = b.aid(s)[g.wide_i];
    __syncwarp();
    if (id == g.pending_id) { agent_remove_at(b, w, s, g.wide_i); g.pending_id = 0; continue; } // keep books consistent
    const bool on_ladder = __ballot_sync(FULL_MASK, b.lane < g.Q && myprice == ap) != 0;
    if (on_ladder) { g.wide_i++; continue; }
    g.pending_id = id;
    type = LOBSIM_MSG_CANCEL; side = s; price = ap; vol = av; ref = LOBSIM_REF_AGENT | id;
    return true;
  }
}

// ---- agents, rl4mm/agents/baseline_agents.py -----------------------------------------------------------------------
__device__ __forceinline__ double clamp_to_unit(double x) { const double eps = 0.00001; return fmax(fmin(x, 1 - eps), -1 + eps); }
// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11): counter c[4], key (k0, k1)
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll 1
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
// RandomAgent (baseline_agents.py:9-18): action_space.sample() for the env's Box(0, high) -- uniform in [0, high_i) per
// dimension, 53 random bits each, from the stream keyed by (seed, env, grid step)
__device__ __forceinline__ void random_action(const lobsim_agent_t& ag, int env, int now_step, double* a) {
#pragma unroll 1
  for (int blk = 0; blk < 3; blk++) {
    uint32_t c[4] = {(uint32_t)now_step, (uint32_t)env, (uint32_t)blk, 0u};
    philox4x32_10(c, (uint32_t)ag.reserved, 0x4C4F4253u);
    const double u0 = (double)((((unsigned long long)c[0] << 32) | c[1]) >> 11) * (1.0 / 9007199254740992.0);
    const double u1 = (double)((((unsigned long long)c[2] << 32) | c[3]) >> 11) * (1.0 / 9007199254740992.0);
    a[2 * blk] = ag.fixed_action[2 * blk] * u0;
    if (2 * blk + 1 < 5) a[2 * blk + 1] = ag.fixed_action[2 * blk + 1] * u1;
  }
}
__device__ __forceinline__ void agent_action(const lobsim_agent_t& ag, double inventory_obs, double* a, int env, int now_step) {
  if (ag.kind == LOBSIM_AGENT_FIXED) {
#pragma unroll
    for (int i = 0; i < 5; i++) a[i] = ag.fixed_action[i];
  } else if (ag.kind == LOBSIM_AGENT_RANDOM) {
    random_action(ag, env, now_step, a);
  } else { // Teradactyl.get_action :76-87
    double denom = ag.max_inventory > 0 ? ag.max_inventory : 100.0;
    double wd = ag.default_omega, ob, oa;
    double cu = clamp_to_unit(inventory_obs / denom);
    if (inventory_obs >= 0) {
      ob = wd * (1 + (1 / wd - 1) * pow(cu, ag.exponent));
      oa = wd * (1 - pow(cu, ag.exponent));
    } else {
      ob = wd * (1 - pow(fabs(cu), ag.exponent));
      oa = wd * (1 + (1 / wd - 1) * pow(fabs(cu), ag.exponent));
    }
    double kappa = (ag.max_kappa - ag.default_kappa) * pow(fabs(inventory_obs / ag.max_inventory), ag.exponent) + ag.default_kappa;
    a[0] = (ob * (kappa - 2)) + 1; a[1] = (1 - ob) * (kappa - 2) + 1;
    a[2] = (oa * (kappa - 2)) + 1; a[3] = (1 - oa) * (kappa - 2) + 1;
    a[4] = ag.max_inventory * 2;
  }
}

// ---- rewards, rl4mm/rewards/RewardFunctions.py:97-118 ----------------------------------------------------------------
__device__ __forceinline__ double reward_calc(const lobsim_reward_t& r, double cash0, long long inv0, double p0, double cash1, long long inv1, double p1) {
  double cur = cash0 + (double)inv0 * p0;
  double nxt = cash1 + (double)inv1 * p1;
  double pnl = nxt - cur;
  if (r.kind == LOBSIM_REWARD_PNL) return pnl;
  double delta = p1 - p0;
  double term = r.inventory_aversion * (double)inv1 * delta;
  if (r.asymmetric) term = term > 0.0 ? term : 0.0;
  return pnl - term;
}

// ---- features, rl4mm/features/Features.py : one feature per lane ----------------------------------------------------
struct StepView { // uniform inputs of the feature updates
  int have_tops; int bb, bs, bv, sv;
  double price; long long inventory; long long now_us;
  int us_in_min;   // now_us % 60 s (32-bit: the update-frequency gate of every feature, Features.py:102-105)
  int n_ext0, n_ext1, vol_ext0, vol_ext1, n_int0, n_int1, vol_int0, vol_int1;
};

// Feature._update of the concrete classes; `ring` is this (env, feature)'s circular buffer in global memory
__device__ __forceinline__ void feature_update_raw(const lobsim_feature_t& fc, FeatState& f, double* ring, const StepView& v, long long aux) {
  const int k = fc.lookback;
  switch (fc.kind) {
    case LOBSIM_FEAT_SPREAD: f.cur = v.have_tops ? (double)(v.bs - v.bb) : NAN; break;
    case LOBSIM_FEAT_BOOK_IMBALANCE: f.cur = v.have_tops ? (double)(v.bv - v.sv) / (double)(v.bv + v.sv) : NAN; break;
    case LOBSIM_FEAT_PRICE: f.cur = v.price; break;
    case LOBSIM_FEAT_INVENTORY: f.cur = (double)v.inventory; break;
    case LOBSIM_FEAT_EPISODE_PROPORTION: f.cur += fc.dparam; break;
    case LOBSIM_FEAT_TIME_OF_DAY: {
      const long long min_time = 10LL * 3600 * 1000000;
      const long long bucket = aux;   // (15:30 - 10:00) / n_buckets, rounded like timedelta division (host: time_of_day_bucket_us)
      long long d = v.now_us - min_time;
      long long q = d >= 0 ? d / bucket : -((-d + bucket - 1) / bucket);
      f.cur = (double)(q > 0 ? q : 0);
      break;
    }
    case LOBSIM_FEAT_PRICE_MOVE:
    case LOBSIM_FEAT_PRICE_RANGE: { // deque(maxlen=k+1).appendleft(price)
      const int cap = k + 1;
      ring[f.head] = v.price;
      f.head = f.head + 1 == cap ? 0 : f.head + 1;
      if (f.len < cap) f.len++;
      if (fc.kind == LOBSIM_FEAT_PRICE_MOVE) {
        double oldest = f.len < cap ? ring[0] : ring[f.head];
        f.cur = v.price - oldest;
      } else {
        double mx = v.price, mn = v.price;
        for (int i = 0; i < f.len; i++) { double x = ring[i]; mx = fmax(mx, x); mn = fmin(mn, x); }
        f.cur = mx - mn;
      }
      break;
    }
    case LOBSIM_FEAT_VOLATILITY: {
      const int cap = k + 1;
      if (f.len < k) { ring[f.len++] = v.price; f.head = f.len == cap ? 0 : f.len; f.cur = 0.0; }
      else if (f.len == k) {
        ring[f.len++] = v.price; f.head = 0;
        double s = 0.0, first = ring[0];
        for (int i = 0; i < k; i++) { double r = (ring[i + 1] - ring[i]) / first; s += r * r; }
        f.cur = s / (double)k;
      } else {
        int h = f.head, h1 = h + 1 == cap ? 0 : h + 1, hn = h == 0 ? cap - 1 : h - 1;
        double oldest = ring[h], second = ring[h1], newest = ring[hn];
        double oldest_ret = (second - oldest) / oldest;
        double new_ret = (v.price - newest) / newest;
        ring[h] = v.price; f.head = h1;
        double ss = f.cur * (double)k - oldest_ret * oldest_ret + new_ret * new_ret;
        f.cur = ss / (double)k;
      }
      break;
    }
    case LOBSIM_FEAT_TRADE_DIR_IMBALANCE:
    case LOBSIM_FEAT_TRADE_VOL_IMBALANCE: {
      int nb, ns;
      if (fc.kind == LOBSIM_FEAT_TRADE_DIR_IMBALANCE) { nb = v.n_ext0; ns = v.n_ext1; if (fc.iparam) { nb += v.n_int0; ns += v.n_int1; } }
      else { nb = v.vol_ext0; ns = v.vol_ext1; if (fc.iparam) { nb += v.vol_int0; ns += v.vol_int1; } }
      int2* pr = reinterpret_cast<int2*>(ring);
      int len = f.len & ~FEAT_SUMS_VALID;
      if (len < k) {
        pr[len] = make_int2(nb, ns);
        f.len = (f.len & FEAT_SUMS_VALID) | (len + 1);
        f.head = len + 1 == k ? 0 : len + 1;
        f.cur = 0.0;
      } else {
        int h = f.head;
        int2 old = pr[h];
        pr[h] = make_int2(nb, ns);
        f.head = h + 1 == k ? 0 : h + 1;
        if (f.total == 0) {
          if (f.len & FEAT_SUMS_VALID) { f.total = (long long)nb + ns; f.diff = (long long)nb - ns; } // window was all zero
          else {
            long long sb = 0, ss = 0;
            for (int i = 0; i < k; i++) { int2 e = pr[i]; sb += e.x; ss += e.y; }
            f.total = sb + ss; f.diff = sb - ss; f.len |= FEAT_SUMS_VALID;
          }
        } else {
          f.total -= (long long)old.x + old.y; f.total += (long long)nb + ns;
          f.diff -= (long long)old.x - old.y; f.diff += (long long)nb - ns;
        }
        f.cur = f.total != 0 ? (double)f.diff / (double)f.total : 0.5;
      }
      break;
    }
    case LOBSIM_FEAT_AMIHUD_LAMBDA: { // Features.py:285-324; ring[0..kk] prices (oldest first), ring[kk+1..2kk] dollar volumes
      const int sf = fc.iparam, kk = fc.lookback / sf - 1;
      int plen = f.len & 0xffff, until = (f.len >> 16) & 0x3fff, dvlen = f.head;
      long long* dv = reinterpret_cast<long long*>(ring + kk + 1);
      if (until > 0) {
        until -= 1;
        f.diff = __double_as_longlong(__longlong_as_double(f.diff) + v.price);   // partial_price_sum
        f.total += (long long)v.vol_ext0 + v.vol_ext1;                            // partial_dollar_volume
      } else {
        until = sf - 1;
        const double new_price = __longlong_as_double(f.diff) / (double)sf;
        const long long new_dv = f.total;
        if (plen <= kk) { // prices deque not full yet: both deques append (the full dollar-volume deque drops its oldest)
          ring[plen] = new_price;
          if (dvlen < kk) dv[dvlen++] = new_dv; else { for (int i = 0; i + 1 < kk; i++) dv[i] = dv[i + 1]; dv[kk - 1] = new_dv; }
          plen += 1;
          if (plen <= kk) f.cur = 0.0;
          else {
            double sacc = 0.0; const double first = ring[0];
            for (int i = 0; i < kk; i++) {
              const double r = (ring[i + 1] - ring[i]) / first;
              const long long d = dv[i];
              if (d > 0) sacc += fabs(r) / (double)d;
            }
            f.cur = sacc / (double)kk;
          }
        } else {
          const double oldest = ring[0];
          for (int i = 0; i < kk; i++) ring[i] = ring[i + 1];
          const double oldest_ret = (ring[0] - oldest) / oldest;
          const long long oldest_dv = dv[0];
          for (int i = 0; i + 1 < kk; i++) dv[i] = dv[i + 1];
          const double last = ring[kk - 1];
          const double new_ret = (new_price - last) / last;
          ring[kk] = new_price; dv[kk - 1] = new_dv;
          const double new_ratio = new_dv > 0 ? fabs(new_ret) / (double)new_dv : 0.0;
          const double old_ratio = oldest_dv > 0 ? fabs(oldest_ret) / (double)oldest_dv : 0.0;
          const double sum_of_ratio = f.cur * (double)kk + new_ratio - old_ratio;
          f.cur = sum_of_ratio / (double)kk;
        }
        f.diff = __double_as_longlong(0.0); f.total = 0;
      }
      f.len = plen | (until << 16); f.head = dvlen;
      break;
    }
    default: break;
  }
}

// ---- Feature.normalise, Features.py:67-74: scipy.stats.zscore(history)[-1] over a deque(maxlen) of the clamped values ----
// scipy (1.18.1, the version the goldens were generated with; zmap in scipy/stats/_stats_py.py):
//   mean = np.mean(a); std = np.mean((a - mean) * (a - mean)) ** 0.5; z = (a - mean) / std; z = NaN where std <= |eps * mean|
// with numpy's pairwise summation.  The reference recomputes this from scratch every step (O(history)).  Here:
//   * normal regime (std > 1e-8 |mean|, numpy's own rounding error < 1e-7 relative): shifted running sums, O(1);
//   * constant window: numpy's pairwise sum of n equal values is replayed without touching memory (the mean may be off
//     by an ulp or more, which decides between NaN and +-1);
//   * noise-dominated window (|std| <= 1e-8 |mean|, e.g. [p + 1e-06, p, p, ...] for a price p ~ 4e6): the numpy arithmetic
//     is replayed over the ring, O(history) like the reference, because there the result IS the rounding error.
// mode 0: x_i, mode 1: (x_i - mean)^2, mode 2: the constant cval (no memory access)
// Frames of the explicit post-order stack below: one per level of numpy's split tree (leaf included).  A child holds at most
// n/2 + 8 entries, so the tree of n <= LOBSIM_MAX_NORM_LEN (10 M) entries is 18 levels deep (tests/test_zscore_cpu.py).
#define NP_PAIRWISE_STACK 18
static __device__ __noinline__ double np_pairwise_sum_ring(const double* hist, int maxlen, int start, int n, int mode, double mean, double cval) {
  auto el = [&](int i) -> double {
    if (mode == 2) return cval;
    int k = start + i; if (k >= maxlen) k -= maxlen;
    const double x = hist[k];
    if (mode == 1) { const double d = x - mean; return d * d; }
    return x;
  };
  auto leaf = [&](int off, int m) -> double {        // numpy pairwise_sum_DOUBLE for n <= PW_BLOCKSIZE (128)
    if (m < 8) { double r = -0.0; for (int i = 0; i < m; i++) r += el(off + i); return r; }
    const int body = m - (m % 8);
    double res;
    if (mode == 2) {                                  // eight identical accumulators
      double r = cval;
      for (int i = 8; i < body; i += 8) r += cval;
      const double r2 = r + r, r4 = r2 + r2;
      res = r4 + r4;
    } else {
      double r0 = el(off), r1 = el(off + 1), r2 = el(off + 2), r3 = el(off + 3), r4 = el(off + 4), r5 = el(off + 5), r6 = el(off + 6), r7 = el(off + 7);
      for (int i = 8; i < body; i += 8) {
        r0 += el(off + i); r1 += el(off + i + 1); r2 += el(off + i + 2); r3 += el(off + i + 3);
        r4 += el(off + i + 4); r5 += el(off + i + 5); r6 += el(off + i + 6); r7 += el(off + i + 7);
      }
      res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
    }
    for (int i = body; i < m; i++) res += el(off + i);
    return res;
  };
  if (n <= 128) return leaf(0, n);
  int f_off[NP_PAIRWISE_STACK], f_n[NP_PAIRWISE_STACK], f_stage[NP_PAIRWISE_STACK]; double f_left[NP_PAIRWISE_STACK];
  int sp = 1; double ret = 0.0;
  f_off[0] = 0; f_n[0] = n; f_stage[0] = 0; f_left[0] = 0.0;
  while (sp > 0) {
    const int t = sp - 1;
    if (f_n[t] <= 128) { ret = leaf(f_off[t], f_n[t]); sp--; continue; }
    int n2 = f_n[t] / 2; n2 -= n2 % 8;
    if (f_stage[t] == 0) { f_stage[t] = 1; f_off[sp] = f_off[t]; f_n[sp] = n2; f_stage[sp] = 0; sp++; }
    else if (f_stage[t] == 1) { f_left[t] = ret; f_stage[t] = 2; f_off[sp] = f_off[t] + n2; f_n[sp] = f_n[t] - n2; f_stage[sp] = 0; sp++; }
    else { ret = f_left[t] + ret; sp--; }
  }
  return ret;
}

// scipy's zscore of the last element, replayed exactly; `start` = ring index of the oldest of the n window entries
static __device__ __noinline__ double zscore_exact(const double* hist, int maxlen, int start, int n, double value, int constant) {
  const int m0 = constant ? 2 : 0;
  const double mean = np_pairwise_sum_ring(hist, maxlen, start, n, m0, 0.0, value) / (double)n;
  double var;
  if (constant) { const double d = value - mean; var = np_pairwise_sum_ring(hist, maxlen, start, n, 2, 0.0, d * d) / (double)n; }
  else var = np_pairwise_sum_ring(hist, maxlen, start, n, 1, mean, 0.0) / (double)n;
  const double sd = sqrt(var);
  if (sd <= fabs(2.220446049250313e-16 * mean)) return NAN;   // zmap: "zero = std <= abs(eps * mn)" -> NaN
  return (value - mean) / sd;
}

// exact shifted sums of the window around a new centre (sheds accumulated rounding and cancellation)
static __device__ __noinline__ void zscore_recenter(NormState& f, const double* hist, int maxlen, int start, int n, double centre) {
  double s1 = 0.0, s2 = 0.0;
  for (int i = 0; i < n; i++) {
    int k = start + i; if (k >= maxlen) k -= maxlen;
    const double d = hist[k] - centre;
    s1 += d; s2 += d * d;
  }
  f.nK = centre; f.nS1 = s1; f.nS2 = s2; f.nS2max = s2;
}

// Cold and out of line, working on the NormState in global memory: nothing of the caller stays live across the (rare) calls
// into the exact paths, so the per-step feature code keeps its registers.  Returns the normalised current value.
static __device__ __noinline__ double feature_normalise(NormState* fg, double* hist, int maxlen, double value) {
  NormState f = *fg;
  double cur;
  int n = f.nlen;
  int head = f.nhead;
  double last = NAN;
  if (n == 0) { // "to prevent a NaN value from being returned if the queue is empty" :68-72
    const double x0 = value + 1e-06;
    f.nK = x0; f.nS1 = 0.0; f.nS2 = 0.0; f.nS2max = 0.0; f.nrun = 1;
    hist[0] = x0; n = 1; head = maxlen > 1 ? 1 : 0; last = x0;
  } else last = hist[head == 0 ? maxlen - 1 : head - 1];
  if (n == maxlen) { const double old = hist[head] - f.nK; f.nS1 -= old; f.nS2 -= old * old; n -= 1; }
  hist[head] = value;
  head = head + 1 == maxlen ? 0 : head + 1;
  n += 1;
  f.nrun = value == last ? (f.nrun < 0x7fffffff ? f.nrun + 1 : f.nrun) : 1;
  f.nlen = n; f.nhead = head;
  int start = head - n; if (start < 0) start += maxlen;      // ring index of the oldest entry
  if (f.nrun >= n) {                                          // the whole window holds one value
    f.nK = value; f.nS1 = 0.0; f.nS2 = 0.0; f.nS2max = 0.0;   // exact sums around the value itself
    cur = zscore_exact(hist, maxlen, start, n, value, 1);
    *fg = f;
    return cur;
  }
  double d = value - f.nK;
  f.nS1 += d; f.nS2 += d * d;
  f.nS2max = fmax(f.nS2max, f.nS2);
  double m1 = f.nS1 / (double)n, msq = f.nS2 / (double)n;
  double var = msq - m1 * m1;
  // the running sums carry an absolute error ~ eps * nS2max per update, and it accumulates: recompute them exactly (around
  // the current mean) when nS2max exceeds 100 n * var -- a dominant entry (e.g. the 1e-06 offset of the first one) left the
  // window or dominates it, or the mean drifted far from the centre -- when a NaN got in, and every 512 updates (ring
  // positions 0, 512, ...: once per lap of a shorter ring).  This keeps the normal-regime z-score within 256 eps * kappa of
  // the exact one (tests/test_gpu_zscore.py); a bound of 1e6 n * var and one recentre per lap left windows of 1 000 to
  // 20 000 entries up to 400 eps * kappa off.
  if (!(var * (double)n > 1e-2 * f.nS2max) || (head & 511) == 0) {
    double centre = f.nK + m1;
    if (!isfinite(centre)) centre = isfinite(value) ? value : 0.0;
    zscore_recenter(f, hist, maxlen, start, n, centre);
    d = value - f.nK; m1 = f.nS1 / (double)n; msq = f.nS2 / (double)n; var = msq - m1 * m1;
  }
  const double sd = sqrt(var);
  if (!(sd > 1e-8 * fabs(f.nK + m1))) cur = zscore_exact(hist, maxlen, start, n, value, 0);   // noise-dominated (or NaN)
  else cur = (d - m1) / sd;
  *fg = f;
  return cur;
}

// Feature.reset/_reset, Features.py:92-96 (the normalisation history is cleared by features_step)
__device__ __forceinline__ void feature_reset(const lobsim_feature_t& fc, FeatState& f, double* ring, const StepView& v, long long aux) {
  f.len = 0; f.head = 0; f.total = 0; f.diff = 0;
  if (fc.kind == LOBSIM_FEAT_AMIHUD_LAMBDA) { f.len = (fc.iparam - 1) << 16; f.diff = __double_as_longlong(0.0); } // AmihudLambda.reset :278-283
  feature_update_raw(fc, f, ring, v, aux);
  if (fc.kind == LOBSIM_FEAT_EPISODE_PROPORTION) f.cur = 0.0;
}

// Feature.update, Features.py:80-86,102-105
// returns true when the (clamped) value still has to go through Feature.normalise (done by the caller, out of line)
__device__ __forceinline__ bool feature_update(const lobsim_feature_t& fc, FeatState& f, double* ring, const StepView& v, long long episode_start_us, long long aux) {
  long long first_usage = episode_start_us - (long long)fc.lookback * fc.update_us;
  if (v.now_us < first_usage) return false;
  if (v.us_in_min % (int)fc.update_us != 0) return false;   // (second * 1e6 + microsecond) % update_frequency, update_us <= 60 s
  feature_update_raw(fc, f, ring, v, aux);
  f.cur = fmax(fmin(f.cur, fc.max_value), fc.min_value);
  return fc.norm_len > 0;
}

// Cold per-step feature phase: lane f < F loads its feature state from HBM, resets (mode 1) or updates (mode 0) it,
// stores it back and returns Feature.current_value.  Keeping this out of line keeps the fp64 / 64-bit-division heavy
// code (and its registers) away from the order-processing loop.
// NORM == false instantiations contain no call into the z-score code: a callee subtree that is never executed still costs
// the calling kernel registers around the call and I-cache footprint (measured: 3.7 % of the env step).
// With normalisation the value a feature's recurrences continue from (Feature.current_value, e.g. Volatility) IS the
// normalised one (Features.py:80-86 overwrites current_value), so it is written back into the FeatState.
template <bool NORM>
static __device__ __noinline__ double features_step(const EnvConst* ecp, FeatState* fstate_env, NormState* nstate_env, double* rings_env, int lane, const StepView v, long long episode_start_us, int mode) {
  const EnvConst& ec = *ecp;
  double cur = 0.0;
  if (lane < ec.cfg.n_features) {
    const lobsim_feature_t fc = ec.cfg.features[lane];
    FeatState fs = fstate_env[lane];
    double* ring = rings_env + ec.ring_off[lane];
    bool norm = false;
    if (mode == 1) {
      feature_reset(fc, fs, ring, v, ec.feat_aux[lane]);
      if (NORM && fc.norm_len > 0) { NormState z; z.nK = z.nS1 = z.nS2 = z.nS2max = 0.0; z.nlen = z.nhead = z.nrun = z.pad = 0; nstate_env[lane] = z; } // history.clear()
    } else norm = feature_update(fc, fs, ring, v, episode_start_us, ec.feat_aux[lane]);
    if (NORM && norm) fs.cur = feature_normalise(&nstate_env[lane], rings_env + ec.hist_off[lane], fc.norm_len, fs.cur);
    fstate_env[lane] = fs;
    cur = fs.cur;
  }
  return cur;
}

// Agent.get_action for the fused rollout (cold)
static __device__ __noinline__ void agent_action_cold(const lobsim_agent_t* ag, double inventory_obs, double* out5_smem, int env, int now_step) {
  double a[5] = {0, 0, 0, 0, 0};
  agent_action(*ag, inventory_obs, a, env, now_step);
#pragma unroll
  for (int i = 0; i < 5; i++) out5_smem[i] = a[i];
}

// ---- agent_next for the straight-line path -----------------------------------------------------------------------------
// Same order sequence as agent_next (the reference's convert_action_to_orders, HOE.py:206-258), but the generator never walks
// over things that yield nothing: the ladder levels whose volume difference is non-zero are a bitmask (one __ffs per yielded
// order instead of a loop over all Q levels), and the agent's off-ladder ("wide") orders are found by ONE lane-parallel pass
// over the agent table when the ladder stage of a side ends (instead of one scalar iteration per resting agent order).
// The per-level differences live in the per-warp scratch (int[64]: buy levels, sell levels); the agent table counters in the
// shared-memory header.
struct AgentGenFast {
  int side, stage, need;        // cursor: side 0/1 (2 = market order stage, 3 = done); stage 0 = ladder, 1 = wide cancels
  unsigned todo0, todo1;        // ladder levels with a non-zero volume difference, per side
  unsigned wm0, wm1;            // wide stage of the current side: off-ladder entries of the agent table (original indices 0..63)
  int wide_removed, wide_pos;   // entries removed so far in this wide stage; table position of the cancel yielded last
  uint32_t pending_id;          // id of that cancel (0: none)
  int base0, base1;             // first ladder price per side: price of level k = base0 - k * tick / base1 + k * tick
  int clear_vol, clear_side;    // inventory-clearing market order (clear_vol < 0: none)
};

// AgentGen (agent_prepare: one quote level per lane) -> the compact form; diffs go to the per-warp scratch
__device__ __forceinline__ AgentGenFast agent_gen_fast_init(const AgentGen& g, int lane, int* diff_scratch) {
  AgentGenFast a;
  a.side = g.side; a.stage = 0; a.need = 0;
  a.todo0 = __ballot_sync(FULL_MASK, lane < g.Q && g.diff0 != 0);
  a.todo1 = __ballot_sync(FULL_MASK, lane < g.Q && g.diff1 != 0);
  a.wm0 = a.wm1 = 0; a.wide_removed = 0; a.wide_pos = 0; a.pending_id = 0;
  a.base0 = __shfl_sync(FULL_MASK, g.price0, 0); a.base1 = __shfl_sync(FULL_MASK, g.price1, 0);
  a.clear_vol = g.clearing ? g.clear_vol : -1; a.clear_side = g.clear_side;
  __syncwarp();
  diff_scratch[lane] = g.diff0; diff_scratch[32 + lane] = g.diff1;
  __syncwarp();
  return a;
}

template <class LT>
__device__ __forceinline__ bool agent_next_fast(const FastBook<LT>& fb, FastState& f, AgentGenFast& g, const int* diff_scratch, int Q, int tick,
                                                int& type, int& side, int& price, int& vol, uint32_t& ref) {
  BookHdr* h = reinterpret_cast<BookHdr*>(fb.blob);
  for (;;) {
    if (f.dead || g.side >= 3) return false;
    if (g.side == 2) { // _get_inventory_clearing_market_order :260-266
      g.side = 3;
      if (g.clear_vol < 0) return false;
      if (g.clear_vol == 0) { f.err |= LOBSIM_ERR_BAD_VOLUME; return false; }
      type = LOBSIM_MSG_MARKET; side = g.clear_side; price = 0; vol = g.clear_vol; ref = 0;
      return true;
    }
    const int s = g.side;
    const int32_t* ap = reinterpret_cast<const int32_t*>(fb.blob + LT::agent_off + s * LT::NA * 12);
    const int32_t* av = ap + LT::NA;
    const uint32_t* ai = reinterpret_cast<const uint32_t*>(ap + 2 * LT::NA);
    const int nag = h->nag[s];
    const int base = s ? g.base1 : g.base0;
    if (g.stage == 0) {
      const unsigned todo = s ? g.todo1 : g.todo0;
      if (todo == 0) {
        // ladder done: agent orders off the ladder are cancelled in full, :250-257.  One pass: entry i is on the ladder iff its
        // distance from the first ladder price is k * tick with 0 <= k < Q (orders placed during the ladder stage are).
        __syncwarp();
        bool off0 = false, off1 = false;
        if (fb.lane < nag) { const int d = s ? ap[fb.lane] - base : base - ap[fb.lane]; const int q = d / tick; off0 = !(d >= 0 && q * tick == d && q < Q); }
        if (fb.lane + 32 < nag) { const int d = s ? ap[fb.lane + 32] - base : base - ap[fb.lane + 32]; const int q = d / tick; off1 = !(d >= 0 && q * tick == d && q < Q); }
        g.wm0 = __ballot_sync(FULL_MASK, off0); g.wm1 = __ballot_sync(FULL_MASK, off1);
        g.stage = 1; g.wide_removed = 0; g.pending_id = 0;
        continue;
      }
      const int k = __ffs(todo) - 1;
      const int p = s ? base + k * tick : base - k * tick;
      if (g.need == 0) {
        const int d = diff_scratch[s * 32 + k];
        if (d > 0) {
          if (s) g.todo1 = todo & (todo - 1); else g.todo0 = todo & (todo - 1);
          type = LOBSIM_MSG_LIMIT; side = s; price = p; vol = d; ref = 0;
          return true;
        }
        g.need = -d;
      }
      // cancel from the back of the agent's queue at this price, :239-249 (NA <= 64)
      const unsigned m1 = __ballot_sync(FULL_MASK, fb.lane + 32 < nag && ap[fb.lane + 32] == p);
      const unsigned m0 = __ballot_sync(FULL_MASK, fb.lane < nag && ap[fb.lane] == p);
      if (!(m0 | m1)) { g.need = 0; if (s) g.todo1 = todo & (todo - 1); else g.todo0 = todo & (todo - 1); continue; }
      const int hit = m1 ? 63 - __clz(m1) : 31 - __clz(m0);
      const int a = av[hit];
      const uint32_t id = ai[hit];
      const int v = a < g.need ? a : g.need;
      g.need -= v;
      if (g.need == 0) { if (s) g.todo1 = todo & (todo - 1); else g.todo0 = todo & (todo - 1); }
      type = LOBSIM_MSG_CANCEL; side = s; price = p; vol = v; ref = LOBSIM_REF_AGENT | id;
      return true;
    }
    // ---- wide stage --------------------------------------------------------------------------------------------------------
    if (g.pending_id) {   // the cancel yielded last: if the book could not apply it, drop the entry here (keeps the books consistent)
      const bool still = g.wide_pos < nag && ai[g.wide_pos] == g.pending_id;
      __syncwarp();
      if (still) fast_agent_reduce(fb, s, g.pending_id, 0, true);
      g.pending_id = 0; g.wide_removed++;
      continue;
    }
    if (!(g.wm0 | g.wm1)) { g.side = s + 1; g.stage = 0; g.need = 0; continue; }
    int i;
    if (g.wm0) { i = __ffs(g.wm0) - 1; g.wm0 &= g.wm0 - 1; } else { i = 32 + __ffs(g.wm1) - 1; g.wm1 &= g.wm1 - 1; }
    const int pos = i - g.wide_removed;
    if (pos < 0 || pos >= nag) continue;   // cannot happen while every wide cancel removes exactly its own entry
    const int wp = ap[pos], wv = av[pos];
    const uint32_t id = ai[pos];
    g.pending_id = id; g.wide_pos = pos;
    type = LOBSIM_MSG_CANCEL; side = s; price = wp; vol = wv; ref = LOBSIM_REF_AGENT | id;
    return true;
  }
}

// ---- RollingSharpe.calculate, rl4mm/rewards/RewardFunctions.py:10-22,64-94 (cold; warp-collective) -------------------
// ring: maxw doubles (circular, logical order oldest -> newest), state[0] = n_filled, state[1] = head (next write).
// Returns the reward; *err_out gets LOBSIM_ERR_AUM_NONPOSITIVE when an AUM in the window is <= 0 (the reference raises).
struct SharpeOut { double reward; uint32_t err; };
// get_sharpe (RewardFunctions.py:10-22): np.mean and np.std(ddof=1) of the simple returns.  The returns are written to a scratch
// row (`tmp`) by all lanes and then summed by lane 0 in numpy's pairwise order (np_pairwise_sum_ring) -- mean / std of tiny
// returns amplifies any other summation order beyond the 1e-6 tolerance.
static __device__ __noinline__ SharpeOut rolling_sharpe_step(double* ring, int* state, int packed_windows, double new_aum, int lane, double* tmp) {
  const int maxw = packed_windows & 0xffff, minw = (packed_windows >> 16) & 0xffff;
  int n = state[0], head = state[1];
  __syncwarp();
  if (lane == 0) { ring[head] = new_aum; state[0] = n + 1 < maxw ? n + 1 : maxw; state[1] = head + 1 == maxw ? 0 : head + 1; }
  __syncwarp();
  n = n + 1 < maxw ? n + 1 : maxw; head = head + 1 == maxw ? 0 : head + 1;
  SharpeOut out; out.reward = 0.0; out.err = 0;
  if (n < minw) return out;
  const int first = n < maxw ? 0 : head;     // physical index of the oldest entry (the ring starts at 0 after create)
  const int m = n - 1;                       // number of returns
  int bad = 0;
  for (int i = lane; i < n; i += 32) { int k = first + i; if (k >= maxw) k -= maxw; if (ring[k] <= 0.0) bad = 1; }
  if (__any_sync(FULL_MASK, bad)) { out.reward = NAN; out.err = LOBSIM_ERR_AUM_NONPOSITIVE; return out; }
  for (int i = lane; i < m; i += 32) {
    int k0 = first + i; if (k0 >= maxw) k0 -= maxw;
    int k1 = k0 + 1 == maxw ? 0 : k0 + 1;
    tmp[i] = cr_exp(cr_log(ring[k1]) - cr_log(ring[k0])) - 1.0;   // correctly rounded: crmath.cuh
  }
  __syncwarp();
  double r = 0.0;
  if (lane == 0) {
    const double mean = np_pairwise_sum_ring(tmp, m, 0, m, 0, 0.0, 0.0) / (double)m;
    const double sd = sqrt(np_pairwise_sum_ring(tmp, m, 0, m, 1, mean, 0.0) / (double)(m - 1));
    r = mean / (sd + 2.2250738585072014e-308);
  }
  out.reward = __shfl_sync(FULL_MASK, r, 0);
  return out;
}
