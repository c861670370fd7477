// book.cuh -- the device limit order book: one warp per book, the whole book in shared memory.
//
// Data layout (DESIGN.md "Data layout").  A book is one contiguous blob (HBM <-> shared memory by TMA bulk copy):
//
//   BookHdr (128 B)
//   per side s in {buy, sell}  (side stride SS):
//     lvp  [NL] int32   level prices, sorted WORST -> BEST (the best level is lvp[nlv-1])
//     lvend[NL] uint16  cumulative end offset of the level's FIFO segment inside ord[]
//     ord  [NO] uint2   resting orders (x = volume, y = ref), level segments in the same worst -> best order and,
//                       inside a segment, FIFO order (segment start = queue head = highest time priority)
//   agent table per side (the reference's internal_orderbook): aprice/avol/aid [NA], ascending agent id
//
// This is the reference's `SortedDict[price -> deque[LimitOrder]]` (rl4mm/orderbook/models.py:64-69) flattened so
// that every operation is a handful of warp-wide loads, ballots and <=32-entry shifts:
//   * level lookup      = 32 prices per load + __ballot_sync            (Exchange.py:80-82, :202-205)
//   * order lookup      = 32 (volume, ref) pairs per load + ballot      (Exchange.py:196-217; the reference's
//                         ext-id dict + binary search by internal id finds exactly the entry whose ref matches)
//   * append at the best level costs no shift at all, a pop of the best head shifts only the best queue
// `ref` identifies the order: 0 = snapshot aggregate (internal_id -1), 1..2^31-1 = dense external id,
// 0x80000000|id = the agent's own order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lobsim.h"

#define FULL_MASK 0xffffffffu

struct __align__(16) BookHdr {
  int32_t cnt[2][2]; // cnt[side] = {number of levels, number of orders}
  int32_t nag[2];
  uint32_t next_agent_id;
  uint32_t err;
  int32_t now_step;
  int32_t episode_start_step;
  int32_t stream_id;
  int32_t dead;
  int32_t min_buy, max_sell, init_buy_range, init_sell_range;
  int64_t inventory;
  double cash;
  double price;
  int32_t has_reset;
  int32_t flow[8];   // per-step fill flow: n_ext[2], vol_ext[2], n_int[2], vol_int[2] (by recorded direction)
  int32_t n_fills;   // fills recorded during the current launch (tracked fast path)
};
static_assert(sizeof(BookHdr) == 128, "BookHdr must be 128 bytes");

struct Layout {
  int32_t NL, NO, NA;
  int32_t side_off;    // offset of side 0 block
  int32_t side_stride; // SS
  int32_t ord_off;     // offset of ord[] inside a side block
  int32_t lvend_off;   // offset of lvend[] inside a side block
  int32_t agent_off;   // offset of the agent tables
  int32_t blob_bytes;  // multiple of 16
};

__host__ __device__ inline Layout make_layout(int NL, int NO, int NA) {
  Layout l;
  l.NL = NL; l.NO = NO; l.NA = NA;
  l.side_off = (int)sizeof(BookHdr);
  l.lvend_off = NL * 4;
  l.ord_off = (NL * 4 + NL * 2 + 7) & ~7;
  l.side_stride = (l.ord_off + NO * 8 + 15) & ~15;
  l.agent_off = l.side_off + 2 * l.side_stride;
  l.blob_bytes = (l.agent_off + 2 * NA * 12 + 15) & ~15;
  return l;
}

// uniform per-warp register state (every lane holds the same values)
struct WarpState {
  int nlv0, nlv1, nord0, nord1, nag0, nag1;
  uint32_t next_agent_id, err;
  int dead;
  long long inventory;
  double cash;
  // flow of the current step: [recorded direction]
  int n_ext0, n_ext1, vol_ext0, vol_ext1, n_int0, n_int1, vol_int0, vol_int1;
  // optional fill log (global memory)
  lobsim_fill_t* fill_log;
  int fill_cap, n_fills;
};

struct Book {
  unsigned char* blob; // shared memory
  Layout L;
  int lane;

  __device__ __forceinline__ BookHdr* hdr() const { return reinterpret_cast<BookHdr*>(blob); }
  __device__ __forceinline__ int32_t* lvp(int s) const { return reinterpret_cast<int32_t*>(blob + L.side_off + s * L.side_stride); }
  __device__ __forceinline__ uint16_t* lvend(int s) const { return reinterpret_cast<uint16_t*>(blob + L.side_off + s * L.side_stride + L.lvend_off); }
  __device__ __forceinline__ uint2* ord(int s) const { return reinterpret_cast<uint2*>(blob + L.side_off + s * L.side_stride + L.ord_off); }
  __device__ __forceinline__ int32_t* aprice(int s) const { return reinterpret_cast<int32_t*>(blob + L.agent_off + s * L.NA * 12); }
  __device__ __forceinline__ int32_t* avol(int s) const { return aprice(s) + L.NA; }
  __device__ __forceinline__ uint32_t* aid(int s) const { return reinterpret_cast<uint32_t*>(aprice(s) + 2 * L.NA); }
};

__device__ __forceinline__ int key_of(int side, int price) { return side ? -price : price; }
// uniform two-way register select / update (no addresses taken: the state must stay in registers)
#define GET2(side, a0, a1) ((side) ? (a1) : (a0))
#define SET2(side, a0, a1, v) do { if (side) (a1) = (v); else (a0) = (v); } while (0)
#define NLV(w, s) GET2(s, (w).nlv0, (w).nlv1)
#define NORD(w, s) GET2(s, (w).nord0, (w).nord1)
#define NAG(w, s) GET2(s, (w).nag0, (w).nag1)
#define SET_NLV(w, s, v) SET2(s, (w).nlv0, (w).nlv1, v)
#define SET_NORD(w, s, v) SET2(s, (w).nord0, (w).nord1, v)
#define SET_NAG(w, s, v) SET2(s, (w).nag0, (w).nag1, v)

// ---- warp-wide shifts ----------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void shift_up1(T* a, int pos, int n, int lane) { // a[pos+1..n] = a[pos..n-1]
  for (int hi = n; hi > pos; hi -= 32) {
    int i = hi - 32 + lane;
    bool act = i >= pos;
    T v;
    if (act) v = a[i];
    __syncwarp();
    if (act) a[i + 1] = v;
    __syncwarp();
  }
}
template <typename T>
__device__ __forceinline__ void shift_down(T* a, int pos, int d, int n, int lane) { // drop a[pos..pos+d)
  for (int lo = pos + d; lo < n; lo += 32) {
    int i = lo + lane;
    bool act = i < n;
    T v;
    if (act) v = a[i];
    __syncwarp();
    if (act) a[i - d] = v;
    __syncwarp();
  }
}
__device__ __forceinline__ void bump_lvend(uint16_t* le, int j, int nlv, int delta, int lane) {
  for (int i = j + lane; i < nlv; i += 32) le[i] = (uint16_t)(le[i] + delta);
  __syncwarp();
}

// ---- level lookup: index of the level with `price`, or the insertion index when absent ------------------------
__device__ __forceinline__ int find_level(const Book& b, int side, int nlv, int price, bool& found) {
  const int32_t* p = b.lvp(side);
  int tkey = key_of(side, price);
  for (int base = 0;; base += 32) {
    int idx = nlv - 1 - base - b.lane;
    bool valid = idx >= 0;
    int k = valid ? key_of(side, p[idx]) : INT32_MIN;
    unsigned eq = __ballot_sync(FULL_MASK, valid && k == tkey);
    if (eq) { found = true; return nlv - 1 - base - (__ffs(eq) - 1); }
    unsigned gt = __ballot_sync(FULL_MASK, valid && k > tkey);
    int c = __popc(gt);
    if (c < 32) { found = false; return nlv - base - c; }
  }
}

__device__ __forceinline__ int level_start(const Book& b, int side, int j) { return j > 0 ? (int)b.lvend(side)[j - 1] : 0; }

// insert an empty level at index j (shifts better levels up)
__device__ __forceinline__ bool insert_level(const Book& b, WarpState& w, int side, int j, int price) {
  int nlv = NLV(w, side);
  if (nlv >= b.L.NL) { w.err |= LOBSIM_ERR_LEVEL_OVERFLOW; return false; }
  int32_t* p = b.lvp(side);
  uint16_t* le = b.lvend(side);
  int start = level_start(b, side, j);
  __syncwarp();
  shift_up1(p, j, nlv, b.lane);
  shift_up1(le, j, nlv, b.lane);
  if (b.lane == 0) { p[j] = price; le[j] = (uint16_t)start; }
  __syncwarp();
  SET_NLV(w, side, nlv + 1);
  return true;
}

// append an order to the FIFO of level j
__device__ __forceinline__ bool add_order(const Book& b, WarpState& w, int side, int j, int vol, uint32_t ref) {
  int n = NORD(w, side);
  if (n >= b.L.NO) { w.err |= LOBSIM_ERR_ORDER_OVERFLOW; return false; }
  uint16_t* le = b.lvend(side);
  uint2* o = b.ord(side);
  int pos = le[j];
  __syncwarp();
  shift_up1(o, pos, n, b.lane);
  if (b.lane == 0) o[pos] = make_uint2((unsigned)vol, ref);
  bump_lvend(le, j, NLV(w, side), 1, b.lane);
  SET_NORD(w, side, n + 1);
  return true;
}

// remove `d` consecutive entries of level j starting at pos; drops the level when it becomes empty
__device__ __forceinline__ void remove_entries(const Book& b, WarpState& w, int side, int j, int pos, int d) {
  int n = NORD(w, side);
  int nlv = NLV(w, side);
  uint16_t* le = b.lvend(side);
  shift_down(b.ord(side), pos, d, n, b.lane);
  bump_lvend(le, j, nlv, -d, b.lane);
  SET_NORD(w, side, n - d);
  int start = level_start(b, side, j);
  if ((int)le[j] == start) { // level empty => pop the price
    __syncwarp();
    shift_down(b.lvp(side), j, 1, nlv, b.lane);
    shift_down(le, j, 1, nlv, b.lane);
    SET_NLV(w, side, nlv - 1);
  }
}

// ---- agent table (Exchange.internal_orderbook) ---------------------------------------------------------------
__device__ __forceinline__ int agent_find(const Book& b, int side, int nag, uint32_t id) {
  const uint32_t* ids = b.aid(side);
  for (int base = 0; base < nag; base += 32) {
    int i = base + b.lane;
    unsigned m = __ballot_sync(FULL_MASK, i < nag && ids[i] == id);
    if (m) return base + __ffs(m) - 1;
  }
  return -1;
}
__device__ __forceinline__ void agent_remove_at(const Book& b, WarpState& w, int side, int i) {
  int nag = NAG(w, side);
  shift_down(b.aprice(side), i, 1, nag, b.lane);
  shift_down(b.avol(side), i, 1, nag, b.lane);
  shift_down(b.aid(side), i, 1, nag, b.lane);
  SET_NAG(w, side, nag - 1);
}
// reduce the agent's order `id` by v (removing it at zero); no-op when it is not in the table
__device__ __forceinline__ void agent_reduce(const Book& b, WarpState& w, int side, uint32_t id, int v, bool full) {
  int i = agent_find(b, side, NAG(w, side), id);
  if (i < 0) return;
  int32_t* av = b.avol(side);
  int nv = full ? 0 : av[i] - v;
  __syncwarp();
  if (nv <= 0) agent_remove_at(b, w, side, i);
  else { if (b.lane == 0) av[i] = nv; __syncwarp(); }
}

// ---- fills ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ void log_fill(const Book& b, WarpState& w, int list, int dir, int price, int vol, int is_market, uint32_t ref) {
  if (w.fill_log) {
    if (w.n_fills < w.fill_cap) {
      if (b.lane == 0) {
        lobsim_fill_t f; f.list = list; f.direction = dir; f.price = price; f.volume = vol; f.is_market = is_market; f.ref = ref;
        w.fill_log[w.n_fills] = f;
      }
    } else w.err |= LOBSIM_ERR_FILL_LOG_FULL;
    w.n_fills++;
  }
}
// FilledOrders.internal entry => portfolio (HOE.py:280-289) + flow counters
__device__ __forceinline__ void record_internal(WarpState& w, int dir, int price, int vol) {
  long long notional = (long long)vol * (long long)price;
  if (dir == 1) { w.inventory -= vol; w.cash += (double)notional; w.n_int1++; w.vol_int1 += vol; }
  else { w.inventory += vol; w.cash -= (double)notional; w.n_int0++; w.vol_int0 += vol; }
}
__device__ __forceinline__ void record_external(WarpState& w, int dir, int vol) {
  if (dir == 1) { w.n_ext1++; w.vol_ext1 += vol; } else { w.n_ext0++; w.vol_ext0 += vol; }
}

// ---- Exchange.submit_order (no-cross branch), Exchange.py:74-83 ------------------------------------------------
// returns the agent id given to the order, 0xffffffff for an external order that rested, 0 on overflow
__device__ __forceinline__ uint32_t rest_order(const Book& b, WarpState& w, int side, int price, int vol, uint32_t ref, bool is_agent) {
  int nag = NAG(w, side);
  if (is_agent && nag >= b.L.NA) { w.err |= LOBSIM_ERR_AGENT_OVERFLOW; return 0; }
  if (NORD(w, side) >= b.L.NO) { w.err |= LOBSIM_ERR_ORDER_OVERFLOW; return 0; }
  bool found;
  int j = find_level(b, side, NLV(w, side), price, found);
  if (!found && !insert_level(b, w, side, j, price)) return 0;
  uint32_t id = 0;
  if (is_agent) { // OrderIdConvertor.add_internal_id_to_order_and_track + internal book append
    id = w.next_agent_id++;
    ref = LOBSIM_REF_AGENT | id;
    if (b.lane == 0) { b.aprice(side)[nag] = price; b.avol(side)[nag] = vol; b.aid(side)[nag] = id; }
    SET_NAG(w, side, nag + 1);
    __syncwarp();
  }
  add_order(b, w, side, j, vol, ref);
  return is_agent ? id : 0xffffffffu; // external order rested (the reference assigns it an internal id here)
}

// ---- Exchange.submit_order / execute_order, Exchange.py:71-120 --------------------------------------------------
// is_limit: LimitOrder (crosses only while price allows, remainder rests); else MarketOrder.
__device__ __forceinline__ uint32_t submit_or_execute(const Book& b, WarpState& w, int side, int price, int vol, uint32_t ref, bool is_limit, bool is_agent) {
  int rem = vol;
  const int opp = side ^ 1;
  while (rem > 0) {
    int nl = NLV(w, opp);
    if (nl == 0) {
      if (!is_limit) { w.err |= LOBSIM_ERR_EMPTY_BOOK; w.dead = 1; return 0; } // EmptyOrderbookError :183-186
      break;                                                               // best = inf / 0 => no cross
    }
    int j = nl - 1;
    int bp = b.lvp(opp)[j];
    if (is_limit && !(side == 0 ? price >= bp : price <= bp)) break;     // _does_order_cross_spread :188-194
    int start = level_start(b, opp, j);
    uint2 head = b.ord(opp)[start];
    const bool hagent = (head.y & LOBSIM_REF_AGENT) != 0;
    __syncwarp();
    if (is_agent && hagent) { // cannot fill our own order => delete it, :91-94
      remove_entries(b, w, opp, j, start, 1);
      agent_reduce(b, w, opp, head.y & 0x7fffffffu, 0, true);
      continue;
    }
    int hv = (int)head.x;
    int v = rem < hv ? rem : hv;
    if (hv - v == 0) remove_entries(b, w, opp, j, start, 1);
    else { if (b.lane == 0) b.ord(opp)[start].x = (unsigned)(hv - v); __syncwarp(); }
    if (hagent) {
      agent_reduce(b, w, opp, head.y & 0x7fffffffu, v, false);
      record_internal(w, opp, bp, v);
      log_fill(b, w, 0, opp, bp, v, 0, head.y);
    } else {
      record_external(w, opp, v);
      log_fill(b, w, 1, opp, bp, v, 0, head.y);
    }
    rem -= v;
    if (is_agent) { // the synthetic MarketOrder fill of the aggressing agent, :111-115
      record_internal(w, side, bp, v);
      log_fill(b, w, 0, side, bp, v, 1, head.y);
    }
  }
  if (rem > 0 && is_limit) return rest_order(b, w, side, price, rem, ref, is_agent); // :116-119 / :74-83
  return 0;
}

// ---- Exchange.remove_order, Exchange.py:122-147 ------------------------------------------------------------------
// has_vol == false: Deletion with volume None (full delete).
__device__ __forceinline__ void remove_order(const Book& b, WarpState& w, int side, int price, int vol, bool has_vol, uint32_t ref, bool is_agent) {
  bool found;
  int j = find_level(b, side, NLV(w, side), price, found);
  if (!found) return;                                  // KeyError => continue, :129-132
  int start = level_start(b, side, j);
  int end = b.lvend(side)[j];
  const uint2* o = b.ord(side);
  int pos = -1;
  for (int base = start; base < end; base += 32) {    // _find_queue_position :196-217
    int i = base + b.lane;
    unsigned m = __ballot_sync(FULL_MASK, i < end && o[i].y == ref);
    if (m) { pos = base + __ffs(m) - 1; break; }
  }
  bool aggregate = false;
  if (pos < 0) {
    if (o[start].y != LOBSIM_REF_AGGREGATE) return;   // already filled, :138-139
    if (!has_vol) { w.err |= LOBSIM_ERR_BAD_VOLUME; return; } // assert :134
    pos = start; aggregate = true;                    // initial orders remain in book, :133-137
  }
  int cur = (int)o[pos].x;
  int rv = has_vol ? (vol < cur ? vol : cur) : cur;   // :140-146 (over-size => the resting volume)
  __syncwarp();
  if (cur - rv == 0) remove_entries(b, w, side, j, pos, 1);
  else { if (b.lane == 0) b.ord(side)[pos].x = (unsigned)(cur - rv); __syncwarp(); }
  if (is_agent && !aggregate) agent_reduce(b, w, side, ref & 0x7fffffffu, rv, false);
}

// ---- Exchange.process_order, Exchange.py:58-69: the ONE call site of the general book routines in a kernel ---------
__device__ __forceinline__ void process_order(const Book& b, WarpState& w, int type, int side, int price, int vol, uint32_t ref, bool is_agent) {
  if (w.dead) return;
  if (vol <= 0) { w.err |= LOBSIM_ERR_BAD_VOLUME; return; }
  if (type == LOBSIM_MSG_LIMIT || type == LOBSIM_MSG_MARKET) submit_or_execute(b, w, side, price, vol, ref, type == LOBSIM_MSG_LIMIT, is_agent);
  else remove_order(b, w, side, price, vol, true, ref, is_agent);
}

// ---- Orderbook properties, rl4mm/orderbook/models.py:72-101 -------------------------------------------------------
__device__ __forceinline__ int best_level_volume(const Book& b, int side, int nlv) {
  int j = nlv - 1;
  int start = level_start(b, side, j), end = b.lvend(side)[j];
  const uint2* o = b.ord(side);
  int s = 0;
  for (int i = start + b.lane; i < end; i += 32) s += (int)o[i].x;
  for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(FULL_MASK, s, d);
  return s;
}

__device__ __forceinline__ double microprice(int bb, int bs, int bv, int sv, double& imbalance) {
  imbalance = (double)(bv - sv) / (double)(bv + sv);
  return (1.0 + imbalance) / 2.0 * (double)bs + (1.0 - imbalance) / 2.0 * (double)bb;
}

// ---- WarpState <-> header ----------------------------------------------------------------------------------------
__device__ __forceinline__ void load_state(const Book& b, WarpState& w) {
  const BookHdr* h = b.hdr();
  w.nlv0 = h->cnt[0][0]; w.nlv1 = h->cnt[1][0]; w.nord0 = h->cnt[0][1]; w.nord1 = h->cnt[1][1];
  w.err = h->err; w.dead = h->dead;
  w.nag0 = h->nag[0]; w.nag1 = h->nag[1]; w.next_agent_id = h->next_agent_id; w.inventory = h->inventory; w.cash = h->cash;
  w.n_ext0 = w.n_ext1 = w.vol_ext0 = w.vol_ext1 = w.n_int0 = w.n_int1 = w.vol_int0 = w.vol_int1 = 0;
}
__device__ __forceinline__ void store_state(const Book& b, const WarpState& w) {
  __syncwarp();
  if (b.lane == 0) {
    BookHdr* h = b.hdr();
    h->cnt[0][0] = w.nlv0; h->cnt[1][0] = w.nlv1; h->cnt[0][1] = w.nord0; h->cnt[1][1] = w.nord1;
    h->err = w.err; h->dead = w.dead;
    h->nag[0] = w.nag0; h->nag[1] = w.nag1; h->next_agent_id = w.next_agent_id; h->inventory = w.inventory; h->cash = w.cash;
  }
  __syncwarp();
}
__device__ __forceinline__ void reset_flow(WarpState& w) {
  w.n_ext0 = w.n_ext1 = w.vol_ext0 = w.vol_ext1 = w.n_int0 = w.n_int1 = w.vol_int0 = w.vol_int1 = 0;
}
