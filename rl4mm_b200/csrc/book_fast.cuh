// book_fast.cuh -- the straight-line order path (the sorted books of the replay kernels, k_env_fast): same semantics as process_order in
// book.cuh, specialised for the overwhelmingly common shapes -- the touched level is among the 32 best, at most 32
// (64 for removals) queue entries have to move, no capacity is exhausted -- as straight-line warp-wide code without
// search / shift loops.  Anything else goes, BEFORE the book is mutated, to the any-depth routines at the end of this file
// (chunked whole-side searches and shifts, still static layout, still no call): fast_order_full is the entry point.
//
// Differences from the general path, all for instruction count (the kernel is issue-bound, DESIGN.md section 3):
//   * the layout is a compile-time constant (StaticLayout<NL,NO,NA>), so every array access is base + immediate;
//   * the per-side counters {nlv, nord} stay in the shared-memory header and are read / written with one 64-bit
//     access keyed by the side, instead of living in registers behind per-side selects;
//   * the best price of each side is cached in registers for the crossing test.
#pragma once
#include "book.cuh"

template <int NL_, int NO_, int NA_>
struct StaticLayout {
  static constexpr int NL = NL_, NO = NO_, NA = NA_;
  static constexpr int side_off = (int)sizeof(BookHdr);
  static constexpr int lvend_off = NL * 4;
  static constexpr int ord_off = (NL * 4 + NL * 2 + 7) & ~7;
  static constexpr int side_stride = (ord_off + NO * 8 + 15) & ~15;
  static constexpr int agent_off = side_off + 2 * side_stride;
  static constexpr int blob_bytes = (agent_off + 2 * NA * 12 + 15) & ~15;
  __host__ __device__ static bool matches(const Layout& l) {
    return l.NL == NL && l.NO == NO && l.NA == NA && l.side_off == side_off && l.lvend_off == lvend_off && l.ord_off == ord_off &&
           l.side_stride == side_stride && l.agent_off == agent_off && l.blob_bytes == blob_bytes;
  }
};

struct FastState {
  int best0, best1; // INT32_MIN / INT32_MAX when the side is empty
  uint32_t err;
  int dead;
  // tracked mode only: optional fill log (global memory); the fill counter lives in the header
  lobsim_fill_t* fill_log;
  int fill_cap;
  // fast_order handles the common cases and leaves the rare order to fast_order_full -- bail = 1: rest `bail_vol` (the whole
  // order, or the unfilled remainder of a crossing limit order whose fills have been applied), bail = 2: cancel / delete
  int bail, bail_vol;
};

template <class LT>
struct FastBook {
  unsigned char* blob;
  int lane;
  __device__ __forceinline__ int2* cnt(int s) const { return reinterpret_cast<int2*>(blob) + s; }
  __device__ __forceinline__ unsigned char* side(int s) const { return blob + LT::side_off + s * LT::side_stride; }
  static __device__ __forceinline__ int32_t* P(unsigned char* sb) { return reinterpret_cast<int32_t*>(sb); }
  static __device__ __forceinline__ uint16_t* LE(unsigned char* sb) { return reinterpret_cast<uint16_t*>(sb + LT::lvend_off); }
  static __device__ __forceinline__ uint2* O(unsigned char* sb) { return reinterpret_cast<uint2*>(sb + LT::ord_off); }
};

// (err | dead << 31) word exchanged with the cold noinline routines of the kernels
__device__ __forceinline__ uint32_t pack_errdead(uint32_t err, int dead) { return err | ((uint32_t)dead << 31); }

// ---- tracked mode: fills -> per-step flow, portfolio (HOE.py:280-289) and the optional fill log; all by lane 0 on the
//      shared-memory header --------------------------------------------------------------------------------------------
// (real functions with by-value arguments: one copy of each in the instruction cache, no address-taken locals)
static __device__ __noinline__ void fast_record_fn(unsigned char* blob, int lane, lobsim_fill_t* fill_log, int fill_cap, int list, int dir, int price, int vol, int is_market, uint32_t ref) {
  if (lane == 0) {
    BookHdr* h = reinterpret_cast<BookHdr*>(blob);
    if (list == 0) { // FilledOrders.internal
      const long long notional = (long long)vol * (long long)price;
      if (dir == 1) { h->inventory -= vol; h->cash += (double)notional; } else { h->inventory += vol; h->cash -= (double)notional; }
      h->flow[4 + dir] += 1; h->flow[6 + dir] += vol;
    } else { h->flow[dir] += 1; h->flow[2 + dir] += vol; }
    const int n = h->n_fills;
    if (fill_log && n < fill_cap) {
      lobsim_fill_t r; r.list = list; r.direction = dir; r.price = price; r.volume = vol; r.is_market = is_market; r.ref = ref;
      fill_log[n] = r;
    }
    h->n_fills = n + 1;
  }
}
template <class LT>
__device__ __forceinline__ void fast_record(const FastBook<LT>& fb, FastState& f, int list, int dir, int price, int vol, int is_market, uint32_t ref) {
  fast_record_fn(fb.blob, fb.lane, f.fill_log, f.fill_cap, list, dir, price, vol, is_market, ref);
}

// the agent's order `id` loses v (or everything): Exchange.internal_orderbook mirror.  NA <= 64.
static __device__ __noinline__ void fast_agent_reduce_fn(unsigned char* blob, int lane, int agent_off, int NA, int side, uint32_t id, int v, int full) {
  BookHdr* h = reinterpret_cast<BookHdr*>(blob);
  int32_t* ap = reinterpret_cast<int32_t*>(blob + agent_off + side * NA * 12);
  int32_t* av = ap + NA;
  uint32_t* ai = reinterpret_cast<uint32_t*>(ap + 2 * NA);
  const int nag = h->nag[side];
  const unsigned m0 = __ballot_sync(FULL_MASK, lane < nag && ai[lane] == id);
  const unsigned m1 = __ballot_sync(FULL_MASK, lane + 32 < nag && ai[lane + 32] == id);
  if (!(m0 | m1)) return;
  const int i = m0 ? __ffs(m0) - 1 : 32 + __ffs(m1) - 1;
  const int nv = full ? 0 : av[i] - v;
  __syncwarp();
  if (nv > 0) { if (lane == 0) av[i] = nv; __syncwarp(); return; }
  const int tail = nag - i - 1; // <= 63 entries move down by one
  int p0 = 0, p1 = 0, v0 = 0, v1 = 0; uint32_t i0 = 0, i1 = 0;
  if (lane < tail) { p0 = ap[i + 1 + lane]; v0 = av[i + 1 + lane]; i0 = ai[i + 1 + lane]; }
  if (lane + 32 < tail) { p1 = ap[i + 33 + lane]; v1 = av[i + 33 + lane]; i1 = ai[i + 33 + lane]; }
  __syncwarp();
  if (lane < tail) { ap[i + lane] = p0; av[i + lane] = v0; ai[i + lane] = i0; }
  if (lane + 32 < tail) { ap[i + 32 + lane] = p1; av[i + 32 + lane] = v1; ai[i + 32 + lane] = i1; }
  if (lane == 0) h->nag[side] = nag - 1;
  __syncwarp();
}
template <class LT>
__device__ __forceinline__ void fast_agent_reduce(const FastBook<LT>& fb, int side, uint32_t id, int v, bool full) {
  static_assert(LT::NA <= 64, "the straight-line agent table code handles at most 64 agent orders per side");
  fast_agent_reduce_fn(fb.blob, fb.lane, LT::agent_off, LT::NA, side, id, v, full ? 1 : 0);
}

template <class LT>
__device__ __forceinline__ void fast_refresh_best(const FastBook<LT>& fb, FastState& f) {
  __syncwarp();
  const int n0 = fb.cnt(0)->x, n1 = fb.cnt(1)->x;
  f.best0 = n0 ? fb.P(fb.side(0))[n0 - 1] : INT32_MIN;
  f.best1 = n1 ? fb.P(fb.side(1))[n1 - 1] : INT32_MAX;
}

// TR: fills / flows / agent orders are tracked (env kernels); TR == false is the pure replay.
template <class LT, bool TR>
__device__ __forceinline__ void fast_order(const FastBook<LT>& fb, FastState& f, int type, int side, int price, int vol, uint32_t ref, bool is_agent) {
  if (!TR) is_agent = false;
  const int lane = fb.lane;
  if (vol <= 0) { f.err |= LOBSIM_ERR_BAD_VOLUME; return; }
  const bool crosses = side ? price <= f.best0 : price >= f.best1;
  if (type == LOBSIM_MSG_MARKET || (type == LOBSIM_MSG_LIMIT && crosses)) {
    // ---- execution against the opposite best queue (Exchange.py:85-120) -------------------------------------------
    const int opp = side ^ 1;
    unsigned char* sb = fb.side(opp);
    int2 c = *fb.cnt(opp);
    int rem = vol;
#pragma unroll 1
    while (rem > 0) {
      if (c.x == 0) {
        if (type == LOBSIM_MSG_MARKET) { f.err |= LOBSIM_ERR_EMPTY_BOOK; f.dead = 1; } // EmptyOrderbookError :183-186
        break;
      }
      const int bp = opp ? f.best1 : f.best0;
      if (type == LOBSIM_MSG_LIMIT && !(side ? price <= bp : price >= bp)) break;
      const int j = c.x - 1;
      const int start = j > 0 ? (int)fb.LE(sb)[j - 1] : 0;   // the best level is the last segment: [start, nord)
      const int len = c.y - start;
      uint2 e = make_uint2(0u, 0u);
      if (lane < len) e = fb.O(sb)[start + lane];           // first 32 entries of the best queue
      const int hv = (int)__shfl_sync(FULL_MASK, e.x, 0);
      const uint32_t href = TR ? __shfl_sync(FULL_MASK, e.y, 0) : 0u;
      const bool hagent = TR && (href & LOBSIM_REF_AGENT) != 0;
      const bool self_match = TR && is_agent && hagent;      // cannot fill our own order => delete it, :91-94
      if (!self_match) {
        const int v = rem < hv ? rem : hv;
        if (TR) {
          if (hagent) { fast_record(fb, f, 0, opp, bp, v, 0, href); }
          else fast_record(fb, f, 1, opp, bp, v, 0, href);
          if (is_agent) fast_record(fb, f, 0, side, bp, v, 1, href);   // the synthetic MarketOrder fill, :111-115
        }
        if (rem < hv) {                                      // partial fill of the head
          if (lane == 0) fb.O(sb)[start].x = (unsigned)(hv - rem);
          if (TR && hagent) { __syncwarp(); fast_agent_reduce(fb, opp, href & 0x7fffffffu, rem, false); }
          rem = 0;
          break;
        }
        rem -= hv;                                           // the head is consumed
      }
      if (len > 33) { __syncwarp(); shift_down(fb.O(sb), start, 1, c.y, lane); }
      else {
        uint2 e32 = make_uint2(0u, 0u);
        if (len == 33 && lane == 0) e32 = fb.O(sb)[start + 32];
        __syncwarp();
        if (lane >= 1 && lane < len) fb.O(sb)[start + lane - 1] = e;
        if (len == 33 && lane == 0) fb.O(sb)[start + 31] = e32;
      }
      c.y -= 1;
      if (len == 1) {                                        // level emptied: it is the last one, nothing to shift
        c.x -= 1;
        const int nb = c.x ? fb.P(sb)[c.x - 1] : (opp ? INT32_MAX : INT32_MIN);
        if (opp) f.best1 = nb; else f.best0 = nb;
      } else if (lane == 0) fb.LE(sb)[j] = (uint16_t)c.y;
      __syncwarp();
      if (TR && hagent) fast_agent_reduce(fb, opp, href & 0x7fffffffu, 0, true);   // the resting agent order is gone
    }
    __syncwarp();   // every lane has read the counters (WAR) before lane 0 rewrites them
    if (lane == 0) *fb.cnt(opp) = c;
    __syncwarp();
    if (rem > 0 && type == LOBSIM_MSG_LIMIT && !f.dead) {    // the remainder rests (Exchange.py:116-119); rare
      f.bail = 1; f.bail_vol = rem;                        // -> fast_rest_any (fast_order_full)
    }
    return;
  }
  unsigned char* sb = fb.side(side);
  const int2 c = *fb.cnt(side);
  const int nlv = c.x, nord = c.y;
  // ---- level search among the 32 best levels (prices compared as keys: bids p, asks -p) ---------------------------
  const int sm = -side;                                      // 0 or 0xffffffff
  const int idx = nlv - 1 - lane;
  const int tkey = (price ^ sm) - sm;
  int k = INT32_MIN;
  if (idx >= 0) k = (fb.P(sb)[idx] ^ sm) - sm;
  const unsigned eq = __ballot_sync(FULL_MASK, k == tkey);
  const unsigned gt = __ballot_sync(FULL_MASK, k > tkey);
  if (type == LOBSIM_MSG_LIMIT) {
    // ---- a non-crossing limit order rests (Exchange.py:74-83) -------------------------------------------------------
    const int cb = __popc(gt);
    int nag = 0;
    if (TR && is_agent) nag = reinterpret_cast<BookHdr*>(fb.blob)->nag[side];
    if ((!eq && (cb == 32 || nlv >= LT::NL)) || nord >= LT::NO || (TR && is_agent && nag >= LT::NA)) { // deep level or a capacity limit
      f.bail = 1; f.bail_vol = vol;                        // -> fast_rest_any (fast_order_full)
      return;
    }
    int j, pos;
    if (eq) {
      j = nlv - __ffs(eq);
      pos = fb.LE(sb)[j];
    } else {
      j = nlv - cb;                                          // insertion index; the cb better levels move up by one
      pos = j > 0 ? (int)fb.LE(sb)[j - 1] : 0;
      int pv = 0; unsigned short ev = 0;
      const int i = j + lane;
      if (i < nlv) { pv = fb.P(sb)[i]; ev = fb.LE(sb)[i]; }
      __syncwarp();
      if (i < nlv) { fb.P(sb)[i + 1] = pv; fb.LE(sb)[i + 1] = ev; }
      if (lane == 0) { fb.P(sb)[j] = price; fb.LE(sb)[j] = (uint16_t)pos; }
      if (cb == 0) { if (side) f.best1 = price; else f.best0 = price; }
      __syncwarp();
    }
    const int nlv2 = eq ? nlv : nlv + 1;
    const int above = nord - pos;                            // entries of better levels that move up by one
    if (above > 32) { __syncwarp(); shift_up1(fb.O(sb), pos, nord, lane); }
    else if (above > 0) {
      uint2 v = make_uint2(0u, 0u);
      if (lane < above) v = fb.O(sb)[pos + lane];
      __syncwarp();
      if (lane < above) fb.O(sb)[pos + lane + 1] = v;
    }
    if (TR && is_agent) {   // OrderIdConvertor.add_internal_id_to_order_and_track + internal book append
      BookHdr* h = reinterpret_cast<BookHdr*>(fb.blob);
      const uint32_t id = h->next_agent_id;
      ref = LOBSIM_REF_AGENT | id;
      __syncwarp();
      if (lane == 0) {
        int32_t* ap = reinterpret_cast<int32_t*>(fb.blob + LT::agent_off + side * LT::NA * 12);
        ap[nag] = price; ap[LT::NA + nag] = vol; reinterpret_cast<uint32_t*>(ap)[2 * LT::NA + nag] = id;
        h->nag[side] = nag + 1; h->next_agent_id = id + 1;
      }
    }
    __syncwarp();   // every lane has read the counters / level ends (WAR) before they are rewritten
    if (lane == 0) { fb.O(sb)[pos] = make_uint2((unsigned)vol, ref); *fb.cnt(side) = make_int2(nlv2, nord + 1); }
    { const int i = j + lane; if (i < nlv2) fb.LE(sb)[i] = (uint16_t)(fb.LE(sb)[i] + 1); }   // nlv2 - j <= 32
    __syncwarp();
    return;
  }
  // ---- cancellation / deletion (Exchange.py:122-147) ------------------------------------------------------------------
  if (!eq) {
    if (__popc(gt) == 32) {                                  // the level may be deeper than the 32 best
      f.bail = 2;                                          // -> fast_remove_any (fast_order_full)
    }
    return;                                                  // level absent: nothing to do (:129-132)
  }
  const int j = nlv - __ffs(eq);
  const int start = j > 0 ? (int)fb.LE(sb)[j - 1] : 0, end = fb.LE(sb)[j];
  const int len = end - start;
  if (len > 32 || nord - start > 64) {                       // long queue / long shift: general path
    f.bail = 2;                                            // -> fast_remove_any (fast_order_full)
    return;
  }
  uint2 e = make_uint2(0u, 0xffffffffu);
  if (lane < len) e = fb.O(sb)[start + lane];
  const unsigned m = __ballot_sync(FULL_MASK, lane < len && e.y == ref);   // _find_queue_position :196-217
  int l;
  bool aggregate = false;
  if (m) l = __ffs(m) - 1;
  else {
    if (__shfl_sync(FULL_MASK, e.y, 0) != LOBSIM_REF_AGGREGATE) return;    // already filled (:138-139)
    l = 0; aggregate = true;                                              // hit the aggregate at the head (:133-137)
  }
  const int cur = (int)__shfl_sync(FULL_MASK, e.x, l);
  const int pos = start + l;
  if (vol < cur) {                                           // partial: reduce in place
    if (lane == l) fb.O(sb)[pos].x = (unsigned)(cur - vol);
    __syncwarp();
    if (TR && is_agent && !aggregate) fast_agent_reduce(fb, side, ref & 0x7fffffffu, vol, false);
    return;
  }
  // full removal (over-size requests remove the resting volume, :142-146): entries (pos, nord) move down by one
  const int tail = nord - pos - 1;                           // <= 63
  uint2 v0 = make_uint2(0u, 0u), v1 = make_uint2(0u, 0u);
  if (lane < tail) v0 = fb.O(sb)[pos + 1 + lane];
  if (lane + 32 < tail) v1 = fb.O(sb)[pos + 33 + lane];
  __syncwarp();
  if (lane < tail) fb.O(sb)[pos + lane] = v0;
  if (lane + 32 < tail) fb.O(sb)[pos + 32 + lane] = v1;
  if (len == 1) {                                            // the level disappears: better levels move down by one
    int pv = 0; unsigned short ev = 0;
    const int i = j + 1 + lane;
    if (i < nlv) { pv = fb.P(sb)[i]; ev = fb.LE(sb)[i]; }
    __syncwarp();
    if (i < nlv) { fb.P(sb)[i - 1] = pv; fb.LE(sb)[i - 1] = (uint16_t)(ev - 1); }
    if (lane == 0) *fb.cnt(side) = make_int2(nlv - 1, nord - 1);
    if (j == nlv - 1) {                                      // it was the best level
      const int nb = nlv > 1 ? fb.P(sb)[nlv - 2] : (side ? INT32_MAX : INT32_MIN);
      if (side) f.best1 = nb; else f.best0 = nb;
    }
  } else {
    if (lane < nlv - j) fb.LE(sb)[j + lane] = (uint16_t)(fb.LE(sb)[j + lane] - 1);   // nlv - j <= 32
    if (lane == 0) *fb.cnt(side) = make_int2(nlv, nord - 1);
  }
  __syncwarp();
  if (TR && is_agent && !aggregate) fast_agent_reduce(fb, side, ref & 0x7fffffffu, cur, true);
}

// ---- OrderbookSimulator.update_outer_levels (OrderbookSimulator.py:105-135) for books WITHOUT agent orders (pure replay) ----
// One snapshot level beyond the tracked price range: central[side][price] = deque([aggregate]) -- the level's queue is replaced by
// one aggregate order, or the level is inserted (anywhere, typically at the WORST end, i.e. the front of the arrays).  Static
// layout, whole-side searches and shifts in 32-wide chunks, no call.
template <class LT>
__device__ __forceinline__ void fast_resync_level(const FastBook<LT>& fb, FastState& f, int side, int price, int vol) {
  const int lane = fb.lane;
  unsigned char* sb = fb.side(side);
  const int2 c = *fb.cnt(side);
  const int nlv = c.x, nord = c.y;
  const int sm = -side;
  const int tkey = (price ^ sm) - sm;                        // keys ascend from the worst to the best level on both sides
  int j = 0, jeq = -1;
#pragma unroll
  for (int q = 0; q < LT::NL / 32; q++) {
    const int i = q * 32 + lane;
    int k = INT32_MAX;
    if (i < nlv) k = (fb.P(sb)[i] ^ sm) - sm;
    j += __popc(__ballot_sync(FULL_MASK, i < nlv && k < tkey));
    const unsigned eq = __ballot_sync(FULL_MASK, i < nlv && k == tkey);
    if (eq) jeq = q * 32 + __ffs(eq) - 1;
  }
  __syncwarp();
  if (jeq >= 0) {                                            // the level exists: keep one entry, make it the aggregate
    const int start = jeq > 0 ? (int)fb.LE(sb)[jeq - 1] : 0, end = fb.LE(sb)[jeq];
    const int extra = end - start - 1;
    __syncwarp();
    if (extra > 0) {
      for (int base = end; base < nord; base += 32) {       // entries behind the level move down by `extra`, ascending chunks
        uint2 v = make_uint2(0u, 0u);
        if (base + lane < nord) v = fb.O(sb)[base + lane];
        __syncwarp();
        if (base + lane < nord) fb.O(sb)[base + lane - extra] = v;
        __syncwarp();
      }
#pragma unroll
      for (int q = 0; q < LT::NL / 32; q++) {
        const int i = q * 32 + lane;
        if (i >= jeq && i < nlv) fb.LE(sb)[i] = (uint16_t)(fb.LE(sb)[i] - extra);
      }
    }
    if (lane == 0) { fb.O(sb)[start] = make_uint2((unsigned)vol, LOBSIM_REF_AGGREGATE); *fb.cnt(side) = make_int2(nlv, nord - (extra > 0 ? extra : 0)); }
    __syncwarp();
    return;
  }
  if (nord >= LT::NO) { f.err |= LOBSIM_ERR_ORDER_OVERFLOW; return; }                       // same flags as the general routine
  if (nlv >= LT::NL) { f.err |= LOBSIM_ERR_LEVEL_OVERFLOW; return; }
  const int pos = j > 0 ? (int)fb.LE(sb)[j - 1] : 0;         // the new level's (one-entry) segment starts where level j-1 ends
  __syncwarp();
  for (int base = pos + ((nord - pos + 31) / 32 - 1) * 32; base >= pos; base -= 32) {   // entries [pos, nord) move up by one, descending chunks
    uint2 v = make_uint2(0u, 0u);
    if (base + lane < nord) v = fb.O(sb)[base + lane];
    __syncwarp();
    if (base + lane < nord) fb.O(sb)[base + lane + 1] = v;
    __syncwarp();
  }
  for (int base = j + ((nlv - j + 31) / 32 - 1) * 32; base >= j; base -= 32) {          // levels [j, nlv) move up by one
    int pv = 0; unsigned short ev = 0;
    if (base + lane < nlv) { pv = fb.P(sb)[base + lane]; ev = fb.LE(sb)[base + lane]; }
    __syncwarp();
    if (base + lane < nlv) { fb.P(sb)[base + lane + 1] = pv; fb.LE(sb)[base + lane + 1] = (uint16_t)(ev + 1); }
    __syncwarp();
  }
  if (lane == 0) {
    fb.P(sb)[j] = price; fb.LE(sb)[j] = (uint16_t)(pos + 1);
    fb.O(sb)[pos] = make_uint2((unsigned)vol, LOBSIM_REF_AGGREGATE);
    *fb.cnt(side) = make_int2(nlv + 1, nord + 1);
  }
  __syncwarp();
}

// The whole update for a replay book: every snapshot level beyond [min_buy, max_sell] in the reference's order (buy side best ->
// worst, then sell side), then the price-range trackers (:134-135).  `row` = the snapshot row of this second.
template <class LT>
__device__ __forceinline__ void fast_resync(const FastBook<LT>& fb, FastState& f, const int32_t* __restrict__ row, int L) {
  const int lane = fb.lane;
  BookHdr* h = reinterpret_cast<BookHdr*>(fb.blob);
  const int min_buy = h->min_buy, max_sell = h->max_sell;   // the filter uses the range at entry (_initial_prices_filter_function)
  for (int base = 0; base < 2 * L; base += 32) {
    const int idx = base + lane;
    int price = LOBSIM_NO_PRICE, vol = 0;
    if (idx < 2 * L) { price = __ldg(&row[idx * 2]); vol = __ldg(&row[idx * 2 + 1]); }
    unsigned hits = __ballot_sync(FULL_MASK, price != LOBSIM_NO_PRICE && (idx < L ? price < min_buy : price > max_sell));
    while (hits) {
      const int src = __ffs(hits) - 1;
      hits &= hits - 1;
      const int pr = __shfl_sync(FULL_MASK, price, src), vo = __shfl_sync(FULL_MASK, vol, src);
      fast_resync_level(fb, f, base + src >= L ? 1 : 0, pr, vo);
    }
  }
  __syncwarp();
  if (lane == 0) {
    const int n0 = fb.cnt(0)->x, n1 = fb.cnt(1)->x;
    if (n0 && fb.P(fb.side(0))[0] < h->min_buy) h->min_buy = fb.P(fb.side(0))[0];
    if (n1 && fb.P(fb.side(1))[0] > h->max_sell) h->max_sell = fb.P(fb.side(1))[0];
  }
  __syncwarp();
  fast_refresh_best(fb, f);
}

// ---- the rare orders of a pure replay (no agent orders in the book), straight-line at any depth / queue length ----------------
// whole-side level search: j = number of levels worse than `price` (insertion index), jeq = index of the level or -1
template <class LT>
__device__ __forceinline__ void fast_find_any(const FastBook<LT>& fb, unsigned char* sb, int side, int nlv, int price, int& j, int& jeq) {
  const int sm = -side;
  const int tkey = (price ^ sm) - sm;
  j = 0; jeq = -1;
#pragma unroll 1
  for (int q = 0; q * 32 < nlv; q++) {                       // only the chunks that hold levels (deep books: 40-60 of 128)
    const int i = q * 32 + fb.lane;
    int k = INT32_MAX;
    if (i < nlv) k = (fb.P(sb)[i] ^ sm) - sm;
    j += __popc(__ballot_sync(FULL_MASK, i < nlv && k < tkey));
    const unsigned eq = __ballot_sync(FULL_MASK, i < nlv && k == tkey);
    if (eq) jeq = q * 32 + __ffs(eq) - 1;
  }
  __syncwarp();
}
// Exchange.submit_order, no-cross branch (Exchange.py:74-83) = book.cuh rest_order: same result, same overflow flags
template <class LT, bool TR>
__device__ __forceinline__ void fast_rest_any(const FastBook<LT>& fb, FastState& f, int side, int price, int vol, uint32_t ref, bool is_agent) {
  if (!TR) is_agent = false;
  const int lane = fb.lane;
  unsigned char* sb = fb.side(side);
  BookHdr* h = reinterpret_cast<BookHdr*>(fb.blob);
  const int2 c = *fb.cnt(side);
  const int nlv = c.x, nord = c.y;
  int nag = 0;
  if (TR && is_agent) { nag = h->nag[side]; if (nag >= LT::NA) { f.err |= LOBSIM_ERR_AGENT_OVERFLOW; return; } }
  if (nord >= LT::NO) { f.err |= LOBSIM_ERR_ORDER_OVERFLOW; return; }
  int j, jeq;
  fast_find_any(fb, sb, side, nlv, price, j, jeq);
  int nlv2 = nlv, pos;
  if (jeq < 0) {
    if (nlv >= LT::NL) { f.err |= LOBSIM_ERR_LEVEL_OVERFLOW; return; }
    pos = j > 0 ? (int)fb.LE(sb)[j - 1] : 0;
    __syncwarp();
    for (int base = j + ((nlv - j + 31) / 32 - 1) * 32; base >= j; base -= 32) {   // levels [j, nlv) move up by one, descending chunks
      int pv = 0; unsigned short ev = 0;
      if (base + lane < nlv) { pv = fb.P(sb)[base + lane]; ev = fb.LE(sb)[base + lane]; }
      __syncwarp();
      if (base + lane < nlv) { fb.P(sb)[base + lane + 1] = pv; fb.LE(sb)[base + lane + 1] = ev; }
      __syncwarp();
    }
    if (lane == 0) { fb.P(sb)[j] = price; fb.LE(sb)[j] = (uint16_t)pos; }
    nlv2 = nlv + 1;
    __syncwarp();
  } else { j = jeq; pos = fb.LE(sb)[jeq]; __syncwarp(); }
  if (TR && is_agent) {   // OrderIdConvertor.add_internal_id_to_order_and_track + internal book append (after the level exists)
    const uint32_t id = h->next_agent_id;
    ref = LOBSIM_REF_AGENT | id;
    __syncwarp();
    if (lane == 0) {
      int32_t* ap = reinterpret_cast<int32_t*>(fb.blob + LT::agent_off + side * LT::NA * 12);
      ap[nag] = price; ap[LT::NA + nag] = vol; reinterpret_cast<uint32_t*>(ap)[2 * LT::NA + nag] = id;
      h->nag[side] = nag + 1; h->next_agent_id = id + 1;
    }
    __syncwarp();
  }
  for (int base = pos + ((nord - pos + 31) / 32 - 1) * 32; base >= pos; base -= 32) {   // entries [pos, nord) move up by one
    uint2 v = make_uint2(0u, 0u);
    if (base + lane < nord) v = fb.O(sb)[base + lane];
    __syncwarp();
    if (base + lane < nord) fb.O(sb)[base + lane + 1] = v;
    __syncwarp();
  }
#pragma unroll 1
  for (int q = j >> 5; q * 32 < nlv2; q++) {                 // level ends from the touched level on
    const int i = q * 32 + lane;
    if (i >= j && i < nlv2) fb.LE(sb)[i] = (uint16_t)(fb.LE(sb)[i] + 1);
  }
  if (lane == 0) { fb.O(sb)[pos] = make_uint2((unsigned)vol, ref); *fb.cnt(side) = make_int2(nlv2, nord + 1); }
  __syncwarp();
  fast_refresh_best(fb, f);
}
// Exchange.remove_order (Exchange.py:122-147) = book.cuh remove_order with a volume
template <class LT, bool TR>
__device__ __forceinline__ void fast_remove_any(const FastBook<LT>& fb, FastState& f, int side, int price, int vol, uint32_t ref, bool is_agent) {
  if (!TR) is_agent = false;
  const int lane = fb.lane;
  unsigned char* sb = fb.side(side);
  const int2 c = *fb.cnt(side);
  const int nlv = c.x, nord = c.y;
  int j, jeq;
  fast_find_any(fb, sb, side, nlv, price, j, jeq);
  if (jeq < 0) return;                                       // KeyError => continue, :129-132
  const int start = jeq > 0 ? (int)fb.LE(sb)[jeq - 1] : 0, end = fb.LE(sb)[jeq];
  int pos = -1;
  for (int base = start; base < end; base += 32) {           // _find_queue_position :196-217
    const int i = base + lane;
    const unsigned m = __ballot_sync(FULL_MASK, i < end && fb.O(sb)[i < end ? i : start].y == ref);
    if (m) { pos = base + __ffs(m) - 1; break; }
  }
  bool aggregate = false;
  if (pos < 0) {
    if (fb.O(sb)[start].y != LOBSIM_REF_AGGREGATE) return;   // already filled, :138-139
    pos = start; aggregate = true;                           // initial orders remain in book, :133-137
  }
  const int cur = (int)fb.O(sb)[pos].x;
  const int rv = vol < cur ? vol : cur;                      // over-size => the resting volume, :142-146
  __syncwarp();
  if (cur - rv > 0) {
    if (lane == 0) fb.O(sb)[pos].x = (unsigned)(cur - rv);
    __syncwarp();
    if (TR && is_agent && !aggregate) fast_agent_reduce(fb, side, ref & 0x7fffffffu, rv, false);
    return;
  }
  for (int base = pos + 1; base < nord; base += 32) {       // entries behind it move down by one, ascending chunks
    uint2 v = make_uint2(0u, 0u);
    if (base + lane < nord) v = fb.O(sb)[base + lane];
    __syncwarp();
    if (base + lane < nord) fb.O(sb)[base + lane - 1] = v;
    __syncwarp();
  }
  const bool level_gone = end - start == 1;
  if (!level_gone) {
#pragma unroll 1
    for (int q = jeq >> 5; q * 32 < nlv; q++) {
      const int i = q * 32 + lane;
      if (i >= jeq && i < nlv) fb.LE(sb)[i] = (uint16_t)(fb.LE(sb)[i] - 1);
    }
    if (lane == 0) *fb.cnt(side) = make_int2(nlv, nord - 1);
  } else {                                                   // the level disappears: levels above it move down by one
    for (int base = jeq + 1; base < nlv; base += 32) {
      int pv = 0; unsigned short ev = 0;
      if (base + lane < nlv) { pv = fb.P(sb)[base + lane]; ev = fb.LE(sb)[base + lane]; }
      __syncwarp();
      if (base + lane < nlv) { fb.P(sb)[base + lane - 1] = pv; fb.LE(sb)[base + lane - 1] = (uint16_t)(ev - 1); }
      __syncwarp();
    }
    if (lane == 0) *fb.cnt(side) = make_int2(nlv - 1, nord - 1);
  }
  __syncwarp();
  if (TR && is_agent && !aggregate) fast_agent_reduce(fb, side, ref & 0x7fffffffu, rv, false);
  fast_refresh_best(fb, f);
}

// One order through the straight-line path: the common cases in fast_order (no call), the rare ones (level beyond the
// 32 best, queue longer than 32, shift longer than 64, remainder of a crossing limit order, capacity limits) in the any-depth
// routines above.  This is the only entry point the kernels use.
template <class LT, bool TR>
__device__ __forceinline__ void fast_order_full(const FastBook<LT>& fb, FastState& f, int type, int side, int price, int vol, uint32_t ref, bool is_agent) {
  fast_order<LT, TR>(fb, f, type, side, price, vol, ref, is_agent);
  if (f.bail) {
    if (f.bail == 1) fast_rest_any<LT, TR>(fb, f, side, price, f.bail_vol, ref, is_agent);
    else fast_remove_any<LT, TR>(fb, f, side, price, vol, ref, is_agent);
    f.bail = 0;
  }
}

// update_outer_levels for a book WITH agent orders (env kernels), OrderbookSimulator.py:105-135: as fast_resync, plus -- the
// agent's orders at an overwritten price are cancelled first (:116-129) and re-submitted, behind the new aggregate, after all
// levels are done (:132-133, a normal limit order of the agent: it may cross).  scratch: per-warp int2[2*NA] = {price | side, vol}.
template <class LT>
__device__ __forceinline__ void fast_resync_tracked(const FastBook<LT>& fb, FastState& f, const int32_t* __restrict__ row, int L, int2* scratch) {
  const int lane = fb.lane;
  BookHdr* h = reinterpret_cast<BookHdr*>(fb.blob);
  const int min_buy = h->min_buy, max_sell = h->max_sell;
  int nrepl = 0, nrepl_buy = -1;
  for (int base = 0; base < 2 * L; base += 32) {
    const int idx = base + lane;
    int price = LOBSIM_NO_PRICE, vol = 0;
    if (idx < 2 * L) { price = __ldg(&row[idx * 2]); vol = __ldg(&row[idx * 2 + 1]); }
    unsigned hits = __ballot_sync(FULL_MASK, price != LOBSIM_NO_PRICE && (idx < L ? price < min_buy : price > max_sell));
    while (hits) {
      const int src = __ffs(hits) - 1;
      hits &= hits - 1;
      const int pr = __shfl_sync(FULL_MASK, price, src), vo = __shfl_sync(FULL_MASK, vol, src);
      const int side = base + src >= L ? 1 : 0;
      if (side == 1 && nrepl_buy < 0) nrepl_buy = nrepl;       // everything saved so far belongs to the buy side
      const int32_t* ap = reinterpret_cast<const int32_t*>(fb.blob + LT::agent_off + side * LT::NA * 12);
      const int32_t* av = ap + LT::NA;
      const uint32_t* ai = reinterpret_cast<const uint32_t*>(ap + 2 * LT::NA);
      for (int i = 0; i < h->nag[side];) {
        const int p_i = ap[i], v_i = av[i];
        const uint32_t id = ai[i];
        __syncwarp();
        if (p_i != pr) { i++; continue; }
        if (lane == 0) scratch[nrepl] = make_int2(pr, v_i);
        nrepl++;
        const int before = h->nag[side];
        fast_order_full<LT, true>(fb, f, LOBSIM_MSG_CANCEL, side, pr, v_i, LOBSIM_REF_AGENT | id, true);
        __syncwarp();
        if (h->nag[side] == before) fast_agent_reduce(fb, side, id, 0, true);   // keep internal and central consistent
        __syncwarp();
      }
      fast_resync_level(fb, f, side, pr, vo);
    }
  }
  if (nrepl_buy < 0) nrepl_buy = nrepl;
  __syncwarp();
  for (int i = 0; i < nrepl; i++) {                          // :132-133
    const int2 r = scratch[i];
    __syncwarp();
    fast_order_full<LT, true>(fb, f, LOBSIM_MSG_LIMIT, i < nrepl_buy ? 0 : 1, r.x, r.y, 0u, true);
  }
  __syncwarp();
  if (lane == 0) {
    const int n0 = fb.cnt(0)->x, n1 = fb.cnt(1)->x;
    if (n0 && fb.P(fb.side(0))[0] < h->min_buy) h->min_buy = fb.P(fb.side(0))[0];
    if (n1 && fb.P(fb.side(1))[0] > h->max_sell) h->max_sell = fb.P(fb.side(1))[0];
  }
  __syncwarp();
  fast_refresh_best(fb, f);
}

// the replay form: a packed historical message.  The common cases run in fast_order (no call); the rare ones (level
// beyond the 32 best, queue longer than 32, shift longer than 64, remainder of a crossing limit order) in the any-depth routines.
template <class LT>
__device__ __forceinline__ void fast_message(const FastBook<LT>& fb, FastState& f, int price, int vol, uint32_t ref, uint32_t meta) {
  fast_order_full<LT, false>(fb, f, (int)(meta & 7u), (int)((meta >> 3) & 1u), price, vol, ref, false);
}
