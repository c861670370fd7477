// book_flat.cuh -- the FLAT book: a side is an unordered pool of resting orders
//
//     pool[s][i] = { price, ref, volume, seq }      i < n[s] <= FLAT_CAP, 16 bytes per order, no gaps
//
// with NO level structure at all.  It is the reference's `SortedDict[price -> deque[LimitOrder]]` (rl4mm/orderbook/models.py:64-69)
// for books that are small enough that a few warp-wide compares see every resting order of a side (BASELINE config 2: 8-12
// levels and 30-55 orders per side; configs 3 / 4 with the agent's ladders: 60-100):
//   * price-time priority is carried by `seq`, a per-book counter stamped when an order starts resting (Exchange.py:78-83 appends
//     to the level's deque): the head of a level = the order with the smallest seq at that price (one REDUX.MIN);
//   * a new order is ONE 16-byte store at pool[n] (no level search, no level insert, no queue shift, no prefix-end update);
//   * a cancellation / deletion finds (price, ref) with one 8-byte load per lane and 32-order chunk + ballots and fills the hole
//     with the last order (one load + one store) -- Exchange.remove_order / _find_queue_position, Exchange.py:122-147,196-217;
//   * the best price of a side lives in a register and is recomputed (REDUX.MAX / MIN over the prices already in registers)
//     only when the last order at the best price leaves.
// 69 warp instructions per message against 110 for the sorted level arrays of book_fast.cuh (profiles/r02_replay_ab.md).
//
// FLAT_CAP = 32 * NCH orders per side, NCH = 2 or 4 chunks by the handle's capacities (flat_nch<LT>): a flat side may hold
// FLAT_CAP distinct prices, so the sorted layout must have room for as many levels, and the pool lives in the side's order array.
//
// The flat form is the replay's (k_replay_flat, kernels.cuh).  A book is flat or sorted PER BOOK: in shared memory during a launch,
// and in HBM between launches (header marker, kernels.cuh), so that consecutive replay launches do not convert every book twice each.
// Conversions: flat_enter (sorted -> flat: trivial, seq = position in the sorted order array) when a book fits with some slack;
// flat_leave (flat -> sorted: rank-by-counting sort on (price, seq)) when a pool is full, when update_outer_levels
// (OrderbookSimulator.py:105-135) really has a level to overwrite (leave -> resync on the sorted form -> enter), on load by the env
// and hybrid replay kernels, and by k_to_sorted before anything else reads a book.
#pragma once
#include "book_fast.cuh"

struct FlatState {
  int n0, n1;      // resting orders per side
  uint32_t seq;    // next time-priority stamp
};

// chunks of 32 orders per side that the flat form of this layout may use
template <class LT>
__host__ __device__ constexpr int flat_nch() { return (LT::NL >= 128 && LT::NO >= 256) ? 4 : 2; }
template <class LT>
__host__ __device__ constexpr int flat_cap() { return 32 * flat_nch<LT>(); }

template <class LT>
__device__ __forceinline__ uint4* flat_pool(unsigned char* blob, int s) {
  static_assert(LT::NO * 8 >= flat_cap<LT>() * 16, "the flat pool (FLAT_CAP x 16 B) lives in the order array of the side");
  static_assert(LT::NO * 8 >= flat_cap<LT>() * 12, "flat_leave: sorted orders (8 B) + one price per order (4 B) in the order array");
  static_assert(LT::NL >= flat_cap<LT>(), "a flat side may hold FLAT_CAP distinct prices");
  static_assert(LT::ord_off % 16 == 0 && LT::side_stride % 16 == 0 && LT::side_off % 16 == 0, "16-byte aligned pool");
  return reinterpret_cast<uint4*>(blob + LT::side_off + s * LT::side_stride + LT::ord_off);
}

// (price, ref) of every order of a side, one order per lane and chunk; lanes beyond n: a ref that no resting order has
template <int NCH>
__device__ __forceinline__ void flat_keys(const uint4* pool, int n, int lane, uint2 (&k)[NCH]) {
#pragma unroll
  for (int c = 0; c < NCH; c++) {
    k[c] = make_uint2(0u, 0xffffffffu);
    if (c * 32 + lane < n) k[c] = *reinterpret_cast<const uint2*>(&pool[c * 32 + lane]);
  }
}
// the same without the sentinel: every lane loads its slot (always inside the pool, CAP = 32 x NCH), slots beyond n hold stale
// orders -- every use must test `c * 32 + lane < n` itself (saves the per-search register initialisation)
template <int NCH>
__device__ __forceinline__ void flat_keys_raw(const uint4* pool, int lane, uint2 (&k)[NCH]) {
#pragma unroll
  for (int c = 0; c < NCH; c++) k[c] = *reinterpret_cast<const uint2*>(&pool[c * 32 + lane]);
}
// first set bit of a per-chunk ballot array -> order index (the array is not all zero)
template <int NCH>
__device__ __forceinline__ int flat_first(const unsigned (&m)[NCH]) {
  int i = 0;
#pragma unroll
  for (int c = NCH - 1; c >= 0; c--) if (m[c]) i = c * 32 + __ffs(m[c]) - 1;
  return i;
}
// best price of side S over the keys in registers, leaving out order `skip` (-1: none)
template <int S, int NCH>
__device__ __forceinline__ int flat_best_of(const uint2 (&k)[NCH], int n, int lane, int skip) {
  int b = S ? INT32_MAX : INT32_MIN;
#pragma unroll
  for (int c = 0; c < NCH; c++) {
    const int i = c * 32 + lane;
    if (i < n && i != skip) b = S ? min(b, (int)k[c].x) : max(b, (int)k[c].x);
  }
  return S ? __reduce_min_sync(FULL_MASK, b) : __reduce_max_sync(FULL_MASK, b);
}
template <class LT, int S>
__device__ __forceinline__ int flat_best_scan(unsigned char* blob, int lane, int n) {
  uint2 k[flat_nch<LT>()];
  flat_keys(flat_pool<LT>(blob, S), n, lane, k);
  return flat_best_of<S>(k, n, lane, -1);
}

// One historical order of side S (0 buy, 1 sell) through the flat book.  Same results as fast_order_full<LT,false> on the sorted book:
// a replay book holds no agent orders, so nothing is tracked.
// Sets f.bail = FLAT_BAIL_FULL -- with the book untouched -- when the order may have to rest and the pool of its side is full: the
// caller converts the book to the sorted form and runs the order there.  Returns true when the caller's message loop has to stop
// (f.bail or f.dead set) -- a constant per return site, so the compiler threads the rare exits straight out of the loop and the
// common paths carry no status register.
#define FLAT_BAIL_FULL 3
template <class LT, int S, bool VCHK = true>
__device__ __forceinline__ bool flat_order(unsigned char* blob, int lane, FastState& f, FlatState& st, int type, int price, int vol, uint32_t ref) {
  constexpr int OPP = S ^ 1;
  constexpr int NCH = flat_nch<LT>();
  int& n_own = S ? st.n1 : st.n0;
  int& n_opp = S ? st.n0 : st.n1;
  int& best_own = S ? f.best1 : f.best0;
  int& best_opp = S ? f.best0 : f.best1;
  uint4* own = flat_pool<LT>(blob, S);
  uint4* opp = flat_pool<LT>(blob, OPP);
  if (VCHK && __builtin_expect(vol <= 0, 0)) { f.err |= LOBSIM_ERR_BAD_VOLUME; return false; }   // assert order.volume > 0, Exchange.py:59-60
  // (!VCHK: the caller has checked the volume)
  // Pool stores: every lane stores the same value to the same address, so each lane's own later loads see it whatever the other
  // lanes do, and the paths need no barrier (control flow is warp-uniform: every value it depends on is the same in all lanes).
  // ---- the order rests at the back of its price's queue (Exchange.py:74-83) --------------------------------------------
  auto rest = [&](int rem) -> bool {
    own[n_own] = make_uint4((unsigned)price, ref, (unsigned)rem, st.seq);
    n_own += 1; st.seq += 1;
    if (S ? price < best_own : price > best_own) best_own = price;
    return false;
  };
  auto remove = [&]() -> bool {
    // ---- cancellation / deletion (Exchange.py:122-147) ----------------------------------------------------------------------
    uint2 k[NCH];
    flat_keys_raw(own, lane, k);
    // (price, ref) names at most one resting order: the lane that holds it announces its index (one warp reduction)
    int mine = -1;
#pragma unroll
    for (int c = 0; c < NCH; c++) if (c * 32 + lane < n_own && (int)k[c].x == price && k[c].y == ref) mine = c * 32 + lane;
    int i = __reduce_max_sync(FULL_MASK, mine);
    if (i < 0) {
      // unknown id: the level's snapshot aggregate (internal_id -1, always the head of its level) takes the hit (:133-137);
      // no such level, or no aggregate left at it: nothing happens (:129-132,138-139)
      mine = INT32_MAX;
#pragma unroll
      for (int c = NCH - 1; c >= 0; c--) if (c * 32 + lane < n_own && (int)k[c].x == price && k[c].y == LOBSIM_REF_AGGREGATE) mine = c * 32 + lane;
      i = __reduce_min_sync(FULL_MASK, mine);
      if (i == INT32_MAX) return false;
    }
    const int cur = (int)own[i].z;
    if (vol < cur) {                                                         // partial: reduce in place
      own[i].z = (unsigned)(cur - vol);
      return false;
    }
    // full removal (over-size requests remove the resting volume, :142-146): the last order of the pool fills the hole
    if (price == best_own) best_own = flat_best_of<S>(k, n_own, lane, i);
    own[i] = own[n_own - 1];
    n_own -= 1;
    return false;
  };
  // dispatch, the common cases first: a limit order that neither crosses nor finds the pool full, then cancellations / deletions.
  // (The second test reads an opaque copy of `type`: two plain tests of one variable become a jump table -- LDC + BRX, measured
  // 8 % slower than the two compares.)
  int type2 = type;
  asm volatile("" : "+r"(type2));
  if (__builtin_expect(type == LOBSIM_MSG_LIMIT, 1)) {                     // (the previous order's stores are visible: above)
    const bool crosses = S ? price <= best_opp : price >= best_opp;        // empty opposite side: INT32_MIN / INT32_MAX
    if (__builtin_expect(!crosses & (n_own < flat_cap<LT>()), 1)) return rest(vol);   // (one branch for the common case)
    if (n_own >= flat_cap<LT>()) { f.bail = FLAT_BAIL_FULL; return true; }
  } else if (type2 != LOBSIM_MSG_MARKET) return remove();
  {
    int rem = vol;
    {
      // ---- execution against the opposite side, best price first, oldest order first (Exchange.py:85-120) -------------
#pragma unroll 1
      while (rem > 0) {
        if (n_opp == 0) {
          if (type == LOBSIM_MSG_MARKET) { f.err |= LOBSIM_ERR_EMPTY_BOOK; f.dead = 1; return true; }   // EmptyOrderbookError :183-186
          break;
        }
        const int bp = best_opp;
        if (type == LOBSIM_MSG_LIMIT && !(S ? price <= bp : price >= bp)) break;
        unsigned q[NCH], qmin = 0xffffffffu;                                // seq of the orders at the best price, ~0 elsewhere
#pragma unroll
        for (int c = 0; c < NCH; c++) {
          q[c] = 0xffffffffu;
          if (c * 32 + lane < n_opp) { const uint4 e = opp[c * 32 + lane]; if ((int)e.x == bp) q[c] = e.w; }
          qmin = min(qmin, q[c]);
        }
        const unsigned head_seq = __reduce_min_sync(FULL_MASK, qmin);
        int at_best = 0, head = -1;                                         // seq is unique: the head's lane announces its index
#pragma unroll
        for (int c = 0; c < NCH; c++) {
          if (q[c] == head_seq) head = c * 32 + lane;
          at_best += __popc(__ballot_sync(FULL_MASK, q[c] != 0xffffffffu));
        }
        const int i = __reduce_max_sync(FULL_MASK, head);                                       // the head of the best queue
        const int hv = (int)opp[i].z;
        if (rem < hv) {                                                    // partial fill of the head
          opp[i].z = (unsigned)(hv - rem);
          rem = 0;
          break;
        }
        rem -= hv;                                                         // the head is consumed
        if (at_best == 1) {                                                // the level emptied: next best price
          uint2 k[NCH];
          flat_keys(opp, n_opp, lane, k);
          best_opp = flat_best_of<OPP>(k, n_opp, lane, i);
        }
        opp[i] = opp[n_opp - 1];
        n_opp -= 1;
      }
    }
    if (!(rem > 0 && type == LOBSIM_MSG_LIMIT)) return false;
    return rest(rem);                                                       // the remainder of a crossing limit order rests (:116-119)
  }
  return remove();
}

// the replay form: a packed historical message
// (VCHK = false: the caller has looked at the volumes of the whole message tile at once)
template <class LT, bool VCHK = true>
__device__ __forceinline__ bool flat_message(unsigned char* blob, int lane, FastState& f, FlatState& st, int price, int vol, uint32_t ref, uint32_t meta) {
  const int type = (int)(meta & 7u);
  if (meta & 8u) return flat_order<LT, 1, VCHK>(blob, lane, f, st, type, price, vol, ref);
  return flat_order<LT, 0, VCHK>(blob, lane, f, st, type, price, vol, ref);
}

// ---- sorted -> flat (kernel entry, after a reset / resync, when a book has shrunk) ----------------------------------------------
template <class LT>
__device__ __forceinline__ bool flat_fits(const FastBook<LT>& fb, int slack) {
  return fb.cnt(0)->y <= flat_cap<LT>() - slack && fb.cnt(1)->y <= flat_cap<LT>() - slack;
}
// precondition: flat_fits(fb, 0).  Returns {n0, n1}; seq restarts at FLAT_CAP (above every position stamp).
template <class LT>
static __device__ __noinline__ int2 flat_enter_fn(unsigned char* blob, int lane) {
  constexpr int NCH = flat_nch<LT>();
  FastBook<LT> fb; fb.blob = blob; fb.lane = lane;
  int2 out = make_int2(0, 0);
  __syncwarp();
#pragma unroll 1
  for (int s = 0; s < 2; s++) {
    unsigned char* sb = fb.side(s);
    const int2 c = *fb.cnt(s);
    const int nlv = c.x, n = c.y;
    uint2 o[NCH]; int pr[NCH];
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      const int i = ch * 32 + lane;
      o[ch] = make_uint2(0u, 0u); pr[ch] = 0;
      if (i < n) {
        o[ch] = fb.O(sb)[i];
        int lo = 0, hi = nlv - 1;                 // the level of order i = the first level whose end offset is beyond i
#pragma unroll 1
        while (lo < hi) { const int mid = (lo + hi) >> 1; if ((int)fb.LE(sb)[mid] > i) hi = mid; else lo = mid + 1; }
        pr[ch] = fb.P(sb)[lo];
      }
    }
    __syncwarp();                                                           // the pool overlays the order array
    uint4* pool = flat_pool<LT>(blob, s);
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      const int i = ch * 32 + lane;
      if (i < n) pool[i] = make_uint4((unsigned)pr[ch], o[ch].y, o[ch].x, (unsigned)i);
    }
    if (s) out.y = n; else out.x = n;
  }
  __syncwarp();
  return out;
}
template <class LT>
__device__ __forceinline__ void flat_enter(const FastBook<LT>& fb, FlatState& st) {
  const int2 n = flat_enter_fn<LT>(fb.blob, fb.lane);
  st.n0 = n.x; st.n1 = n.y; st.seq = (uint32_t)flat_cap<LT>();
}

// ---- flat -> sorted: rank every order by (price worst -> best, seq), scatter, rebuild the level prices / ends ---------------
template <class LT>
static __device__ __noinline__ void flat_leave_fn(unsigned char* blob, int lane, int n0, int n1) {
  constexpr int NCH = flat_nch<LT>();
  FastBook<LT> fb; fb.blob = blob; fb.lane = lane;
  __syncwarp();
#pragma unroll 1
  for (int s = 0; s < 2; s++) {
    unsigned char* sb = fb.side(s);
    const uint4* pool = flat_pool<LT>(blob, s);
    const int n = s ? n1 : n0;
    const unsigned flip = s ? 0xffffffffu : 0u;                             // ascending key = worst -> best price, then oldest first
    uint4 e[NCH]; unsigned long long k[NCH]; int r[NCH];
#pragma unroll
    for (int c = 0; c < NCH; c++) {
      e[c] = make_uint4(0u, 0u, 0u, 0u);
      if (c * 32 + lane < n) e[c] = pool[c * 32 + lane];
      k[c] = ((unsigned long long)((e[c].x ^ 0x80000000u) ^ flip) << 32) | e[c].w;
      r[c] = 0;
    }
#pragma unroll 1
    for (int m = 0; m < n; m++) {
      const uint4 em = pool[m];
      const unsigned long long km = ((unsigned long long)((em.x ^ 0x80000000u) ^ flip) << 32) | em.w;
#pragma unroll
      for (int c = 0; c < NCH; c++) r[c] += km < k[c] ? 1 : 0;
    }
    __syncwarp();                                                           // every lane holds its orders: the arrays can be rewritten
    int32_t* tmp = reinterpret_cast<int32_t*>(fb.O(sb) + flat_cap<LT>());     // one sorted price per ORDER, behind the sorted orders
#pragma unroll
    for (int c = 0; c < NCH; c++)
      if (c * 32 + lane < n) { fb.O(sb)[r[c]] = make_uint2(e[c].z, e[c].y); tmp[r[c]] = (int)e[c].x; }
    __syncwarp();
    int t[NCH]; unsigned nb[NCH + 1]; int below = 0;
#pragma unroll
    for (int c = 0; c < NCH; c++) {
      const int i = c * 32 + lane;
      t[c] = 0; int pv = 0;
      if (i < n) t[c] = tmp[i];
      if (i > 0 && i < n) pv = tmp[i - 1];
      nb[c] = __ballot_sync(FULL_MASK, i < n && (i == 0 || t[c] != pv));   // first order of a level
    }
    nb[NCH] = 0;
    const unsigned le_mask = 0xffffffffu >> (31 - lane);                    // lanes <= this lane
#pragma unroll
    for (int c = 0; c < NCH; c++) {
      const int i = c * 32 + lane;
      const int lvl = below + __popc(nb[c] & le_mask) - 1;
      const bool is_new = (nb[c] >> lane) & 1u;
      // last order of a level: the next order starts a new level, or there is no next order
      const bool next_new = lane == 31 ? (nb[c + 1] & 1u) != 0 : ((nb[c] >> (lane + 1)) & 1u) != 0;
      if (is_new) fb.P(sb)[lvl] = t[c];
      if (i < n && (i == n - 1 || next_new)) fb.LE(sb)[lvl] = (uint16_t)(i + 1);
      below += __popc(nb[c]);
    }
    if (lane == 0) *fb.cnt(s) = make_int2(below, n);
    __syncwarp();
  }
}
template <class LT>
__device__ __forceinline__ void flat_leave(const FastBook<LT>& fb, const FlatState& st) { flat_leave_fn<LT>(fb.blob, fb.lane, st.n0, st.n1); }

// does the snapshot row of this second hold a level beyond the tracked price range (OrderbookSimulator.py:99-103,113-115)?
__device__ __forceinline__ bool flat_resync_needed(const BookHdr* h, const int32_t* __restrict__ row, int L, int lane) {
  const int min_buy = h->min_buy, max_sell = h->max_sell;
  unsigned any = 0;
  for (int base = 0; base < 2 * L; base += 32) {
    const int idx = base + lane;
    int price = LOBSIM_NO_PRICE;
    if (idx < 2 * L) price = __ldg(&row[idx * 2]);
    any |= __ballot_sync(FULL_MASK, price != LOBSIM_NO_PRICE && (idx < L ? price < min_buy : price > max_sell));
  }
  return any != 0;
}
// the price-range trackers when no level is overwritten (OrderbookSimulator.py:134-135): worst resting price of each side
template <class LT>
__device__ __forceinline__ void flat_update_trackers(unsigned char* blob, int lane, const FlatState& st) {
  BookHdr* h = reinterpret_cast<BookHdr*>(blob);
  __syncwarp();
  uint2 k[flat_nch<LT>()];
  flat_keys(flat_pool<LT>(blob, 0), st.n0, lane, k);
  const int w0 = flat_best_of<1>(k, st.n0, lane, -1);                     // lowest bid
  flat_keys(flat_pool<LT>(blob, 1), st.n1, lane, k);
  const int w1 = flat_best_of<0>(k, st.n1, lane, -1);                     // highest ask
  if (lane == 0) {
    if (st.n0 && w0 < h->min_buy) h->min_buy = w0;
    if (st.n1 && w1 > h->max_sell) h->max_sell = w1;
  }
  __syncwarp();
}
