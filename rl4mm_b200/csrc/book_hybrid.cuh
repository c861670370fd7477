// book_hybrid.cuh -- the HYBRID book of the replay kernel for deep books: flat near the touch, sorted beyond.
//
// The flat order pools of book_flat.cuh are the cheapest structure when a warp can look at every resting order of a side at once
// (<= 128 orders); a 50-level book with deep queues (BASELINE config 5: ~450-600 orders per side) does not fit, but its activity does:
// limit prices are placed geometrically from the best, executions only touch the best level.  So each side is split at a floor price:
//   HOT  -- every order at or better than the floor: an unordered pool of <= HYB_CAP (128) orders {price, ref, volume, seq}
//           (exactly book_flat.cuh: ~60 instructions per message, no level structure);
//   COLD -- everything worse than the floor: the sorted level arrays of book.cuh / book_fast.cuh, worst -> best, so that the level
//           next to the floor is the LAST one -- moving a whole level across the floor costs no shift at all:
//             hot -> cold (pool full): the worst hot level, ranked by seq, is appended as the best cold level;
//             cold -> hot (pool empty / low): the best cold level is popped off the end and stamped with fresh seq.
// A level is hot or cold as a whole, so price-time priority inside it is never split.  The best price of a side is always hot
// (the pool is refilled the moment it runs empty), so the crossing test and executions are the flat ones.  Orders beyond the floor
// take the any-depth routines of book_fast.cuh on the cold arrays (what a deep book pays for most orders today).
// The pool lives in the LAST 2 KB of the side's order array (the cold part may use the first NO - 256 order slots); the blob in HBM is
// always the canonical sorted layout: hyb_enter peels levels off the end, hyb_leave sorts the pool (<= 128 orders) and appends it.
// What cannot be represented (a single level longer than the pool at the touch, a cold part beyond NO - 256 orders) hands the book --
// and the unfinished part of the order, if any -- to the sorted path of the same kernel.
#pragma once
#include "book_flat.cuh"

#ifndef HYB_COLD_ATTR
#define HYB_COLD_ATTR __forceinline__   // the cold-array routines: inline (measured: 3.47e9 msgs/s vs 2.75e9 out of line, BASELINE config 5)
#endif
#ifndef HYB_REFILL_ATTR
#define HYB_REFILL_ATTR __noinline__    // the level moves: out of line (inline: 2.71e9)
#endif
#ifndef HYB_SPILL_ATTR
#define HYB_SPILL_ATTR __noinline__
#endif
#define HYB_CAP 128
#define HYB_NCH 4
#define HYB_BAIL_DONE 4          // leave the hybrid form; the order itself is complete
#ifndef HYB_REFILL_BELOW
#define HYB_REFILL_BELOW 96      // refill the pool from the cold levels at step boundaries when it holds fewer orders than this
                                 // (measured on BASELINE config 5: 16/64 3.39e9, 32/80 3.48e9, 96/120 3.65e9 msgs/s)
#endif
#ifndef HYB_REFILL_TO
#define HYB_REFILL_TO 120
#endif

template <class LT>
__host__ __device__ constexpr bool hyb_layout() { return LT::NO >= 512 && LT::NL >= 64; }
template <class LT>
__host__ __device__ constexpr int hyb_cold_max() { return LT::NO - 2 * HYB_CAP; }     // order slots left to the cold part

template <class LT>
__device__ __forceinline__ uint4* hyb_pool(unsigned char* blob, int s) {
  static_assert(LT::ord_off % 16 == 0 && LT::side_stride % 16 == 0 && (LT::NO * 8) % 16 == 0, "16-byte aligned pool");
  return reinterpret_cast<uint4*>(blob + LT::side_off + s * LT::side_stride + LT::ord_off + LT::NO * 8 - HYB_CAP * 16);
}

struct HybState {
  int n0, n1;          // orders in the pools
  int floor0, floor1;  // bids at or above floor0 / asks at or below floor1 are hot (INT32_MIN / INT32_MAX: the whole side)
  uint32_t seq;
};

// ---- cold -> hot: the best cold level moves into the pool (if the pool has room).  Keeps f.best of the side current. ----------
// (out of line: called from half a dozen places of hyb_order, rarely)   returns {orders moved or -1, the level's price}
template <class LT, int S>
static __device__ HYB_REFILL_ATTR int2 hyb_refill_fn(unsigned char* blob, int lane, int n, unsigned seq) {
  FastBook<LT> fb; fb.blob = blob; fb.lane = lane;
  unsigned char* sb = fb.side(S);
  __syncwarp();
  const int2 c = *fb.cnt(S);
  if (c.x == 0) return make_int2(-1, 0);
  const int j = c.x - 1;
  const int start = j > 0 ? (int)fb.LE(sb)[j - 1] : 0, len = c.y - start;
  if (n + len > HYB_CAP) return make_int2(-1, 0);
  const int price = fb.P(sb)[j];
  uint4* pool = hyb_pool<LT>(blob, S);
  for (int i = lane; i < len; i += 32) {
    const uint2 o = fb.O(sb)[start + i];
    pool[n + i] = make_uint4((unsigned)price, o.y, o.x, seq + (unsigned)i);
  }
  __syncwarp();
  if (lane == 0) *fb.cnt(S) = make_int2(c.x - 1, start);
  __syncwarp();
  return make_int2(len, price);
}
template <class LT, int S>
__device__ __forceinline__ bool hyb_refill_one(const FastBook<LT>& fb, FastState& f, HybState& hs) {
  int& n = S ? hs.n1 : hs.n0;
  int& floor_ = S ? hs.floor1 : hs.floor0;
  int& best = S ? f.best1 : f.best0;
  const int2 r = hyb_refill_fn<LT, S>(fb.blob, fb.lane, n, hs.seq);
  if (r.x < 0) return false;
  if (n == 0) best = r.y;                                    // (otherwise the level is worse than everything hot)
  hs.seq += (unsigned)r.x; n += r.x;
  floor_ = fb.cnt(S)->x > 0 ? r.y : (S ? INT32_MAX : INT32_MIN);   // nothing cold left: the whole side is hot
  return true;
}

// the any-depth routines of book_fast.cuh on the cold arrays, out of line (one copy for both sides); return the error bits
template <class LT>
static __device__ HYB_COLD_ATTR uint32_t hyb_cold_rest_fn(unsigned char* blob, int lane, int side, int price, int vol, uint32_t ref) {
  FastBook<LT> fb; fb.blob = blob; fb.lane = lane;
  FastState t; t.err = 0; t.dead = 0; t.bail = 0; t.bail_vol = 0; t.best0 = t.best1 = 0;
  fast_rest_any<LT, false>(fb, t, side, price, vol, ref, false);
  return t.err;
}
template <class LT>
static __device__ HYB_COLD_ATTR uint32_t hyb_cold_remove_fn(unsigned char* blob, int lane, int side, int price, int vol, uint32_t ref) {
  FastBook<LT> fb; fb.blob = blob; fb.lane = lane;
  FastState t; t.err = 0; t.dead = 0; t.bail = 0; t.bail_vol = 0; t.best0 = t.best1 = 0;
  fast_remove_any<LT, false>(fb, t, side, price, vol, ref, false);
  return t.err;
}

// ---- hot -> cold: the worst hot level, in time priority, becomes the best cold level.  false: no room in the cold arrays. --------
template <class LT, int S>
static __device__ HYB_SPILL_ATTR int hyb_spill_fn(unsigned char* blob, int lane, int n) {   // returns the new pool size, or -1
  FastBook<LT> fb; fb.blob = blob; fb.lane = lane;
  unsigned char* sb = fb.side(S);
  uint4* pool = hyb_pool<LT>(blob, S);
  __syncwarp();
  uint4 e[HYB_NCH]; uint2 k[HYB_NCH];
#pragma unroll
  for (int c = 0; c < HYB_NCH; c++) {
    e[c] = make_uint4(0u, 0xffffffffu, 0u, 0xffffffffu);
    if (c * 32 + lane < n) e[c] = pool[c * 32 + lane];
    k[c] = make_uint2(e[c].x, e[c].y);
  }
  const int w = flat_best_of<S ^ 1>(k, n, lane, -1);        // the WORST hot price: lowest bid / highest ask
  unsigned mk[HYB_NCH]; int m = 0;
#pragma unroll
  for (int c = 0; c < HYB_NCH; c++) { mk[c] = __ballot_sync(FULL_MASK, c * 32 + lane < n && (int)e[c].x == w); m += __popc(mk[c]); }
  const int2 cc = *fb.cnt(S);
  if (cc.y + m > hyb_cold_max<LT>() || cc.x >= LT::NL) return -1;
  // rank of every member among the members by seq (queue order), new index of every other order (compaction)
  int r[HYB_NCH], keep_before = 0, ni[HYB_NCH];
#pragma unroll
  for (int c = 0; c < HYB_NCH; c++) r[c] = 0;
#pragma unroll
  for (int c2 = 0; c2 < HYB_NCH; c2++) {
    unsigned bits = mk[c2];
    while (bits) {
      const int src = __ffs(bits) - 1;
      bits &= bits - 1;
      const unsigned sq = __shfl_sync(FULL_MASK, e[c2].w, src);
#pragma unroll
      for (int c = 0; c < HYB_NCH; c++) r[c] += sq < e[c].w ? 1 : 0;
    }
  }
  const unsigned lt_mask = (1u << lane) - 1u;
#pragma unroll
  for (int c = 0; c < HYB_NCH; c++) {
    const unsigned valid = __ballot_sync(FULL_MASK, c * 32 + lane < n);
    const unsigned keep = valid & ~mk[c];
    ni[c] = keep_before + __popc(keep & lt_mask);
    keep_before += __popc(keep);
  }
  __syncwarp();
#pragma unroll
  for (int c = 0; c < HYB_NCH; c++) {
    if (c * 32 + lane < n) {
      if ((mk[c] >> lane) & 1u) fb.O(sb)[cc.y + r[c]] = make_uint2(e[c].z, e[c].y);
      else pool[ni[c]] = e[c];
    }
  }
  if (lane == 0) { fb.P(sb)[cc.x] = w; fb.LE(sb)[cc.x] = (uint16_t)(cc.y + m); *fb.cnt(S) = make_int2(cc.x + 1, cc.y + m); }
  __syncwarp();
  return n - m;
}
template <class LT, int S>
__device__ __forceinline__ bool hyb_spill_one(const FastBook<LT>& fb, HybState& hs) {
  int& n = S ? hs.n1 : hs.n0;
  int& floor_ = S ? hs.floor1 : hs.floor0;
  const int before = fb.cnt(S)->x;
  const int nn = hyb_spill_fn<LT, S>(fb.blob, fb.lane, n);
  if (nn < 0) return false;
  n = nn;
  const int w = FastBook<LT>::P(fb.side(S))[before];        // the price that just went cold
  floor_ = S ? w - 1 : w + 1;                                // everything at or beyond it is cold now
  return true;
}

// ---- sorted -> hybrid: peel the best levels off the end of the sorted arrays into the pool ----------------------------------------
// false: the book cannot be hybrid (too many orders for the cold part, or the best level alone is longer than the pool)
template <class LT>
__device__ __forceinline__ bool hyb_enter(const FastBook<LT>& fb, FastState& f, HybState& hs) {
  if (fb.cnt(0)->y > hyb_cold_max<LT>() || fb.cnt(1)->y > hyb_cold_max<LT>()) return false;
  hs.n0 = hs.n1 = 0; hs.seq = 0;
  hs.floor0 = fb.cnt(0)->x ? INT32_MAX : INT32_MIN;          // everything cold to begin with (an empty side: everything hot)
  hs.floor1 = fb.cnt(1)->x ? INT32_MIN : INT32_MAX;
  while (hs.n0 < HYB_REFILL_TO && hyb_refill_one<LT, 0>(fb, f, hs)) {}
  while (hs.n1 < HYB_REFILL_TO && hyb_refill_one<LT, 1>(fb, f, hs)) {}
  const bool ok = (hs.n0 > 0 || fb.cnt(0)->x == 0) && (hs.n1 > 0 || fb.cnt(1)->x == 0);
  return ok;                                                 // (!ok: nothing was moved on that side; whatever the other side moved is
}                                                            //  put back by the caller's hyb_leave)

// ---- hybrid -> sorted: the pool, sorted by (price worst -> best, seq), is appended behind the cold levels ---------------------------
template <class LT>
static __device__ __noinline__ uint32_t hyb_leave_fn(unsigned char* blob, int lane, int n0, int n1) {
  FastBook<LT> fb; fb.blob = blob; fb.lane = lane;
  uint32_t err = 0;
  __syncwarp();
#pragma unroll 1
  for (int s = 0; s < 2; s++) {
    unsigned char* sb = fb.side(s);
    const uint4* pool = hyb_pool<LT>(blob, s);
    const int n = s ? n1 : n0;
    if (n == 0) continue;
    const int2 cc = *fb.cnt(s);
    const unsigned flip = s ? 0xffffffffu : 0u;
    uint4 e[HYB_NCH]; unsigned long long k[HYB_NCH]; int r[HYB_NCH];
#pragma unroll
    for (int c = 0; c < HYB_NCH; c++) {
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
      for (int c = 0; c < HYB_NCH; c++) r[c] += km < k[c] ? 1 : 0;
    }
    __syncwarp();                                            // every lane holds its orders: the pool region can be rewritten
    int32_t* tmp = reinterpret_cast<int32_t*>(sb + LT::ord_off + LT::NO * 8 - HYB_CAP * 4);   // one sorted price per hot ORDER
#pragma unroll
    for (int c = 0; c < HYB_NCH; c++)
      if (c * 32 + lane < n) { fb.O(sb)[cc.y + r[c]] = make_uint2(e[c].z, e[c].y); tmp[r[c]] = (int)e[c].x; }
    __syncwarp();
    int t[HYB_NCH]; unsigned nb[HYB_NCH + 1]; int below = 0;
#pragma unroll
    for (int c = 0; c < HYB_NCH; c++) {
      const int i = c * 32 + lane;
      t[c] = 0; int pv = 0;
      if (i < n) t[c] = tmp[i];
      if (i > 0 && i < n) pv = tmp[i - 1];
      nb[c] = __ballot_sync(FULL_MASK, i < n && (i == 0 || t[c] != pv));
    }
    nb[HYB_NCH] = 0;
    int n_new = 0;
#pragma unroll
    for (int c = 0; c < HYB_NCH; c++) n_new += __popc(nb[c]);
    if (cc.x + n_new > LT::NL) { err |= LOBSIM_ERR_LEVEL_OVERFLOW; n_new = LT::NL - cc.x; }   // capacity of the sorted form
    const unsigned le_mask = 0xffffffffu >> (31 - lane);
#pragma unroll
    for (int c = 0; c < HYB_NCH; c++) {
      const int i = c * 32 + lane;
      const int lvl = below + __popc(nb[c] & le_mask) - 1;
      const bool is_new = (nb[c] >> lane) & 1u;
      const bool next_new = lane == 31 ? (nb[c + 1] & 1u) != 0 : ((nb[c] >> (lane + 1)) & 1u) != 0;
      if (lvl < n_new) {
        if (is_new) fb.P(sb)[cc.x + lvl] = t[c];
        if (i < n && (i == n - 1 || next_new)) fb.LE(sb)[cc.x + lvl] = (uint16_t)(cc.y + i + 1);
      }
      below += __popc(nb[c]);
    }
    if (lane == 0) *fb.cnt(s) = make_int2(cc.x + n_new, cc.y + n);
    __syncwarp();
  }
  return err;
}
template <class LT>
__device__ __forceinline__ void hyb_leave(const FastBook<LT>& fb, FastState& f, const HybState& hs) {
  f.err |= hyb_leave_fn<LT>(fb.blob, fb.lane, hs.n0, hs.n1);
  fast_refresh_best(fb, f);
}

// ---- one historical message through the hybrid book (results == fast_order_full<LT,false> on the sorted book) -----------------
// Returns true when the message loop has to stop (f.bail or f.dead set; a constant per return site, as in flat_order).
// f.bail = FLAT_BAIL_FULL: leave the hybrid form and run a (type, side, price, f.bail_vol, ref) order on the sorted book (the
// unfinished part of this one); f.bail = HYB_BAIL_DONE: leave the hybrid form, the order is complete.
template <class LT, int S>
__device__ __forceinline__ bool hyb_order(const FastBook<LT>& fb, FastState& f, HybState& hs, int type, int price, int vol, uint32_t ref) {
  constexpr int OPP = S ^ 1;
  const int lane = fb.lane;
  int& n_own = S ? hs.n1 : hs.n0;
  int& n_opp = S ? hs.n0 : hs.n1;
  int& best_own = S ? f.best1 : f.best0;
  int& best_opp = S ? f.best0 : f.best1;
  const int floor_own = S ? hs.floor1 : hs.floor0;
  uint4* own = hyb_pool<LT>(fb.blob, S);
  uint4* opp = hyb_pool<LT>(fb.blob, OPP);
  // (vol > 0: the caller looks at the volumes of a whole message segment at once and runs a segment with a bad one on the sorted book)
  __syncwarp();
  const bool hot = S ? price <= floor_own : price >= floor_own;
  if (type == LOBSIM_MSG_LIMIT || type == LOBSIM_MSG_MARKET) {
    int rem = vol;
    const bool crosses = S ? price <= best_opp : price >= best_opp;
    if (type == LOBSIM_MSG_MARKET || crosses) {
#pragma unroll 1
      while (rem > 0) {
        if (n_opp == 0) {                                     // pool empty: more levels beyond the floor?
          if (fb.cnt(OPP)->x == 0) {
            if (type == LOBSIM_MSG_MARKET) { f.err |= LOBSIM_ERR_EMPTY_BOOK; f.dead = 1; return true; }   // EmptyOrderbookError :183-186
            break;
          }
          if (!hyb_refill_one<LT, OPP>(fb, f, hs)) { f.bail = FLAT_BAIL_FULL; f.bail_vol = rem; return true; }   // a level longer than the pool
        }
        const int bp = best_opp;
        if (type == LOBSIM_MSG_LIMIT && !(S ? price <= bp : price >= bp)) break;
        unsigned q[HYB_NCH], qmin = 0xffffffffu;
#pragma unroll
        for (int c = 0; c < HYB_NCH; c++) {
          q[c] = 0xffffffffu;
          if (c * 32 + lane < n_opp) { const uint4 e = opp[c * 32 + lane]; if ((int)e.x == bp) q[c] = e.w; }
          qmin = min(qmin, q[c]);
        }
        const unsigned head_seq = __reduce_min_sync(FULL_MASK, qmin);
        int at_best = 0, head = -1;                                         // seq is unique: the head's lane announces its index
#pragma unroll
        for (int c = 0; c < HYB_NCH; c++) {
          if (q[c] == head_seq) head = c * 32 + lane;
          at_best += __popc(__ballot_sync(FULL_MASK, q[c] != 0xffffffffu));
        }
        const int i = __reduce_max_sync(FULL_MASK, head);
        const int hv = (int)opp[i].z;
        __syncwarp();
        if (rem < hv) {
          if (lane == 0) opp[i].z = (unsigned)(hv - rem);
          rem = 0;
          break;
        }
        rem -= hv;
        if (at_best == 1) {
          uint2 k[HYB_NCH];
          flat_keys(opp, n_opp, lane, k);
          best_opp = flat_best_of<OPP>(k, n_opp, lane, i);  // (sentinel when the pool runs empty: refilled at the loop top / below)
        }
        __syncwarp();
        if (lane == 0) opp[i] = opp[n_opp - 1];
        n_opp -= 1;
        __syncwarp();
      }
      if (n_opp == 0 && fb.cnt(OPP)->x != 0) {     // keep the best price of the side in the pool
        if (!hyb_refill_one<LT, OPP>(fb, f, hs)) {
          if (rem > 0 && type == LOBSIM_MSG_LIMIT) { f.bail = FLAT_BAIL_FULL; f.bail_vol = rem; }   // the remainder rests on the sorted book
          else f.bail = HYB_BAIL_DONE;
          return true;
        }
      }
      if (!(rem > 0 && type == LOBSIM_MSG_LIMIT)) return false;
      // the remainder of a crossing limit order rests: it is the new best of its side => hot
    } else if (!hot) {
      // ---- beyond the floor: the any-depth routine on the cold arrays ------------------------------------------------------
      if (fb.cnt(S)->y >= hyb_cold_max<LT>()) { f.bail = FLAT_BAIL_FULL; f.bail_vol = rem; return true; }
      f.err |= hyb_cold_rest_fn<LT>(fb.blob, lane, S, price, rem, ref);
      if (n_own == 0) { if (!hyb_refill_one<LT, S>(fb, f, hs)) { f.bail = HYB_BAIL_DONE; return true; } }   // (the side was empty: its best must be hot)
      return false;
    }
    if (n_own >= HYB_CAP && !hyb_spill_one<LT, S>(fb, hs)) { f.bail = FLAT_BAIL_FULL; f.bail_vol = rem; return true; }
    const int floor_now = S ? hs.floor1 : hs.floor0;          // the spill may have moved the floor past this price
    if (!(S ? price <= floor_now : price >= floor_now)) {
      if (fb.cnt(S)->y >= hyb_cold_max<LT>()) { f.bail = FLAT_BAIL_FULL; f.bail_vol = rem; return true; }
      f.err |= hyb_cold_rest_fn<LT>(fb.blob, lane, S, price, rem, ref);
      if (n_own == 0) { if (!hyb_refill_one<LT, S>(fb, f, hs)) { f.bail = HYB_BAIL_DONE; return true; } }
      return false;
    }
    __syncwarp();
    if (lane == 0) own[n_own] = make_uint4((unsigned)price, ref, (unsigned)rem, hs.seq);
    n_own += 1; hs.seq += 1;
    if (S ? price < best_own : price > best_own) best_own = price;
    return false;
  }
  // ---- cancellation / deletion ---------------------------------------------------------------------------------------------
  if (!hot) {
    f.err |= hyb_cold_remove_fn<LT>(fb.blob, lane, S, price, vol, ref);
    return false;
  }
  uint2 k[HYB_NCH];
  flat_keys_raw(own, lane, k);                               // (slots beyond n_own are stale: every test below checks the index)
  int mine = -1;                                             // (price, ref) names at most one order: its lane announces the index
#pragma unroll
  for (int c = 0; c < HYB_NCH; c++) if (c * 32 + lane < n_own && (int)k[c].x == price && k[c].y == ref) mine = c * 32 + lane;
  int i = __reduce_max_sync(FULL_MASK, mine);
  if (i < 0) {                                               // unknown id: the level's snapshot aggregate, if it is still there
    mine = INT32_MAX;
#pragma unroll
    for (int c = HYB_NCH - 1; c >= 0; c--) if (c * 32 + lane < n_own && (int)k[c].x == price && k[c].y == LOBSIM_REF_AGGREGATE) mine = c * 32 + lane;
    i = __reduce_min_sync(FULL_MASK, mine);
    if (i == INT32_MAX) return false;
  }
  const int cur = (int)own[i].z;
  __syncwarp();
  if (vol < cur) { if (lane == 0) own[i].z = (unsigned)(cur - vol); return false; }
  if (price == best_own) best_own = flat_best_of<S>(k, n_own, lane, i);
  if (lane == 0) own[i] = own[n_own - 1];
  n_own -= 1;
  if (n_own == 0 && fb.cnt(S)->x != 0) { if (!hyb_refill_one<LT, S>(fb, f, hs)) { f.bail = HYB_BAIL_DONE; return true; } }
  return false;
}

template <class LT>
__device__ __forceinline__ bool hyb_message(const FastBook<LT>& fb, FastState& f, HybState& hs, int price, int vol, uint32_t ref, uint32_t meta) {
  const int type = (int)(meta & 7u);
  if (meta & 8u) return hyb_order<LT, 1>(fb, f, hs, type, price, vol, ref);
  return hyb_order<LT, 0>(fb, f, hs, type, price, vol, ref);
}
// step boundary: top the pools up from the cold levels when they run low (keeps most of the flow on the flat path)
template <class LT>
__device__ __forceinline__ void hyb_top_up(const FastBook<LT>& fb, FastState& f, HybState& hs) {
  if (hs.n0 < HYB_REFILL_BELOW) while (hs.n0 < HYB_REFILL_TO && hyb_refill_one<LT, 0>(fb, f, hs)) {}
  if (hs.n1 < HYB_REFILL_BELOW) while (hs.n1 < HYB_REFILL_TO && hyb_refill_one<LT, 1>(fb, f, hs)) {}
}

// the price-range trackers when no level is overwritten (OrderbookSimulator.py:134-135): worst resting price of each side = the
// first cold level, or the worst hot order when nothing is cold
template <class LT>
__device__ __forceinline__ void hyb_update_trackers(const FastBook<LT>& fb, const HybState& hs) {
  BookHdr* h = reinterpret_cast<BookHdr*>(fb.blob);
  const int lane = fb.lane;
  __syncwarp();
  uint2 k[HYB_NCH];
  flat_keys(hyb_pool<LT>(fb.blob, 0), hs.n0, lane, k);
  int w0 = flat_best_of<1>(k, hs.n0, lane, -1);            // lowest hot bid
  flat_keys(hyb_pool<LT>(fb.blob, 1), hs.n1, lane, k);
  int w1 = flat_best_of<0>(k, hs.n1, lane, -1);            // highest hot ask
  const int c0 = fb.cnt(0)->x, c1 = fb.cnt(1)->x;
  if (c0) w0 = FastBook<LT>::P(fb.side(0))[0];
  if (c1) w1 = FastBook<LT>::P(fb.side(1))[0];
  if (lane == 0) {
    if ((hs.n0 || c0) && w0 < h->min_buy) h->min_buy = w0;
    if ((hs.n1 || c1) && w1 > h->max_sell) h->max_sell = w1;
  }
  __syncwarp();
}
