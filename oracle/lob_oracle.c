/*
 * lob_oracle.c -- TEST INFRASTRUCTURE: a plain-C, single-environment CPU restatement of the rl4mm hot path.
 *
 * This file is the parity oracle for the CUDA path.  It is NOT part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it.
 *
 * It follows the reference literally (unbounded containers, a shared internal-id counter, the external-id map and
 * the binary search by internal id) rather than the device data structure, so that agreement between the two is
 * evidence and not a tautology.  Every function cites the reference file:line it restates (paths relative to the
 * reference tree).  Parity of this file against the reference itself is pinned by tests/golden/ (vectors generated
 * from the unmodified reference by oracle/gen_golden.py) -- see tests/test_oracle_golden.py.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off -shared -fPIC).
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../include/lobsim.h"
#include "lob_oracle.h"

/* ------------------------------------------------------------------------------------------------------------ */
/*  containers                                                                                                    */
/* ------------------------------------------------------------------------------------------------------------ */

typedef struct {
  int64_t vol;
  int64_t iid;    /* internal_id; -1 = snapshot aggregate */
  int64_t ext;    /* external_id; -1 = None */
  int is_ext;
} o_order;

typedef struct {
  int64_t price;
  o_order* q;     /* FIFO, index 0 = head */
  int n, cap;
} o_level;

typedef struct {
  o_level* lv;    /* ascending price (SortedDict) */
  int n, cap;
  int nord;              /* resting orders on the side (snapshot aggregates included) */
  int peak_lv, peak_ord; /* high-water marks of n / nord since the last lo_reset_book / lo_set_book */
} o_side;

typedef struct {
  o_side s[2];    /* 0 = buy, 1 = sell */
} o_book;

/* external_to_internal_lookup: rl4mm/orderbook/OrderIDConvertor.py:7-37 (open addressing, never reset) */
typedef struct {
  int64_t* key;
  int64_t* val;
  uint8_t* st;    /* 0 empty, 1 used, 2 tombstone */
  size_t cap, used, filled;
} o_map;

static uint64_t mix64(uint64_t x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
  return x;
}
static void map_init(o_map* m, size_t cap) {
  m->cap = cap; m->used = m->filled = 0;
  m->key = (int64_t*)calloc(cap, sizeof(int64_t));
  m->val = (int64_t*)calloc(cap, sizeof(int64_t));
  m->st = (uint8_t*)calloc(cap, 1);
}
static void map_free(o_map* m) { free(m->key); free(m->val); free(m->st); }
static void map_put(o_map* m, int64_t k, int64_t v);
static void map_grow(o_map* m) {
  o_map n; map_init(&n, m->cap * 2);
  for (size_t i = 0; i < m->cap; i++) if (m->st[i] == 1) map_put(&n, m->key[i], m->val[i]);
  map_free(m); *m = n;
}
static void map_put(o_map* m, int64_t k, int64_t v) {
  if ((m->filled + 1) * 2 > m->cap) map_grow(m);
  size_t i = mix64((uint64_t)k) & (m->cap - 1), tomb = (size_t)-1;
  while (m->st[i] != 0) {
    if (m->st[i] == 1 && m->key[i] == k) { m->val[i] = v; return; }
    if (m->st[i] == 2 && tomb == (size_t)-1) tomb = i;
    i = (i + 1) & (m->cap - 1);
  }
  if (tomb != (size_t)-1) i = tomb; else m->filled++;
  m->st[i] = 1; m->key[i] = k; m->val[i] = v; m->used++;
}
static int map_get(const o_map* m, int64_t k, int64_t* v) {
  size_t i = mix64((uint64_t)k) & (m->cap - 1);
  while (m->st[i] != 0) {
    if (m->st[i] == 1 && m->key[i] == k) { *v = m->val[i]; return 1; }
    i = (i + 1) & (m->cap - 1);
  }
  return 0;
}
static void map_del(o_map* m, int64_t k) {
  size_t i = mix64((uint64_t)k) & (m->cap - 1);
  while (m->st[i] != 0) {
    if (m->st[i] == 1 && m->key[i] == k) { m->st[i] = 2; m->used--; return; }
    i = (i + 1) & (m->cap - 1);
  }
}

static void side_clear(o_side* s) {
  for (int i = 0; i < s->n; i++) free(s->lv[i].q);
  s->n = 0; s->nord = 0;
}
static void book_clear(o_book* b) { side_clear(&b->s[0]); side_clear(&b->s[1]); }
static void book_free(o_book* b) { book_clear(b); free(b->s[0].lv); free(b->s[1].lv); }

static int side_find(const o_side* s, int64_t price) { /* index of the level or -1 */
  int lo = 0, hi = s->n - 1;
  while (lo <= hi) {
    int mid = (lo + hi) / 2;
    if (s->lv[mid].price == price) return mid;
    if (s->lv[mid].price < price) lo = mid + 1; else hi = mid - 1;
  }
  return -1;
}
static o_level* side_get_or_insert(o_side* s, int64_t price) {
  int pos = 0;
  while (pos < s->n && s->lv[pos].price < price) pos++;
  if (pos < s->n && s->lv[pos].price == price) return &s->lv[pos];
  if (s->n == s->cap) { s->cap = s->cap ? s->cap * 2 : 16; s->lv = (o_level*)realloc(s->lv, s->cap * sizeof(o_level)); }
  memmove(&s->lv[pos + 1], &s->lv[pos], (size_t)(s->n - pos) * sizeof(o_level));
  s->lv[pos].price = price; s->lv[pos].q = NULL; s->lv[pos].n = s->lv[pos].cap = 0;
  s->n++;
  if (s->n > s->peak_lv) s->peak_lv = s->n;
  return &s->lv[pos];
}
static void side_remove_level(o_side* s, int idx) {
  s->nord -= s->lv[idx].n;
  free(s->lv[idx].q);
  memmove(&s->lv[idx], &s->lv[idx + 1], (size_t)(s->n - idx - 1) * sizeof(o_level));
  s->n--;
}
static void level_append(o_side* s, o_level* l, o_order o) {
  if (l->n == l->cap) { l->cap = l->cap ? l->cap * 2 : 4; l->q = (o_order*)realloc(l->q, (size_t)l->cap * sizeof(o_order)); }
  l->q[l->n++] = o;
  if (++s->nord > s->peak_ord) s->peak_ord = s->nord;
}
static void level_erase(o_side* s, o_level* l, int pos) {
  memmove(&l->q[pos], &l->q[pos + 1], (size_t)(l->n - pos - 1) * sizeof(o_order));
  l->n--; s->nord--;
}
/* deque([order]): the level's queue is replaced by one order */
static void level_replace(o_side* s, o_level* l, o_order o) { s->nord -= l->n; l->n = 0; level_append(s, l, o); }

/* ------------------------------------------------------------------------------------------------------------ */
/*  feature state                                                                                                 */
/* ------------------------------------------------------------------------------------------------------------ */

typedef struct {
  double cur;               /* Feature.current_value */
  int64_t first_usage_us;   /* Feature.first_usage_time, absolute us after midnight (may be negative) */
  double* ring;             /* deque of doubles (prices) */
  int64_t* iring[2];        /* deques of ints (trades / volumes), [buy, sell] */
  int len;                  /* current deque length */
  int64_t total, diff;      /* total_trades / trade_diff, total_volume / volume_imbalance */
  double partial_price_sum; /* AmihudLambda */
  int64_t partial_dollar_volume;
  int steps_until_update, dv_len;
  double* hist;             /* Feature.history (deque(maxlen=max_norm_len)) */
  int hist_len;
} o_feat;

/* RollingSharpe.aum_array / n_filled -- rl4mm/rewards/RewardFunctions.py:50-59 (never reset by the env) */
typedef struct { double aum[LOBSIM_MAX_SHARPE_WINDOW]; int n_filled; } o_sharpe;

struct lo {
  lobsim_cfg_t cfg;
  lobsim_stream_t stream;   /* host pointers */
  int has_stream;
  o_book central, internal;
  o_map ext2int;
  int64_t counter;          /* OrderIdConvertor.counter */
  /* simulator */
  int64_t now_step;
  int32_t env_index;   /* which env of the batch this oracle stands for: part of the RandomAgent stream key */
  int64_t min_buy_price, max_sell_price, init_buy_range, init_sell_range;
  /* env */
  int64_t episode_start_step;
  int64_t inventory;
  double cash;
  double price;
  uint32_t err;
  int dead;
  o_feat feat[LOBSIM_MAX_FEATURES];
  o_sharpe sharpe[2];       /* [per-step reward, terminal reward] */
  /* fills of the current step */
  lobsim_fill_t* fills;
  int n_fills, cap_fills;
  int call_fills, peak_fills; /* fills since the start of the current API call; its high-water mark since lo_reset_book */
  double prev_action[8];
  int has_reset;
};

/* ------------------------------------------------------------------------------------------------------------ */
/*  Exchange                                                                                                      */
/* ------------------------------------------------------------------------------------------------------------ */

typedef struct {
  int type;       /* LOBSIM_MSG_* */
  int dir;
  int64_t price;
  int64_t vol;
  int has_vol;    /* volume is not None */
  int is_ext;
  int64_t ext;    /* external_id or -1 */
  int64_t iid;    /* internal_id or 0 (None) */
} o_msg;

static void add_fill(lo_t* o, int list, int dir, int64_t price, int64_t vol, int is_market, uint32_t ref) {
  if (o->n_fills == o->cap_fills) {
    o->cap_fills = o->cap_fills ? o->cap_fills * 2 : 64;
    o->fills = (lobsim_fill_t*)realloc(o->fills, (size_t)o->cap_fills * sizeof(lobsim_fill_t));
  }
  lobsim_fill_t* f = &o->fills[o->n_fills++];
  f->list = list; f->direction = dir; f->price = (int32_t)price; f->volume = (int32_t)vol; f->is_market = is_market;
  f->ref = ref;
  if (++o->call_fills > o->peak_fills) o->peak_fills = o->call_fills;
}

static uint32_t order_ref(const o_order* r) {
  if (!r->is_ext) return LOBSIM_REF_AGENT | (uint32_t)r->iid;
  if (r->iid == -1) return LOBSIM_REF_AGGREGATE;
  return (uint32_t)r->ext;
}

/* Exchange.best_buy_price / best_sell_price -- rl4mm/orderbook/Exchange.py:152-158 (0 / inf when empty) */
static int best_buy(const lo_t* o, int64_t* p) { const o_side* s = &o->central.s[0]; if (!s->n) { *p = 0; return 0; } *p = s->lv[s->n - 1].price; return 1; }
static int best_sell(const lo_t* o, int64_t* p) { const o_side* s = &o->central.s[1]; if (!s->n) { *p = INT64_MAX; return 0; } *p = s->lv[0].price; return 1; }

/* Exchange._does_order_cross_spread -- Exchange.py:188-194 */
static int crosses(const lo_t* o, const o_msg* m) {
  int64_t p;
  if (m->type == LOBSIM_MSG_MARKET) return 1;
  if (m->dir == 0) { best_sell(o, &p); return m->price >= p; }
  best_buy(o, &p);
  return m->price <= p;
}

static void process_order(lo_t* o, o_msg* m, uint32_t* ref_out);

/* Exchange._reduce_order_with_queue_position + _clear_empty_orders_and_prices -- Exchange.py:219-247.
 * Returns 0 and leaves the book untouched when volume_to_remove exceeds the resting volume
 * (CancellationVolumeExceededError, :227-230). */
static int reduce_at(lo_t* o, o_book* book, int dir, int64_t price, int pos, int64_t v) {
  o_side* s = &book->s[dir];
  int li = side_find(s, price);
  o_level* l = &s->lv[li];
  if (v > l->q[pos].vol) return 0;
  l->q[pos].vol -= v;
  if (l->q[pos].vol == 0) {
    if (l->q[pos].is_ext && l->q[pos].ext >= 0) map_del(&o->ext2int, l->q[pos].ext); /* :243-244 */
    level_erase(s, l, pos);
  }
  if (l->n == 0) side_remove_level(s, li);
  return 1;
}

/* Exchange.submit_order -- Exchange.py:71-83; OrderIdConvertor.add_internal_id_to_order_and_track :12-18 */
static void execute_order(lo_t* o, o_msg* m, uint32_t* ref_out);
static void submit_order(lo_t* o, o_msg* m, uint32_t* ref_out) {
  if (crosses(o, m)) { execute_order(o, m, ref_out); return; }
  o_order r;
  r.iid = ++o->counter; r.vol = m->vol; r.ext = m->ext; r.is_ext = m->is_ext;
  if (m->is_ext) map_put(&o->ext2int, m->ext, r.iid);
  level_append(&o->central.s[m->dir], side_get_or_insert(&o->central.s[m->dir], m->price), r);
  if (!m->is_ext) level_append(&o->internal.s[m->dir], side_get_or_insert(&o->internal.s[m->dir], m->price), r);
  if (ref_out) *ref_out = m->is_ext ? 0xffffffffu : (uint32_t)r.iid;
}

/* Exchange.execute_order -- Exchange.py:85-120 */
static void execute_order(lo_t* o, o_msg* m, uint32_t* ref_out) {
  int64_t remaining = m->vol;
  int opp = m->dir ^ 1;
  while (remaining > 0 && crosses(o, m)) {
    o_side* s = &o->central.s[opp];
    if (s->n == 0) { o->err |= LOBSIM_ERR_EMPTY_BOOK; o->dead = 1; return; } /* EmptyOrderbookError :183-186 */
    o_level* l = opp == 1 ? &s->lv[0] : &s->lv[s->n - 1];
    o_order head = l->q[0];
    int64_t hprice = l->price;
    if (!m->is_ext && !head.is_ext) { /* cannot fill our own order => delete it, :91-94 */
      o_msg d; d.type = LOBSIM_MSG_DELETE; d.dir = opp; d.price = hprice; d.vol = head.vol; d.has_vol = 1;
      d.is_ext = 0; d.ext = head.ext; d.iid = head.iid;
      process_order(o, &d, NULL);
      if (o->dead) return;
      continue;
    }
    int64_t v = remaining < head.vol ? remaining : head.vol;
    uint32_t href = order_ref(&head);
    if (!head.is_ext) reduce_at(o, &o->internal, opp, hprice, 0, v); /* internal first, :97-98 */
    reduce_at(o, &o->central, opp, hprice, 0, v);
    add_fill(o, head.is_ext ? 1 : 0, opp, hprice, v, 0, href);
    remaining -= v;
    if (!m->is_ext) add_fill(o, 0, m->dir, hprice, v, 1, href); /* :111-115 */
  }
  if (remaining > 0 && m->type == LOBSIM_MSG_LIMIT) { /* :116-119 */
    o_msg r = *m; r.vol = remaining;
    submit_order(o, &r, ref_out);
  }
}

/* Exchange._find_queue_position -- Exchange.py:196-217 ; OrderIdConvertor.get_internal_order_id :20-27 */
static int find_queue_position(lo_t* o, const o_msg* m, o_book* book) {
  int64_t iid = m->iid;
  if (iid == 0) {
    if (m->is_ext) { if (!map_get(&o->ext2int, m->ext, &iid)) return -1; }
    else return -1; /* (the reference would raise a TypeError; unreachable through the env) */
  }
  o_side* s = &book->s[m->dir];
  int li = side_find(s, m->price);
  if (li < 0) return -1;
  o_level* l = &s->lv[li];
  int left = 0, right = l->n - 1;
  while (left <= right) {
    int middle = (left + right) / 2;
    int64_t mid_id = l->q[middle].iid;
    if (mid_id == iid) return middle;
    if (mid_id < iid) left = middle + 1; else right = middle - 1;
  }
  return -1;
}

/* Exchange.remove_order -- Exchange.py:122-147 */
static void remove_order(lo_t* o, o_msg* m) {
  o_book* books[2] = {&o->central, &o->internal};
  int nb = m->is_ext ? 1 : 2;
  for (int b = 0; b < nb; b++) {
    o_book* book = books[b];
    int pos = find_queue_position(o, m, book);
    if (pos < 0) {
      o_side* s = &book->s[m->dir];
      int li = side_find(s, m->price);
      if (li < 0) continue;
      if (s->lv[li].q[0].iid == -1) {
        if (!m->has_vol) { o->err |= LOBSIM_ERR_BAD_VOLUME; continue; } /* assert :134 */
        m->iid = -1; pos = 0;
      } else continue;
    } else if (!m->has_vol) {
      o_side* s = &book->s[m->dir];
      m->vol = s->lv[side_find(s, m->price)].q[pos].vol; m->has_vol = 1;
    }
    if (!reduce_at(o, book, m->dir, m->price, pos, m->vol)) {
      o_side* s = &book->s[m->dir];
      int64_t resting = s->lv[side_find(s, m->price)].q[pos].vol;
      reduce_at(o, book, m->dir, m->price, pos, resting);
    }
  }
}

/* Exchange.process_order -- Exchange.py:58-69 */
static void process_order(lo_t* o, o_msg* m, uint32_t* ref_out) {
  if (o->dead) return;
  if (m->has_vol && m->vol <= 0) { o->err |= LOBSIM_ERR_BAD_VOLUME; return; } /* assert :59-60 */
  if (m->type == LOBSIM_MSG_LIMIT) submit_order(o, m, ref_out);
  else if (m->type == LOBSIM_MSG_MARKET) execute_order(o, m, ref_out);
  else remove_order(o, m);
}

/* ------------------------------------------------------------------------------------------------------------ */
/*  Orderbook properties -- rl4mm/orderbook/models.py:64-101                                                      */
/* ------------------------------------------------------------------------------------------------------------ */

static int64_t level_volume(const o_level* l) { int64_t v = 0; for (int i = 0; i < l->n; i++) v += l->q[i].vol; return v; }

static int book_tops(const lo_t* o, int64_t* bb, int64_t* bs, int64_t* bv, int64_t* sv) {
  const o_side* b = &o->central.s[0]; const o_side* s = &o->central.s[1];
  if (!b->n || !s->n) return 0;
  *bb = b->lv[b->n - 1].price; *bs = s->lv[0].price;
  *bv = level_volume(&b->lv[b->n - 1]); *sv = level_volume(&s->lv[0]);
  return 1;
}
static double book_imbalance(int64_t bv, int64_t sv) { return (double)(bv - sv) / (double)(bv + sv); } /* :92 */
static double book_microprice(int64_t bb, int64_t bs, int64_t bv, int64_t sv) { /* :96 */
  double I = book_imbalance(bv, sv);
  return (1.0 + I) / 2.0 * (double)bs + (1.0 - I) / 2.0 * (double)bb;
}

/* ------------------------------------------------------------------------------------------------------------ */
/*  OrderbookSimulator                                                                                            */
/* ------------------------------------------------------------------------------------------------------------ */

static int64_t now_us(const lo_t* o) { return o->stream.t0_us + o->now_step * o->cfg.step_us; }

static const int32_t* snapshot_row(const lo_t* o, int64_t sec_idx) {
  if (sec_idx < 0 || sec_idx > (int64_t)o->stream.n_seconds || !o->stream.snap_valid[sec_idx]) return NULL;
  return o->stream.snapshots + (size_t)sec_idx * 2 * (size_t)o->cfg.n_levels * 2;
}

/* Exchange.orderbook_price_range -- Exchange.py:160-170 (dummy levels are never materialised here) */
static void price_range(const lo_t* o, int64_t* worst_buy, int64_t* worst_sell) {
  const o_side* b = &o->central.s[0]; const o_side* s = &o->central.s[1];
  *worst_buy = b->n ? b->lv[0].price : 0;
  *worst_sell = s->n ? s->lv[s->n - 1].price : 0;
}

/* capacity high-water marks (lo_peaks): restart from the current book */
static void reset_peaks(lo_t* o) {
  for (int side = 0; side < 2; side++) {
    o_side* c = &o->central.s[side]; o_side* a = &o->internal.s[side];
    c->peak_lv = c->n; c->peak_ord = c->nord; a->peak_lv = a->n; a->peak_ord = a->nord;
  }
  o->call_fills = 0; o->peak_fills = 0;
}

/* OrderbookSimulator.reset_episode -- OrderbookSimulator.py:55-68 (+ get_historical_start_book :90-97,
 * _get_initial_orders_from_snapshot :156-175, Exchange.get_initial_orderbook_from_orders Exchange.py:172-178,
 * _reset_initial_price_ranges :185-188) */
int lo_reset_book(lo_t* o, int start_step) {
  if (!o->has_stream) return LOBSIM_E_STATE;
  int64_t t = o->stream.t0_us + (int64_t)start_step * o->cfg.step_us;
  if (t % 1000000) return LOBSIM_E_INVALID; /* "Episodes must be started on the second." :61 */
  book_clear(&o->central); book_clear(&o->internal);
  reset_peaks(o);
  o->dead = 0; o->err = 0;
  o->now_step = start_step;
  const int32_t* row = snapshot_row(o, (t - o->stream.t0_us) / 1000000);
  if (!row) { o->err |= LOBSIM_ERR_NO_SNAPSHOT; o->dead = 1; return LOBSIM_OK; }
  int L = o->cfg.n_levels;
  for (int side = 0; side < 2; side++)
    for (int lvl = 0; lvl < L; lvl++) {
      int32_t price = row[(side * L + lvl) * 2], vol = row[(side * L + lvl) * 2 + 1];
      if (price == LOBSIM_NO_PRICE) continue;
      o_order r; r.iid = -1; r.ext = -1; r.is_ext = 1; r.vol = vol;
      level_replace(&o->central.s[side], side_get_or_insert(&o->central.s[side], price), r); /* deque([order]) */
    }
  int64_t bb, bs;
  price_range(o, &o->min_buy_price, &o->max_sell_price);
  best_buy(o, &bb); best_sell(o, &bs);
  o->init_buy_range = bb - o->min_buy_price;
  o->init_sell_range = o->max_sell_price - bs;
  return LOBSIM_OK;
}

/* OrderbookSimulator._near_exiting_initial_price_range -- OrderbookSimulator.py:177-183 */
static int near_exiting(const lo_t* o) {
  double prop = (double)o->cfg.outer_levels / (double)o->cfg.n_levels;
  int64_t bb, bs; int hb = best_buy(o, &bb), hs = best_sell(o, &bs);
  double lhs_b = (double)bb, lhs_s = hs ? (double)bs : INFINITY;
  (void)hb;
  return lhs_b < (double)o->min_buy_price + prop * (double)o->init_buy_range ||
         lhs_s > (double)o->max_sell_price - prop * (double)o->init_sell_range;
}

/* OrderbookSimulator.update_outer_levels -- OrderbookSimulator.py:105-135 */
static void update_outer_levels(lo_t* o) {
  const int32_t* row = snapshot_row(o, (now_us(o) - o->stream.t0_us) / 1000000);
  if (!row) return;
  int L = o->cfg.n_levels;
  o_msg* repl = NULL; int nrepl = 0, caprepl = 0;
  for (int side = 0; side < 2; side++)
    for (int lvl = 0; lvl < L; lvl++) {
      int64_t price = row[(side * L + lvl) * 2], vol = row[(side * L + lvl) * 2 + 1];
      if (price == LOBSIM_NO_PRICE) continue;
      /* _initial_prices_filter_function :99-103 */
      if (!((side == 0 && price < o->min_buy_price) || (side == 1 && price > o->max_sell_price))) continue;
      int li = side_find(&o->internal.s[side], price);
      if (li >= 0) {
        o_level* il = &o->internal.s[side].lv[li];
        int n = il->n;
        o_msg* canc = (o_msg*)malloc((size_t)n * sizeof(o_msg));
        for (int i = 0; i < n; i++) {
          o_msg c; c.type = LOBSIM_MSG_CANCEL; c.dir = side; c.price = price; c.vol = il->q[i].vol; c.has_vol = 1;
          c.is_ext = 0; c.ext = -1; c.iid = il->q[i].iid;
          canc[i] = c;
          if (nrepl == caprepl) { caprepl = caprepl ? caprepl * 2 : 8; repl = (o_msg*)realloc(repl, (size_t)caprepl * sizeof(o_msg)); }
          c.type = LOBSIM_MSG_LIMIT; repl[nrepl++] = c;
        }
        for (int i = 0; i < n; i++) process_order(o, &canc[i], NULL);
        free(canc);
      }
      o_order r; r.iid = -1; r.ext = -1; r.is_ext = 1; r.vol = vol;
      level_replace(&o->central.s[side], side_get_or_insert(&o->central.s[side], price), r); /* central[dir][price] = deque([order]) :130 */
    }
  for (int i = 0; i < nrepl; i++) { repl[i].iid = 0; process_order(o, &repl[i], NULL); }
  free(repl);
  int64_t wb, ws; price_range(o, &wb, &ws);
  if (wb < o->min_buy_price) o->min_buy_price = wb;
  if (ws > o->max_sell_price) o->max_sell_price = ws;
}

/* OrderbookSimulator.forward_step -- OrderbookSimulator.py:70-88; messages of the step come from the packed stream
 * (HistoricalOrderGenerator.generate_orders, HistoricalOrderGenerator.py:32-46, get_order_from_external_message
 * :77-90). */
static void forward_step_ex(lo_t* o, o_msg* internal_orders, int n_internal, int resync_check) {
  if (o->dead) return;
  if (o->now_step < 0 || o->now_step >= (int64_t)o->stream.n_grid_steps) { o->err |= LOBSIM_ERR_END_OF_STREAM; o->dead = 1; return; }
  for (int i = 0; i < n_internal && !o->dead; i++) process_order(o, &internal_orders[i], NULL);
  uint32_t m0 = o->stream.step_off[o->now_step], m1 = o->stream.step_off[o->now_step + 1];
  for (uint32_t i = m0; i < m1 && !o->dead; i++) {
    const lobsim_msg_t* r = &o->stream.msgs[i];
    o_msg m; m.type = (int)LOBSIM_META_TYPE(r->meta); m.dir = (int)LOBSIM_META_DIR(r->meta); m.price = r->price;
    m.vol = r->volume; m.has_vol = 1; m.is_ext = 1; m.ext = r->ref; m.iid = 0;
    process_order(o, &m, NULL);
  }
  if (o->dead) return;
  o->now_step += 1;
  if (resync_check && o->cfg.resync && near_exiting(o) && now_us(o) % 1000000 == 0) update_outer_levels(o);
}
static void forward_step(lo_t* o, o_msg* internal_orders, int n_internal) { forward_step_ex(o, internal_orders, n_internal, 1); }

int lo_replay(lo_t* o, int n_steps) {
  if (!o->has_stream) return LOBSIM_E_STATE;
  o->n_fills = 0; o->call_fills = 0;
  for (int i = 0; i < n_steps; i++) forward_step(o, NULL, 0);
  return LOBSIM_OK;
}

/* ONE OrderbookSimulator.forward_step(until = now + n_steps * step_size) -- OrderbookSimulator.py:70-88: the messages of the
 * n_steps grid intervals, then the resync condition (:86-87) evaluated once, at `until` */
int lo_forward_step(lo_t* o, int n_steps) {
  if (!o->has_stream) return LOBSIM_E_STATE;
  o->n_fills = 0; o->call_fills = 0;
  for (int i = 0; i < n_steps; i++) forward_step_ex(o, NULL, 0, i == n_steps - 1);
  return LOBSIM_OK;
}

/* ------------------------------------------------------------------------------------------------------------ */
/*  Features -- rl4mm/features/Features.py                                                                        */
/* ------------------------------------------------------------------------------------------------------------ */

typedef struct {
  int64_t n_ext[2], vol_ext[2], n_int[2], vol_int[2]; /* per direction of the recorded order */
} o_flow;

static o_flow step_flow(const lo_t* o) {
  o_flow f; memset(&f, 0, sizeof f);
  for (int i = 0; i < o->n_fills; i++) {
    const lobsim_fill_t* x = &o->fills[i];
    if (x->list == 1) { f.n_ext[x->direction]++; f.vol_ext[x->direction] += x->volume; }
    else { f.n_int[x->direction]++; f.vol_int[x->direction] += x->volume; }
  }
  return f;
}

static double clampd(double x, double lo_, double hi) { double m = x < hi ? x : hi; return m > lo_ ? m : lo_; } /* :99 */

/* Feature._update of each concrete class */
static void feature_update_raw(lo_t* o, int fi) {
  const lobsim_feature_t* fc = &o->cfg.features[fi];
  o_feat* f = &o->feat[fi];
  int k = fc->lookback;
  int64_t bb = 0, bs = 0, bv = 0, sv = 0;
  int tops = book_tops(o, &bb, &bs, &bv, &sv);
  switch (fc->kind) {
    case LOBSIM_FEAT_SPREAD: f->cur = tops ? (double)(bs - bb) : NAN; break;             /* :128 */
    case LOBSIM_FEAT_BOOK_IMBALANCE: f->cur = tops ? book_imbalance(bv, sv) : NAN; break; /* :142 */
    case LOBSIM_FEAT_PRICE: f->cur = o->price; break;                                     /* :342 */
    case LOBSIM_FEAT_INVENTORY: f->cur = (double)o->inventory; break;                     /* :489 */
    case LOBSIM_FEAT_EPISODE_PROPORTION: f->cur += fc->dparam; break;                     /* :511 */
    case LOBSIM_FEAT_TIME_OF_DAY: {                                                       /* :526-536 */
      int64_t min_time = 10LL * 3600 * 1000000, max_time = (15LL * 3600 + 1800) * 1000000;
      int64_t tot = max_time - min_time, nb_ = fc->iparam;
      int64_t bucket = tot / nb_, rem = tot % nb_; /* timedelta / int rounds half to even (in us) */
      if (2 * rem > nb_ || (2 * rem == nb_ && (bucket & 1))) bucket++;
      int64_t d = now_us(o) - min_time;
      int64_t q = d >= 0 ? d / bucket : -((-d + bucket - 1) / bucket); /* floor division */
      f->cur = (double)(q > 0 ? q : 0);
      break;
    }
    case LOBSIM_FEAT_PRICE_MOVE:   /* :173-175 deque(maxlen=k+1), appendleft; ring[0] = newest */
    case LOBSIM_FEAT_PRICE_RANGE: { /* :198-200 */
      int n = f->len < k + 1 ? f->len + 1 : k + 1;
      memmove(&f->ring[1], &f->ring[0], (size_t)(n - 1) * sizeof(double));
      f->ring[0] = o->price; f->len = n;
      if (fc->kind == LOBSIM_FEAT_PRICE_MOVE) f->cur = f->ring[0] - f->ring[n - 1];
      else {
        double mx = f->ring[0], mn = f->ring[0];
        for (int i = 1; i < n; i++) { if (f->ring[i] > mx) mx = f->ring[i]; if (f->ring[i] < mn) mn = f->ring[i]; }
        f->cur = mx - mn;
      }
      break;
    }
    case LOBSIM_FEAT_VOLATILITY: { /* :226-242; ring[0] = oldest */
      if (f->len < k) { f->ring[f->len++] = o->price; f->cur = 0.0; }
      else if (f->len == k) {
        f->ring[f->len++] = o->price;
        double s = 0.0; /* python sum() starts from int 0 and adds left to right */
        for (int i = 0; i < k; i++) { double r = (f->ring[i + 1] - f->ring[i]) / f->ring[0]; s += r * r; }
        f->cur = s / (double)k;
      } else {
        double oldest = f->ring[0];
        memmove(&f->ring[0], &f->ring[1], (size_t)k * sizeof(double));
        double oldest_ret = (f->ring[0] - oldest) / oldest;
        double new_ret = (o->price - f->ring[k - 1]) / f->ring[k - 1];
        f->ring[k] = o->price;
        double ss = f->cur * (double)k - oldest_ret * oldest_ret + new_ret * new_ret;
        f->cur = ss / (double)k;
      }
      break;
    }
    case LOBSIM_FEAT_TRADE_DIR_IMBALANCE:   /* :376-407 */
    case LOBSIM_FEAT_TRADE_VOL_IMBALANCE: { /* :435-466 */
      o_flow fl = step_flow(o);
      int64_t nb, ns;
      if (fc->kind == LOBSIM_FEAT_TRADE_DIR_IMBALANCE) { nb = fl.n_ext[0]; ns = fl.n_ext[1]; if (fc->iparam) { nb += fl.n_int[0]; ns += fl.n_int[1]; } }
      else { nb = fl.vol_ext[0]; ns = fl.vol_ext[1]; if (fc->iparam) { nb += fl.vol_int[0]; ns += fl.vol_int[1]; } }
      if (f->len < k) {
        f->iring[0][f->len] = nb; f->iring[1][f->len] = ns; f->len++;
        f->cur = 0.0;
      } else {
        if (f->total == 0) {
          /* deque(maxlen=k).append on a full deque drops the oldest */
          memmove(&f->iring[0][0], &f->iring[0][1], (size_t)(k - 1) * sizeof(int64_t));
          memmove(&f->iring[1][0], &f->iring[1][1], (size_t)(k - 1) * sizeof(int64_t));
          f->iring[0][k - 1] = nb; f->iring[1][k - 1] = ns;
          int64_t sb = 0, ss = 0;
          for (int i = 0; i < k; i++) { sb += f->iring[0][i]; ss += f->iring[1][i]; }
          f->total = sb + ss; f->diff = sb - ss;
        } else {
          int64_t ob = f->iring[0][0], os = f->iring[1][0];
          memmove(&f->iring[0][0], &f->iring[0][1], (size_t)(k - 1) * sizeof(int64_t));
          memmove(&f->iring[1][0], &f->iring[1][1], (size_t)(k - 1) * sizeof(int64_t));
          f->total -= ob + os; f->total += nb + ns;
          f->diff -= ob - os; f->diff += nb - ns;
          f->iring[0][k - 1] = nb; f->iring[1][k - 1] = ns;
        }
        f->cur = f->total != 0 ? (double)f->diff / (double)f->total : 0.5;
      }
      break;
    }
    case LOBSIM_FEAT_AMIHUD_LAMBDA: { /* :285-324; ring = prices (oldest first), iring[0] = dollar volumes */
      const int sf = fc->iparam, kk = fc->lookback / sf - 1; /* true_lookback_periods */
      if (f->steps_until_update > 0) {
        f->steps_until_update -= 1;
        f->partial_price_sum += o->price;
        o_flow fl = step_flow(o);
        f->partial_dollar_volume += fl.vol_ext[0] + fl.vol_ext[1];
      } else {
        f->steps_until_update = sf - 1;
        const double new_price = f->partial_price_sum / (double)sf;
        const int64_t new_dv = f->partial_dollar_volume;
        if (f->len < kk) {
          f->ring[f->len++] = new_price;
          if (f->dv_len < kk) f->iring[0][f->dv_len++] = new_dv; else { memmove(&f->iring[0][0], &f->iring[0][1], (size_t)(kk - 1) * sizeof(int64_t)); f->iring[0][kk - 1] = new_dv; }
          f->cur = 0.0;
        } else if (f->len == kk) {
          f->ring[f->len++] = new_price;
          if (f->dv_len < kk) f->iring[0][f->dv_len++] = new_dv; else { memmove(&f->iring[0][0], &f->iring[0][1], (size_t)(kk - 1) * sizeof(int64_t)); f->iring[0][kk - 1] = new_dv; }
          double sacc = 0.0;
          for (int i = 0; i < kk; i++) {
            double r = (f->ring[i + 1] - f->ring[i]) / f->ring[0];
            if (f->iring[0][i] > 0) sacc += fabs(r) / (double)f->iring[0][i];
          }
          f->cur = sacc / (double)kk;
        } else {
          double oldest = f->ring[0];
          memmove(&f->ring[0], &f->ring[1], (size_t)kk * sizeof(double));
          double oldest_ret = (f->ring[0] - oldest) / oldest;
          int64_t oldest_dv = f->iring[0][0];
          memmove(&f->iring[0][0], &f->iring[0][1], (size_t)(kk - 1) * sizeof(int64_t));
          double new_ret = (new_price - f->ring[kk - 1]) / f->ring[kk - 1];
          f->ring[kk] = new_price; f->iring[0][kk - 1] = new_dv;
          double new_ratio = new_dv > 0 ? fabs(new_ret) / (double)new_dv : 0.0;
          double old_ratio = oldest_dv > 0 ? fabs(oldest_ret) / (double)oldest_dv : 0.0;
          double sum_of_ratio = f->cur * (double)kk + new_ratio - old_ratio;
          f->cur = sum_of_ratio / (double)kk;
        }
        f->partial_price_sum = 0.0; f->partial_dollar_volume = 0;
      }
      break;
    }
    default: break;
  }
}

/* Feature.reset / _reset -- Features.py:92-96 (+ concrete reset methods) */
static void feature_reset(lo_t* o, int fi, int64_t first_usage_us) {
  const lobsim_feature_t* fc = &o->cfg.features[fi];
  o_feat* f = &o->feat[fi];
  f->first_usage_us = first_usage_us;
  f->len = 0; f->total = 0; f->diff = 0;
  f->hist_len = 0; /* history.clear() :94-95 */
  if (fc->kind == LOBSIM_FEAT_AMIHUD_LAMBDA) { /* AmihudLambda.reset :278-283 */
    f->dv_len = 0; f->partial_price_sum = 0.0; f->partial_dollar_volume = 0; f->steps_until_update = fc->iparam - 1;
  }
  feature_update_raw(o, fi);
  if (fc->kind == LOBSIM_FEAT_EPISODE_PROPORTION) f->cur = 0.0; /* :507-509 */
}

/* Feature.normalise -- Features.py:67-74: scipy.stats.zscore(history)[-1] = (value - mean) / std (ddof 0), numpy's
 * pairwise mean and two-pass variance (np.mean of the squared deviations), NaN when std <= |eps * mean| */
static double np_pairwise_sum(const double* a, int n);
static double feature_normalise(o_feat* f, int maxlen, double value) {
  if (f->hist_len == 0) f->hist[f->hist_len++] = value + 1e-06;
  if (f->hist_len == maxlen) { memmove(&f->hist[0], &f->hist[1], (size_t)(maxlen - 1) * sizeof(double)); f->hist_len--; }
  f->hist[f->hist_len++] = value;
  const int n = f->hist_len;
  double mean = np_pairwise_sum(f->hist, n) / (double)n;
  double* sq = (double*)malloc((size_t)n * sizeof(double));
  for (int i = 0; i < n; i++) { double d = f->hist[i] - mean; sq[i] = d * d; }
  double sd = sqrt(np_pairwise_sum(sq, n) / (double)n);
  free(sq);
  /* scipy.stats.zmap (scipy 1.18.1, the version installed where the goldens were generated; _stats_py.py):
   * "zero = std <= xp.abs(eps * mn); z[zero] = nan" -- (nearly) constant windows give NaN, not +-1 */
  if (sd <= fabs(2.220446049250313e-16 * mean)) return NAN;
  return (value - mean) / sd;
}

/* Feature.update -- Features.py:80-86, _now_is_multiple_of_update_freq :102-105 */
static void feature_update(lo_t* o, int fi) {
  const lobsim_feature_t* fc = &o->cfg.features[fi];
  o_feat* f = &o->feat[fi];
  int64_t t = now_us(o);
  if (t < f->first_usage_us) return;
  if ((t % 60000000LL) % fc->update_us != 0) return;
  feature_update_raw(o, fi);
  f->cur = clampd(f->cur, fc->min_value, fc->max_value);
  if (fc->norm_len > 0) f->cur = feature_normalise(f, fc->norm_len, f->cur);
}

/* ------------------------------------------------------------------------------------------------------------ */
/*  Action interpretation                                                                                         */
/* ------------------------------------------------------------------------------------------------------------ */

static double round_half_even(double x) { return nearbyint(x); } /* np.round; default FE_TONEAREST */

/* BetaOrderDistributor.convert_action/_convert_action -- rl4mm/gym/action_interpretation/OrderDistributors.py:23-56.
 * scipy.stats.beta.pdf(x; a, b) = exp(xlogy(a-1, x) + xlog1py(b-1, -x) - betaln(a, b)); betaln is common to all
 * midpoints and cancels in the normalisation up to rounding, so it is omitted (documented deviation, see
 * tests/golden/beta_ladders.json for the pinned lot sizes). */
static void beta_ladder(const lo_t* o, double a, double b, int64_t* out) {
  int Q = o->cfg.max_quote_level - o->cfg.min_quote_level;
  double w[64], s = 0.0, amax = -INFINITY;
  for (int i = 0; i < Q; i++) {
    double x = 1.0 / (double)Q * ((double)i + 0.5); /* midpoints :37 */
    double lx = (a - 1.0) == 0.0 ? 0.0 : (a - 1.0) * log(x);
    double l1 = (b - 1.0) == 0.0 ? 0.0 : (b - 1.0) * log1p(-x);
    w[i] = lx + l1;
    if (w[i] > amax) amax = w[i];
  }
  /* the common factor exp(-amax) (like 1/B(a,b)) cancels in the normalisation; it keeps exp() in range */
  for (int i = 0; i < Q; i++) { w[i] = exp(w[i] - amax); s += w[i]; }
  if (Q > 8) { /* numpy pairwise summation: blocks of 8 accumulators for n >= 8 */
    double r[8];
    int i;
    for (i = 0; i < 8; i++) r[i] = w[i];
    for (i = 8; i + 8 <= Q; i += 8) for (int j = 0; j < 8; j++) r[j] += w[i + j];
    s = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < Q; i++) s += w[i];
  } else if (Q == 8) {
    s = ((w[0] + w[1]) + (w[2] + w[3])) + ((w[4] + w[5]) + (w[6] + w[7]));
  }
  for (int i = 0; i < Q; i++) {
    double lots = round_half_even(w[i] / s * (double)o->cfg.active_volume);
    out[i] = isfinite(lots) ? (int64_t)lots : INT64_MIN; /* np.round(nan).astype(int) */
  }
}

static void action_to_ladders(const lo_t* o, const double* action, int64_t* buy, int64_t* sell) {
  const double EPS = 0.000001;
  double a[8];
  int ad = lo_action_dim(&o->cfg);
  for (int i = 0; i < ad; i++) a[i] = action[i] + EPS; /* :24 */
  double ab, bbeta, as, bs;
  if (o->cfg.concentration >= 0) {
    double c = o->cfg.concentration;
    ab = a[0]; bbeta = c - a[0] + EPS; as = a[1]; bs = c - a[1] + EPS;
  } else { ab = a[0]; bbeta = a[1]; as = a[2]; bs = a[3]; }
  beta_ladder(o, ab, bbeta, buy);
  beta_ladder(o, as, bs, sell);
}

void lo_action_to_ladders(const lo_t* o, const double* action, int64_t* buy, int64_t* sell) { action_to_ladders(o, action, buy, sell); }

typedef struct { o_msg* v; int n, cap; } o_msgs;
static void msgs_push(o_msgs* l, o_msg m) {
  if (l->n == l->cap) { l->cap = l->cap ? l->cap * 2 : 32; l->v = (o_msg*)realloc(l->v, (size_t)l->cap * sizeof(o_msg)); }
  l->v[l->n++] = m;
}

static int in_ladder(const int64_t* prices, int Q, int64_t p) { for (int i = 0; i < Q; i++) if (prices[i] == p) return 1; return 0; }

/* HistoricalOrderbookEnvironment.convert_action_to_orders -- HOE.py:206-216 (+ _get_best_prices :298-322,
 * _get_current_internal_order_volumes :291-296, _volume_diff_to_orders :227-258,
 * _get_inventory_clearing_market_order :260-266) */
static void convert_action_to_orders(lo_t* o, const double* action, o_msgs* out) {
  int Q = o->cfg.max_quote_level - o->cfg.min_quote_level;
  int64_t desired[2][64];
  action_to_ladders(o, action, desired[0], desired[1]);
  int ad = lo_action_dim(&o->cfg);
  int64_t absinv = o->inventory < 0 ? -o->inventory : o->inventory;
  int clearing = o->cfg.market_order_clearing && (double)absinv > action[ad - 1];
  if (clearing) { memset(desired, 0, sizeof desired); }
  for (int i = 0; i < Q; i++) /* a NaN ladder is INT64_MIN lots: _volume_diff_to_orders raises (KeyError / pop from an empty deque) */
    if (desired[0][i] == INT64_MIN || desired[1][i] == INT64_MIN) { o->err |= LOBSIM_ERR_BAD_ACTION; o->dead = 1; return; }
  int64_t bb, bs; int hb = best_buy(o, &bb), hs = best_sell(o, &bs);
  int64_t tick = o->cfg.tick_size;
  if (!hb || !hs) { o->err |= LOBSIM_ERR_EMPTY_BOOK; o->dead = 1; return; }
  if (o->cfg.enter_spread) {
    double mid = (double)(bs + bb) / 2.0; /* models.py:88 */
    int64_t nb = (int64_t)(floor(mid / (double)tick) * (double)tick);
    int64_t ns = (int64_t)(ceil(mid / (double)tick) * (double)tick);
    bb = nb; bs = ns;
  }
  int64_t prices[2][64];
  for (int i = 0; i < Q; i++) {
    prices[0][i] = bb - (o->cfg.min_quote_level + i) * tick;
    prices[1][i] = bs + (o->cfg.min_quote_level + i) * tick;
  }
  for (int side = 0; side < 2; side++) {
    o_side* is = &o->internal.s[side];
    for (int lvl = 0; lvl < Q; lvl++) {
      int64_t price = prices[side][lvl];
      int li = side_find(is, price);
      int64_t cur = li >= 0 ? level_volume(&is->lv[li]) : 0;
      int64_t diff = desired[side][lvl] - cur;
      o_msg m; m.dir = side; m.price = price; m.is_ext = 0; m.ext = -1; m.iid = 0; m.has_vol = 1;
      if (diff > 0) { m.type = LOBSIM_MSG_LIMIT; m.vol = diff; msgs_push(out, m); }
      if (diff < 0) {
        o_level* l = &is->lv[li];
        int j = l->n - 1;
        while (diff < 0) {
          int64_t wv = l->q[j].vol, v = wv < -diff ? wv : -diff;
          m.type = LOBSIM_MSG_CANCEL; m.vol = v; m.iid = l->q[j].iid;
          msgs_push(out, m);
          diff += v; j--;
        }
      }
    }
    for (int li = 0; li < is->n; li++) { /* wide orders: set(internal prices) - set(ladder), :250-257 */
      if (in_ladder(prices[side], Q, is->lv[li].price)) continue;
      for (int j = 0; j < is->lv[li].n; j++) {
        o_msg m; m.type = LOBSIM_MSG_CANCEL; m.dir = side; m.price = is->lv[li].price; m.vol = is->lv[li].q[j].vol;
        m.has_vol = 1; m.is_ext = 0; m.ext = -1; m.iid = is->lv[li].q[j].iid;
        msgs_push(out, m);
      }
    }
  }
  if (clearing) {
    o_msg m; m.type = LOBSIM_MSG_MARKET; m.dir = o->inventory < 0 ? 0 : 1; m.price = 0;
    m.vol = (int64_t)round_half_even((double)absinv * o->cfg.market_order_fraction_of_inventory);
    m.has_vol = 1; m.is_ext = 0; m.ext = -1; m.iid = 0;
    msgs_push(out, m);
  }
}

/* ------------------------------------------------------------------------------------------------------------ */
/*  HistoricalOrderbookEnvironment                                                                                */
/* ------------------------------------------------------------------------------------------------------------ */

/* _update_portfolio -- HOE.py:280-289 ; update_internal_state :199-204 */
static void update_internal_state(lo_t* o) {
  for (int i = 0; i < o->n_fills; i++) {
    const lobsim_fill_t* f = &o->fills[i];
    if (f->list != 0) continue;
    if (f->direction == 1) { o->inventory -= f->volume; o->cash += (double)((int64_t)f->volume * (int64_t)f->price); }
    else { o->inventory += f->volume; o->cash -= (double)((int64_t)f->volume * (int64_t)f->price); }
  }
  int64_t bb, bs, bv, sv;
  if (book_tops(o, &bb, &bs, &bv, &sv)) o->price = book_microprice(bb, bs, bv, sv);
  else { o->price = NAN; o->err |= LOBSIM_ERR_EMPTY_BOOK; }
}

static void env_forward(lo_t* o, o_msg* orders, int n) {
  o->n_fills = 0;
  forward_step(o, orders, n);
  update_internal_state(o);
}

static void get_observation(const lo_t* o, const double* prev_action, double* obs) {
  int F = o->cfg.n_features;
  for (int i = 0; i < F; i++) obs[i] = o->feat[i].cur;
  if (o->cfg.inc_prev_action_in_obs) {
    int ad = lo_action_dim(&o->cfg);
    for (int i = 0; i < ad; i++) obs[F + i] = prev_action ? prev_action[i] : 0.0;
  }
}

/* numpy's pairwise summation (np.add.reduce on a contiguous double array) */
static double np_pairwise_sum(const double* a, int n) {
  if (n < 8) { double r = -0.0; for (int i = 0; i < n; i++) r += a[i]; return r; }
  if (n <= 128) {
    double r[8]; int i;
    for (i = 0; i < 8; i++) r[i] = a[i];
    for (i = 8; i < n - (n % 8); i += 8) for (int j = 0; j < 8; j++) r[j] += a[i + j];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
  }
  int n2 = n / 2; n2 -= n2 % 8;
  return np_pairwise_sum(a, n2) + np_pairwise_sum(a + n2, n - n2);
}

/* get_sharpe -- rl4mm/rewards/RewardFunctions.py:10-22 */
static double get_sharpe(lo_t* o, const double* aum, int n) {
  double simple[LOBSIM_MAX_SHARPE_WINDOW] = {0};
  for (int i = 0; i < n; i++) if (aum[i] <= 0) { o->err |= LOBSIM_ERR_AUM_NONPOSITIVE; return NAN; } /* raise Exception */
  for (int i = 0; i + 1 < n; i++) simple[i] = exp(log(aum[i + 1]) - log(aum[i])) - 1.0;
  int m = n - 1;
  double mean = np_pairwise_sum(simple, m) / (double)m;
  double sq[LOBSIM_MAX_SHARPE_WINDOW];
  for (int i = 0; i < m; i++) { double d = simple[i] - mean; sq[i] = d * d; }
  double sd = sqrt(np_pairwise_sum(sq, m) / (double)(m - 1));
  return mean / (sd + 2.2250738585072014e-308);
}

/* RollingSharpe.calculate -- RewardFunctions.py:64-94 */
static double rolling_sharpe_calc(lo_t* o, const lobsim_reward_t* r, o_sharpe* st, double cash1, int64_t inv1, double p1) {
  const int maxw = r->asymmetric & 0xffff, minw = (r->asymmetric >> 16) & 0xffff;
  double new_aum = cash1 + p1 * (double)inv1; /* calculate_aum :61-62 */
  memmove(&st->aum[0], &st->aum[1], (size_t)(maxw - 1) * sizeof(double)); /* overwrite oldest + roll */
  st->aum[maxw - 1] = new_aum;
  st->n_filled = st->n_filled + 1 < maxw ? st->n_filled + 1 : maxw;
  if (st->n_filled < minw) return 0.0;
  return get_sharpe(o, &st->aum[maxw - st->n_filled], st->n_filled);
}

/* RewardFunctions.py:97-118 */
static double reward_calc(const lobsim_reward_t* r, double cash0, int64_t inv0, double p0, double cash1, int64_t inv1, double p1) {
  double cur = cash0 + (double)inv0 * p0;
  double nxt = cash1 + (double)inv1 * p1;
  double pnl = nxt - cur;
  if (r->kind == LOBSIM_REWARD_PNL) return pnl;
  double delta = p1 - p0;
  double term = r->inventory_aversion * (double)inv1 * delta;
  if (r->asymmetric) term = term > 0.0 ? term : 0.0;
  return pnl - term;
}

/* HistoricalOrderbookEnvironment.reset -- HOE.py:147-161 */
int lo_reset(lo_t* o, int episode_start_step, double* obs_out) {
  if (!o->has_stream) return LOBSIM_E_STATE;
  int start = episode_start_step - o->cfg.warmup_steps;
  int rc = lo_reset_book(o, start);
  if (rc) return rc;
  o->episode_start_step = episode_start_step;
  /* State.portfolio aliases env.initial_portfolio (HOE.py:153): inventory and cash carry over across resets */
  if (!o->cfg.portfolio_carryover) { o->inventory = o->cfg.initial_inventory; o->cash = o->cfg.initial_cash; }
  memset(o->prev_action, 0, sizeof o->prev_action);
  o->has_reset = 1;
  o->n_fills = 0; o->call_fills = 0;
  int64_t bb, bs, bv, sv;
  if (book_tops(o, &bb, &bs, &bv, &sv)) o->price = book_microprice(bb, bs, bv, sv); else o->price = NAN;
  int64_t ep_start_us = o->stream.t0_us + (int64_t)episode_start_step * o->cfg.step_us;
  for (int i = 0; i < o->cfg.n_features; i++) { /* _reset_features :218-221 */
    const lobsim_feature_t* fc = &o->cfg.features[i];
    feature_reset(o, i, ep_start_us - (int64_t)fc->lookback * fc->update_us);
  }
  for (int s = 0; s < o->cfg.warmup_steps; s++) { /* :155-157 */
    env_forward(o, NULL, 0);
    for (int i = 0; i < o->cfg.n_features; i++) feature_update(o, i);
  }
  if (obs_out) get_observation(o, NULL, obs_out);
  return LOBSIM_OK;
}

/* HistoricalOrderbookEnvironment.step -- HOE.py:163-178 */
static int step_impl(lo_t* o, const double* action, double* obs, double* reward, uint8_t* done);
int lo_step(lo_t* o, const double* action, double* obs, double* reward, uint8_t* done) {
  o->call_fills = 0;
  return step_impl(o, action, obs, reward, done);
}
static int step_impl(lo_t* o, const double* action, double* obs, double* reward, uint8_t* done) {
  if (!o->has_stream || !o->has_reset) return LOBSIM_E_STATE;
  o_msgs orders = {0};
  if (!o->dead) convert_action_to_orders(o, action, &orders);
  double cash0 = o->cash, p0 = o->price; int64_t inv0 = o->inventory; /* deepcopy(self.state) :166 */
  env_forward(o, orders.v, orders.n);
  free(orders.v);
  for (int i = 0; i < o->cfg.n_features; i++) feature_update(o, i);
  double r = o->cfg.step_reward.kind == LOBSIM_REWARD_ROLLING_SHARPE
                 ? rolling_sharpe_calc(o, &o->cfg.step_reward, &o->sharpe[0], o->cash, o->inventory, o->price)
                 : reward_calc(&o->cfg.step_reward, cash0, inv0, p0, o->cash, o->inventory, o->price);
  int d = 0;
  /* terminal_time - now < step/2  <=>  now_step >= episode_start + episode_steps (integers) */
  if (o->now_step >= o->episode_start_step + o->cfg.episode_steps) {
    r = o->cfg.terminal_reward.kind == LOBSIM_REWARD_ROLLING_SHARPE
            ? rolling_sharpe_calc(o, &o->cfg.terminal_reward, &o->sharpe[1], o->cash, o->inventory, o->price)
            : reward_calc(&o->cfg.terminal_reward, cash0, inv0, p0, o->cash, o->inventory, o->price);
    d = 1;
  }
  if (obs) get_observation(o, action, obs);
  if (reward) *reward = r;
  if (done) *done = (uint8_t)d;
  return LOBSIM_OK;
}

/* Agents -- rl4mm/agents/baseline_agents.py */
static double clamp_to_unit(double x) { const double eps = 0.00001; double m = x < 1 - eps ? x : 1 - eps; return m > -1 + eps ? m : -1 + eps; } /* :96-100 */
/* Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11), written from the paper:
 * ten rounds of  (L, R) pairs  c0,c1,c2,c3 -> hi(M1*c2)^c1^k0, lo(M1*c2), hi(M0*c0)^c3^k1, lo(M0*c0), keys bumped by the Weyl
 * constants.  Known-answer vectors of the Random123 distribution are checked in tests/test_oracle_golden.py. */
void lo_philox4x32_10(uint32_t ctr[4], uint32_t key0, uint32_t key1) {
  for (int round = 0; round < 10; round++) {
    uint64_t prod0 = (uint64_t)0xD2511F53u * (uint64_t)ctr[0];
    uint64_t prod1 = (uint64_t)0xCD9E8D57u * (uint64_t)ctr[2];
    uint32_t out0 = (uint32_t)(prod1 >> 32) ^ ctr[1] ^ key0;
    uint32_t out1 = (uint32_t)prod1;
    uint32_t out2 = (uint32_t)(prod0 >> 32) ^ ctr[3] ^ key1;
    uint32_t out3 = (uint32_t)prod0;
    ctr[0] = out0; ctr[1] = out1; ctr[2] = out2; ctr[3] = out3;
    key0 += 0x9E3779B9u; key1 += 0xBB67AE85u;
  }
}
/* RandomAgent.get_action = action_space.sample() (baseline_agents.py:9-18) for Box(0, high): uniform in [0, high_i).  The
 * device kernels have no global numpy RNG to share, so "random" is DEFINED as: dimension 2b / 2b+1 = the two 53-bit uniforms
 * of Philox(counter = (grid step, env index, b, 0), key = (seed, "LOBS")).  No reference parity target; this twin pins the
 * device implementation bit for bit. */
void lo_random_action(const lobsim_agent_t* ag, int32_t env_index, int64_t now_step, double* action) {
  for (uint32_t b = 0; b < 3; b++) {
    uint32_t ctr[4] = {(uint32_t)now_step, (uint32_t)env_index, b, 0u};
    lo_philox4x32_10(ctr, (uint32_t)ag->reserved, 0x4C4F4253u);
    uint64_t w0 = ((uint64_t)ctr[0] << 32) | ctr[1], w1 = ((uint64_t)ctr[2] << 32) | ctr[3];
    action[2 * b] = ag->fixed_action[2 * b] * ((double)(w0 >> 11) / 9007199254740992.0);
    if (2 * b + 1 < 5) action[2 * b + 1] = ag->fixed_action[2 * b + 1] * ((double)(w1 >> 11) / 9007199254740992.0);
  }
}
void lo_set_env_index(lo_t* o, int32_t env_index) { o->env_index = env_index; }

void lo_agent_action(const lobsim_agent_t* ag, const double* obs, double* action) {
  if (ag->kind == LOBSIM_AGENT_FIXED) { for (int i = 0; i < 5; i++) action[i] = ag->fixed_action[i]; return; }
  if (ag->kind == LOBSIM_AGENT_TERADACTYL) { /* :51-87 */
    double inventory = obs[ag->inventory_index];
    double denom = ag->max_inventory > 0 ? ag->max_inventory : 100.0;
    double w = ag->default_omega, ob, oa;
    if (inventory >= 0) {
      ob = w * (1 + (1 / w - 1) * pow(clamp_to_unit(inventory / denom), ag->exponent));
      oa = w * (1 - pow(clamp_to_unit(inventory / denom), ag->exponent));
    } else {
      ob = w * (1 - pow(fabs(clamp_to_unit(inventory / denom)), ag->exponent));
      oa = w * (1 + (1 / w - 1) * pow(fabs(clamp_to_unit(inventory / denom)), ag->exponent));
    }
    double kappa = (ag->max_kappa - ag->default_kappa) * pow(fabs(inventory / ag->max_inventory), ag->exponent) + ag->default_kappa;
    action[0] = (ob * (kappa - 2)) + 1;
    action[1] = (1 - ob) * (kappa - 2) + 1;
    action[2] = (oa * (kappa - 2)) + 1;
    action[3] = (1 - oa) * (kappa - 2) + 1;
    action[4] = ag->max_inventory * 2;
  }
}

/* generate_trajectory -- rl4mm/gym/utils.py:100-117 (without the reset; obs_t is the observation after step t) */
/* one row of the info series: what SimpleInfoCalculator.calculate (InfoCalculators.py:31-43) reads from the state at
 * the end of HistoricalOrderbookEnvironment.step (HOE.py:175-177) */
static void info_row(const lo_t* o, double* row) {
  const o_side* b = &o->central.s[0]; const o_side* s = &o->central.s[1];
  int tops = b->n > 0 && s->n > 0;
  row[LOBSIM_INFO_ASSET_PRICE] = o->price; row[LOBSIM_INFO_INVENTORY] = (double)o->inventory; row[LOBSIM_INFO_CASH] = o->cash;
  row[LOBSIM_INFO_AUM] = o->cash + o->price * (double)o->inventory;
  row[LOBSIM_INFO_BEST_BUY] = tops ? (double)b->lv[b->n - 1].price : NAN;
  row[LOBSIM_INFO_BEST_SELL] = tops ? (double)s->lv[0].price : NAN;
  row[LOBSIM_INFO_MARKET_SPREAD] = tops ? (double)(s->lv[0].price - b->lv[b->n - 1].price) : NAN;
  row[LOBSIM_INFO_ERR] = (double)o->err;
}

int lo_rollout(lo_t* o, int T, const lobsim_agent_t* ag, double* obs, double* act, double* rew, uint8_t* done) {
  return lo_rollout_info(o, T, ag, obs, act, rew, done, NULL);
}

int lo_rollout_info(lo_t* o, int T, const lobsim_agent_t* ag, double* obs, double* act, double* rew, uint8_t* done, double* info) {
  int od = lo_obs_dim(&o->cfg), ad = lo_action_dim(&o->cfg);
  double cur_obs[LOBSIM_MAX_FEATURES + 8], a[8];
  get_observation(o, o->prev_action, cur_obs);
  o->call_fills = 0;   /* one call: the device's per-call fill log spans all T steps */
  for (int t = 0; t < T; t++) {
    if (ag->kind == LOBSIM_AGENT_NONE) {
      env_forward(o, NULL, 0);
      for (int i = 0; i < o->cfg.n_features; i++) feature_update(o, i);
      if (obs) get_observation(o, NULL, obs + (size_t)t * od);
      continue;
    }
    if (ag->kind == LOBSIM_AGENT_EXTERNAL) memcpy(a, act + (size_t)t * ad, sizeof(double) * (size_t)ad);
    else if (ag->kind == LOBSIM_AGENT_RANDOM) lo_random_action(ag, o->env_index, o->now_step, a);
    else lo_agent_action(ag, cur_obs, a);
    double r; uint8_t d;
    step_impl(o, a, cur_obs, &r, &d);
    memcpy(o->prev_action, a, sizeof(double) * (size_t)ad);
    if (obs) memcpy(obs + (size_t)t * od, cur_obs, sizeof(double) * (size_t)od);
    if (act && ag->kind != LOBSIM_AGENT_EXTERNAL) memcpy(act + (size_t)t * ad, a, sizeof(double) * (size_t)ad);
    if (rew) rew[t] = r;
    if (done) done[t] = d;
    if (info) info_row(o, info + (size_t)t * LOBSIM_INFO_DIM);
  }
  return LOBSIM_OK;
}

/* ------------------------------------------------------------------------------------------------------------ */
/*  plumbing                                                                                                      */
/* ------------------------------------------------------------------------------------------------------------ */

int lo_obs_dim(const lobsim_cfg_t* c) { return c->n_features + (c->inc_prev_action_in_obs ? lo_action_dim(c) : 0); }
int lo_action_dim(const lobsim_cfg_t* c) { return (c->concentration >= 0 ? 2 : 4) + (c->market_order_clearing ? 1 : 0); }

lo_t* lo_create(const lobsim_cfg_t* cfg) {
  lo_t* o = (lo_t*)calloc(1, sizeof(lo_t));
  o->cfg = *cfg;
  map_init(&o->ext2int, 1024);
  for (int i = 0; i < cfg->n_features; i++) {
    int k = cfg->features[i].lookback + 2;
    o->feat[i].ring = (double*)calloc((size_t)k, sizeof(double));
    o->feat[i].iring[0] = (int64_t*)calloc((size_t)k, sizeof(int64_t));
    o->feat[i].iring[1] = (int64_t*)calloc((size_t)k, sizeof(int64_t));
    o->feat[i].hist = (double*)calloc((size_t)(cfg->features[i].norm_len > 0 ? cfg->features[i].norm_len : 1), sizeof(double));
  }
  o->inventory = cfg->initial_inventory; o->cash = cfg->initial_cash;
  return o;
}

void lo_destroy(lo_t* o) {
  if (!o) return;
  book_free(&o->central); book_free(&o->internal); map_free(&o->ext2int);
  for (int i = 0; i < o->cfg.n_features; i++) { free(o->feat[i].ring); free(o->feat[i].iring[0]); free(o->feat[i].iring[1]); free(o->feat[i].hist); }
  free(o->fills); free(o);
}

void lo_set_stream(lo_t* o, const lobsim_stream_t* s) { o->stream = *s; o->has_stream = 1; }

int lo_process_order(lo_t* o, const lobsim_order_t* ord, uint32_t* ref_out) {
  o_msg m; m.type = ord->type; m.dir = ord->direction; m.price = ord->price; m.vol = ord->volume;
  m.has_vol = !((ord->type == LOBSIM_MSG_DELETE || ord->type == LOBSIM_MSG_CANCEL) && ord->volume <= 0);
  m.is_ext = ord->is_external;
  if (ord->is_external) { m.ext = ord->ref; m.iid = 0; } else { m.ext = -1; m.iid = (int64_t)(ord->ref & 0x7fffffffu); }
  if (ord->type == LOBSIM_MSG_LIMIT || ord->type == LOBSIM_MSG_MARKET) m.iid = 0;
  if (ref_out) *ref_out = 0;
  const int peak_fills = o->peak_fills;
  process_order(o, &m, ref_out);
  o->peak_fills = peak_fills;   /* lobsim_process_orders returns its fills to the caller: they never enter the fill log */
  return LOBSIM_OK;
}

/* Exchange(central_orderbook=..., internal_orderbook=...) -- Exchange.py:40-49, with L3 entries in the lobsim_dump_book format
 * (per side best level first, FIFO inside a level; ref = LOBSIM_REF_AGENT | id marks the agent's orders, which also form the
 * internal book).  A new Exchange has a new OrderIdConvertor, so the external-id map is rebuilt from the given book; the id
 * counter moves above the largest id.  The clock, the portfolio and the price-range trackers stay; the error bits (and the
 * capacity high-water marks, which explain them) restart, as on the device (lobsim_set_book).
 * External orders carry no internal id in the dump: each gets the smallest id above its predecessor in the level, so that the
 * binary search by internal id (Exchange._find_queue_position) stays valid.  Returns LOBSIM_E_INVALID (book unchanged) for
 * unsorted levels, negative volumes, or agent ids that leave no room for the external orders queued before them. */
int lo_set_book(lo_t* o, const lobsim_book_entry_t* buy, int n_buy, const lobsim_book_entry_t* sell, int n_sell) {
  for (int side = 0; side < 2; side++) {   /* validate first: the book is only replaced by a valid one */
    const lobsim_book_entry_t* e = side ? sell : buy;
    const int n = side ? n_sell : n_buy;
    int64_t last = INT64_MIN;
    for (int i = 0; i < n; i++) {
      if (e[i].volume < 0) return LOBSIM_E_INVALID;
      if (i > 0 && e[i].price != e[i - 1].price) {
        if (side == 0 ? e[i].price >= e[i - 1].price : e[i].price <= e[i - 1].price) return LOBSIM_E_INVALID;
        last = INT64_MIN;
      }
      if (e[i].ref & LOBSIM_REF_AGENT) {
        const int64_t id = (int64_t)(e[i].ref & 0x7fffffffu);
        if (id <= last || id < 1) return LOBSIM_E_INVALID;
        last = id;
      } else if (e[i].ref == LOBSIM_REF_AGGREGATE) {
        if (last != INT64_MIN) return LOBSIM_E_INVALID;   /* a snapshot aggregate heads its level */
        last = -1;
      } else last = last < 1 ? 1 : last + 1;
    }
  }
  book_clear(&o->central); book_clear(&o->internal);
  map_free(&o->ext2int); map_init(&o->ext2int, 1024);
  int64_t max_id = 0;
  for (int side = 0; side < 2; side++) {
    const lobsim_book_entry_t* e = side ? sell : buy;
    const int n = side ? n_sell : n_buy;
    o_level* l = NULL; o_level* il = NULL;
    int64_t last = INT64_MIN;
    for (int i = 0; i < n; i++) {
      if (i == 0 || e[i].price != e[i - 1].price) { l = side_get_or_insert(&o->central.s[side], e[i].price); il = NULL; last = INT64_MIN; }
      o_order r; r.vol = e[i].volume;
      if (e[i].ref & LOBSIM_REF_AGENT) { r.iid = (int64_t)(e[i].ref & 0x7fffffffu); r.ext = -1; r.is_ext = 0; }
      else if (e[i].ref == LOBSIM_REF_AGGREGATE) { r.iid = -1; r.ext = -1; r.is_ext = 1; }
      else { r.iid = last < 1 ? 1 : last + 1; r.ext = e[i].ref; r.is_ext = 1; map_put(&o->ext2int, r.ext, r.iid); }
      last = r.iid;
      if (r.iid > max_id) max_id = r.iid;
      level_append(&o->central.s[side], l, r);
      if (!r.is_ext) {
        if (!il) il = side_get_or_insert(&o->internal.s[side], e[i].price);
        level_append(&o->internal.s[side], il, r);
      }
    }
  }
  if (o->counter < max_id) o->counter = max_id;
  reset_peaks(o);
  o->err = 0; o->dead = 0;
  return LOBSIM_OK;
}

void lo_peaks(const lo_t* o, int32_t* out) {
  for (int side = 0; side < 2; side++) {
    out[side] = o->central.s[side].peak_lv;
    out[2 + side] = o->central.s[side].peak_ord;
    out[4 + side] = o->internal.s[side].peak_ord;
  }
  out[6] = o->peak_fills;
}

void lo_clear_fills(lo_t* o) { o->n_fills = 0; }

int lo_get_fills(const lo_t* o, lobsim_fill_t* out, int cap) {
  int n = o->n_fills < cap ? o->n_fills : cap;
  memcpy(out, o->fills, (size_t)n * sizeof(lobsim_fill_t));
  return o->n_fills;
}

static int dump_side(const o_book* b, int side, lobsim_book_entry_t* out, int cap) {
  const o_side* s = &b->s[side];
  int n = 0;
  for (int k = 0; k < s->n; k++) {
    const o_level* l = side == 0 ? &s->lv[s->n - 1 - k] : &s->lv[k];
    for (int j = 0; j < l->n; j++) {
      if (n < cap) { out[n].price = (int32_t)l->price; out[n].volume = (int32_t)l->q[j].vol; out[n].ref = order_ref(&l->q[j]); out[n].level = k; }
      n++;
    }
  }
  return n;
}
int lo_dump_book(const lo_t* o, int side, lobsim_book_entry_t* out, int cap) { return dump_side(&o->central, side, out, cap); }

static int cmp_entry_ref(const void* a, const void* b) {
  uint32_t x = ((const lobsim_book_entry_t*)a)->ref, y = ((const lobsim_book_entry_t*)b)->ref;
  return x < y ? -1 : x > y;
}
int lo_dump_agent_orders(const lo_t* o, int side, lobsim_book_entry_t* out, int cap) {
  int n = dump_side(&o->internal, side, out, cap);
  qsort(out, (size_t)(n < cap ? n : cap), sizeof(lobsim_book_entry_t), cmp_entry_ref);
  return n;
}

void lo_get_state(const lo_t* o, lobsim_env_state_t* st) {
  memset(st, 0, sizeof *st);
  st->inventory = o->inventory; st->cash = o->cash; st->price = o->price;
  st->now_step = (int32_t)o->now_step; st->episode_start_step = (int32_t)o->episode_start_step;
  st->min_buy_price = (int32_t)o->min_buy_price; st->max_sell_price = (int32_t)o->max_sell_price;
  int64_t bb = 0, bs = 0, bv = 0, sv = 0;
  const o_side* b = &o->central.s[0]; const o_side* s = &o->central.s[1];
  if (b->n) { bb = b->lv[b->n - 1].price; bv = level_volume(&b->lv[b->n - 1]); }
  if (s->n) { bs = s->lv[0].price; sv = level_volume(&s->lv[0]); } else bs = INT32_MAX;
  st->best_buy = (int32_t)bb; st->best_sell = (int32_t)bs; st->best_buy_volume = (int32_t)bv; st->best_sell_volume = (int32_t)sv;
  st->err = o->err;
  for (int side = 0; side < 2; side++) {
    uint32_t n = 0;
    for (int k = 0; k < o->internal.s[side].n; k++) n += (uint32_t)o->internal.s[side].lv[k].n;
    st->n_agent_orders[side] = n;
  }
  st->next_agent_id = (uint32_t)o->counter;
}
