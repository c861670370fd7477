// lobsim.cu -- kernels and the C ABI (include/lobsim.h) of the B200-native LOB simulation step.
//
// Kernel design (DESIGN.md):
//   * one warp per book; a CTA is `warps_per_cta` independent warps, no block-level synchronisation at all;
//   * the book blob lives in shared memory for the whole launch: HBM -> smem by one TMA bulk copy
//     (cp.async.bulk + mbarrier) at the start, smem -> HBM by one bulk store at the end;
//   * historical messages are streamed by TMA bulk copies of 512-byte tiles (32 x 16 B records) into a per-warp
//     double buffer, prefetched one tile ahead; all 32 lanes read a record with one broadcast LDS.128;
//   * book operations are warp-collective (ballot / popc / ffs level and order search, <=32-entry shifts);
//   * features run one per lane, the reward and the rollout tensors are written straight from the kernel.
// fp64 everywhere the reference uses Python floats, compiled with --fmad=false (no FMA contraction).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <utility>
#include <new>
#include <string>
#include <vector>

#include "lobsim.h"

#include "kernels.cuh"


#include "layouts.h"

// ---- the compiled straight-line layouts (layouts.h; one pair of translation units each, fast_layout.cu) -------------
struct FastLayoutOps {
  int NL, NO, NA;
  bool env_hot;
  cudaError_t (*attrs)(int dyn_replay, int dyn_env);
  cudaError_t (*attrs_rare)(int dyn_env);
  void (*replay)(int grid, int block, size_t dyn, cudaStream_t stream, const AdvParams& p, const EnvConst& ec);
  void (*replay_flat)(int grid, int block, size_t dyn, cudaStream_t stream, const AdvParams& p, const EnvConst& ec);
  void (*to_sorted)(unsigned char* blobs, int n_envs, cudaStream_t stream);
  void (*env)(int mode, bool sync, int grid, int block, size_t dyn, cudaStream_t stream, const AdvParams& p, const EnvConst& ec);
  void (*env_rare)(int mode, bool sync, int grid, int block, size_t dyn, cudaStream_t stream, const AdvParams& p, const EnvConst& ec);
};
#define X(i, nl, no, na)                                                                                                   \
  cudaError_t lobsim_fast##i##_attrs(int, int);                                                                            \
  cudaError_t lobsim_fast##i##_attrs_rare(int);                                                                            \
  void lobsim_fast##i##_replay(int, int, size_t, cudaStream_t, const AdvParams&, const EnvConst&);                         \
  void lobsim_fast##i##_replay_flat(int, int, size_t, cudaStream_t, const AdvParams&, const EnvConst&);                    \
  void lobsim_fast##i##_to_sorted(unsigned char*, int, cudaStream_t);                                                      \
  void lobsim_fast##i##_env(int, bool, int, int, size_t, cudaStream_t, const AdvParams&, const EnvConst&);                 \
  void lobsim_fast##i##_env_rare(int, bool, int, int, size_t, cudaStream_t, const AdvParams&, const EnvConst&);
LOBSIM_FAST_LAYOUTS(X)
#undef X
#define X(i, nl, no, na) {nl, no, na, LOBSIM_LAYOUT_ENV_HOT(nl, no, na), lobsim_fast##i##_attrs, lobsim_fast##i##_attrs_rare, lobsim_fast##i##_replay, lobsim_fast##i##_replay_flat, lobsim_fast##i##_to_sorted, lobsim_fast##i##_env, lobsim_fast##i##_env_rare},
static const FastLayoutOps g_fast_layouts[LOBSIM_N_FAST_LAYOUTS] = {LOBSIM_FAST_LAYOUTS(X)};
#undef X
static const FastLayoutOps* find_fast_layout(const Layout& L) {
  for (int i = 0; i < LOBSIM_N_FAST_LAYOUTS; i++)
    if (g_fast_layouts[i].NL == L.NL && g_fast_layouts[i].NO == L.NO && g_fast_layouts[i].NA == L.NA) return &g_fast_layouts[i];
  return nullptr;
}

// ====================================================================================================================
//  Exchange.process_order for a list of orders (drop-in / test entry point; one warp, sequential)
// ====================================================================================================================
struct OrdParams {
  unsigned char* blobs; Layout L; int32_t n_envs; int32_t blob_in_global;
  const lobsim_order_t* orders; int32_t n;
  lobsim_fill_t* fills; int32_t max_fills; int32_t* n_fills; uint32_t* refs_out;
};

__global__ void __launch_bounds__(32) k_process_orders(const __grid_constant__ OrdParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int lane = threadIdx.x;
  Book b; b.blob = smem; b.L = p.L; b.lane = lane;
  WarpState w;
  int cur_env = -1, total_fills = 0;
  long long inventory_in = 0; double cash_in = 0.0;
  auto load_env = [&](int env) {
    if (p.blob_in_global) b.blob = p.blobs + (size_t)env * p.L.blob_bytes;   // deep-book mode: in place
    else {
      const uint4* src = reinterpret_cast<const uint4*>(p.blobs + (size_t)env * p.L.blob_bytes);
      uint4* dst = reinterpret_cast<uint4*>(smem);
      for (int i = lane; i < p.L.blob_bytes / 16; i += 32) dst[i] = src[i];
    }
    __syncwarp();
    load_state<true>(b, w);
    inventory_in = w.inventory; cash_in = w.cash;
    w.fill_log = p.fills ? p.fills + total_fills : nullptr;
    w.fill_cap = p.max_fills - total_fills; w.n_fills = 0;
  };
  auto store_env = [&](int env) {
    // Exchange.process_order only returns the fills: the portfolio belongs to the env and moves in its step (HOE.py:280-289)
    w.inventory = inventory_in; w.cash = cash_in;
    store_state<true>(b, w);
    if (!p.blob_in_global) {
      uint4* dst = reinterpret_cast<uint4*>(p.blobs + (size_t)env * p.L.blob_bytes);
      const uint4* src = reinterpret_cast<const uint4*>(smem);
      for (int i = lane; i < p.L.blob_bytes / 16; i += 32) dst[i] = src[i];
    }
    __syncwarp();
    total_fills += w.n_fills < w.fill_cap ? w.n_fills : w.fill_cap;
  };
  for (int k = 0; k < p.n; k++) {
    const lobsim_order_t o = p.orders[k];
    if (o.env < 0 || o.env >= p.n_envs) continue;
    if (o.env != cur_env) { if (cur_env >= 0) store_env(cur_env); load_env(o.env); cur_env = o.env; }
    uint32_t id = 0;
    const bool is_agent = !o.is_external;
    const bool has_vol = !((o.type == LOBSIM_MSG_DELETE || o.type == LOBSIM_MSG_CANCEL) && o.volume <= 0);
    if (!w.dead) {
      if (has_vol && o.volume <= 0) w.err |= LOBSIM_ERR_BAD_VOLUME;
      else if (o.type == LOBSIM_MSG_LIMIT || o.type == LOBSIM_MSG_MARKET)
        id = submit_or_execute<true>(b, w, o.direction, o.price, o.volume, is_agent ? 0u : o.ref, o.type == LOBSIM_MSG_LIMIT, is_agent);
      else remove_order<true>(b, w, o.direction, o.price, o.volume, has_vol, is_agent ? (LOBSIM_REF_AGENT | (o.ref & 0x7fffffffu)) : o.ref, is_agent);
    }
    if (p.refs_out && lane == 0) p.refs_out[k] = id;
  }
  if (cur_env >= 0) store_env(cur_env);
  if (lane == 0 && p.n_fills) *p.n_fills = total_fills;
}

// ====================================================================================================================
//  per-env state summary (one thread per env, reads the blob in HBM)
// ====================================================================================================================
__global__ void k_get_state(const unsigned char* blobs, Layout L, int first, int n, lobsim_env_state_t* out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned char* blob = blobs + (size_t)(first + i) * L.blob_bytes;
  const BookHdr* h = reinterpret_cast<const BookHdr*>(blob);
  lobsim_env_state_t s;
  s.inventory = h->inventory; s.cash = h->cash; s.price = h->price; s.now_step = h->now_step;
  s.episode_start_step = h->episode_start_step; s.min_buy_price = h->min_buy; s.max_sell_price = h->max_sell;
  s.err = h->err; s.stream_id = h->stream_id; s.n_agent_orders[0] = h->nag[0]; s.n_agent_orders[1] = h->nag[1];
  s.next_agent_id = h->next_agent_id; s.reserved = 0;   // book form, set below
  int best[2] = {0, INT32_MAX}, bvol[2] = {0, 0};
  const bool flat = h->cnt[0][0] < 0;   // the flat form (book_flat.cuh): cnt[side][1] orders {price, ref, volume, seq} at the order array
  for (int side = 0; flat && side < 2; side++) {
    const int n = h->cnt[side][1];
    const uint4* pool = reinterpret_cast<const uint4*>(blob + L.side_off + side * L.side_stride + L.ord_off);
    int bp = side ? INT32_MAX : INT32_MIN, v = 0;
    for (int k = 0; k < n; k++) { const int pr = (int)pool[k].x; if (side ? pr < bp : pr > bp) bp = pr; }
    for (int k = 0; k < n; k++) if ((int)pool[k].x == bp) v += (int)pool[k].z;
    if (n) { best[side] = bp; bvol[side] = v; }
  }
  for (int side = 0; !flat && side < 2; side++) {
    int nlv = h->cnt[side][0];
    if (!nlv) continue;
    const unsigned char* sb = blob + L.side_off + side * L.side_stride;
    const int32_t* lvp = reinterpret_cast<const int32_t*>(sb);
    const uint16_t* lvend = reinterpret_cast<const uint16_t*>(sb + L.lvend_off);
    const uint2* ord = reinterpret_cast<const uint2*>(sb + L.ord_off);
    best[side] = lvp[nlv - 1];
    int start = nlv > 1 ? lvend[nlv - 2] : 0, end = lvend[nlv - 1], v = 0;
    for (int k = start; k < end; k++) v += (int)ord[k].x;
    bvol[side] = v;
  }
  s.best_buy = best[0]; s.best_sell = best[1]; s.best_buy_volume = bvol[0]; s.best_sell_volume = bvol[1];
  { const unsigned n0 = (unsigned)h->cnt[0][1], n1 = (unsigned)h->cnt[1][1];
    s.reserved = (flat ? 1u : 0u) | ((n0 > 4095u ? 4095u : n0) << 8) | ((n1 > 4095u ? 4095u : n1) << 20); }
  out[i] = s;
}

__global__ void k_init_blobs(unsigned char* blobs, Layout L, int n, long long inventory, double cash) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  BookHdr* h = reinterpret_cast<BookHdr*>(blobs + (size_t)i * L.blob_bytes);
  memset(h, 0, sizeof(BookHdr));
  h->next_agent_id = 1; h->inventory = inventory; h->cash = cash; h->stream_id = 0;
}

// ====================================================================================================================
//  host side: handle + C ABI
// ====================================================================================================================
static thread_local std::string g_last_error;
static int fail(int code, const std::string& msg) { g_last_error = msg; return code; }
#define CUDA_TRY(expr)                                                                                             \
  do {                                                                                                             \
    cudaError_t e__ = (expr);                                                                                      \
    if (e__ != cudaSuccess) return fail(LOBSIM_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));       \
  } while (0)

struct lobsim {
  lobsim_cfg_t cfg;
  EnvConst ec;
  Layout L;
  int device;
  int warps_per_cta;
  int env_warps_per_cta;
  int warp_smem;
  int replay_warp_smem;              // straight-line replay kernels: the blob WITHOUT the agent tables + message tiles + barriers
  int replay_warps_per_cta;
  unsigned char* blobs = nullptr;
  FeatState* fstate = nullptr;
  NormState* nstate = nullptr;          // rolling z-score state: only with normalisation_on features
  double* beta_tab = nullptr;           // [2][32] ln x_k, ln(1 - x_k) at the quote-level midpoints (BetaOrderDistributor)
  double* rings = nullptr;
  double* rs_ring = nullptr;
  int32_t* rs_state = nullptr;
  lobsim_fill_t* fill_log = nullptr;
  int32_t* fill_count = nullptr;
  lobsim_agent_t* agents_dev = nullptr; // per-env agents of lobsim_rollout_agents (allocated on first use)
  bool rare_paths = false;              // z-score normalisation or a RollingSharpe reward configured: kernels with that code
  std::vector<lobsim_stream_t> streams;
  lobsim_stream_t* streams_dev = nullptr;
  int streams_cap = 0;
  // staging for the *_host entry points
  double* st_actions = nullptr; double* st_obs = nullptr; double* st_rew = nullptr; uint8_t* st_done = nullptr;
  lobsim_env_state_t* st_state = nullptr;
  lobsim_msg_t* st_msgs = nullptr; uint64_t st_msgs_cap = 0;
  bool has_reset = false;
  bool force_general = false;         // LOBSIM_FORCE_GENERAL=1: always use the runtime-layout kernels (testing)
  int replay_hybrid = -1;             // k_replay_hyb (book_hybrid.cuh) as the replay launch of a deep compiled layout (NL >= 64, NO >= 512):
                                      // -1 (default) when NO >= 1024, LOBSIM_REPLAY_HYBRID=1 on every such layout, =0 never
  bool replay_flat = true;            // LOBSIM_REPLAY_FLAT=0: the replay fast path keeps every book in the sorted level arrays (A/B, testing)
  bool flat_blobs = true;             // LOBSIM_FLAT_BLOBS=0: the fast kernels never keep a book in the flat order pools across launches
                                      // (env kernels: sorted path only; replay: converts back at the end of every launch)
  lobsim_order_t* po_orders = nullptr; uint32_t* po_refs = nullptr; lobsim_fill_t* po_fills = nullptr; int32_t* po_nf = nullptr;   // lobsim_process_orders staging
  int po_cap = 0, po_fill_cap = 0;
  int32_t* defer_count = nullptr; int2* defer_list = nullptr;   // env HOT kernel -> DEFERRED kernel hand-over (kernels.cuh ENV_HOT)
  bool blob_in_global = false;        // deep-book mode: the blob exceeds the shared memory of an SM and is worked on in place in HBM
  bool maybe_flat = false;            // some blob in HBM may be in the flat form: ensure_sorted() before anything that reads level arrays
  bool agent_orders_possible = false; // an agent order may rest in some book (disables the replay fast path)
  const FastLayoutOps* fast = nullptr; // compiled straight-line kernels for these capacities, or null: general kernel
  int64_t launches = 0;
};

extern "C" {

const char* lobsim_last_error(void) { return g_last_error.c_str(); }
int lobsim_abi_version(void) { return LOBSIM_ABI_VERSION; }
int lobsim_action_dim(const lobsim_cfg_t* c) { return (c->concentration >= 0 ? 2 : 4) + (c->market_order_clearing ? 1 : 0); }
int lobsim_obs_dim(const lobsim_cfg_t* c) { return c->n_features + (c->inc_prev_action_in_obs ? lobsim_action_dim(c) : 0); }

static int validate_cfg(const lobsim_cfg_t* c) {
  if (!c) return fail(LOBSIM_E_INVALID, "cfg is null");
  if (c->abi_version != LOBSIM_ABI_VERSION) return fail(LOBSIM_E_INVALID, "abi_version mismatch");
  if (c->n_envs <= 0 || c->n_levels <= 0 || c->tick_size <= 0 || c->step_us <= 0) return fail(LOBSIM_E_INVALID, "n_envs, n_levels, tick_size, step_us must be positive");
  if (1000000 % c->step_us) return fail(LOBSIM_E_INVALID, "step_us must divide one second");
  int Q = c->max_quote_level - c->min_quote_level;
  if (Q <= 0 || Q > 32) return fail(LOBSIM_E_INVALID, "1 <= max_quote_level - min_quote_level <= 32");
  if (c->n_features < 0 || c->n_features > LOBSIM_MAX_FEATURES) return fail(LOBSIM_E_INVALID, "too many features");
  if (c->max_levels_per_side < 4 || c->max_levels_per_side % 4 || c->max_levels_per_side > 4096) return fail(LOBSIM_E_INVALID, "max_levels_per_side must be a multiple of 4 in [4, 4096]");
  if (c->max_orders_per_side < c->max_levels_per_side || c->max_orders_per_side > 65535) return fail(LOBSIM_E_INVALID, "max_orders_per_side must be in [max_levels_per_side, 65535]");
  if (c->max_agent_orders < 1 || c->max_agent_orders > 1024) return fail(LOBSIM_E_INVALID, "max_agent_orders must be in [1, 1024]");
  if (c->n_levels > c->max_levels_per_side) return fail(LOBSIM_E_INVALID, "n_levels exceeds max_levels_per_side");
  if (c->warmup_steps < 0 || c->episode_steps <= 0) return fail(LOBSIM_E_INVALID, "bad episode_steps / warmup_steps");
  const lobsim_reward_t* rw[2] = {&c->step_reward, &c->terminal_reward};
  for (int i = 0; i < 2; i++) {
    if (rw[i]->kind < 0 || rw[i]->kind > LOBSIM_REWARD_ROLLING_SHARPE) return fail(LOBSIM_E_INVALID, "unknown reward kind");
    if (rw[i]->kind == LOBSIM_REWARD_ROLLING_SHARPE) {
      const int maxw = rw[i]->asymmetric & 0xffff, minw = (rw[i]->asymmetric >> 16) & 0xffff;
      if (minw < 2 || minw > maxw || maxw > LOBSIM_MAX_SHARPE_WINDOW) return fail(LOBSIM_E_INVALID, "ROLLING_SHARPE: need 2 <= min_window <= max_window <= 256");
    }
  }
  for (int i = 0; i < c->n_features; i++) {
    const lobsim_feature_t& f = c->features[i];
    if (f.kind < 0 || f.kind > LOBSIM_FEAT_AMIHUD_LAMBDA) return fail(LOBSIM_E_INVALID, "unknown feature kind");
    if (f.kind == LOBSIM_FEAT_AMIHUD_LAMBDA && (f.iparam < 1 || f.iparam > 16383 || f.lookback % f.iparam || f.lookback / f.iparam < 2 || f.lookback / f.iparam > 65535))
      return fail(LOBSIM_E_INVALID, "AMIHUD_LAMBDA: lookback must be (true_lookback + 1) * slowing_factor with true_lookback >= 1");
    if (f.update_us <= 0 || f.update_us > 60000000 || f.lookback < 0) return fail(LOBSIM_E_INVALID, "bad feature update_us / lookback");
    if (f.norm_len < 0 || f.norm_len > 10000000) return fail(LOBSIM_E_INVALID, "bad feature norm_len");
    if (f.kind == LOBSIM_FEAT_TIME_OF_DAY && f.iparam <= 0) return fail(LOBSIM_E_INVALID, "TIME_OF_DAY needs n_buckets > 0");
    if ((f.kind == LOBSIM_FEAT_VOLATILITY || f.kind == LOBSIM_FEAT_TRADE_DIR_IMBALANCE || f.kind == LOBSIM_FEAT_TRADE_VOL_IMBALANCE) && f.lookback < 1)
      return fail(LOBSIM_E_INVALID, "windowed feature needs lookback >= 1");
  }
  return LOBSIM_OK;
}

int64_t lobsim_state_bytes(const lobsim_cfg_t* c) {
  if (validate_cfg(c)) return LOBSIM_E_INVALID;
  return make_layout(c->max_levels_per_side, c->max_orders_per_side, c->max_agent_orders).blob_bytes;
}

static int warp_smem_bytes(const Layout& L) { return (L.blob_bytes + 2 * MSG_TILE_BYTES + scratch_bytes(L.NA) + 32 + 128 + 127) & ~127; }
static int replay_warp_smem_bytes(const Layout& L) { return (L.agent_off + 2 * MSG_TILE_BYTES + 32 + 127) & ~127; }

int lobsim_create(const lobsim_cfg_t* cfg, int device, lobsim_t** out) {
  if (!out) return fail(LOBSIM_E_INVALID, "out is null");
  int rc = validate_cfg(cfg);
  if (rc) return rc;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(LOBSIM_E_CUDA, "no CUDA device: the lobsim hot path has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(LOBSIM_E_INVALID, "bad device index");
  CUDA_TRY(cudaSetDevice(device));
  lobsim* h = new (std::nothrow) lobsim();
  if (!h) return fail(LOBSIM_E_NOMEM, "out of host memory");
  h->cfg = *cfg; h->device = device;
  { const char* e = getenv("LOBSIM_FORCE_GENERAL"); h->force_general = e && e[0] == '1'; }
  { const char* e = getenv("LOBSIM_REPLAY_FLAT"); h->replay_flat = !(e && e[0] == '0'); }
  { const char* e = getenv("LOBSIM_REPLAY_HYBRID"); h->replay_hybrid = e && e[0] == '1' ? 1 : e && e[0] == '0' ? 0 : -1; }
  { const char* e = getenv("LOBSIM_FLAT_BLOBS"); h->flat_blobs = !(e && e[0] == '0'); }
  h->rare_paths = cfg->step_reward.kind == LOBSIM_REWARD_ROLLING_SHARPE || cfg->terminal_reward.kind == LOBSIM_REWARD_ROLLING_SHARPE;
  for (int i = 0; i < cfg->n_features; i++) h->rare_paths = h->rare_paths || cfg->features[i].norm_len > 0;
  h->L = make_layout(cfg->max_levels_per_side, cfg->max_orders_per_side, cfg->max_agent_orders);
  h->warp_smem = warp_smem_bytes(h->L);
  int max_smem = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  if (h->L.NO > 65535 || h->L.NL > 65535) { delete h; return fail(LOBSIM_E_INVALID, "at most 65535 levels / orders per side (16-bit level ends)"); }
  if (h->warp_smem > max_smem - 1024) {
    // deep-book mode: the blob stays in HBM / L2 and the general kernel works on it in place (k_advance, blob_in_global)
    h->blob_in_global = true;
    h->force_general = true;
    h->warp_smem = (2 * MSG_TILE_BYTES + scratch_bytes(h->L.NA) + 32 + 128 + 127) & ~127;
    static bool warned_deep = false;
    if (!warned_deep) {
      warned_deep = true;
      fprintf(stderr, "lobsim: capacities {levels %d, orders %d, agent orders %d} = %d bytes per book exceed the shared memory of an SM: "
                      "deep-book mode, the books are worked on in place in HBM (same results, several times slower per order)\n",
              h->L.NL, h->L.NO, h->L.NA, h->L.blob_bytes);
    }
  }
  // warps (= books) per CTA: as many resident books per SM as the shared memory allows -- deep books are smem-bound, and a CTA
  // size that does not divide the SM's shared memory wastes up to half of it (128/1536/64 capacities: 30 KB per book, 4 books
  // per CTA = one CTA = 4 books per SM, 1 book per CTA = 7 books per SM).  Ties go to the larger CTA.
  int sm_smem = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&sm_smem, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device));
  // `keep`: the largest CTA within that fraction of the best residency wins (the env kernel prefers large CTAs: its warps move
  // through the phases of a step together, kernels.cuh).
  h->replay_warp_smem = replay_warp_smem_bytes(h->L);
  auto best_wpc = [&](int max_wpc, double keep, int ws) {
    int books_of[65] = {0}, best_books = 0;
    for (int w = 1; w <= max_wpc && w <= 64; w++) {
      if ((long long)w * ws > max_smem - 1024) break;
      const int ctas = sm_smem / (w * ws + 1024);               // 1 KB per CTA is reserved by the driver
      books_of[w] = (ctas > 32 ? 32 : ctas) * w;
      if (books_of[w] > best_books) best_books = books_of[w];
    }
    int best = 1;
    for (int w = 1; w <= max_wpc && w <= 64; w++) if (books_of[w] > 0 && books_of[w] >= keep * best_books) best = w;
    return best;
  };
  h->warps_per_cta = best_wpc(4, 1.0, h->warp_smem);
  h->replay_warps_per_cta = best_wpc(4, 1.0, h->replay_warp_smem);
  h->env_warps_per_cta = best_wpc(LOBSIM_ENVFAST_WARPS, 0.95, h->warp_smem);   // (deep 128/1024/64 books: 5 warps x 2 CTAs = 10 resident, +11 % over 8 x 1)
  { const char* e = getenv("LOBSIM_ENV_WPC"); const int w = e ? atoi(e) : 0;   // A/B override (tools/)
    if (w >= 1 && w <= LOBSIM_ENVFAST_WARPS && (long long)w * h->warp_smem <= max_smem - 1024) h->env_warps_per_cta = w; }
  CUDA_TRY((cudaFuncSetAttribute(k_advance<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->warps_per_cta * h->warp_smem)));
  CUDA_TRY((cudaFuncSetAttribute(k_advance<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->warps_per_cta * h->warp_smem)));
  h->fast = h->force_general ? nullptr : find_fast_layout(h->L);
  if (h->fast && h->fast->env_hot) {   // (allocated here, not at the first launch: that one may be inside a CUDA-graph capture)
    CUDA_TRY(cudaMalloc(&h->defer_count, sizeof(int32_t)));
    CUDA_TRY(cudaMalloc(&h->defer_list, (size_t)cfg->n_envs * sizeof(int2)));
  }
  if (h->fast) {
    CUDA_TRY(h->fast->attrs(h->replay_warps_per_cta * h->replay_warp_smem, h->env_warps_per_cta * h->warp_smem));
    if (h->rare_paths) CUDA_TRY(h->fast->attrs_rare(h->env_warps_per_cta * h->warp_smem));
  } else if (!h->force_general) {
    static bool warned = false;   // once per process
    if (!warned) {
      warned = true;
      fprintf(stderr, "lobsim: no compiled straight-line kernel for capacities {levels %d, orders %d, agent orders %d}: using the "
                      "general runtime-layout kernel (same results, slower); compiled triples are listed in csrc/layouts.h\n",
              h->L.NL, h->L.NO, h->L.NA);
    }
  }
  CUDA_TRY((cudaFuncSetAttribute(k_advance<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)));
  CUDA_TRY((cudaFuncSetAttribute(k_advance<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)));
  if (!h->blob_in_global) CUDA_TRY(cudaFuncSetAttribute(k_process_orders, cudaFuncAttributeMaxDynamicSharedMemorySize, h->L.blob_bytes));
  // feature rings
  memset(&h->ec, 0, sizeof h->ec);
  h->ec.cfg = *cfg;
  int slots = 0;
  for (int i = 0; i < cfg->n_features; i++) {
    const lobsim_feature_t& ft = cfg->features[i];
    int need = ft.lookback + 2;
    if (ft.kind == LOBSIM_FEAT_AMIHUD_LAMBDA) { const int kk = ft.lookback / ft.iparam - 1; if (2 * kk + 2 > need) need = 2 * kk + 2; }
    h->ec.ring_off[i] = slots; slots += need;
    h->ec.hist_off[i] = slots; slots += ft.norm_len > 0 ? ft.norm_len : 0;
  }
  h->ec.ring_stride = (slots + 1) & ~1;
  h->ec.action_dim = lobsim_action_dim(cfg); h->ec.obs_dim = lobsim_obs_dim(cfg);
  h->ec.steps_per_sec = (int)(1000000 / cfg->step_us); h->ec.outer_prop = (double)cfg->outer_levels / (double)cfg->n_levels;
  h->ec.steps_per_min = (int)(60000000 / cfg->step_us);
  bool any_norm = false;
  for (int i = 0; i < cfg->n_features; i++) {
    const lobsim_feature_t& ft = cfg->features[i];
    any_norm = any_norm || ft.norm_len > 0;
    if (ft.kind == LOBSIM_FEAT_TIME_OF_DAY) { // bucket_size = (15:30 - 10:00) / n_buckets: timedelta division rounds half to even (Features.py:526-536)
      const long long tot = (15LL * 3600 + 1800 - 10LL * 3600) * 1000000, nb = ft.iparam;
      long long bucket = tot / nb, rem = tot % nb;
      if (2 * rem > nb || (2 * rem == nb && (bucket & 1))) bucket++;
      h->ec.feat_aux[i] = bucket;
    }
  }
  {
    const int Q = cfg->max_quote_level - cfg->min_quote_level;
    double tab[64];
    for (int k = 0; k < 32; k++) {   // OrderDistributors.py:37: midpoints 1 / Q * (k + 0.5)
      const double x = 1.0 / (double)Q * ((double)k + 0.5);
      tab[k] = k < Q ? log(x) : 0.0; tab[32 + k] = k < Q ? log1p(-x) : 0.0;
    }
    CUDA_TRY(cudaMalloc(&h->beta_tab, sizeof tab));
    CUDA_TRY(cudaMemcpy(h->beta_tab, tab, sizeof tab, cudaMemcpyHostToDevice));
  }
  const size_t n = (size_t)cfg->n_envs;
  CUDA_TRY(cudaMalloc(&h->blobs, n * h->L.blob_bytes));
  CUDA_TRY(cudaMalloc(&h->fstate, n * LOBSIM_MAX_FEATURES * sizeof(FeatState)));
  CUDA_TRY(cudaMemset(h->fstate, 0, n * LOBSIM_MAX_FEATURES * sizeof(FeatState)));
  if (any_norm) {
    CUDA_TRY(cudaMalloc(&h->nstate, n * LOBSIM_MAX_FEATURES * sizeof(NormState)));
    CUDA_TRY(cudaMemset(h->nstate, 0, n * LOBSIM_MAX_FEATURES * sizeof(NormState)));
  }
  {
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    const size_t ring_bytes = n * (size_t)(h->ec.ring_stride > 0 ? h->ec.ring_stride : 2) * sizeof(double);
    if (ring_bytes > free_b) { lobsim_destroy(h); return fail(LOBSIM_E_NOMEM, "feature windows / normalisation histories (n_envs x sum(lookback + max_norm_len) x 8 B) exceed the free HBM"); }
    CUDA_TRY(cudaMalloc(&h->rings, ring_bytes));
  }
  CUDA_TRY(cudaMemset(h->blobs, 0, n * h->L.blob_bytes));
  if (cfg->step_reward.kind == LOBSIM_REWARD_ROLLING_SHARPE || cfg->terminal_reward.kind == LOBSIM_REWARD_ROLLING_SHARPE) {
    CUDA_TRY(cudaMalloc(&h->rs_ring, n * 3 * LOBSIM_MAX_SHARPE_WINDOW * sizeof(double)));
    CUDA_TRY(cudaMalloc(&h->rs_state, n * 4 * sizeof(int32_t)));
    CUDA_TRY(cudaMemset(h->rs_state, 0, n * 4 * sizeof(int32_t)));
  }
  if (cfg->fill_log_capacity > 0) {
    CUDA_TRY(cudaMalloc(&h->fill_log, n * (size_t)cfg->fill_log_capacity * sizeof(lobsim_fill_t)));
    CUDA_TRY(cudaMalloc(&h->fill_count, n * sizeof(int32_t)));
    CUDA_TRY(cudaMemset(h->fill_count, 0, n * sizeof(int32_t)));
  }
  k_init_blobs<<<(cfg->n_envs + 127) / 128, 128>>>(h->blobs, h->L, cfg->n_envs, cfg->initial_inventory, cfg->initial_cash);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  h->launches++;
  *out = h;
  return LOBSIM_OK;
}

int lobsim_destroy(lobsim_t* h) {
  if (!h) return LOBSIM_OK;
  cudaSetDevice(h->device);
  cudaFree(h->blobs); cudaFree(h->fstate); cudaFree(h->nstate); cudaFree(h->beta_tab); cudaFree(h->rings); cudaFree(h->rs_ring); cudaFree(h->rs_state); cudaFree(h->fill_log); cudaFree(h->fill_count); cudaFree(h->agents_dev);
  cudaFree(h->streams_dev); cudaFree(h->st_actions); cudaFree(h->st_obs); cudaFree(h->st_rew); cudaFree(h->st_done);
  cudaFree(h->st_state); cudaFree(h->st_msgs);
  cudaFree(h->po_orders); cudaFree(h->po_refs); cudaFree(h->po_fills); cudaFree(h->po_nf); cudaFree(h->defer_count); cudaFree(h->defer_list);
  delete h;
  return LOBSIM_OK;
}

int lobsim_load_stream(lobsim_t* h, int stream_id, const lobsim_stream_t* s) {
  if (!h || !s) return fail(LOBSIM_E_INVALID, "null argument");
  if (stream_id < 0 || stream_id > 65535) return fail(LOBSIM_E_INVALID, "bad stream id");
  if (!s->step_off || !s->snapshots || !s->snap_valid || (!s->msgs && s->n_msgs)) return fail(LOBSIM_E_INVALID, "stream arrays missing");
  if (s->t0_us % 1000000) return fail(LOBSIM_E_INVALID, "t0_us must be a whole second");
  if (s->n_msgs >= 0xffffffffull) return fail(LOBSIM_E_INVALID, "more than 2^32-1 messages in one stream");
  if (((uintptr_t)s->msgs & 15) != 0) return fail(LOBSIM_E_INVALID, "msgs must be 16-byte aligned");
  CUDA_TRY(cudaSetDevice(h->device));
  if ((int)h->streams.size() <= stream_id) {
    lobsim_stream_t empty; memset(&empty, 0, sizeof empty);
    h->streams.resize(stream_id + 1, empty);
  }
  h->streams[stream_id] = *s;
  h->streams[stream_id].reserved = (uint32_t)(s->t0_us % 60000000);   // the kernels' 32-bit update-frequency gate (us_in_minute)
  if (h->streams_cap < (int)h->streams.size()) {
    CUDA_TRY(cudaDeviceSynchronize());
    cudaFree(h->streams_dev);
    h->streams_cap = (int)h->streams.size() * 2;
    CUDA_TRY(cudaMalloc(&h->streams_dev, h->streams_cap * sizeof(lobsim_stream_t)));
  }
  CUDA_TRY(cudaMemcpy(h->streams_dev, h->streams.data(), h->streams.size() * sizeof(lobsim_stream_t), cudaMemcpyHostToDevice));
  return LOBSIM_OK;
}

static void base_params(lobsim* h, AdvParams& p) {
  memset(&p, 0, sizeof p);
  p.blobs = h->blobs; p.fstate = h->fstate; p.nstate = h->nstate; p.beta_tab = h->beta_tab; p.rings = h->rings; p.rs_ring = h->rs_ring; p.rs_state = h->rs_state; p.streams = h->streams_dev; p.n_streams = (int)h->streams.size();
  p.fill_log = h->fill_log; p.fill_count = h->fill_count; p.fill_cap = h->cfg.fill_log_capacity;
  p.n_envs = h->cfg.n_envs; p.n_sel = h->cfg.n_envs; p.L = h->L; p.warp_smem = h->warp_smem;
  p.allow_flat = h->fast && h->flat_blobs ? 1 : 0;
  p.blob_in_global = h->blob_in_global ? 1 : 0;
}

// Flat blobs (book_flat.cuh) exist only between launches of the straight-line kernels; everything else reads the level arrays.
static int ensure_sorted(lobsim* h, cudaStream_t stream) {
  if (!h->maybe_flat || !h->fast) return LOBSIM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  h->fast->to_sorted(h->blobs, h->cfg.n_envs, stream);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  h->maybe_flat = false;
  return LOBSIM_OK;
}

} // extern "C"

template <bool kEnv, bool kTrack>
static int launch_advance(lobsim* h, const AdvParams& p, cudaStream_t stream) {
  { int rc = ensure_sorted(h, stream); if (rc) return rc; }
  if (h->streams.empty()) return fail(LOBSIM_E_STATE, "no stream loaded");
  CUDA_TRY(cudaSetDevice(h->device));
  int wpc = h->warps_per_cta;
  int grid = (p.n_sel + wpc - 1) / wpc;
  if (grid <= 0) return LOBSIM_OK;
  k_advance<kEnv, kTrack><<<grid, wpc * 32, (size_t)wpc * h->warp_smem, stream>>>(p, h->ec);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return LOBSIM_OK;
}

static int launch_replay_fast(lobsim* h, const AdvParams& p, cudaStream_t stream) {
  if (h->streams.empty()) return fail(LOBSIM_E_STATE, "no stream loaded");
  if (!h->fast) return 1;
  CUDA_TRY(cudaSetDevice(h->device));
  const int wpc = h->replay_warps_per_cta, grid = (p.n_sel + wpc - 1) / wpc;
  if (grid <= 0) return LOBSIM_OK;
  AdvParams pr = p;
  pr.warp_smem = h->replay_warp_smem;
  pr.hybrid = h->replay_flat && h->fast->NL >= 64 && h->fast->NO >= 512 && (h->replay_hybrid > 0 || (h->replay_hybrid < 0 && h->fast->NO >= 1024)) ? 1 : 0;
  if (pr.hybrid) pr.allow_flat = 0;
  if (!h->replay_flat || pr.hybrid) { int rc = ensure_sorted(h, stream); if (rc) return rc; }
  else if (p.allow_flat) h->maybe_flat = true;
  (h->replay_flat ? h->fast->replay_flat : h->fast->replay)(grid, wpc * 32, (size_t)wpc * h->replay_warp_smem, stream, pr, h->ec);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return LOBSIM_OK;
}

// env launches (reset / step / rollout): the straight-line kernel when a compiled StaticLayout matches the capacities,
// the general runtime-layout kernel otherwise
static int launch_env(lobsim* h, const AdvParams& p, cudaStream_t stream) {
  if (h->streams.empty()) return fail(LOBSIM_E_STATE, "no stream loaded");
  if (!h->fast) return launch_advance<true, true>(h, p, stream);
  CUDA_TRY(cudaSetDevice(h->device));
  const int wpc = h->env_warps_per_cta;
  const size_t dyn = (size_t)wpc * h->warp_smem;
  const int full = p.n_sel / wpc, tail = p.n_sel % wpc;
  auto launch = h->rare_paths ? h->fast->env_rare : h->fast->env;
  // Step / rollout launches of an ENV_HOT layout: the flat-only kernel for every env, then the deferred (sorted) kernel for the env
  // steps it handed over (usually none).  Resets, fill-logged handles and LOBSIM_FLAT_BLOBS=0 take the classic kernel, which reads both
  // book forms and stores the sorted one.
  const bool hot = h->fast->env_hot && h->defer_list && p.allow_flat && p.reset_mode == 0 && !h->fill_log && p.T > 0;
  AdvParams q = p;
  if (hot) {
    CUDA_TRY(cudaMemsetAsync(h->defer_count, 0, sizeof(int32_t), stream));
    q.defer_count = h->defer_count; q.defer_list = h->defer_list;
    h->maybe_flat = true;
  }
  const int mode = hot ? ENV_HOT : ENV_CLASSIC;
  if (full > 0) { // full CTAs: phase-synchronous
    launch(mode, true, full, wpc * 32, dyn, stream, q, h->ec);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  if (tail > 0) { // the remaining n_sel % wpc envs: one partially filled CTA without block-level barriers
    AdvParams pt = q;
    pt.sel_offset = full * wpc;
    launch(mode, false, 1, wpc * 32, dyn, stream, pt, h->ec);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  if (hot) {
    launch(ENV_DEFERRED, false, (p.n_sel + wpc - 1) / wpc, wpc * 32, dyn, stream, q, h->ec);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  return LOBSIM_OK;
}

extern "C" {

int lobsim_reset_book(lobsim_t* h, const int32_t* env_ids, int32_t n, const int32_t* stream_ids, const int32_t* start_steps, void* stream) {
  if (!h || !stream_ids || !start_steps) return fail(LOBSIM_E_INVALID, "null argument");
  AdvParams p; base_params(h, p);
  p.env_ids = env_ids; p.n_sel = env_ids ? n : h->cfg.n_envs;
  p.T = 0; p.reset_mode = 1; p.reset_stream_ids = stream_ids; p.reset_steps = start_steps; p.agent_kind = LOBSIM_AGENT_NONE;
  if (!env_ids) h->agent_orders_possible = false; // every book is a fresh snapshot again
  return launch_advance<false, true>(h, p, (cudaStream_t)stream);
}

int lobsim_reset(lobsim_t* h, const int32_t* env_ids, int32_t n, const int32_t* stream_ids, const int32_t* episode_start_steps, double* obs_out, void* stream) {
  if (!h || !stream_ids || !episode_start_steps) return fail(LOBSIM_E_INVALID, "null argument");
  AdvParams p; base_params(h, p);
  p.env_ids = env_ids; p.n_sel = env_ids ? n : h->cfg.n_envs;
  p.T = h->cfg.warmup_steps; p.reset_mode = 2; p.reset_stream_ids = stream_ids; p.reset_steps = episode_start_steps;
  p.agent_kind = LOBSIM_AGENT_NONE; p.obs = obs_out; p.out_final_obs_only = 1;
  h->has_reset = true;
  return launch_env(h, p, (cudaStream_t)stream);
}

int lobsim_step(lobsim_t* h, const double* actions, double* obs_out, double* reward_out, uint8_t* done_out, void* stream) {
  if (!h || !actions) return fail(LOBSIM_E_INVALID, "null argument");
  if (!h->has_reset) return fail(LOBSIM_E_STATE, "step before reset");
  AdvParams p; base_params(h, p);
  p.T = 1; p.agent_kind = LOBSIM_AGENT_EXTERNAL; p.actions_in = actions; p.obs = obs_out; p.rew = reward_out; p.done = done_out;
  h->agent_orders_possible = true;
  return launch_env(h, p, (cudaStream_t)stream);
}

static int ensure_staging(lobsim* h) {
  if (h->st_actions) return LOBSIM_OK;
  const size_t n = (size_t)h->cfg.n_envs;
  CUDA_TRY(cudaMalloc(&h->st_actions, n * 8 * sizeof(double)));
  CUDA_TRY(cudaMalloc(&h->st_obs, n * (LOBSIM_MAX_FEATURES + 8) * sizeof(double)));
  CUDA_TRY(cudaMalloc(&h->st_rew, n * sizeof(double)));
  CUDA_TRY(cudaMalloc(&h->st_done, n));
  CUDA_TRY(cudaMalloc(&h->st_state, n * sizeof(lobsim_env_state_t)));
  return LOBSIM_OK;
}

int lobsim_step_host(lobsim_t* h, const double* actions, double* obs_out, double* reward_out, uint8_t* done_out) {
  if (!h || !actions) return fail(LOBSIM_E_INVALID, "null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = ensure_staging(h);
  if (rc) return rc;
  const size_t n = (size_t)h->cfg.n_envs;
  CUDA_TRY(cudaMemcpyAsync(h->st_actions, actions, n * h->ec.action_dim * sizeof(double), cudaMemcpyHostToDevice, 0));
  rc = lobsim_step(h, h->st_actions, h->st_obs, h->st_rew, h->st_done, nullptr);
  if (rc) return rc;
  if (obs_out) CUDA_TRY(cudaMemcpyAsync(obs_out, h->st_obs, n * h->ec.obs_dim * sizeof(double), cudaMemcpyDeviceToHost, 0));
  if (reward_out) CUDA_TRY(cudaMemcpyAsync(reward_out, h->st_rew, n * sizeof(double), cudaMemcpyDeviceToHost, 0));
  if (done_out) CUDA_TRY(cudaMemcpyAsync(done_out, h->st_done, n, cudaMemcpyDeviceToHost, 0));
  CUDA_TRY(cudaStreamSynchronize(0));
  return LOBSIM_OK;
}

int lobsim_rollout(lobsim_t* h, int32_t T, const lobsim_agent_t* agent, double* obs, double* act, double* rew, uint8_t* done, void* stream) {
  return lobsim_rollout_info(h, T, agent, obs, act, rew, done, nullptr, stream);
}

int lobsim_rollout_info(lobsim_t* h, int32_t T, const lobsim_agent_t* agent, double* obs, double* act, double* rew, uint8_t* done, double* info, void* stream) {
  if (!h || !agent || T < 0) return fail(LOBSIM_E_INVALID, "bad argument");
  if (!h->has_reset) return fail(LOBSIM_E_STATE, "rollout before reset");
  if (agent->kind < LOBSIM_AGENT_NONE || agent->kind > LOBSIM_AGENT_RANDOM) return fail(LOBSIM_E_INVALID, "unknown agent kind");
  if (agent->kind == LOBSIM_AGENT_EXTERNAL && !act) return fail(LOBSIM_E_INVALID, "EXTERNAL agent needs the act tensor as input");
  if (agent->kind == LOBSIM_AGENT_TERADACTYL && (agent->inventory_index < 0 || agent->inventory_index >= h->cfg.n_features)) return fail(LOBSIM_E_INVALID, "bad inventory_index");
  AdvParams p; base_params(h, p);
  p.T = T; p.agent_kind = agent->kind; p.agent = *agent; p.obs = obs; p.rew = rew; p.done = done; p.info = info;
  if (agent->kind == LOBSIM_AGENT_EXTERNAL) p.actions_in = act; else p.act = act;
  if (agent->kind != LOBSIM_AGENT_NONE) h->agent_orders_possible = true;
  return launch_env(h, p, (cudaStream_t)stream);
}

int lobsim_rollout_agents(lobsim_t* h, int32_t T, const lobsim_agent_t* agents_host, double* obs, double* act, double* rew, uint8_t* done, double* info, void* stream) {
  if (!h || !agents_host || T < 0) return fail(LOBSIM_E_INVALID, "bad argument");
  if (!h->has_reset) return fail(LOBSIM_E_STATE, "rollout before reset");
  const int n = h->cfg.n_envs;
  for (int i = 0; i < n; i++) {
    const lobsim_agent_t& a = agents_host[i];
    if (a.kind != LOBSIM_AGENT_FIXED && a.kind != LOBSIM_AGENT_TERADACTYL && a.kind != LOBSIM_AGENT_RANDOM) return fail(LOBSIM_E_INVALID, "per-env agents must be FIXED, TERADACTYL or RANDOM");
    if (a.kind == LOBSIM_AGENT_TERADACTYL && (a.inventory_index < 0 || a.inventory_index >= h->cfg.n_features)) return fail(LOBSIM_E_INVALID, "bad inventory_index");
  }
  CUDA_TRY(cudaSetDevice(h->device));
  if (!h->agents_dev) CUDA_TRY(cudaMalloc(&h->agents_dev, (size_t)n * sizeof(lobsim_agent_t)));
  CUDA_TRY(cudaMemcpyAsync(h->agents_dev, agents_host, (size_t)n * sizeof(lobsim_agent_t), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  AdvParams p; base_params(h, p);
  p.T = T; p.agent_kind = LOBSIM_AGENT_TERADACTYL; p.agent = agents_host[0]; p.agents = h->agents_dev;
  p.obs = obs; p.act = act; p.rew = rew; p.done = done; p.info = info;
  h->agent_orders_possible = true;
  return launch_env(h, p, (cudaStream_t)stream);
}

int lobsim_replay(lobsim_t* h, int32_t n_steps, void* stream) {
  if (!h || n_steps < 0) return fail(LOBSIM_E_INVALID, "bad argument");
  AdvParams p; base_params(h, p);
  p.T = n_steps; p.agent_kind = LOBSIM_AGENT_NONE;
  // fast path: no fill log requested and no agent order can be resting in any book
  if (!h->fill_log && !h->agent_orders_possible && h->fast) {
    int rc = launch_replay_fast(h, p, (cudaStream_t)stream);
    if (rc != 1) return rc; // 1: no compiled StaticLayout matches these capacities
  }
  return launch_advance<false, true>(h, p, (cudaStream_t)stream);
}

int lobsim_forward_step(lobsim_t* h, int32_t n_steps, void* stream) {
  if (!h || n_steps < 0) return fail(LOBSIM_E_INVALID, "bad argument");
  AdvParams p; base_params(h, p);
  p.T = n_steps; p.agent_kind = LOBSIM_AGENT_NONE; p.resync_last_only = 1;
  return launch_advance<false, true>(h, p, (cudaStream_t)stream);
}

int lobsim_set_book(lobsim_t* h, int32_t env, const lobsim_book_entry_t* buy, int32_t n_buy, const lobsim_book_entry_t* sell, int32_t n_sell) {
  if (!h || env < 0 || env >= h->cfg.n_envs || n_buy < 0 || n_sell < 0 || (!buy && n_buy) || (!sell && n_sell)) return fail(LOBSIM_E_INVALID, "bad argument");
  const Layout& L = h->L;
  if (n_buy > L.NO || n_sell > L.NO) return fail(LOBSIM_E_INVALID, "more orders than max_orders_per_side");
  CUDA_TRY(cudaSetDevice(h->device));
  { int rc = ensure_sorted(h, 0); if (rc) return rc; }
  CUDA_TRY(cudaDeviceSynchronize());
  std::vector<unsigned char> buf(L.blob_bytes);
  unsigned char* gblob = h->blobs + (size_t)env * L.blob_bytes;
  CUDA_TRY(cudaMemcpy(buf.data(), gblob, L.blob_bytes, cudaMemcpyDeviceToHost));
  BookHdr* hd = reinterpret_cast<BookHdr*>(buf.data());
  uint32_t max_agent_id = 0;
  for (int side = 0; side < 2; side++) {
    const lobsim_book_entry_t* e = side ? sell : buy;
    const int n = side ? n_sell : n_buy;
    unsigned char* sb = buf.data() + L.side_off + side * L.side_stride;
    int32_t* lvp = reinterpret_cast<int32_t*>(sb);
    uint16_t* lvend = reinterpret_cast<uint16_t*>(sb + L.lvend_off);
    uint2* ord = reinterpret_cast<uint2*>(sb + L.ord_off);
    int32_t* ap = reinterpret_cast<int32_t*>(buf.data() + L.agent_off + side * L.NA * 12);
    int32_t* av = ap + L.NA;
    uint32_t* ai = reinterpret_cast<uint32_t*>(ap + 2 * L.NA);
    // entries arrive best level first; storage is worst level first => walk the levels backwards
    std::vector<std::pair<int, int>> levels; // [first, last) index ranges of equal price, best first
    for (int i = 0; i < n;) {
      int j = i;
      while (j < n && e[j].price == e[i].price) j++;
      if (!levels.empty()) {
        int prev = e[levels.back().first].price;
        if (side == 0 ? e[i].price >= prev : e[i].price <= prev) return fail(LOBSIM_E_INVALID, "entries must be sorted best level first");
      }
      levels.push_back({i, j});
      i = j;
    }
    if ((int)levels.size() > L.NL) return fail(LOBSIM_E_INVALID, "more levels than max_levels_per_side");
    int nlv = (int)levels.size(), pos = 0, nag = 0;
    std::vector<std::pair<uint32_t, int>> agent; // (id, entry index)
    for (int k = nlv - 1; k >= 0; k--) {
      int j = nlv - 1 - k;
      lvp[j] = e[levels[k].first].price;
      for (int i = levels[k].first; i < levels[k].second; i++) {
        if (e[i].volume < 0) return fail(LOBSIM_E_INVALID, "negative volume");
        ord[pos++] = make_uint2((unsigned)e[i].volume, e[i].ref);
        if (e[i].ref & LOBSIM_REF_AGENT) agent.push_back({e[i].ref & 0x7fffffffu, i});
      }
      lvend[j] = (uint16_t)pos;
    }
    if ((int)agent.size() > L.NA) return fail(LOBSIM_E_INVALID, "more agent orders than max_agent_orders");
    std::sort(agent.begin(), agent.end());
    for (auto& a : agent) { ap[nag] = e[a.second].price; av[nag] = e[a.second].volume; ai[nag] = a.first; nag++; if (a.first > max_agent_id) max_agent_id = a.first; }
    hd->cnt[side][0] = nlv; hd->cnt[side][1] = pos; hd->nag[side] = nag;
  }
  if (hd->next_agent_id <= max_agent_id) hd->next_agent_id = max_agent_id + 1;
  hd->dead = 0; hd->err = 0;
  CUDA_TRY(cudaMemcpy(gblob, buf.data(), L.blob_bytes, cudaMemcpyHostToDevice));
  h->agent_orders_possible = true;
  return LOBSIM_OK;
}

int lobsim_get_state_dev(lobsim_t* h, lobsim_env_state_t* out_dev, void* stream) {
  if (!h || !out_dev) return fail(LOBSIM_E_INVALID, "null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  k_get_state<<<(h->cfg.n_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->blobs, h->L, 0, h->cfg.n_envs, out_dev);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return LOBSIM_OK;
}

int lobsim_get_state(lobsim_t* h, int32_t first_env, int32_t n, lobsim_env_state_t* out) {
  if (!h || !out || first_env < 0 || n < 0 || first_env + n > h->cfg.n_envs) return fail(LOBSIM_E_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = ensure_staging(h);
  if (rc) return rc;
  if (n == 0) return LOBSIM_OK;
  k_get_state<<<(n + 127) / 128, 128>>>(h->blobs, h->L, first_env, n, h->st_state);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  CUDA_TRY(cudaMemcpy(out, h->st_state, (size_t)n * sizeof(lobsim_env_state_t), cudaMemcpyDeviceToHost));
  return LOBSIM_OK;
}

int lobsim_replay_host(lobsim_t* h, int stream_id, const lobsim_msg_t* msgs_host, uint64_t first_msg, uint64_t n_msgs, int32_t n_steps, lobsim_env_state_t* state_out) {
  if (!h || stream_id < 0 || stream_id >= (int)h->streams.size()) return fail(LOBSIM_E_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = ensure_staging(h);
  if (rc) return rc;
  lobsim_stream_t& s = h->streams[stream_id];
  if (first_msg + n_msgs > s.n_msgs) return fail(LOBSIM_E_INVALID, "segment outside the stream");
  if (n_msgs) { // H2D of the segment straight into the resident stream buffer (same layout, same offsets)
    if (!msgs_host) return fail(LOBSIM_E_INVALID, "msgs_host is null");
    CUDA_TRY(cudaMemcpyAsync(const_cast<lobsim_msg_t*>(s.msgs) + first_msg, msgs_host, n_msgs * sizeof(lobsim_msg_t), cudaMemcpyHostToDevice, 0));
  }
  rc = lobsim_replay(h, n_steps, nullptr);
  if (rc) return rc;
  if (state_out) {
    rc = lobsim_get_state_dev(h, h->st_state, nullptr);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(state_out, h->st_state, (size_t)h->cfg.n_envs * sizeof(lobsim_env_state_t), cudaMemcpyDeviceToHost, 0));
  }
  CUDA_TRY(cudaStreamSynchronize(0));
  return LOBSIM_OK;
}

int lobsim_process_orders(lobsim_t* h, const lobsim_order_t* orders, int32_t n, lobsim_fill_t* fills_out, int32_t max_fills, int32_t* n_fills_out, uint32_t* refs_out) {
  if (!h || (!orders && n) || n < 0 || max_fills < 0) return fail(LOBSIM_E_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(h->device));
  if (n_fills_out) *n_fills_out = 0;
  if (n == 0) return LOBSIM_OK;
  // device staging buffers, kept in the handle and grown on demand (a façade Exchange.process_order call is one order per call)
  if (n > h->po_cap) {
    cudaFree(h->po_orders); cudaFree(h->po_refs); h->po_orders = nullptr; h->po_refs = nullptr; h->po_cap = 0;
    const int cap = n < 64 ? 64 : 2 * n;
    CUDA_TRY(cudaMalloc(&h->po_orders, (size_t)cap * sizeof(lobsim_order_t)));
    CUDA_TRY(cudaMalloc(&h->po_refs, (size_t)cap * sizeof(uint32_t)));
    h->po_cap = cap;
  }
  if (max_fills > h->po_fill_cap || !h->po_fills) {
    cudaFree(h->po_fills); h->po_fills = nullptr; h->po_fill_cap = 0;
    const int cap = max_fills < 256 ? 256 : 2 * max_fills;
    CUDA_TRY(cudaMalloc(&h->po_fills, (size_t)cap * sizeof(lobsim_fill_t)));
    h->po_fill_cap = cap;
  }
  if (!h->po_nf) CUDA_TRY(cudaMalloc(&h->po_nf, sizeof(int32_t)));
  lobsim_order_t* d_orders = h->po_orders; lobsim_fill_t* d_fills = h->po_fills; int32_t* d_nf = h->po_nf; uint32_t* d_refs = h->po_refs;
  CUDA_TRY(cudaMemcpy(d_orders, orders, (size_t)n * sizeof(lobsim_order_t), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemset(d_nf, 0, sizeof(int32_t)));
  OrdParams p; p.blobs = h->blobs; p.L = h->L; p.n_envs = h->cfg.n_envs; p.blob_in_global = h->blob_in_global ? 1 : 0; p.orders = d_orders; p.n = n;
  p.fills = max_fills > 0 ? d_fills : nullptr; p.max_fills = max_fills; p.n_fills = d_nf; p.refs_out = d_refs;
  h->agent_orders_possible = true;
  { int rc = ensure_sorted(h, 0); if (rc) return rc; }
  k_process_orders<<<1, 32, h->blob_in_global ? 16 : h->L.blob_bytes>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  h->launches++;
  int32_t nf = 0;
  if (e == cudaSuccess) e = cudaMemcpy(&nf, d_nf, sizeof nf, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && fills_out && nf > 0) e = cudaMemcpy(fills_out, d_fills, (size_t)nf * sizeof(lobsim_fill_t), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && refs_out) e = cudaMemcpy(refs_out, d_refs, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return fail(LOBSIM_E_CUDA, cudaGetErrorString(e));
  if (n_fills_out) *n_fills_out = nf;
  return LOBSIM_OK;
}

// host-side decode of one env's blob (layout = book.cuh)
static int fetch_blob(lobsim* h, int env, std::vector<unsigned char>& buf) {
  if (env < 0 || env >= h->cfg.n_envs) return fail(LOBSIM_E_INVALID, "bad env index");
  CUDA_TRY(cudaSetDevice(h->device));
  { CUDA_TRY(cudaDeviceSynchronize()); int rc = ensure_sorted(h, 0); if (rc) return rc; }
  buf.resize(h->L.blob_bytes);
  CUDA_TRY(cudaMemcpy(buf.data(), h->blobs + (size_t)env * h->L.blob_bytes, h->L.blob_bytes, cudaMemcpyDeviceToHost));
  return LOBSIM_OK;
}

int lobsim_dump_book(lobsim_t* h, int32_t env, int32_t side, lobsim_book_entry_t* out, int32_t capacity) {
  if (!h || side < 0 || side > 1) return fail(LOBSIM_E_INVALID, "bad argument");
  std::vector<unsigned char> buf;
  int rc = fetch_blob(h, env, buf);
  if (rc) return rc;
  const Layout& L = h->L;
  const BookHdr* hd = reinterpret_cast<const BookHdr*>(buf.data());
  const unsigned char* sb = buf.data() + L.side_off + side * L.side_stride;
  const int32_t* lvp = reinterpret_cast<const int32_t*>(sb);
  const uint16_t* lvend = reinterpret_cast<const uint16_t*>(sb + L.lvend_off);
  const uint2* ord = reinterpret_cast<const uint2*>(sb + L.ord_off);
  int n = 0;
  for (int k = 0; k < hd->cnt[side][0]; k++) { // best level first
    int j = hd->cnt[side][0] - 1 - k;
    int start = j > 0 ? lvend[j - 1] : 0, end = lvend[j];
    for (int i = start; i < end; i++) {
      if (out && n < capacity) { out[n].price = lvp[j]; out[n].volume = (int32_t)ord[i].x; out[n].ref = ord[i].y; out[n].level = k; }
      n++;
    }
  }
  return n;
}

int lobsim_dump_agent_orders(lobsim_t* h, int32_t env, int32_t side, lobsim_book_entry_t* out, int32_t capacity) {
  if (!h || side < 0 || side > 1) return fail(LOBSIM_E_INVALID, "bad argument");
  std::vector<unsigned char> buf;
  int rc = fetch_blob(h, env, buf);
  if (rc) return rc;
  const Layout& L = h->L;
  const BookHdr* hd = reinterpret_cast<const BookHdr*>(buf.data());
  const int32_t* ap = reinterpret_cast<const int32_t*>(buf.data() + L.agent_off + side * L.NA * 12);
  const int32_t* av = ap + L.NA;
  const uint32_t* ai = reinterpret_cast<const uint32_t*>(ap + 2 * L.NA);
  int n = hd->nag[side];
  for (int i = 0; i < n && out && i < capacity; i++) { out[i].price = ap[i]; out[i].volume = av[i]; out[i].ref = LOBSIM_REF_AGENT | ai[i]; out[i].level = -1; }
  return n;
}

int lobsim_get_fills(lobsim_t* h, int32_t env, lobsim_fill_t* out, int32_t capacity, int32_t* n_out) {
  if (!h || env < 0 || env >= h->cfg.n_envs || !n_out) return fail(LOBSIM_E_INVALID, "bad argument");
  *n_out = 0;
  if (!h->fill_log) return LOBSIM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  int32_t n = 0;
  CUDA_TRY(cudaMemcpy(&n, h->fill_count + env, sizeof n, cudaMemcpyDeviceToHost));
  *n_out = n;
  int m = n < h->cfg.fill_log_capacity ? n : h->cfg.fill_log_capacity;
  if (m > capacity) m = capacity;
  if (out && m > 0) CUDA_TRY(cudaMemcpy(out, h->fill_log + (size_t)env * h->cfg.fill_log_capacity, (size_t)m * sizeof(lobsim_fill_t), cudaMemcpyDeviceToHost));
  return LOBSIM_OK;
}

int lobsim_errors(lobsim_t* h, uint32_t* err_out) {
  if (!h || !err_out) return fail(LOBSIM_E_INVALID, "null argument");
  // one strided device-to-host copy of the 4-byte error word of every blob header (both book forms keep it in place): no
  // kernel, no state summary
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpy2D(err_out, sizeof(uint32_t), h->blobs + offsetof(BookHdr, err), (size_t)h->L.blob_bytes, sizeof(uint32_t), (size_t)h->cfg.n_envs,
                        cudaMemcpyDeviceToHost));
  return LOBSIM_OK;
}

int64_t lobsim_launch_count(lobsim_t* h) { return h ? h->launches : 0; }

int lobsim_kernel_path(lobsim_t* h) { return h && h->fast ? LOBSIM_PATH_FAST : (h && h->blob_in_global ? LOBSIM_PATH_DEEP : LOBSIM_PATH_GENERAL); }

#ifndef LOBSIM_SOURCE_HASH
#define LOBSIM_SOURCE_HASH "unstamped"
#endif
const char* lobsim_source_hash(void) { return LOBSIM_SOURCE_HASH; }

} // extern "C"
