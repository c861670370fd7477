// kernels.cuh -- the kernels of the B200-native LOB simulation step.
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
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>
#include "book_flat.cuh"
#include "book_hybrid.cuh"
#include "env.cuh"
#include "lobsim.h"

// ====================================================================================================================
//  PTX helpers: mbarrier + TMA bulk copies (sm_90+; SASS: UBLKCP / SYNCS)
// ====================================================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void tma_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_store(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_part(void* dst_gmem, const void* src_smem, uint32_t bytes) { // no commit: several parts, one group
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ====================================================================================================================
//  kernel parameters
// ====================================================================================================================
#ifndef LOBSIM_ENV_MIN_BLOCKS
#define LOBSIM_ENV_MIN_BLOCKS 3
#endif
#define MSG_TILE 32                      // records per TMA tile
#define MSG_TILE_BYTES (MSG_TILE * 16)
// per-warp scratch behind the message tiles: int2[2 * NA] for update_outer_levels (the agent's re-queued orders), at least
// int[64] for the agent's resting volume per ladder level (agent_prepare) and the 5 action doubles
__host__ __device__ constexpr int scratch_bytes(int NA) { return 2 * NA * 8 > 256 ? 2 * NA * 8 : 256; }

// the replay kernel of a handle with compiled straight-line kernels, fixed by lobsim_create: k_replay_fast (sorted level arrays
// only), k_replay_flat (flat order pools, book_flat.cuh) or k_replay_hyb (hybrid book of deep layouts, book_hybrid.cuh)
enum ReplayKind { REPLAY_SORTED, REPLAY_FLAT, REPLAY_HYBRID };

struct AdvParams {
  unsigned char* blobs;             // [n_envs][blob_bytes]
  FeatState* fstate;                // [n_envs][LOBSIM_MAX_FEATURES]
  NormState* nstate;                // [n_envs][LOBSIM_MAX_FEATURES] rolling z-score state, or null (no normalised feature configured)
  const double* beta_tab;           // [2][32]: ln x_k, ln(1 - x_k) at the quote-level midpoints x_k = (k + 0.5) / Q
  double* rings;                    // [n_envs][ring_stride]
  double* rs_ring;                  // RollingSharpe [n_envs][3][LOBSIM_MAX_SHARPE_WINDOW]: two AUM windows + a scratch row of returns, or null
  int32_t* rs_state;                // [n_envs][2][2] = {n_filled, head}
  const lobsim_stream_t* streams;   // device array [n_streams]
  int32_t n_streams;
  lobsim_fill_t* fill_log;          // [n_envs][fill_cap] or null
  int32_t* fill_count;              // [n_envs]
  int32_t fill_cap;
  int32_t n_envs;                   // total envs of the handle
  int32_t n_sel;                    // number of envs this launch works on
  int32_t sel_offset;               // first selection index handled by this launch (tail launches)
  const int32_t* env_ids;           // [n_sel] or null (identity)
  int32_t T;                        // simulation steps to run
  int32_t reset_mode;               // 0 none, 1 book reset only, 2 full env reset (+ warm-up of T steps)
  const int32_t* reset_stream_ids;  // [n_sel]
  const int32_t* reset_steps;       // [n_sel]: book reset: start step; env reset: episode start step
  int32_t agent_kind;               // LOBSIM_AGENT_*
  int32_t out_final_obs_only;       // reset: write obs once, after the warm-up
  int32_t resync_last_only;         // forward_step over several grid steps: resync check only at the end
  int32_t blob_in_global;           // deep books: the blob does not fit in the shared memory of an SM and is worked on in place in HBM / L2
  int32_t allow_flat;               // fast kernels: books that fit run on -- and are stored in -- the flat order pools (book_flat.cuh)
  const double* actions_in;         // EXTERNAL: [T][n_sel][action_dim]
  double* obs; double* act; double* rew; uint8_t* done; // [T][n_sel][...] (any may be null)
  double* info;                     // [T][n_sel][LOBSIM_INFO_DIM] per-step info series (SimpleInfoCalculator source) or null
  lobsim_agent_t agent;
  const lobsim_agent_t* agents;     // per-env built-in agents [n_sel] (parameter sweeps) or null: every env runs `agent`
  Layout L;
  int32_t warp_smem;                // bytes of shared memory per warp
};

// one row of the per-step info series (InfoCalculators.py:31-59: asset_price, inventory, cash, aum, market_spread) --
// the state the reference's info_calculator sees at the end of HistoricalOrderbookEnvironment.step (HOE.py:175-177)
__device__ __forceinline__ void write_info(double* row, int lane, const StepView& v, double cash, long long inv, uint32_t err) {
  double x = v.price;
  if (lane == LOBSIM_INFO_INVENTORY) x = (double)inv;
  else if (lane == LOBSIM_INFO_CASH) x = cash;
  else if (lane == LOBSIM_INFO_AUM) x = cash + v.price * (double)inv;
  else if (lane == LOBSIM_INFO_MARKET_SPREAD) x = v.have_tops ? (double)(v.bs - v.bb) : NAN;
  else if (lane == LOBSIM_INFO_BEST_BUY) x = v.have_tops ? (double)v.bb : NAN;
  else if (lane == LOBSIM_INFO_BEST_SELL) x = v.have_tops ? (double)v.bs : NAN;
  else if (lane == LOBSIM_INFO_ERR) x = (double)err;
  if (lane < LOBSIM_INFO_DIM) row[lane] = x;
}

// per_step / terminal reward of one env step (HOE.py:170-174); RollingSharpe keeps one AUM window per reward function
template <bool RARE>
__device__ __forceinline__ double step_reward(const AdvParams& p, const lobsim_cfg_t& c, int env, int lane, bool done, double cash0, long long inv0, double p0,
                                              double cash1, long long inv1, double p1, uint32_t& err) {
  double r;
  if (RARE && c.step_reward.kind == LOBSIM_REWARD_ROLLING_SHARPE) {
    SharpeOut o = rolling_sharpe_step(p.rs_ring + ((size_t)env * 3 + 0) * LOBSIM_MAX_SHARPE_WINDOW, p.rs_state + ((size_t)env * 2 + 0) * 2, c.step_reward.asymmetric, cash1 + p1 * (double)inv1, lane, p.rs_ring + ((size_t)env * 3 + 2) * LOBSIM_MAX_SHARPE_WINDOW);
    r = o.reward; err |= o.err;
  } else r = reward_calc(c.step_reward, cash0, inv0, p0, cash1, inv1, p1);
  if (done) {
    if (RARE && c.terminal_reward.kind == LOBSIM_REWARD_ROLLING_SHARPE) {
      SharpeOut o = rolling_sharpe_step(p.rs_ring + ((size_t)env * 3 + 1) * LOBSIM_MAX_SHARPE_WINDOW, p.rs_state + ((size_t)env * 2 + 1) * 2, c.terminal_reward.asymmetric, cash1 + p1 * (double)inv1, lane, p.rs_ring + ((size_t)env * 3 + 2) * LOBSIM_MAX_SHARPE_WINDOW);
      r = o.reward; err |= o.err;
    } else r = reward_calc(c.terminal_reward, cash0, inv0, p0, cash1, inv1, p1);
  }
  return r;
}

// (second * 1e6 + microsecond) of now = t0 + now_step * step_us, in 32-bit arithmetic (t0 % 60 s comes with the stream)
__device__ __forceinline__ int us_in_minute(int t0_mod_min, int now_step, const EnvConst& ec) {
  int u = t0_mod_min + (now_step % ec.steps_per_min) * (int)ec.cfg.step_us;
  return u >= 60000000 ? u - 60000000 : u;
}

__device__ __forceinline__ unsigned char* warp_smem_base(unsigned char* smem, int warp, int warp_smem) { return smem + (size_t)warp * warp_smem; }

// The messages [g, g_end_all) of the T grid steps from now_step.  Steps beyond the end of the grid: the steps that exist are run,
// the first one past the end sets END_OF_STREAM (here: a launch that starts outside the grid).  `err` / `dead` of the caller's state.
__device__ __forceinline__ void stream_window(const uint32_t* __restrict__ step_off, int n_grid, int now_step, int T, uint32_t& err, int& dead,
                                              unsigned& g, unsigned& g_end_all) {
  if ((now_step < 0 || now_step > n_grid) && !dead && T > 0) { err |= LOBSIM_ERR_END_OF_STREAM; dead = 1; }
  g = 0; g_end_all = 0;
  if (!dead && T > 0) { g = __ldg(&step_off[now_step]); g_end_all = __ldg(&step_off[min((long long)now_step + T, (long long)n_grid)]); }
}

// The message tiles of one warp: TMA bulk loads of MSG_TILE records into a double buffer, one tile ahead of the reader.  Tiles are
// MSG_TILE-aligned in the global message index space; relative tile r (rel(g)) lives in buffer r & 1 and completes phase
// (r >> 1) & 1 of that buffer's mbarrier.  Tiles are issued and consumed strictly in order.  All members are warp-uniform.
struct MsgTiles {
  const lobsim_stream_t* stp;
  const lobsim_msg_t* msgs;
  unsigned char* buf;     // 2 x MSG_TILE_BYTES
  uint64_t* bars;         // bars[0], bars[1]: one per buffer
  int lane;
  unsigned tile0, g_end, next_issue, next_wait;
  // (constructed where the stream is known, started where the range is: the kernels' register allocation depends on that order)
  __device__ __forceinline__ explicit MsgTiles(const lobsim_stream_t* s) : stp(s), msgs(s->msgs) {}
  // the first two tiles of [g, g_end_all)
  __device__ __forceinline__ void start(unsigned char* msgbuf, uint64_t* b, int ln, unsigned g, unsigned g_end_all) {
    buf = msgbuf; bars = b; lane = ln;
    tile0 = g / MSG_TILE; g_end = g_end_all; next_issue = next_wait = 0;
    if (g < g_end_all) { issue(); issue(); }
    __syncwarp();
  }
  __device__ __forceinline__ void issue() { // lane 0 talks to the TMA unit
    const unsigned first = (tile0 + next_issue) * MSG_TILE;
    if (first >= g_end) return;
    if (lane == 0) {
      const unsigned n_total = (unsigned)stp->n_msgs;   // (read here, not cached: a cached copy costs the replay kernels spills)
      const unsigned cnt = n_total - first < MSG_TILE ? n_total - first : MSG_TILE;
      uint64_t* bar = &bars[next_issue & 1];
      mbar_expect_tx(bar, cnt * 16);
      tma_load(buf + (next_issue & 1) * MSG_TILE_BYTES, msgs + first, cnt * 16, bar);
    }
    next_issue++;
  }
  __device__ __forceinline__ void wait() { mbar_wait(&bars[next_wait & 1], (next_wait >> 1) & 1); next_wait++; }
  __device__ __forceinline__ unsigned rel(unsigned g) const { return g / MSG_TILE - tile0; }
  __device__ __forceinline__ void drain() { while (next_wait < next_issue) wait(); }   // TMA loads still in flight (aborted episode)
};

// ====================================================================================================================
//  the advance kernel: [reset] + T x ([agent orders] + messages of the step + [resync] + [features, reward])
// ====================================================================================================================
// kEnv: agent + features + rewards (HistoricalOrderbookEnvironment.step); fills / flows / agent orders are tracked either way.
template <bool kEnv>
__global__ void __launch_bounds__(128, kEnv ? LOBSIM_ENV_MIN_BLOCKS : 4) k_advance(const __grid_constant__ AdvParams p, const __grid_constant__ EnvConst ec) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sel = blockIdx.x * (blockDim.x >> 5) + warp;
  if (sel >= p.n_sel) return;
  const int env = p.env_ids ? p.env_ids[sel] : sel;
  const lobsim_cfg_t& c = ec.cfg;

  // Deep-book mode (p.blob_in_global): capacities whose blob exceeds the shared memory of an SM (thousands of resting orders per side,
  // rl4mm/orderbook/models.py:66-67 is unbounded) -- the book is worked on IN PLACE in HBM / L2 through the same routines (generic
  // addressing), only the message tiles / scratch / barriers live in shared memory.  Slower per order, but no capacity cliff.
  unsigned char* wbase = warp_smem_base(smem, warp, p.warp_smem);
  unsigned char* gblob = p.blobs + (size_t)env * p.L.blob_bytes;
  unsigned char* base = p.blob_in_global ? gblob : wbase;
  Book b; b.blob = base; b.L = p.L; b.lane = lane;
  unsigned char* msgbuf = p.blob_in_global ? wbase : wbase + p.L.blob_bytes;       // 2 x 512 B
  int2* scratch = reinterpret_cast<int2*>(msgbuf + 2 * MSG_TILE_BYTES);             // [2*NA]
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(scratch) + scratch_bytes(p.L.NA)); // 3 barriers

  // ---- book blob: HBM -> shared memory ---------------------------------------------------------------------------
  if (lane == 0) {
    mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
    fence_mbar_init();
    if (!p.blob_in_global) {
      mbar_expect_tx(&bars[2], (uint32_t)p.L.blob_bytes);
      tma_load(base, gblob, (uint32_t)p.L.blob_bytes, &bars[2]);
    }
  }
  __syncwarp();
  if (!p.blob_in_global) mbar_wait(&bars[2], 0);

  WarpState w;
  load_state(b, w);
  w.fill_log = p.fill_log ? p.fill_log + (size_t)env * p.fill_cap : nullptr;
  w.fill_cap = p.fill_cap; w.n_fills = 0;
  const long long inventory_in = w.inventory; const double cash_in = w.cash;
  BookHdr* h = b.hdr();
  const int F = c.n_features;

  // ---- reset prologue ----------------------------------------------------------------------------------------------
  int stream_id = h->stream_id;
  if (p.reset_mode) {
    stream_id = p.reset_stream_ids[sel];
    int start = p.reset_steps[sel] - (p.reset_mode == 2 ? c.warmup_steps : 0);
    if (stream_id < 0 || stream_id >= p.n_streams) { stream_id = 0; start = -1; }
    w = init_book_cold(b, w, &ec.cfg, &p.streams[stream_id], stream_id, start);
    if (p.reset_mode == 2 && lane == 0) {
      h->episode_start_step = p.reset_steps[sel];
      if (!c.portfolio_carryover || !h->has_reset) { h->inventory = c.initial_inventory; h->cash = c.initial_cash; }
      h->has_reset = 1;
    }
    __syncwarp();
    w.inventory = h->inventory; w.cash = h->cash;
  }
  const lobsim_stream_t* stp = &p.streams[stream_id];
  MsgTiles mt(stp);
  const uint32_t* __restrict__ st_step_off = stp->step_off;
  const long long st_t0_us = kEnv ? stp->t0_us : 0;
  int now_step = h->now_step;
  const long long episode_start_us = st_t0_us + (long long)h->episode_start_step * c.step_us;

  FeatState* fstate_env = p.fstate + (size_t)env * LOBSIM_MAX_FEATURES;
  NormState* nstate_env = p.nstate ? p.nstate + (size_t)env * LOBSIM_MAX_FEATURES : nullptr;
  double* rings_env = p.rings + (size_t)env * ec.ring_stride;
  double feat_cur = 0.0; // Feature.current_value of this lane's feature
  if (kEnv && lane < F) feat_cur = fstate_env[lane].cur;
  const int t0_mod_min = (int)stp->reserved;   // t0_us % 60 s, filled in by lobsim_load_stream

  // price / tops of the current book
  auto tops = [&](StepView& v) {
    v.have_tops = w.nlv0 > 0 && w.nlv1 > 0;
    if (v.have_tops) {
      v.bb = b.lvp(0)[w.nlv0 - 1]; v.bs = b.lvp(1)[w.nlv1 - 1];
      v.bv = best_level_volume(b, 0, w.nlv0); v.sv = best_level_volume(b, 1, w.nlv1);
      double imb; v.price = microprice(v.bb, v.bs, v.bv, v.sv, imb);
    } else { v.bb = v.bs = v.bv = v.sv = 0; v.price = NAN; }
  };

  double price = h->price;
  if (kEnv && p.reset_mode == 2) { // State(...) + _reset_features, HOE.py:152-154,218-221
    StepView v; tops(v);
    v.inventory = w.inventory; v.now_us = st_t0_us + (long long)now_step * c.step_us;
    v.us_in_min = us_in_minute(t0_mod_min, now_step, ec);
    v.n_ext0 = v.n_ext1 = v.vol_ext0 = v.vol_ext1 = v.n_int0 = v.n_int1 = v.vol_int0 = v.vol_int1 = 0;
    price = v.price;
    feat_cur = features_step<true>(&ec, fstate_env, nstate_env, rings_env, lane, v, episode_start_us, 1);
  }

  // ---- message pipeline ----------------------------------------------------------------------------------------------
  const int T = p.T;
  const int n_grid = (int)stp->n_grid_steps;
  unsigned g, g_end_all;
  stream_window(st_step_off, n_grid, now_step, T, w.err, w.dead, g, g_end_all);
  mt.start(msgbuf, bars, lane, g, g_end_all);

  AgentGen gen; gen.side = 3;
  bool agent_phase = false;
#pragma unroll 1
  for (int t = 0; t < T; t++) {
    // ---- agent: obs -> action -> orders (processed before the step's history, OrderbookSimulator.py:76-77) -------
    double cash0 = w.cash, p0 = price; long long inv0 = w.inventory;
    if (kEnv) {
      reset_flow(w);
      if (p.agent_kind != LOBSIM_AGENT_NONE) {
        double* act_sm = reinterpret_cast<double*>(scratch); // 5 doubles of per-warp scratch
        if (p.agent_kind == LOBSIM_AGENT_EXTERNAL) {
          const double* a = p.actions_in + ((size_t)t * p.n_sel + sel) * ec.action_dim;
          if (lane < 5) act_sm[lane] = lane < ec.action_dim ? __ldg(&a[lane]) : 0.0;
        } else {
          const lobsim_agent_t* agp = p.agents ? p.agents + sel : &p.agent;
          const double inv_obs = __shfl_sync(FULL_MASK, feat_cur, agp->inventory_index & 31);
          if (lane == 0) agent_action_cold(agp, inv_obs, act_sm, env, now_step);
        }
        __syncwarp();
        const double a0 = act_sm[0], a1 = act_sm[1], a2 = act_sm[2], a3 = act_sm[3], a4 = act_sm[4];
        const double mine = lane < 5 ? act_sm[lane] : 0.0;
        __syncwarp();
        if (p.act && p.agent_kind != LOBSIM_AGENT_EXTERNAL && lane < ec.action_dim) p.act[((size_t)t * p.n_sel + sel) * ec.action_dim + lane] = mine;
        if (p.obs && !p.out_final_obs_only && c.inc_prev_action_in_obs && lane < ec.action_dim)
          p.obs[((size_t)t * p.n_sel + sel) * ec.obs_dim + F + lane] = mine; // get_observation(action), HOE.py:171
        gen = agent_prepare(b, w.nlv0 ? b.lvp(0)[w.nlv0 - 1] : INT32_MIN, w.nlv1 ? b.lvp(1)[w.nlv1 - 1] : INT32_MAX, w.nag0, w.nag1, w.inventory, &ec, a0, a1, a2, a3, a4, p.beta_tab, reinterpret_cast<int*>(scratch));
        w.err |= gen.err_out; if (gen.dead_out) w.dead = 1;
        agent_phase = true;
      }
    }
    // ---- the step's orders: the agent's first, then the historical messages of (now, now + step] ------------------
    {
      if (!w.dead && now_step >= n_grid) { w.err |= LOBSIM_ERR_END_OF_STREAM; w.dead = 1; }
      const unsigned g_step_end = w.dead ? g : __ldg(&st_step_off[now_step + 1]);
#pragma unroll 1
      for (;;) {
        int type, side, price, vol; uint32_t ref; bool is_agent;
        if (kEnv && agent_phase) {
          if (!agent_next(b, w, gen, type, side, price, vol, ref)) { agent_phase = false; continue; }
          is_agent = true;
        } else {
          if (w.dead || g >= g_step_end) break;
          const unsigned tile = mt.rel(g);
          if (tile == mt.next_wait) mt.wait();
          const uint4 m = *reinterpret_cast<const uint4*>(msgbuf + (tile & 1) * MSG_TILE_BYTES + (g % MSG_TILE) * 16);
          price = (int)m.x; vol = (int)m.y; ref = m.z; type = (int)LOBSIM_META_TYPE(m.w); side = (int)LOBSIM_META_DIR(m.w);
          is_agent = false;
          g++;
          if (g % MSG_TILE == 0) { __syncwarp(); mt.issue(); } // tile consumed: refill its buffer
        }
        process_order(b, w, type, side, price, vol, ref, is_agent);
      }
    }
    if (!w.dead) {
      now_step++;
      // ---- resync, OrderbookSimulator.py:86-87 ----------------------------------------------------------------------
      if (c.resync && (!p.resync_last_only || t == T - 1)) {
        long long rel = (long long)now_step * c.step_us;
        if (rel % 1000000 == 0 && near_exiting(b, w, c)) {
          long long sec = rel / 1000000;
          if (sec <= (long long)stp->n_seconds && stp->snap_valid[sec]) {
            w = update_outer_levels(b, w, &ec.cfg, stp->snapshots + (size_t)sec * 2 * c.n_levels * 2, scratch);
                    }
        }
      }
    }
    if (kEnv) {
      // ---- update_internal_state + _update_features + reward, HOE.py:163-178,199-204 -------------------------------
      StepView v; tops(v);
      if (!v.have_tops) w.err |= LOBSIM_ERR_EMPTY_BOOK;
      price = v.price;
      v.inventory = w.inventory; v.now_us = st_t0_us + (long long)now_step * c.step_us;
      v.us_in_min = us_in_minute(t0_mod_min, now_step, ec);
      v.n_ext0 = w.n_ext0; v.n_ext1 = w.n_ext1; v.vol_ext0 = w.vol_ext0; v.vol_ext1 = w.vol_ext1;
      v.n_int0 = w.n_int0; v.n_int1 = w.n_int1; v.vol_int0 = w.vol_int0; v.vol_int1 = w.vol_int1;
      feat_cur = features_step<true>(&ec, fstate_env, nstate_env, rings_env, lane, v, episode_start_us, 0);
      const bool write_now = !p.out_final_obs_only || t == T - 1;
      if (p.obs && write_now) {
        double* o = p.obs + ((size_t)(p.out_final_obs_only ? 0 : t) * p.n_sel + sel) * ec.obs_dim;
        if (lane < F) o[lane] = feat_cur;
        if (c.inc_prev_action_in_obs && lane < ec.action_dim && (p.agent_kind == LOBSIM_AGENT_NONE || p.out_final_obs_only)) o[F + lane] = 0.0;
      }
      if (p.agent_kind != LOBSIM_AGENT_NONE) {
        const bool d = now_step >= h->episode_start_step + c.episode_steps; // terminal_time - now < step/2, HOE.py:172
        const double r = step_reward<true>(p, c, env, lane, d, cash0, inv0, p0, w.cash, w.inventory, price, w.err);
        if (lane == 0) {
          if (p.rew) p.rew[(size_t)t * p.n_sel + sel] = r;
          if (p.done) p.done[(size_t)t * p.n_sel + sel] = d ? 1 : 0;
        }
        if (p.info) write_info(p.info + ((size_t)t * p.n_sel + sel) * LOBSIM_INFO_DIM, lane, v, w.cash, w.inventory, w.err);
      }
    }
  }
  if (kEnv && T == 0 && p.obs && p.reset_mode == 2) { // reset with no warm-up: obs straight after _reset_features
    double* o = p.obs + (size_t)sel * ec.obs_dim;
    if (lane < F) o[lane] = feat_cur;
    if (c.inc_prev_action_in_obs && lane < ec.action_dim) o[F + lane] = 0.0;
  }

  mt.drain();

  // ---- write back ----------------------------------------------------------------------------------------------------
  // OrderbookSimulator.forward_step only returns the fills: the portfolio belongs to the env (HOE.py:280-289)
  if (!kEnv && !p.reset_mode) { w.inventory = inventory_in; w.cash = cash_in; }
  if (lane == 0) {
    h->now_step = now_step;
    h->price = price;
    if (p.fill_count) p.fill_count[env] = w.n_fills;
  }
  store_state(b, w);
  fence_proxy_async();
  __syncwarp();
  if (lane == 0 && !p.blob_in_global) { tma_store(gblob, base, (uint32_t)p.L.blob_bytes); tma_store_wait(); }
  __syncwarp();
}

// ====================================================================================================================
//  the frame of the straight-line replay kernels: a replay book holds no agent orders, so the agent tables at the end of the
//  blob stay in HBM (deep books are shared-memory bound: 128/1536/64 capacities = 8 instead of 7 resident books per SM)
// ====================================================================================================================
// the blob up to the agent tables, HBM -> shared memory on bars[2] (bars[0..1]: the message tiles)
template <class LT>
__device__ __forceinline__ void replay_blob_load(unsigned char* base, const unsigned char* gblob, uint64_t* bars, int lane) {
  if (lane == 0) {
    mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
    fence_mbar_init();
    mbar_expect_tx(&bars[2], (uint32_t)LT::agent_off);
    tma_load(base, gblob, (uint32_t)LT::agent_off, &bars[2]);
  }
  __syncwarp();
  mbar_wait(&bars[2], 0);
}
// ... and back: the header fields of the launch, then one bulk store.  `hdr_extra()`: header fields of the kernel's own, written by
// lane 0 with the others
template <class LT, class HdrExtra>
__device__ __forceinline__ void replay_blob_store(unsigned char* gblob, unsigned char* base, int lane, int now_step, const FastState& f, HdrExtra hdr_extra) {
  BookHdr* h = reinterpret_cast<BookHdr*>(base);
  __syncwarp();
  if (lane == 0) { h->now_step = now_step; h->err = f.err; h->dead = f.dead; hdr_extra(); }
  __syncwarp();
  fence_proxy_async();
  __syncwarp();
  if (lane == 0) { tma_store(gblob, base, (uint32_t)LT::agent_off); tma_store_wait(); }
  __syncwarp();
}

// Whole second: the outer-level resync test of OrderbookSimulator.py:86-87 for a book with the best prices best0 / best1 -- the
// snapshot row of the second that now_step ends when a best price has left the inner part of the book's initial range and the
// stream has a snapshot of that second, else nullptr.
__device__ __forceinline__ const int32_t* resync_row(const EnvConst& ec, const BookHdr* h, const lobsim_stream_t* stp, int best0, int best1, int now_step, int steps_per_sec) {
  const double prop = ec.outer_prop;
  const double bb = best0 == INT32_MIN ? 0.0 : (double)best0;
  const double bs = best1 == INT32_MAX ? (double)INFINITY : (double)best1;
  if (bb < (double)h->min_buy + prop * (double)h->init_buy_range || bs > (double)h->max_sell - prop * (double)h->init_sell_range) {
    const int sec = now_step / steps_per_sec;
    if (sec <= (int)stp->n_seconds && stp->snap_valid[sec]) return stp->snapshots + (size_t)sec * 2 * ec.cfg.n_levels * 2;
  }
  return nullptr;
}
__device__ __forceinline__ bool hdr_is_flat(const BookHdr* h) { return h->cnt[0][0] < 0; }

// ---- the flat form of a blob in HBM (book_flat.cuh): header with cnt[0] = {-1, n0}, cnt[1] = {seq, n1}; per side the order pool
//      (n x 16 B at the start of the side's order array); the agent tables as always.  Parts: lanes 0-1 the pools, 2-7 the agent tables.
//      Loads the body of a flat blob whose header is in shared memory; returns the bytes expected on `bar` (0: nothing was issued).
template <class LT>
__device__ __forceinline__ uint32_t flat_body_copy(unsigned char* sm, unsigned char* gm, uint64_t* bar, int lane, int n0, int n1) {
  const BookHdr* h = reinterpret_cast<const BookHdr*>(sm);
  uint32_t off = 0, len = 0;
  if (lane < 2) { off = LT::side_off + lane * LT::side_stride + LT::ord_off; len = (uint32_t)(lane ? n1 : n0) * 16u; }
  else if (lane < 8) {
    const int s = (lane - 2) / 3, part = (lane - 2) % 3;
    off = LT::agent_off + s * LT::NA * 12 + part * LT::NA * 4;
    len = (min((uint32_t)h->nag[s], (uint32_t)LT::NA) * 4 + 15) & ~15u;
  }
  const uint32_t total = __reduce_add_sync(FULL_MASK, len);
  if (total == 0) return 0;
  if (lane == 0) mbar_expect_tx(bar, total);
  __syncwarp();
  if (len) tma_load(sm + off, gm + off, len, bar);
  return total;
}
// FlatState of a flat blob whose header and pools are in shared memory; the best prices are recomputed from the pools
template <class LT>
__device__ __forceinline__ void flat_adopt(unsigned char* sm, int lane, FastState& f, FlatState& fs) {
  const BookHdr* h = reinterpret_cast<const BookHdr*>(sm);
  fs.n0 = h->cnt[0][1]; fs.n1 = h->cnt[1][1]; fs.seq = (uint32_t)h->cnt[1][0];
  f.best0 = flat_best_scan<LT, 0>(sm, lane, fs.n0);
  f.best1 = flat_best_scan<LT, 1>(sm, lane, fs.n1);
}
__device__ __forceinline__ void flat_mark(BookHdr* h, const FlatState& fs) {   // lane 0, before the blob goes back to HBM
  h->cnt[0][0] = -1; h->cnt[0][1] = fs.n0; h->cnt[1][0] = (int32_t)fs.seq; h->cnt[1][1] = fs.n1;
}

// Every flat blob back to the canonical sorted layout, in place (run by the host before anything that reads the level arrays:
// the general kernels, k_process_orders, the sorted-only replay kernel, the L3 dump).  One warp per book; sorted books: nothing.
template <class LT>
__global__ void __launch_bounds__(128) k_to_sorted(unsigned char* blobs, int n_envs) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int env = blockIdx.x * (blockDim.x >> 5) + warp;
  if (env >= n_envs) return;
  unsigned char* gblob = blobs + (size_t)env * LT::blob_bytes;
  if (!hdr_is_flat(reinterpret_cast<const BookHdr*>(gblob))) return;
  unsigned char* base = smem + (size_t)warp * LT::blob_bytes;
  if (lane < 8) reinterpret_cast<uint4*>(base)[lane] = reinterpret_cast<const uint4*>(gblob)[lane];   // the 128-byte header
  __syncwarp();
  const BookHdr* h = reinterpret_cast<const BookHdr*>(base);
  FlatState fs; fs.n0 = h->cnt[0][1]; fs.n1 = h->cnt[1][1]; fs.seq = (uint32_t)h->cnt[1][0];
#pragma unroll
  for (int s = 0; s < 2; s++) {
    const int n = s ? fs.n1 : fs.n0;
    const uint4* gp = flat_pool<LT>(gblob, s); uint4* sp = flat_pool<LT>(base, s);
    for (int i = lane; i < n; i += 32) sp[i] = gp[i];
  }
  __syncwarp();
  FastBook<LT> fb; fb.blob = base; fb.lane = lane;
  flat_leave(fb, fs);
  __syncwarp();
  if (lane == 0) reinterpret_cast<uint4*>(gblob)[0] = reinterpret_cast<const uint4*>(base)[0];          // cnt[2][2]
#pragma unroll
  for (int s = 0; s < 2; s++) {
    const int2 c = *fb.cnt(s);
    unsigned char* ss = fb.side(s); unsigned char* gs = gblob + LT::side_off + s * LT::side_stride;
    for (int i = lane; i < c.x; i += 32) { fb.P(gs)[i] = fb.P(ss)[i]; fb.LE(gs)[i] = fb.LE(ss)[i]; }
    for (int i = lane; i < c.y; i += 32) fb.O(gs)[i] = fb.O(ss)[i];
  }
}

// ====================================================================================================================
//  the straight-line replay kernels: T x (messages of the step + [resync]) with the straight-line message paths.  Used by
//  lobsim_replay when no fill log is requested, no agent order can be resting and the book capacities match one of the compiled
//  StaticLayouts.  kForm is the form a book runs in where it can (per book, re-decided every second); the others run on the sorted
//  straight-line path of book_fast.cuh:
//    REPLAY_SORTED (k_replay_fast): the sorted path for every book;
//    REPLAY_FLAT   (k_replay_flat): the flat order pools of book_flat.cuh for every book that fits them (at most FLAT_CAP resting
//                  orders per side);
//    REPLAY_HYBRID (k_replay_hyb, deep layouts): the hybrid book of book_hybrid.cuh -- the levels near the touch in a flat order
//                  pool, the rest in the sorted arrays -- for every book that can take that form.
//  The blob in HBM is the canonical sorted layout on entry, and on exit unless the flat form may be stored (p.allow_flat).  The
//  kind of a handle is fixed in lobsim_create, only REPLAY_FLAT launches store the flat form, and the host converts every blob
//  to the sorted form (ensure_sorted) before a launch of any other kind: so only the REPLAY_FLAT kernel meets a flat blob.
// ====================================================================================================================
// (forced-inline functions, not lambdas: with lambdas the compiler schedules k_replay_flat differently)
// sorted -> the pool form of kForm, where the book can take it (the flat pools: with `slack` orders to spare per side)
template <class LT, ReplayKind kForm>
__device__ __forceinline__ void pool_enter(const FastBook<LT>& fb, FastState& f, FlatState& fs, HybState& hs, bool& flat, int slack) {
  if constexpr (kForm == REPLAY_HYBRID) {
    if (hyb_enter(fb, f, hs)) flat = true;
    else if (hs.n0 | hs.n1) { hyb_leave(fb, f, hs); hs.n0 = hs.n1 = 0; }   // one side was moved, the other could not be: put it back
  } else if (flat_fits(fb, slack)) { flat_enter(fb, fs); flat = true; }
}
// pool form -> sorted
template <class LT, ReplayKind kForm>
__device__ __forceinline__ void pool_leave(const FastBook<LT>& fb, FastState& f, FlatState& fs, HybState& hs, bool& flat) {
  if constexpr (kForm == REPLAY_HYBRID) { hyb_leave(fb, f, hs); hs.n0 = hs.n1 = 0; }
  else flat_leave(fb, fs);
  flat = false;
}
template <class LT, ReplayKind kForm>
__device__ __forceinline__ void replay_straight(const AdvParams& p, const EnvConst& ec) {
  constexpr bool kHyb = kForm == REPLAY_HYBRID;
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int env = blockIdx.x * (blockDim.x >> 5) + warp;
  if (env >= p.n_sel) return;
  const lobsim_cfg_t& c = ec.cfg;
  unsigned char* base = warp_smem_base(smem, warp, p.warp_smem);
  unsigned char* msgbuf = base + LT::agent_off;
  uint64_t* bars = reinterpret_cast<uint64_t*>(msgbuf + 2 * MSG_TILE_BYTES);
  unsigned char* gblob = p.blobs + (size_t)env * LT::blob_bytes;
  replay_blob_load<LT>(base, gblob, bars, lane);

  FastBook<LT> fb; fb.blob = base; fb.lane = lane;
  BookHdr* h = reinterpret_cast<BookHdr*>(base);
  FastState f; f.err = h->err; f.dead = h->dead; f.bail = 0; f.bail_vol = 0;
  if (kForm != REPLAY_FLAT || !hdr_is_flat(h)) fast_refresh_best(fb, f);
  // flat: the book is in the pool form of kForm (fs: the flat pools; hs: the hybrid book's pools near the touch)
  FlatState fs; fs.n0 = fs.n1 = 0; fs.seq = 0;
  HybState hs; hs.n0 = hs.n1 = 0; hs.floor0 = INT32_MIN; hs.floor1 = INT32_MAX; hs.seq = 0;
  bool flat = false;
  if (kForm == REPLAY_FLAT && hdr_is_flat(h)) { flat_adopt<LT>(base, lane, f, fs); flat = true; }   // the blob was stored in the flat form
  const lobsim_stream_t* stp = &p.streams[h->stream_id];
  MsgTiles mt(stp);
  const uint32_t* __restrict__ st_step_off = stp->step_off;
  int now_step = h->now_step;
  const int T = p.T;
  const int n_grid = (int)stp->n_grid_steps;
  unsigned g, g_end_all;
  stream_window(st_step_off, n_grid, now_step, T, f.err, f.dead, g, g_end_all);
  if (kForm != REPLAY_SORTED && !flat && g < g_end_all) pool_enter<LT, kForm>(fb, f, fs, hs, flat, 0);
  mt.start(msgbuf, bars, lane, g, g_end_all);
  const int steps_per_sec = ec.steps_per_sec;
  int sub = now_step >= 0 ? now_step % steps_per_sec : 0;

  // One pass per second, or per part of a second where the launch (T) or the stream begins or ends inside one: a replay book holds
  // no agent orders, so nothing happens at a step boundary that is not a second boundary, and the message segments run across
  // steps.  The hybrid book walks one grid step per pass instead: its pools are topped up at every step boundary.  now_step
  // advances by the steps a pass covered; where a book dies, it is recovered from the step offsets of that pass.
#pragma unroll 1
  for (int t = 0; t < T && !f.dead;) {
    const int left = n_grid - now_step;                      // grid steps left in the stream
    const int k = kHyb ? 1 : min(min(steps_per_sec - sub, T - t), left);   // steps of this pass
    if (min(k, left) <= 0) { f.err |= LOBSIM_ERR_END_OF_STREAM; f.dead = 1; break; }   // (k <= left in the other forms)
    const unsigned g_pass_end = __ldg(&st_step_off[now_step + k]);
#pragma unroll 1
    while (g < g_pass_end) {
      const unsigned tile = mt.rel(g);
      if (tile == mt.next_wait) mt.wait();
      const unsigned tile_end = (g / MSG_TILE + 1) * MSG_TILE;
      const unsigned lim = g_pass_end < tile_end ? g_pass_end : tile_end;
      const uint4* mp = reinterpret_cast<const uint4*>(msgbuf + (tile & 1) * MSG_TILE_BYTES) + (g % MSG_TILE);
      const unsigned cnt = lim - g;
      unsigned i = 0;
      int redo_vol = 0;                                      // (hybrid) the unfinished part of message i, for the sorted book
      if constexpr (kForm == REPLAY_FLAT) {
        if (flat) {
          // the volumes of the whole segment (<= 32 messages, one per lane) are checked at once; the per-message test is one predicate
          const bool bad_vol = __any_sync(FULL_MASK, (unsigned)lane < cnt && (int)mp[(unsigned)lane < cnt ? lane : 0].y <= 0);
          unsigned off = 0;                                  // (the loop walks a byte offset: no index arithmetic per message)
          const unsigned off_end = cnt * 16u;
          auto run = [&](auto vchk) {                        // (two copies of the loop: the one that runs has no volume test)
#pragma unroll 1
            for (; off != off_end; off += 16u) {
              const uint4 m = *reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(mp) + off);
              if (flat_message<LT, decltype(vchk)::value>(base, lane, f, fs, (int)m.x, (int)m.y, m.z, m.w)) return true;   // pool full
                                                             // (this message runs on the sorted book) or f.dead: EmptyOrderbookError
            }
            return false;
          };
          const bool stopped = __builtin_expect(bad_vol, 0) ? run(std::true_type{}) : run(std::false_type{});
          i = off >> 4;
          f.bail = 0;                                        // (not read: `stopped` without f.dead is the full pool)
          if (stopped && !f.dead) { flat_leave(fb, fs); flat = false; }
        }
      } else if constexpr (kHyb) {
        // the volumes of the whole segment at once: a segment with a bad one (never in valid data) runs on the sorted book, whose
        // routines test every order (assert order.volume > 0, Exchange.py:59-60)
        if (flat && __any_sync(FULL_MASK, (unsigned)lane < cnt && (int)mp[(unsigned)lane < cnt ? lane : 0].y <= 0))
          pool_leave<LT, kForm>(fb, f, fs, hs, flat);
        if (flat) {
#pragma unroll 1
          for (; i < cnt; i++) {
            const uint4 m = mp[i];
            if (hyb_message<LT>(fb, f, hs, (int)m.x, (int)m.y, m.z, m.w)) break;
          }
          if (f.bail) {                                      // this book cannot stay hybrid: back to the sorted form
            const int why = f.bail, rest = f.bail_vol;
            f.bail = 0; f.bail_vol = 0;
            pool_leave<LT, kForm>(fb, f, fs, hs, flat);
            if (why == FLAT_BAIL_FULL) redo_vol = rest;      // the unfinished part of message i runs on the sorted book
            else i++;
          }
        }
      }
      if (!flat && !f.dead) {
#pragma unroll 1
        for (; i < cnt; i++) {
          const uint4 m = mp[i];
          int v = (int)m.y;
          if constexpr (kHyb) { if (redo_vol) v = redo_vol; redo_vol = 0; }
          fast_message(fb, f, (int)m.x, v, m.z, m.w);
          if (f.dead) break;
        }
      }
      if (f.dead) { g += i; break; }                        // g: the message the book died of
      g = lim;
      if (g == tile_end) { __syncwarp(); mt.issue(); }
    }
    if (f.dead) {                                            // now_step: the step that holds message g (a step without messages holds none)
      while (__ldg(&st_step_off[now_step + 1]) <= g) now_step++;
      break;
    }
    now_step += k; t += k; sub += k;
    if constexpr (kHyb) { if (flat) hyb_top_up(fb, f, hs); }
    if (sub == steps_per_sec) {                              // whole second: outer-level resync, OrderbookSimulator.py:86-87
      sub = 0;
      if (c.resync && (!p.resync_last_only || t == T)) {
        if (const int32_t* row = resync_row(ec, h, stp, f.best0, f.best1, now_step, steps_per_sec)) {
          if (flat && !flat_resync_needed(h, row, c.n_levels, lane)) {
            if constexpr (kHyb) hyb_update_trackers(fb, hs);
            else flat_update_trackers<LT>(base, lane, fs);
          } else {
            if (flat) pool_leave<LT, kForm>(fb, f, fs, hs, flat);
            fast_resync(fb, f, row, c.n_levels);
          }
        }
      }
      if constexpr (kForm != REPLAY_SORTED) {
        // (flat pools) renumber the time-priority stamps long before they wrap
        if (kForm == REPLAY_FLAT && flat && fs.seq > 0xE0000000u) pool_leave<LT, kForm>(fb, f, fs, hs, flat);
        if (!flat) pool_enter<LT, kForm>(fb, f, fs, hs, flat, 8);   // back to the pool form once the book has shrunk
      }
    }
  }
  // the hybrid form never goes to HBM; the flat form only where the caller allows it
  if (flat && (kHyb || !p.allow_flat)) pool_leave<LT, kForm>(fb, f, fs, hs, flat);
  mt.drain();
  replay_blob_store<LT>(gblob, base, lane, now_step, f, [&]() { if (flat) flat_mark(h, fs); });
}

// 72 registers: 28 resident warps per SM with the 64/256/32 blob (8 blocks = 64 registers: A/B in profiles/)
template <class LT>
__global__ void __launch_bounds__(128, 7) k_replay_flat(const __grid_constant__ AdvParams p, const __grid_constant__ EnvConst ec) {
  replay_straight<LT, REPLAY_FLAT>(p, ec);
}
template <class LT>
__global__ void __launch_bounds__(128, 7) k_replay_fast(const __grid_constant__ AdvParams p, const __grid_constant__ EnvConst ec) {
  replay_straight<LT, REPLAY_SORTED>(p, ec);
}
template <class LT>
__global__ void __launch_bounds__(128, 3) k_replay_hyb(const __grid_constant__ AdvParams p, const __grid_constant__ EnvConst ec) {
  replay_straight<LT, REPLAY_HYBRID>(p, ec);
}

// ====================================================================================================================
//  the env fast kernel: k_advance<true> with the straight-line tracked order path (book_fast.cuh fast_order<LT,true>)
//  and all per-env scalars (counters, portfolio, per-step flow) in the shared-memory header instead of registers.
// ====================================================================================================================
static __device__ __noinline__ uint32_t reset_book_cold(unsigned char* blob, const Layout* L, int lane, const lobsim_cfg_t* c, const lobsim_stream_t* st, int stream_id, int start_step) {
  Book b; b.blob = blob; b.L = *L; b.lane = lane;
  WarpState w;
  __syncwarp();
  load_state(b, w);
  w.fill_log = nullptr; w.fill_cap = 0; w.n_fills = 0;
  init_book_from_snapshot(b, w, *c, *st, stream_id, start_step);
  store_state(b, w);
  return pack_errdead(w.err, w.dead);
}

// ---- the OCCUPIED part of a book blob (env kernels: one blob round trip per env step when a policy runs between steps) ----
// Only what the counters in the header say is in use moves between HBM and shared memory: per side the level prices, the
// level ends and the order entries up to {nlv, nord}, and the agent tables up to nag -- about 1.5 KB of a 6.5 KB blob for a
// 10-level book.  Sizes are rounded up to the 16-byte granularity of cp.async.bulk; every array of a StaticLayout starts
// 16-byte aligned and its capacity is a multiple of 16 bytes, so a rounded-up part never leaves its array.
// Warp-collective: lane k < 12 owns part k (its offset and length are a few integer operations on the header counters) and
// issues its own bulk copy; lane 0 posts the byte total on the mbarrier first.  LOAD: the header has already arrived in shared
// memory; returns the bytes expected on `bar` (0: nothing was issued).
template <class LT, bool LOAD>
__device__ __forceinline__ uint32_t blob_body_copy(unsigned char* sm, unsigned char* gm, uint64_t* bar, int lane) {
  static_assert(LT::NL % 8 == 0 && LT::NO % 2 == 0 && LT::NA % 4 == 0 && LT::ord_off % 16 == 0 && LT::side_stride % 16 == 0 && LT::agent_off % 16 == 0,
                "StaticLayout arrays must be 16-byte aligned for the partial blob copies");
  const BookHdr* h = reinterpret_cast<const BookHdr*>(sm);
  const int s = lane >= 6 ? 1 : 0, part = lane - s * 6;     // parts 0-2: level prices, level ends, orders; 3-5: agent price / volume / id
  uint32_t off = 0, len = 0;
  if (lane < 12) {
    const uint32_t so = LT::side_off + s * LT::side_stride, ao = LT::agent_off + s * LT::NA * 12;
    if (part == 0)      { off = so;                 len = min((uint32_t)h->cnt[s][0], (uint32_t)LT::NL) * 4; }
    else if (part == 1) { off = so + LT::lvend_off; len = min((uint32_t)h->cnt[s][0], (uint32_t)LT::NL) * 2; }
    else if (part == 2) { off = so + LT::ord_off;   len = min((uint32_t)h->cnt[s][1], (uint32_t)LT::NO) * 8; }
    else                { off = ao + (part - 3) * LT::NA * 4; len = min((uint32_t)h->nag[s], (uint32_t)LT::NA) * 4; }
    len = (len + 15) & ~15u;
  }
  const uint32_t total = __reduce_add_sync(FULL_MASK, len);
  if (total == 0) return 0;
  if (LOAD) { if (lane == 0) mbar_expect_tx(bar, total); __syncwarp(); }
  if (len) { if (LOAD) tma_load(sm + off, gm + off, len, bar); else tma_store_part(gm + off, sm + off, len); }
  return total;
}

#ifndef LOBSIM_ENVFAST_WARPS
#define LOBSIM_ENVFAST_WARPS 8    // warps per CTA of the env fast kernel: the warps of a CTA move through the phases of a step together, so
                                  // fewer, larger CTAs = fewer phases in flight per SM = a warmer instruction cache ("no instruction" is the
                                  // top stall).  Measured at 80 registers / 24 resident warps per SM (profiles/r02_env_ab.txt): 4 warps per CTA
                                  // 4.36e7 env steps/s, 8: 4.77e7, 12: 4.53e7, 24: 4.21e7; no phase sync at all: 3.41e7
#endif
#ifndef LOBSIM_ENVFAST_MINB
#define LOBSIM_ENVFAST_MINB (24 / LOBSIM_ENVFAST_WARPS)   // resident CTAs per SM the register allocation aims at (80 registers: measured
#endif                                                     // +9 % over 128 registers / 16 warps per SM, profiles/r02_env_ab.txt)
// ... but never more CTAs than the shared memory of an SM can hold for this layout (deep 50-level books: 2 CTAs, no register cap)
template <class LT>
constexpr int env_min_blocks() {
  const int warp_bytes = (LT::blob_bytes + 2 * MSG_TILE_BYTES + scratch_bytes(LT::NA) + 32 + 128 + 127) & ~127;
  const int fit = (227 * 1024) / (LOBSIM_ENVFAST_WARPS * warp_bytes);
  return fit < 1 ? 1 : (fit < LOBSIM_ENVFAST_MINB ? fit : LOBSIM_ENVFAST_MINB);
}
// SYNC: the launch consists of full CTAs only, whose warps move through the phases of a step together
// (launch_env puts the n_sel % warps-per-CTA tail into a second, free-running launch).
// Per-warp values that are only needed outside the order-processing phase (B) live in the spare shared memory behind the
// mbarriers instead of in registers: the kernel is register-bound (128 registers at 16 resident warps per SM) and phase B is where it spills.
struct StepSave { double cash0, p0, price; long long inv0, episode_start_us, st_t0_us; };
static_assert(sizeof(StepSave) <= 128, "StepSave must fit the 128-byte per-warp slot behind the mbarriers (warp_smem_bytes)");
// RARE: the configuration uses z-score normalisation or a RollingSharpe reward (their code is compiled out otherwise).
template <class LT, bool SYNC, bool RARE>
__global__ void __launch_bounds__(32 * LOBSIM_ENVFAST_WARPS, env_min_blocks<LT>()) k_env_fast(const __grid_constant__ AdvParams p, const __grid_constant__ EnvConst ec) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // The warps of a CTA move through the phases of a step together (SYNC: a __syncthreads between phases): the instruction
  // working set at any moment is a single phase, which is what keeps the 32 KB L1.5 I-cache warm
  // (profiles/r01_envstep_*: "no instruction" was the top stall with free-running warps).
  const int sel = p.sel_offset + blockIdx.x * (blockDim.x >> 5) + warp;
  if (sel >= p.n_sel) return; // only in SYNC == false launches
  const int env = p.env_ids ? p.env_ids[sel] : sel;
  const lobsim_cfg_t& c = ec.cfg;
  unsigned char* base = warp_smem_base(smem, warp, p.warp_smem);
  unsigned char* msgbuf = base + LT::blob_bytes;
  int2* scratch = reinterpret_cast<int2*>(msgbuf + 2 * MSG_TILE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(scratch) + scratch_bytes(LT::NA));
  unsigned char* gblob = p.blobs + (size_t)env * LT::blob_bytes;
  // ---- book blob, HBM -> shared memory: the 128-byte header first, then only the occupied part of the arrays (a reset rebuilds
  //      the book from the snapshot and needs the header alone)
  if (lane == 0) {
    mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
    fence_mbar_init();
    mbar_expect_tx(&bars[2], (uint32_t)sizeof(BookHdr));
    tma_load(base, gblob, (uint32_t)sizeof(BookHdr), &bars[2]);
  }
  __syncwarp();
  mbar_wait(&bars[2], 0);
  FastBook<LT> fb; fb.blob = base; fb.lane = lane;
  Book b; b.blob = base; b.L = p.L; b.lane = lane;
  BookHdr* h = reinterpret_cast<BookHdr*>(base);
  // a blob in the flat form of book_flat.cuh (stored by k_replay_flat) is converted to the sorted level arrays on load: this kernel
  // runs on the sorted form only
  if (!p.reset_mode) {
    if (hdr_is_flat(h)) {
      if (flat_body_copy<LT>(base, gblob, &bars[2], lane, h->cnt[0][1], h->cnt[1][1])) mbar_wait(&bars[2], 1);
      flat_leave_fn<LT>(base, lane, h->cnt[0][1], h->cnt[1][1]);
    } else if (blob_body_copy<LT, true>(base, gblob, &bars[2], lane)) mbar_wait(&bars[2], 1);
  }
  FastState f; f.err = h->err; f.dead = h->dead; f.bail = 0; f.bail_vol = 0;
  f.fill_log = p.fill_log ? p.fill_log + (size_t)env * p.fill_cap : nullptr; f.fill_cap = p.fill_cap;
  if (lane == 0) h->n_fills = 0;
  const int F = c.n_features;

  // ---- reset prologue ----------------------------------------------------------------------------------------------
  int stream_id = h->stream_id;
  if (p.reset_mode) {
    stream_id = p.reset_stream_ids[sel];
    int start = p.reset_steps[sel] - (p.reset_mode == 2 ? c.warmup_steps : 0);
    if (stream_id < 0 || stream_id >= p.n_streams) { stream_id = 0; start = -1; }
    const uint32_t ed = reset_book_cold(base, &p.L, lane, &ec.cfg, &p.streams[stream_id], stream_id, start);
    f.err = ed & 0x7fffffffu; f.dead = (int)(ed >> 31);
    if (p.reset_mode == 2 && lane == 0) {
      h->episode_start_step = p.reset_steps[sel];
      if (!c.portfolio_carryover || !h->has_reset) { h->inventory = c.initial_inventory; h->cash = c.initial_cash; }
      h->has_reset = 1;
    }
    __syncwarp();
  }
  fast_refresh_best(fb, f);
  const lobsim_stream_t* stp = &p.streams[stream_id];
  MsgTiles mt(stp);
  const uint32_t* __restrict__ st_step_off = stp->step_off;
  StepSave* sv = reinterpret_cast<StepSave*>(bars + 4);
  int now_step = h->now_step;
  if (lane == 0) { sv->st_t0_us = stp->t0_us; sv->episode_start_us = stp->t0_us + (long long)h->episode_start_step * c.step_us; sv->price = h->price; }
  __syncwarp();
  FeatState* fstate_env = p.fstate + (size_t)env * LOBSIM_MAX_FEATURES;
  NormState* nstate_env = RARE && p.nstate ? p.nstate + (size_t)env * LOBSIM_MAX_FEATURES : nullptr;
  double* rings_env = p.rings + (size_t)env * ec.ring_stride;
  double feat_cur = 0.0;
  if (lane < F) feat_cur = fstate_env[lane].cur;
  const int t0_mod_min = (int)stp->reserved;   // t0_us % 60 s, filled in by lobsim_load_stream

  auto tops = [&](StepView& v) { // Orderbook.best_* / microprice, models.py:72-101
    v.have_tops = f.best0 != INT32_MIN && f.best1 != INT32_MAX;
    if (v.have_tops) {
      v.bb = f.best0; v.bs = f.best1;
      __syncwarp();
      v.bv = best_level_volume(b, 0, h->cnt[0][0]); v.sv = best_level_volume(b, 1, h->cnt[1][0]);
      double imb; v.price = microprice(v.bb, v.bs, v.bv, v.sv, imb);
    } else { v.bb = v.bs = v.bv = v.sv = 0; v.price = NAN; }
  };
  if (p.reset_mode == 2) { // State(...) + _reset_features, HOE.py:152-154,218-221
    StepView v; tops(v);
    v.inventory = h->inventory; v.now_us = sv->st_t0_us + (long long)now_step * c.step_us;
    v.us_in_min = us_in_minute(t0_mod_min, now_step, ec);
    v.n_ext0 = v.n_ext1 = v.vol_ext0 = v.vol_ext1 = v.n_int0 = v.n_int1 = v.vol_int0 = v.vol_int1 = 0;
    __syncwarp();
    if (lane == 0) sv->price = v.price;
    feat_cur = features_step<RARE>(&ec, fstate_env, nstate_env, rings_env, lane, v, sv->episode_start_us, 1);
    __syncwarp();
  }

  // ---- message pipeline ----------------------------------------------------------------------------------------------
  const int T = p.T;
  unsigned g, g_end_all;
  stream_window(st_step_off, (int)stp->n_grid_steps, now_step, T, f.err, f.dead, g, g_end_all);
  mt.start(msgbuf, bars, lane, g, g_end_all);
  if (SYNC) __syncthreads();
  const int steps_per_sec = ec.steps_per_sec;
  int sub = now_step >= 0 ? now_step % steps_per_sec : 0;

  AgentGenFast gen; gen.side = 3; gen.stage = 0; gen.need = 0; gen.todo0 = gen.todo1 = gen.wm0 = gen.wm1 = 0; gen.wide_removed = gen.wide_pos = 0;
  gen.pending_id = 0; gen.base0 = gen.base1 = 0; gen.clear_vol = -1; gen.clear_side = 0;
  const int Q = c.max_quote_level - c.min_quote_level;
  int* diff_scratch = reinterpret_cast<int*>(scratch);
  bool agent_phase = false;
#pragma unroll 1
  for (int t = 0; t < T; t++) {
    if (SYNC) __syncthreads(); // ---- phase A: action -> ladders (fp64) -----------------------------------------------------
    __syncwarp();
    if (lane == 0) { sv->cash0 = h->cash; sv->p0 = sv->price; sv->inv0 = h->inventory; } // deepcopy(self.state), HOE.py:166
    if (lane < 8) h->flow[lane] = 0;
    __syncwarp();
    if (p.agent_kind != LOBSIM_AGENT_NONE) {
      double* act_sm = reinterpret_cast<double*>(scratch);
      if (p.agent_kind == LOBSIM_AGENT_EXTERNAL) {
        const double* a = p.actions_in + ((size_t)t * p.n_sel + sel) * ec.action_dim;
        if (lane < 5) act_sm[lane] = lane < ec.action_dim ? __ldg(&a[lane]) : 0.0;
      } else {
        const lobsim_agent_t* agp = p.agents ? p.agents + sel : &p.agent;
        const double inv_obs = __shfl_sync(FULL_MASK, feat_cur, agp->inventory_index & 31);
        if (lane == 0) agent_action_cold(agp, inv_obs, act_sm, env, now_step);
      }
      __syncwarp();
      const double a0 = act_sm[0], a1 = act_sm[1], a2 = act_sm[2], a3 = act_sm[3], a4 = act_sm[4];
      const double mine = lane < 5 ? act_sm[lane] : 0.0;
      __syncwarp();
      if (p.act && p.agent_kind != LOBSIM_AGENT_EXTERNAL && lane < ec.action_dim) p.act[((size_t)t * p.n_sel + sel) * ec.action_dim + lane] = mine;
      if (p.obs && !p.out_final_obs_only && c.inc_prev_action_in_obs && lane < ec.action_dim)
        p.obs[((size_t)t * p.n_sel + sel) * ec.obs_dim + F + lane] = mine;
      if (!f.dead) {
        const AgentGen g0 = agent_prepare(b, f.best0, f.best1, h->nag[0], h->nag[1], h->inventory, &ec, a0, a1, a2, a3, a4, p.beta_tab, diff_scratch);
        f.err |= g0.err_out; if (g0.dead_out) f.dead = 1;
        gen = agent_gen_fast_init(g0, lane, diff_scratch);
        agent_phase = true;
      }
    }
    if (SYNC) __syncthreads(); // ---- phase B: the step's orders: the agent's first, then the historical messages of (now, now + step]
    {
      if (!f.dead && now_step >= (int)stp->n_grid_steps) { f.err |= LOBSIM_ERR_END_OF_STREAM; f.dead = 1; } // re-read: keeps a register free
      const unsigned g_step_end = f.dead ? g : __ldg(&st_step_off[now_step + 1]);
#pragma unroll 1
      for (;;) {
        int type, side, oprice, vol; uint32_t ref; bool is_agent;
        if (agent_phase) {
          if (!agent_next_fast(fb, f, gen, diff_scratch, Q, c.tick_size, type, side, oprice, vol, ref)) { agent_phase = false; continue; }
          is_agent = true;
        } else {
          if (f.dead || g >= g_step_end) break;
          const unsigned tile = mt.rel(g);
          if (tile == mt.next_wait) mt.wait();
          const uint4 m = *reinterpret_cast<const uint4*>(msgbuf + (tile & 1) * MSG_TILE_BYTES + (g % MSG_TILE) * 16);
          oprice = (int)m.x; vol = (int)m.y; ref = m.z; type = (int)(m.w & 7u); side = (int)((m.w >> 3) & 1u);
          is_agent = false;
          g++;
          if (g % MSG_TILE == 0) { __syncwarp(); mt.issue(); }
        }
        if (!f.dead) fast_order_full<LT, true>(fb, f, type, side, oprice, vol, ref, is_agent);
      }
    }
    if (!f.dead) {
      now_step++;
      if (++sub == steps_per_sec) {                          // whole second: outer-level resync, OrderbookSimulator.py:86-87
        sub = 0;
        if (c.resync && (!p.resync_last_only || t == T - 1)) {
          const double prop = ec.outer_prop;
          const double bbd = f.best0 == INT32_MIN ? 0.0 : (double)f.best0;
          const double bsd = f.best1 == INT32_MAX ? (double)INFINITY : (double)f.best1;
          if (bbd < (double)h->min_buy + prop * (double)h->init_buy_range || bsd > (double)h->max_sell - prop * (double)h->init_sell_range) {
            const int sec = now_step / steps_per_sec;
            if (sec <= (int)stp->n_seconds && stp->snap_valid[sec]) {
              const int32_t* row = stp->snapshots + (size_t)sec * 2 * c.n_levels * 2;
              fast_resync_tracked(fb, f, row, c.n_levels, scratch);
            }
          }
        }
      }
    }
    if (SYNC) __syncthreads(); // ---- phase C: update_internal_state + _update_features + reward, HOE.py:163-178,199-204 -------------
    StepView v; tops(v);
    if (!v.have_tops) f.err |= LOBSIM_ERR_EMPTY_BOOK;
    const double price = v.price;
    if (lane == 0) sv->price = price;
    v.inventory = h->inventory; v.now_us = sv->st_t0_us + (long long)now_step * c.step_us;
    v.us_in_min = us_in_minute(t0_mod_min, now_step, ec);
    v.n_ext0 = h->flow[0]; v.n_ext1 = h->flow[1]; v.vol_ext0 = h->flow[2]; v.vol_ext1 = h->flow[3];
    v.n_int0 = h->flow[4]; v.n_int1 = h->flow[5]; v.vol_int0 = h->flow[6]; v.vol_int1 = h->flow[7];
    __syncwarp(); // every lane has read this step's flow counters before lanes 0-7 zero them for the next step
    feat_cur = features_step<RARE>(&ec, fstate_env, nstate_env, rings_env, lane, v, sv->episode_start_us, 0);
    const bool write_now = !p.out_final_obs_only || t == T - 1;
    if (p.obs && write_now) {
      double* o = p.obs + ((size_t)(p.out_final_obs_only ? 0 : t) * p.n_sel + sel) * ec.obs_dim;
      if (lane < F) o[lane] = feat_cur;
      if (c.inc_prev_action_in_obs && lane < ec.action_dim && (p.agent_kind == LOBSIM_AGENT_NONE || p.out_final_obs_only)) o[F + lane] = 0.0;
    }
    if (p.agent_kind != LOBSIM_AGENT_NONE) {
      const double cash1 = h->cash; const long long inv1 = h->inventory;
      const bool d = now_step >= h->episode_start_step + c.episode_steps; // terminal_time - now < step/2, HOE.py:172
      const double r = step_reward<RARE>(p, c, env, lane, d, sv->cash0, sv->inv0, sv->p0, cash1, inv1, price, f.err);
      if (lane == 0) {
        if (p.rew) p.rew[(size_t)t * p.n_sel + sel] = r;
        if (p.done) p.done[(size_t)t * p.n_sel + sel] = d ? 1 : 0;
      }
      if (p.info) write_info(p.info + ((size_t)t * p.n_sel + sel) * LOBSIM_INFO_DIM, lane, v, cash1, inv1, f.err);
    }
  }
  if (T == 0 && p.obs && p.reset_mode == 2) { // reset with no warm-up: obs straight after _reset_features
    double* o = p.obs + (size_t)sel * ec.obs_dim;
    if (lane < F) o[lane] = feat_cur;
    if (c.inc_prev_action_in_obs && lane < ec.action_dim) o[F + lane] = 0.0;
  }
  mt.drain();

  // ---- shared memory -> HBM: the header and the occupied part of the arrays; every issuing lane commits and waits for its own copy
  __syncwarp();
  if (lane == 0) {
    if (f.fill_log && h->n_fills > f.fill_cap) f.err |= LOBSIM_ERR_FILL_LOG_FULL;
    h->now_step = now_step; h->price = sv->price; h->err = f.err; h->dead = f.dead;
    if (p.fill_count) p.fill_count[env] = h->n_fills;
  }
  __syncwarp();
  fence_proxy_async();
  __syncwarp();
  if (lane == 12) tma_store_part(gblob, base, (uint32_t)sizeof(BookHdr));
  blob_body_copy<LT, false>(base, gblob, nullptr, lane);
  if (lane <= 12) { tma_store_commit(); tma_store_wait(); }
  __syncwarp();
}

// ====================================================================================================================
//  lobsim_submit_orders_dev: Exchange.process_order for every env's own row of orders, one warp per env -- k_submit_orders<LT>
//  (the compiled layouts) and k_submit_orders_general (lobsim.cu: every other handle)
// ====================================================================================================================
struct SubmitParams {
  unsigned char* blobs; Layout L; int32_t n_envs; int32_t blob_in_global;
  int32_t max_orders;
  const lobsim_order_t* orders;   // [n_envs][max_orders], 16-byte aligned
  const int32_t* count;           // [n_envs]
  uint32_t* refs;                 // [n_envs][max_orders] or null
  int32_t max_fills;
  lobsim_fill_t* fills;           // [n_envs][max_fills]; null when max_fills == 0 (then no fill is logged or counted)
  int32_t* n_fills;               // [n_envs] or null
};

// the number of orders of env's row: count clamped to [0, max_orders]
__device__ __forceinline__ int submit_count(const SubmitParams& p, int env) {
  const int n = p.count[env];
  return n < 0 ? 0 : n > p.max_orders ? p.max_orders : n;
}

// The first n orders of env's row, in order, through apply(order) -> its ref (warp-collective, uniform).  The row is read 32
// orders at a time, one per lane (two 16-byte loads), and each order is broadcast to the warp; the refs of a group are stored
// by the lanes that read the orders, and the refs beyond n are 0.  Orders with a type outside 1..4 or a direction outside 0..1
// are skipped (ref 0).
template <class Apply>
__device__ __forceinline__ void submit_row(const SubmitParams& p, int env, int n, int lane, Apply apply) {
  const int4* row = reinterpret_cast<const int4*>(p.orders + (size_t)env * p.max_orders);
  uint32_t* refs = p.refs ? p.refs + (size_t)env * p.max_orders : nullptr;
  const int kend = refs ? p.max_orders : n;
#pragma unroll 1
  for (int k0 = 0; k0 < kend; k0 += 32) {
    const int m = min(32, n - k0);
    int4 a = make_int4(0, 0, 0, 0), c = a;   // {env, type, direction, price}, {volume, is_external, ref, reserved}
    if (lane < m) { a = row[2 * (k0 + lane)]; c = row[2 * (k0 + lane) + 1]; }
    uint32_t my_ref = 0;
#pragma unroll 1
    for (int i = 0; i < m; i++) {
      lobsim_order_t o;
      o.env = env; o.type = __shfl_sync(FULL_MASK, a.y, i); o.direction = __shfl_sync(FULL_MASK, a.z, i);
      o.price = __shfl_sync(FULL_MASK, a.w, i); o.volume = __shfl_sync(FULL_MASK, c.x, i);
      o.is_external = __shfl_sync(FULL_MASK, c.y, i); o.ref = (uint32_t)__shfl_sync(FULL_MASK, c.z, i); o.reserved = 0;
      uint32_t id = 0;
      if ((unsigned)(o.type - LOBSIM_MSG_LIMIT) <= LOBSIM_MSG_MARKET - LOBSIM_MSG_LIMIT && (unsigned)o.direction <= 1u) id = apply(o);
      if (lane == i) my_ref = id;
    }
    if (refs && k0 + lane < p.max_orders) refs[k0 + lane] = my_ref;
  }
}

// Volume None (Exchange.py:140) on the straight-line path, which takes removals with a volume only: a removal of at least the
// resting volume removes the whole order (:142-146), which is what volume None does -- except where book.cuh
// remove_order(has_vol = false) differs: `ref` is not in the level and the level's head is a snapshot aggregate, which a removal
// with a volume reduces and volume None may not (the assert of :134, BAD_VOLUME).  True in that case.
template <class LT>
__device__ __forceinline__ bool fast_none_hits_aggregate(const FastBook<LT>& fb, int side, int price, uint32_t ref) {
  unsigned char* sb = fb.side(side);
  int j, jeq;
  fast_find_any(fb, sb, side, fb.cnt(side)->x, price, j, jeq);
  if (jeq < 0) return false;                                 // no level: nothing happens either way (:129-132)
  const int start = jeq > 0 ? (int)fb.LE(sb)[jeq - 1] : 0, end = fb.LE(sb)[jeq];
  for (int base = start; base < end; base += 32) {
    const int i = base + fb.lane;
    if (__any_sync(FULL_MASK, i < end && fb.O(sb)[i].y == ref)) return false;
  }
  return fb.O(sb)[start].y == LOBSIM_REF_AGGREGATE;
}

// One order record through the tracked straight-line path (fast_order_full<LT, true>), with what that path does not report
// itself: the ref of a limit order that rested (an agent order rested iff next_agent_id moved, and got its old value; an
// external one iff its own side gained an order -- fills only remove orders from the opposite side) and volume None.
template <class LT>
__device__ __forceinline__ uint32_t fast_submit_order(const FastBook<LT>& fb, FastState& f, const lobsim_order_t& o) {
  if (f.dead) return 0;
  const bool is_agent = !o.is_external;
  const int side = o.direction;
  BookHdr* h = reinterpret_cast<BookHdr*>(fb.blob);
  __syncwarp();
  if (o.type == LOBSIM_MSG_DELETE || o.type == LOBSIM_MSG_CANCEL) {
    const uint32_t ref = is_agent ? (LOBSIM_REF_AGENT | (o.ref & 0x7fffffffu)) : o.ref;
    int vol = o.volume;
    if (vol <= 0) {
      if (fast_none_hits_aggregate(fb, side, o.price, ref)) { f.err |= LOBSIM_ERR_BAD_VOLUME; return 0; }
      vol = INT32_MAX;
    }
    fast_order_full<LT, true>(fb, f, o.type, side, o.price, vol, ref, is_agent);
    return 0;
  }
  if (o.volume <= 0) { f.err |= LOBSIM_ERR_BAD_VOLUME; return 0; }
  const uint32_t id0 = h->next_agent_id;
  const int n0 = fb.cnt(side)->y;
  fast_order_full<LT, true>(fb, f, o.type, side, o.price, o.volume, is_agent ? 0u : o.ref, is_agent);
  __syncwarp();
  if (o.type != LOBSIM_MSG_LIMIT) return 0;
  if (is_agent) return h->next_agent_id != id0 ? id0 : 0u;
  return fb.cnt(side)->y == n0 + 1 ? 0xffffffffu : 0u;
}

template <class LT>
__host__ __device__ constexpr int submit_warp_bytes() { return (LT::blob_bytes + 8 + 127) & ~127; }   // the blob and one mbarrier
#define LOBSIM_SUBMIT_WARPS 4

// The frame of k_env_fast: the header first, then only the occupied part of the blob (a flat blob left by k_replay_flat is
// converted on load), the orders, and the occupied part back in the sorted form.  Like Exchange.process_order, the call moves
// only the books and the agent tables: the portfolio, the per-step flow and the fill counter that fast_record_fn moves in the
// header are restored before the store.  An env with count 0 is neither read nor written.
template <class LT>
__global__ void __launch_bounds__(32 * LOBSIM_SUBMIT_WARPS) k_submit_orders(const __grid_constant__ SubmitParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int env = blockIdx.x * (blockDim.x >> 5) + warp;
  if (env >= p.n_envs) return;
  const int n = submit_count(p, env);
  if (n == 0) {
    submit_row(p, env, 0, lane, [](const lobsim_order_t&) { return 0u; });
    if (p.n_fills && lane == 0) p.n_fills[env] = 0;
    return;
  }
  unsigned char* base = smem + (size_t)warp * submit_warp_bytes<LT>();
  uint64_t* bar = reinterpret_cast<uint64_t*>(base + LT::blob_bytes);
  unsigned char* gblob = p.blobs + (size_t)env * LT::blob_bytes;
  if (lane == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
    mbar_expect_tx(bar, (uint32_t)sizeof(BookHdr));
    tma_load(base, gblob, (uint32_t)sizeof(BookHdr), bar);
  }
  __syncwarp();
  mbar_wait(bar, 0);
  BookHdr* h = reinterpret_cast<BookHdr*>(base);
  if (hdr_is_flat(h)) {
    if (flat_body_copy<LT>(base, gblob, bar, lane, h->cnt[0][1], h->cnt[1][1])) mbar_wait(bar, 1);
    flat_leave_fn<LT>(base, lane, h->cnt[0][1], h->cnt[1][1]);
  } else if (blob_body_copy<LT, true>(base, gblob, bar, lane)) mbar_wait(bar, 1);
  __syncwarp();
  const long long inventory_in = h->inventory;
  const double cash_in = h->cash;
  const int flow_in = lane < 8 ? h->flow[lane] : 0, n_fills_in = h->n_fills;
  __syncwarp();
  if (lane == 0) h->n_fills = 0;
  FastBook<LT> fb; fb.blob = base; fb.lane = lane;
  FastState f; f.err = h->err; f.dead = h->dead; f.bail = 0; f.bail_vol = 0;
  f.fill_log = p.max_fills > 0 ? p.fills + (size_t)env * p.max_fills : nullptr; f.fill_cap = p.max_fills;
  fast_refresh_best(fb, f);
  submit_row(p, env, n, lane, [&](const lobsim_order_t& o) { return fast_submit_order<LT>(fb, f, o); });
  __syncwarp();
  const int n_fills = f.fill_log ? h->n_fills : 0;
  __syncwarp();
  if (lane < 8) h->flow[lane] = flow_in;
  if (lane == 0) {
    if (n_fills > f.fill_cap) f.err |= LOBSIM_ERR_FILL_LOG_FULL;
    h->inventory = inventory_in; h->cash = cash_in; h->n_fills = n_fills_in;
    h->err = f.err; h->dead = f.dead;
    if (p.n_fills) p.n_fills[env] = n_fills;
  }
  __syncwarp();
  fence_proxy_async();
  __syncwarp();
  if (lane == 12) tma_store_part(gblob, base, (uint32_t)sizeof(BookHdr));
  blob_body_copy<LT, false>(base, gblob, nullptr, lane);
  if (lane <= 12) { tma_store_commit(); tma_store_wait(); }
  __syncwarp();
}
