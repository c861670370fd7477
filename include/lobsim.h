/*
 * lobsim.h -- C ABI of the B200-native limit-order-book simulation step.
 *
 * This is the drop-in boundary for the one hot path of JJJerome/rl4mm that this repository accelerates:
 * batched replay of LOBSTER message streams through a price-time-priority book, the agent's own resting
 * orders filling against historical flow, and the gym environment's features and rewards.
 *
 * The reference has no FFI of its own (it is pure Python); each entry point below names the reference
 * interface (file:line under the reference tree) that it replaces.  A maintainer binds this library with
 * ctypes (see INTEGRATION.md); rl4mm_b200/_lib.py is exactly that binding.
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in any signature.  `stream` is a cudaStream_t passed as void*
 *     (NULL = the legacy default stream).
 *   - pointers named *_dev are device pointers (e.g. torch tensor .data_ptr()); pointers named *_host are host
 *     pointers (pinned memory recommended).  Functions with the _host suffix do the H2D / D2H copies themselves.
 *   - every function returns 0 on success or a negative LOBSIM_E_* code; per-environment conditions that raise
 *     Python exceptions in the reference are reported through a sticky per-env error bitmask (lobsim_errors).
 *   - prices are LOBSTER integers (dollars x 10000), volumes are shares, both int32 on the device.
 *   - side / direction: 0 = buy, 1 = sell.
 */
#ifndef LOBSIM_H
#define LOBSIM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LOBSIM_ABI_VERSION 1

/* ---- return codes ------------------------------------------------------------------------------------------ */
#define LOBSIM_OK 0
#define LOBSIM_E_INVALID -1   /* bad argument / configuration                         */
#define LOBSIM_E_CUDA -2      /* a CUDA runtime call failed (see lobsim_last_error)   */
#define LOBSIM_E_NOMEM -3
#define LOBSIM_E_STATE -4     /* call order violated (e.g. step before reset)         */

/* ---- per-env sticky error bits (replace the reference's Python exceptions) ----------------------------------
 * Capacity bits: the book of every kernel family flags the capacity that an order (or a snapshot level of a reset or a resync)
 * would have to exceed, and only that one: LEVEL_OVERFLOW for one price level more than max_levels_per_side on a side,
 * ORDER_OVERFLOW for one resting order more than max_orders_per_side (snapshot aggregates count as orders), AGENT_OVERFLOW for one
 * agent order more than max_agent_orders, FILL_LOG_FULL for one fill more than fill_log_capacity in one call.  The order that
 * does not fit is dropped, so a flagged book no longer follows the reference.  Straight-line and general kernels flag in the
 * call in which the capacity is first exceeded; the hybrid replay book (csrc/book_hybrid.cuh) may hold a temporary level excess
 * in its order pool and flags it when it leaves that form, at the latest at the end of the call.                        */
#define LOBSIM_ERR_EMPTY_BOOK 1u        /* EmptyOrderbookError, rl4mm/orderbook/Exchange.py:32,183-186            */
#define LOBSIM_ERR_LEVEL_OVERFLOW 2u    /* more price levels on a side than max_levels_per_side                  */
#define LOBSIM_ERR_ORDER_OVERFLOW 4u    /* more resting orders on a side than max_orders_per_side                */
#define LOBSIM_ERR_AGENT_OVERFLOW 8u    /* more resting agent orders than max_agent_orders                       */
#define LOBSIM_ERR_BAD_VOLUME 16u       /* assert volume > 0, Exchange.py:59-60                                   */
#define LOBSIM_ERR_NO_SNAPSHOT 32u      /* "There is no data before the episode start time", OrderbookSimulator.py:92 */
#define LOBSIM_ERR_END_OF_STREAM 64u    /* stepped past the loaded message grid                                  */
#define LOBSIM_ERR_FILL_LOG_FULL 128u   /* fill log capacity exceeded (log truncated, simulation unaffected)     */
#define LOBSIM_ERR_AUM_NONPOSITIVE 256u  /* "AUM has gone non_positive", rl4mm/rewards/RewardFunctions.py:12-13      */
#define LOBSIM_ERR_BAD_ACTION 512u       /* non-finite Beta ladder (NaN action): np.round(nan).astype(int) is INT64_MIN in the
                                            reference and _volume_diff_to_orders (HOE.py:227-258) then raises -> episode dead */

/* ---- packed message record (16 B) -- device-resident replacement of the `messages` table ---------------------
 * rl4mm/database/models.py:10-22 + rl4mm/simulation/HistoricalOrderGenerator.py:77-90.
 * Hidden executions (LOBSTER type 5) are dropped by the packer (HistoricalOrderGenerator.py:49-57); executions
 * (type 4) carry the *aggressor* direction (database_population_helpers.py:132-136).                            */
#define LOBSIM_MSG_LIMIT 1u
#define LOBSIM_MSG_CANCEL 2u   /* partial cancellation ("modify") */
#define LOBSIM_MSG_DELETE 3u   /* deletion carrying the historical remaining size */
#define LOBSIM_MSG_MARKET 4u   /* visible execution => market order of the opposite side */

typedef struct {
  int32_t price;
  int32_t volume;
  uint32_t ref;  /* dense external order reference, 1..2^31-1 (0 = none)        */
  uint32_t meta; /* bits 0-2: LOBSIM_MSG_*, bit 3: direction (0 buy, 1 sell)     */
} lobsim_msg_t;

#define LOBSIM_META(type, dir) ((uint32_t)(type) | ((uint32_t)(dir) << 3))
#define LOBSIM_META_TYPE(m) ((m)&7u)
#define LOBSIM_META_DIR(m) (((m) >> 3) & 1u)

/* order references inside the book */
#define LOBSIM_REF_AGGREGATE 0u       /* snapshot aggregate, internal_id == -1 in the reference        */
#define LOBSIM_REF_AGENT 0x80000000u  /* | agent order id: the agent's own (is_external == False) order */

/* snapshot level entry with this price is absent (LOBSTER dummy level +-9999999999) */
#define LOBSIM_NO_PRICE INT32_MIN

/* ---- features: rl4mm/features/Features.py ------------------------------------------------------------------- */
#define LOBSIM_MAX_FEATURES 16
enum {
  LOBSIM_FEAT_SPREAD = 0,             /* Features.py:113 */
  LOBSIM_FEAT_BOOK_IMBALANCE = 1,     /* :132 */
  LOBSIM_FEAT_PRICE_MOVE = 2,         /* :151 */
  LOBSIM_FEAT_PRICE_RANGE = 3,        /* :178 */
  LOBSIM_FEAT_VOLATILITY = 4,         /* :203 */
  LOBSIM_FEAT_PRICE = 5,              /* :327 */
  LOBSIM_FEAT_TRADE_DIR_IMBALANCE = 6,/* :351 */
  LOBSIM_FEAT_TRADE_VOL_IMBALANCE = 7,/* :410 */
  LOBSIM_FEAT_INVENTORY = 8,          /* :474 */
  LOBSIM_FEAT_EPISODE_PROPORTION = 9, /* :493 */
  LOBSIM_FEAT_TIME_OF_DAY = 10,       /* :515 */
  LOBSIM_FEAT_AMIHUD_LAMBDA = 11      /* :245 (lookback = (true_lookback + 1) * slowing_factor, iparam = slowing_factor) */
};

typedef struct {
  int32_t kind;      /* LOBSIM_FEAT_*                                                        */
  int32_t lookback;  /* lookback_periods                                                     */
  int64_t update_us; /* update_frequency in microseconds (<= 60 s, Features.py:53)           */
  double min_value;  /* clamp, Features.py:83,99                                             */
  double max_value;
  int32_t iparam;    /* TIME_OF_DAY: n_buckets; TRADE_*_IMBALANCE: track_internal; AMIHUD: slowing_factor */
  int32_t norm_len;  /* normalisation_on ? max_norm_len : 0  (rolling z-score over the clamped values, Features.py:67-74) */
  double dparam;     /* EPISODE_PROPORTION: update_frequency / episode_length                */
} lobsim_feature_t;

/* ---- rewards: rl4mm/rewards/RewardFunctions.py -------------------------------------------------------------- */
enum {
  LOBSIM_REWARD_PNL = 0,            /* RewardFunctions.py:97-101  */
  LOBSIM_REWARD_INV_ADJ_PNL = 1,    /* RewardFunctions.py:107-118 */
  LOBSIM_REWARD_ROLLING_SHARPE = 2  /* RewardFunctions.py:38-94   */
};
#define LOBSIM_MAX_SHARPE_WINDOW 256
typedef struct {
  int32_t kind;
  int32_t asymmetric;        /* INV_ADJ_PNL: asymmetrically_dampened; ROLLING_SHARPE: max_window_size | min_window_size << 16 */
  double inventory_aversion; /* INV_ADJ_PNL */
} lobsim_reward_t;

/* ---- built-in agents for the fused rollout: rl4mm/agents/baseline_agents.py --------------------------------- */
enum {
  LOBSIM_AGENT_NONE = 0,       /* empty action list every step (warm-up, replay)       */
  LOBSIM_AGENT_FIXED = 1,      /* FixedActionAgent, baseline_agents.py:21-30            */
  LOBSIM_AGENT_TERADACTYL = 2, /* Teradactyl, baseline_agents.py:33-108                 */
  LOBSIM_AGENT_EXTERNAL = 3,   /* actions supplied by the caller (act tensor is input)  */
  LOBSIM_AGENT_RANDOM = 4      /* RandomAgent, baseline_agents.py:9-18: action_space.sample() = uniform in the action box
                                  [0, fixed_action[i]); here a counter-based stream, Philox4x32-10 keyed by
                                  (seed = `reserved`, env index, absolute grid step), so a rollout does not depend on how it
                                  is cut into launches and the CPU oracle draws the same numbers                       */
};
typedef struct {
  int32_t kind;
  int32_t inventory_index;  /* Teradactyl: index of the inventory feature in obs        */
  double fixed_action[5];   /* FIXED: the action; RANDOM: the upper bounds of the action box (lower bounds are 0, HOE.py:85-93) */
  double max_inventory;     /* Teradactyl (<= 0: None => denom 100)                     */
  double default_kappa, default_omega, max_kappa, exponent;
  int32_t market_clearing;
  int32_t reserved;         /* RANDOM: the seed                                          */
} lobsim_agent_t;

/* ---- environment configuration: kwargs of HistoricalOrderbookEnvironment.__init__ (HOE.py:54-81) and
 *      OrderbookSimulator.__init__ (OrderbookSimulator.py:24-53) ---------------------------------------------- */
typedef struct {
  int32_t abi_version;  /* LOBSIM_ABI_VERSION */
  int32_t n_envs;
  int32_t n_levels;     /* snapshot depth L                                            */
  int32_t tick_size;    /* Exchange.tick_size = 100                                    */
  int64_t step_us;      /* step_size                                                   */
  int32_t episode_steps;
  int32_t warmup_steps; /* int(max_feature_window_size / step_size), HOE.py:155        */
  int32_t min_quote_level, max_quote_level;
  int32_t outer_levels; /* OrderbookSimulator.outer_levels (resync)                    */
  int32_t resync;       /* 1: run update_outer_levels (reference behaviour)            */
  int32_t active_volume;           /* OrderDistributor.active_volume = 100             */
  int32_t market_order_clearing;
  int32_t enter_spread;
  int32_t inc_prev_action_in_obs;
  int32_t portfolio_carryover;     /* 1: State.portfolio aliases initial_portfolio, HOE.py:153 */
  int32_t n_features;
  double concentration;            /* < 0: None                                        */
  double market_order_fraction_of_inventory;
  double initial_cash;
  int64_t initial_inventory;
  lobsim_feature_t features[LOBSIM_MAX_FEATURES];
  lobsim_reward_t step_reward;     /* per_step_reward_function                         */
  lobsim_reward_t terminal_reward; /* terminal_reward_function                         */
  /* capacities of the fixed-size device book (the reference's containers are unbounded) */
  int32_t max_levels_per_side;
  int32_t max_orders_per_side;
  int32_t max_agent_orders;        /* per side                                         */
  int32_t fill_log_capacity;       /* fill records kept per env per call (0 = no log)  */
} lobsim_cfg_t;

/* ---- a message stream (one ticker-day) resident in HBM ------------------------------------------------------
 * step_off has n_grid_steps + 1 entries: the messages of grid step k (timestamps in
 * (t0_us + k*step_us, t0_us + (k+1)*step_us]) are msgs[step_off[k] .. step_off[k+1]).
 * snapshots: [n_seconds + 1][2 sides][n_levels][2] int32 = (price, volume) of the book after the last message with
 * timestamp <= t0 + s seconds (rl4mm/database/HistoricalDatabase.py:46-62 with book_snapshot_freq = "S"), level 0 =
 * best; snap_valid[s] = 0 when no message precedes that second.                                                  */
typedef struct {
  const lobsim_msg_t* msgs;
  uint64_t n_msgs;
  const uint32_t* step_off;
  uint32_t n_grid_steps;
  const int32_t* snapshots;
  const uint8_t* snap_valid;
  uint32_t n_seconds;
  uint32_t reserved;
  int64_t t0_us; /* grid origin, microseconds after midnight, whole second */
} lobsim_stream_t;

/* ---- order record for the Exchange-level entry point -------------------------------------------------------- */
typedef struct {
  int32_t env;
  int32_t type;       /* LOBSIM_MSG_* */
  int32_t direction;
  int32_t price;      /* ignored for market orders                                           */
  int32_t volume;     /* <= 0 with type DELETE: volume None (full delete), Exchange.py:140   */
  int32_t is_external;
  uint32_t ref;       /* external: external_id (dense); agent: internal id returned earlier  */
  uint32_t reserved;
} lobsim_order_t;

/* one fill record: an element of FilledOrders.internal / .external (rl4mm/orderbook/models.py:58-61) */
typedef struct {
  int32_t list;       /* 0 = FilledOrders.internal, 1 = FilledOrders.external                */
  int32_t direction;  /* direction of the recorded order (resting side, or agent aggressor)  */
  int32_t price;
  int32_t volume;
  int32_t is_market;  /* 1: the synthetic MarketOrder fill of Exchange.py:111-115            */
  uint32_t ref;       /* ref of the resting order that was hit                               */
} lobsim_fill_t;

/* L3 dump entry */
typedef struct {
  int32_t price;
  int32_t volume;
  uint32_t ref;
  int32_t level; /* 0 = best */
} lobsim_book_entry_t;

/* per-env scalar state, for parity checks and episode statistics */
typedef struct {
  int64_t inventory;
  double cash;
  double price;        /* microprice after the last step                                    */
  int32_t now_step;    /* grid step index: now_is = t0 + now_step * step_us                  */
  int32_t episode_start_step;
  int32_t min_buy_price, max_sell_price; /* OrderbookSimulator.min_buy_price / max_sell_price */
  int32_t best_buy, best_sell;           /* 0 / INT32_MAX when the side is empty               */
  int32_t best_buy_volume, best_sell_volume;
  uint32_t err;
  int32_t stream_id;
  uint32_t n_agent_orders[2];
  uint32_t next_agent_id;
  uint32_t reserved;   /* book form: bit 0 = the blob is in the flat order-pool form (csrc/book_flat.cuh) between launches;
                          bits 8-19 / 20-31 = resting orders on the buy / sell side (clamped to 4095)              */
} lobsim_env_state_t;

typedef struct lobsim lobsim_t;

const char* lobsim_last_error(void);
int lobsim_abi_version(void);

/* size in bytes of one env's book blob for a configuration (HBM footprint = n_envs * this + feature windows) */
int64_t lobsim_state_bytes(const lobsim_cfg_t* cfg);

/* HistoricalOrderbookEnvironment.__init__ + OrderbookSimulator.__init__ + Exchange.__init__ for n_envs envs */
int lobsim_create(const lobsim_cfg_t* cfg, int device, lobsim_t** out);
int lobsim_destroy(lobsim_t* h);

/* replaces rl4mm/database (HistoricalDatabase.get_messages :103-119, get_last_snapshot :46-62) and
 * HistoricalOrderGenerator.preload_episode_orders (HistoricalOrderGenerator.py:59-63): registers a device-resident
 * stream.  The arrays are NOT copied; they must stay alive while in use.                                        */
int lobsim_load_stream(lobsim_t* h, int stream_id, const lobsim_stream_t* stream_dev);

/* HistoricalOrderbookEnvironment.reset (HOE.py:147-161) = OrderbookSimulator.reset_episode
 * (OrderbookSimulator.py:55-68) at now = (episode_start_steps[i] - warmup_steps), feature reset and the warm-up
 * loop.  env_ids_dev == NULL: all envs, with stream_ids/start_steps of length n_envs.  obs_out_dev may be NULL.
 * obs_out_dev: [n, obs_dim] f64.                                                                                */
int lobsim_reset(lobsim_t* h, const int32_t* env_ids_dev, int32_t n, const int32_t* stream_ids_dev,
                 const int32_t* episode_start_steps_dev, double* obs_out_dev, void* stream);

/* HistoricalOrderbookEnvironment.step (HOE.py:163-178) for every env: actions [n_envs, action_dim] f64 ->
 * obs [n_envs, obs_dim] f64, reward [n_envs] f64, done [n_envs] u8.                                             */
int lobsim_step(lobsim_t* h, const double* actions_dev, double* obs_out_dev, double* reward_out_dev,
                uint8_t* done_out_dev, void* stream);
/* same call with HOST buffers: H2D of the actions, the step, D2H of obs / reward / done                         */
int lobsim_step_host(lobsim_t* h, const double* actions_host, double* obs_out_host, double* reward_out_host,
                     uint8_t* done_out_host);

/* generate_trajectory (rl4mm/gym/utils.py:100-117) fused over T steps with a built-in agent: obs [T, n_envs,
 * obs_dim], act [T, n_envs, action_dim], rew [T, n_envs], done [T, n_envs]; any output may be NULL.  Envs that
 * finish keep stepping (the caller resets them), as a vectorised env without auto-reset would.                 */
int lobsim_rollout(lobsim_t* h, int32_t T, const lobsim_agent_t* agent, double* obs_dev, double* act_dev,
                   double* rew_dev, uint8_t* done_dev, void* stream);

/* lobsim_rollout plus the per-step info series the reference's evaluation path is built from
 * (SimpleInfoCalculator.calculate, rl4mm/gym/order_tracking/InfoCalculators.py:31-59, collected by generate_trajectory,
 * rl4mm/gym/utils.py:100-117, and reduced by append_to_episode_summary_dict :146-190): info [T, n_envs,
 * LOBSIM_INFO_DIM] f64, the state at the END of each env step (after fills, portfolio and price update).
 * The action-derived entries of the info dict (agent spreads / midprice offsets) are functions of `act` alone.     */
#define LOBSIM_INFO_ASSET_PRICE 0   /* microprice of the central book (State.price, HOE.py:203)                 */
#define LOBSIM_INFO_INVENTORY 1
#define LOBSIM_INFO_CASH 2
#define LOBSIM_INFO_AUM 3           /* cash + asset_price * inventory                                           */
#define LOBSIM_INFO_MARKET_SPREAD 4 /* best_sell - best_buy of the central book (NaN when a side is empty)      */
#define LOBSIM_INFO_BEST_BUY 5
#define LOBSIM_INFO_BEST_SELL 6
#define LOBSIM_INFO_ERR 7           /* the env's sticky error bits so far, as a double                          */
#define LOBSIM_INFO_DIM 8
int lobsim_rollout_info(lobsim_t* h, int32_t T, const lobsim_agent_t* agent, double* obs_dev, double* act_dev,
                        double* rew_dev, uint8_t* done_dev, double* info_dev, void* stream);

/* lobsim_rollout_info with ONE BUILT-IN AGENT PER ENV: agents_host [n_envs] (FIXED or TERADACTYL, copied to the device
 * by the call).  This is the batched form of the reference's rule-based-agent tuning (tune_rule_based_agents.py:24-72 runs
 * one Ray trial per Teradactyl parameter set, each trial stepping its own env): K parameter sets x M episodes are one
 * launch.  act_dev is an output.                                                                                  */
int lobsim_rollout_agents(lobsim_t* h, int32_t T, const lobsim_agent_t* agents_host, double* obs_dev, double* act_dev,
                          double* rew_dev, uint8_t* done_dev, double* info_dev, void* stream);

/* OrderbookSimulator.forward_step (OrderbookSimulator.py:70-88) with internal_orders=None, n_steps times, for
 * every env: pure replay of the stream through the book (no features / rewards).                               */
int lobsim_replay(lobsim_t* h, int32_t n_steps, void* stream);
/* replay with HOST buffers: uploads the stream segment needed by the next n_steps into a staging area of the
 * handle (H2D), replays, and downloads one lobsim_env_state_t per env (D2H).                                    */
int lobsim_replay_host(lobsim_t* h, int stream_id, const lobsim_msg_t* msgs_host, uint64_t first_msg,
                       uint64_t n_msgs, int32_t n_steps, lobsim_env_state_t* state_out_host);

/* exactly ONE OrderbookSimulator.forward_step(until = now + n_steps * step_size) for every env: like lobsim_replay
 * but the outer-level resync (OrderbookSimulator.py:86-87) is evaluated once, at `until`, as the reference does when
 * it is stepped over more than one grid interval at a time.                                                     */
int lobsim_forward_step(lobsim_t* h, int32_t n_steps, void* stream);

/* OrderbookSimulator.reset_episode only (no features, no warm-up): book := snapshot at grid step `start_step`   */
int lobsim_reset_book(lobsim_t* h, const int32_t* env_ids_dev, int32_t n, const int32_t* stream_ids_dev,
                      const int32_t* start_steps_dev, void* stream);

/* Exchange.process_order (rl4mm/orderbook/Exchange.py:58-69) for a host list of orders, applied in order.  Like the reference's
 * exchange it only moves the books: the env's portfolio (inventory, cash) changes in its steps, not here.
 * fills_out_host (capacity max_fills) receives FilledOrders in emission order; refs_out_host[i] is, for a limit order
 * (or its unfilled remainder) that RESTED in the book -- i.e. whenever the reference's OrderIdConvertor hands out a
 * new internal id (OrderIDConvertor.py:12-18) --, the agent order id (agent orders) or 0xffffffff (external orders),
 * and 0 otherwise.                                                                                                */
int lobsim_process_orders(lobsim_t* h, const lobsim_order_t* orders_host, int32_t n, lobsim_fill_t* fills_out_host,
                          int32_t max_fills, int32_t* n_fills_out, uint32_t* refs_out_host);

/* Exchange(central_orderbook=..., internal_orderbook=...) (Exchange.py:40-49) / `exchange.central_orderbook = book`:
 * replaces env's books by the given L3 entries (per side: best level first, FIFO order inside a level, exactly the
 * lobsim_dump_book format; ref = LOBSIM_REF_AGENT | id marks the agent's own orders, which also form the internal
 * book).  The simulator clock and portfolio are left untouched.                                                 */
int lobsim_set_book(lobsim_t* h, int32_t env, const lobsim_book_entry_t* buy_host, int32_t n_buy,
                    const lobsim_book_entry_t* sell_host, int32_t n_sell);

/* L3 dump of one env's central book side, best level first, FIFO order within a level
 * (rl4mm/extras/orderbook_comparison.py:6-19 is the L2 projection of this).  Returns the number of entries.     */
int lobsim_dump_book(lobsim_t* h, int32_t env, int32_t side, lobsim_book_entry_t* out_host, int32_t capacity);
/* the agent's internal book side (Exchange.internal_orderbook), ascending internal id */
int lobsim_dump_agent_orders(lobsim_t* h, int32_t env, int32_t side, lobsim_book_entry_t* out_host, int32_t capacity);

int lobsim_get_state(lobsim_t* h, int32_t first_env, int32_t n, lobsim_env_state_t* out_host);
int lobsim_get_state_dev(lobsim_t* h, lobsim_env_state_t* out_dev, void* stream);
/* fills recorded by the last step / rollout / replay / process_orders call of env `env` */
int lobsim_get_fills(lobsim_t* h, int32_t env, lobsim_fill_t* out_host, int32_t capacity, int32_t* n_out);
int lobsim_errors(lobsim_t* h, uint32_t* err_out_host);
int lobsim_obs_dim(const lobsim_cfg_t* cfg);
int lobsim_action_dim(const lobsim_cfg_t* cfg);

/* number of kernel launches issued by this handle so far (bench.py reports it as gpu_launches) */
int64_t lobsim_launch_count(lobsim_t* h);

/* which kernel family serves this handle: the straight-line static-layout kernels exist for the capacity triples
 * {max_levels_per_side, max_orders_per_side, max_agent_orders} listed in rl4mm_b200/csrc/layouts.h; every other triple
 * (and LOBSIM_FORCE_GENERAL=1) runs on the general runtime-layout kernel -- identical results, about 2-3x the
 * instructions per order.  lobsim_create prints one warning per process when it has to select the general kernel.   */
#define LOBSIM_PATH_GENERAL 0
#define LOBSIM_PATH_FAST 1
#define LOBSIM_PATH_DEEP 2   /* capacities whose book exceeds the shared memory of an SM: the general kernel works on the blob in place in HBM */
int lobsim_kernel_path(lobsim_t* h);

/* sha256 (hex) of the sources (rl4mm_b200/csrc/ and include/) this library was built from; rl4mm_b200/_lib.py compares
 * it with the sources next to it, so a stale binary cannot be loaded silently.                                     */
const char* lobsim_source_hash(void);

#ifdef __cplusplus
}
#endif
#endif /* LOBSIM_H */
