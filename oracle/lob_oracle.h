/* lob_oracle.h -- TEST INFRASTRUCTURE: API of the single-environment CPU oracle (see lob_oracle.c). */
#ifndef LOB_ORACLE_H
#define LOB_ORACLE_H
#include "../include/lobsim.h"
#ifdef __cplusplus
extern "C" {
#endif
typedef struct lo lo_t;
lo_t* lo_create(const lobsim_cfg_t* cfg);
void lo_destroy(lo_t* o);
void lo_set_stream(lo_t* o, const lobsim_stream_t* host_stream);
int lo_reset_book(lo_t* o, int start_step);
int lo_reset(lo_t* o, int episode_start_step, double* obs_out);
int lo_step(lo_t* o, const double* action, double* obs, double* reward, uint8_t* done);
int lo_replay(lo_t* o, int n_steps);
int lo_forward_step(lo_t* o, int n_steps);
int lo_set_book(lo_t* o, const lobsim_book_entry_t* buy, int n_buy, const lobsim_book_entry_t* sell, int n_sell);
/* capacity high-water marks since the last lo_reset_book / lo_reset / lo_set_book: out[0..1] price levels per side, [2..3] resting
 * orders per side (snapshot aggregates included), [4..5] agent orders per side, [6] the most fills recorded in one call */
void lo_peaks(const lo_t* o, int32_t* out);
int lo_rollout(lo_t* o, int T, const lobsim_agent_t* agent, double* obs, double* act, double* rew, uint8_t* done);
int lo_rollout_info(lo_t* o, int T, const lobsim_agent_t* agent, double* obs, double* act, double* rew, uint8_t* done, double* info);
void lo_agent_action(const lobsim_agent_t* agent, const double* obs, double* action);
void lo_philox4x32_10(uint32_t ctr[4], uint32_t key0, uint32_t key1);
void lo_random_action(const lobsim_agent_t* agent, int32_t env_index, int64_t now_step, double* action);
void lo_set_env_index(lo_t* o, int32_t env_index);
void lo_action_to_ladders(const lo_t* o, const double* action, int64_t* buy, int64_t* sell);
int lo_process_order(lo_t* o, const lobsim_order_t* order, uint32_t* ref_out);
void lo_clear_fills(lo_t* o);
int lo_get_fills(const lo_t* o, lobsim_fill_t* out, int cap);
int lo_dump_book(const lo_t* o, int side, lobsim_book_entry_t* out, int cap);
int lo_dump_agent_orders(const lo_t* o, int side, lobsim_book_entry_t* out, int cap);
void lo_get_state(const lo_t* o, lobsim_env_state_t* st);
int lo_obs_dim(const lobsim_cfg_t* cfg);
int lo_action_dim(const lobsim_cfg_t* cfg);
#ifdef __cplusplus
}
#endif
#endif
