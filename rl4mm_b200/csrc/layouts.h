// layouts.h -- the book capacities {levels, orders, agent orders per side} that have compiled straight-line kernels
// (k_replay_flat / k_replay_fast / k_replay_hyb / k_env_fast, kernels.cuh).  Any other capacity triple runs on the general runtime-layout kernel
// k_advance (same results, about 2-3x the instructions per order); lobsim_kernel_path() tells which one a handle got.
//
// Each entry is compiled as its own translation units (fast_layout.cu with -DLOBSIM_LAYOUT_INDEX=i, see build.py), in
// parallel; lobsim.cu only sees the launcher functions declared by LOBSIM_DECLARE_FAST_LAYOUT.
#pragma once

#define LOBSIM_FAST_LAYOUTS(X)                                                                       \
  X(0, 64, 256, 32)    /* BASELINE config 2: 10-level books, replay                               */ \
  X(1, 128, 512, 64)   /* the default capacities of lobsim_cfg_t (50-level books)                 */ \
  X(2, 64, 256, 64)    /* 10-level books with a 64-order agent table (configs 3 and 4)            */ \
  X(3, 128, 1536, 64)  /* BASELINE config 5: 50-level books, deep queues, heavy cancel flow (its      \
                          FixedActionAgent holds up to ~45 resting orders per side: 32 overflows) */ \
  X(4, 128, 1024, 64)  /* 50-level books with deep queues and a 64-order agent table              */ \
  X(5, 128, 256, 64)   /* 10-level books + the agent's ladders (configs 3 and 4): 128 levels so that   \
                          the flat form may hold 128 orders per side (book_flat.cuh)               */

#define LOBSIM_N_FAST_LAYOUTS 6
