// fast_layout.cu -- ONE compiled StaticLayout of the straight-line kernels (kernels.cuh): the three instantiations of
// replay_straight (k_replay_flat / k_replay_fast / k_replay_hyb), k_to_sorted and k_env_fast.
// Compiled once per entry of layouts.h and per part (-DLOBSIM_LAYOUT_INDEX=i -DLOBSIM_TU_PART=p, build.py), in parallel:
//   part 0: the replay kernels (k_replay_hyb only for the deep layouts of hyb_layout()) + the env kernels without the z-score /
//           RollingSharpe code
//   part 1: the env kernels with that code (RARE)
// lobsim.cu calls the launchers below through the FastLayoutOps table.
#include "kernels.cuh"
#include "layouts.h"

#if !defined(LOBSIM_LAYOUT_INDEX) || !defined(LOBSIM_TU_PART)
#error "compile with -DLOBSIM_LAYOUT_INDEX=<entry of layouts.h> -DLOBSIM_TU_PART=<0|1>"
#endif

template <int I> struct LayoutAt;
#define X(i, nl, no, na) template <> struct LayoutAt<i> { typedef StaticLayout<nl, no, na> type; };
LOBSIM_FAST_LAYOUTS(X)
#undef X
typedef LayoutAt<LOBSIM_LAYOUT_INDEX>::type LT;

#define LOBSIM_CAT3_(a, b, c) a##b##c
#define LOBSIM_CAT3(a, b, c) LOBSIM_CAT3_(a, b, c)
#define FN(name) LOBSIM_CAT3(lobsim_fast, LOBSIM_LAYOUT_INDEX, name)

static cudaError_t set_attr(const void* k, int dyn) {
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}

template <bool RARE>
static cudaError_t env_attrs(int dyn_env) {
  cudaError_t e = set_attr((const void*)k_env_fast<LT, true, RARE>, dyn_env);
  if (e == cudaSuccess) e = set_attr((const void*)k_env_fast<LT, false, RARE>, dyn_env);
  return e;
}
template <bool RARE>
static void env_launch(bool sync, int grid, int block, size_t dyn, cudaStream_t stream, const AdvParams& p, const EnvConst& ec) {
  if (sync) k_env_fast<LT, true, RARE><<<grid, block, dyn, stream>>>(p, ec);
  else k_env_fast<LT, false, RARE><<<grid, block, dyn, stream>>>(p, ec);
}

#if LOBSIM_TU_PART == 0
cudaError_t FN(_attrs)(int dyn_replay, int dyn_env) {
  cudaError_t e = set_attr((const void*)k_replay_fast<LT>, dyn_replay);
  if (e == cudaSuccess) e = set_attr((const void*)k_replay_flat<LT>, dyn_replay);
  if constexpr (hyb_layout<LT>()) { if (e == cudaSuccess) e = set_attr((const void*)k_replay_hyb<LT>, dyn_replay); }
  if (e == cudaSuccess) e = cudaFuncSetAttribute((const void*)k_to_sorted<LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * LT::blob_bytes <= 227 * 1024 ? 4 * LT::blob_bytes : LT::blob_bytes);
  if (e == cudaSuccess) e = env_attrs<false>(dyn_env);
  return e;
}
void FN(_replay)(ReplayKind kind, int grid, int block, size_t dyn, cudaStream_t stream, const AdvParams& p, const EnvConst& ec) {
  if constexpr (hyb_layout<LT>()) {
    if (kind == REPLAY_HYBRID) { k_replay_hyb<LT><<<grid, block, dyn, stream>>>(p, ec); return; }
  }
  if (kind == REPLAY_SORTED) k_replay_fast<LT><<<grid, block, dyn, stream>>>(p, ec);
  else k_replay_flat<LT><<<grid, block, dyn, stream>>>(p, ec);
}
void FN(_to_sorted)(unsigned char* blobs, int n_envs, cudaStream_t stream) {
  const int wpc = 4 * LT::blob_bytes <= 227 * 1024 ? 4 : 1;
  k_to_sorted<LT><<<(n_envs + wpc - 1) / wpc, wpc * 32, (size_t)wpc * LT::blob_bytes, stream>>>(blobs, n_envs);
}
void FN(_env)(bool sync, int grid, int block, size_t dyn, cudaStream_t stream, const AdvParams& p, const EnvConst& ec) {
  env_launch<false>(sync, grid, block, dyn, stream, p, ec);
}
#else
cudaError_t FN(_attrs_rare)(int dyn_env) { return env_attrs<true>(dyn_env); }
void FN(_env_rare)(bool sync, int grid, int block, size_t dyn, cudaStream_t stream, const AdvParams& p, const EnvConst& ec) {
  env_launch<true>(sync, grid, block, dyn, stream, p, ec);
}
#endif
