// mpc_kernels_tu.cu — one instantiation of K_solve / K_rollout (+ K_step) per translation unit (nvcc -DMPC_TU=n; see mpc_kernels.cuh).
#include "mpc_kernels.cuh"
#ifndef MPC_REG_MAXT
#define MPC_REG_MAXT 256       // register form: threads per CTA the kernel is compiled for (256: 255 registers, 4 problems; 320 / 384: 168 registers)
#endif
#ifndef MPC_REG_STATE
#define MPC_REG_STATE 1      // register form: 1 = stage state in registers inside a block, 0 = state stays in the records
#endif

#define SOLVE_TU(n, ...)                                                                                                     \
  cudaError_t solve_set_smem_##n(int bytes) { return cudaFuncSetAttribute(mpc_solve_kernel<__VA_ARGS__>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); } \
  void solve_launch_##n(int grid, int threads, int smem, cudaStream_t st, const Params& p, const Settings& s, const BatchArgs& a, int P, int F) { \
    mpc_solve_kernel<__VA_ARGS__><<<grid, threads, smem, st>>>(p, s, a, P, F);                                                \
  }
#define SOLVE_REG_TU(n, MAXT, STATE, WPP)                                                                                         \
  cudaError_t solve_set_smem_##n(int bytes) { return cudaFuncSetAttribute(mpc_solve_reg_kernel<MAXT, STATE, WPP>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); } \
  void solve_launch_##n(int grid, int threads, int smem, cudaStream_t st, const Params& p, const Settings& s, const BatchArgs& a, int P, int F) { \
    mpc_solve_reg_kernel<MAXT, STATE, WPP><<<grid, threads, smem, st>>>(p, s, a, P, F);                                            \
  }                                                                                                                          \
  int solve_reg_max_threads_##n() { return MAXT; }
#define ROLLOUT_TU(name, FORM)                                                                                               \
  cudaError_t rollout_set_smem_##name(int bytes) { return cudaFuncSetAttribute(mpc_rollout_kernel<FORM>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); } \
  cudaError_t rollout_occupancy_##name(int bytes, int* n) { return cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, mpc_rollout_kernel<FORM>, 32, bytes); } \
  void rollout_launch_##name(int grid, int smem, cudaStream_t st, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg, const RolloutArgs& a) { \
    mpc_rollout_kernel<FORM><<<grid, 32, smem, st>>>(p, s, cfg, a);                                                          \
  }                                                                                                                          \
  cudaError_t step_set_smem_##name(int bytes) { return cudaFuncSetAttribute(mpc_track_step_kernel<FORM>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); } \
  void step_launch_##name(int grid, int smem, cudaStream_t st, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg, const StepArgs& a) { \
    mpc_track_step_kernel<FORM><<<grid, 32, smem, st>>>(p, s, cfg, a);                                                       \
  }

#if MPC_TU == 0
SOLVE_TU(0, 256, 1, FORM_SHORT)
#elif MPC_TU == 1
SOLVE_TU(1, 256, 1, FORM_GENERAL)
#elif MPC_TU == 2
SOLVE_TU(2, 128, 2, FORM_GENERAL)
#elif MPC_TU == 3
ROLLOUT_TU(short, FORM_SHORT)
#elif MPC_TU == 4
ROLLOUT_TU(general, FORM_GENERAL)
#elif MPC_TU == 5
SOLVE_TU(3, 256, 1, FORM_PAIR)
#elif MPC_TU == 6
ROLLOUT_TU(pair, FORM_PAIR)
#elif MPC_TU == 7
SOLVE_REG_TU(4, MPC_REG_MAXT, MPC_REG_STATE, 2)
#elif MPC_TU == 8
SOLVE_REG_TU(5, 256, MPC_REG_STATE, 1)
#else
#error "MPC_TU must be 0..8"
#endif
