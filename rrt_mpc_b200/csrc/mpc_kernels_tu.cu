// mpc_kernels_tu.cu — one instantiation of K_solve / K_rollout (+ K_step) per translation unit (nvcc -DMPC_TU=n; see mpc_kernels.cuh).
#include "mpc_kernels.cuh"
#ifndef MPC_REG_MAXT
#define MPC_REG_MAXT 256       // register form: threads per CTA the kernel is compiled for (256: 255 registers, 4 problems; 320 / 384: 168 registers)
#endif
#ifndef MPC_REG_STATE
#define MPC_REG_STATE 1      // register form: 1 = stage state in registers inside a block, 0 = state stays in the records
#endif

// name: suffix of the launchers (cudampc.cu); PP: per-problem parameters (mpc_kernels.cuh)
#define SOLVE_TU(name, PP, ...)                                                                                              \
  cudaError_t solve_set_smem_##name(int bytes) { return cudaFuncSetAttribute(mpc_solve_kernel<__VA_ARGS__, PP>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); } \
  void solve_launch_##name(int grid, int threads, int smem, cudaStream_t st, const Params& p, const Settings& s, const BatchArgs& a, int P, int F) { \
    mpc_solve_kernel<__VA_ARGS__, PP><<<grid, threads, smem, st>>>(p, s, a, P, F);                                            \
  }
#define SOLVE_REG_TU(name, PP, MAXT, STATE, WPP)                                                                              \
  cudaError_t solve_set_smem_##name(int bytes) { return cudaFuncSetAttribute(mpc_solve_reg_kernel<MAXT, STATE, WPP, PP>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); } \
  void solve_launch_##name(int grid, int threads, int smem, cudaStream_t st, const Params& p, const Settings& s, const BatchArgs& a, int P, int F) { \
    mpc_solve_reg_kernel<MAXT, STATE, WPP, PP><<<grid, threads, smem, st>>>(p, s, a, P, F);                                        \
  }                                                                                                                          \
  int solve_reg_max_threads_##name() { return MAXT; }
#define ROLLOUT_TU(name, PP, FORM)                                                                                           \
  cudaError_t rollout_set_smem_##name(int bytes) { return cudaFuncSetAttribute(mpc_rollout_kernel<FORM, PP>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); } \
  cudaError_t rollout_occupancy_##name(int bytes, int* n) { return cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, mpc_rollout_kernel<FORM, PP>, 32, bytes); } \
  void rollout_launch_##name(int grid, int smem, cudaStream_t st, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg, const RolloutArgs& a) { \
    mpc_rollout_kernel<FORM, PP><<<grid, 32, smem, st>>>(p, s, cfg, a);                                                      \
  }                                                                                                                          \
  cudaError_t step_set_smem_##name(int bytes) { return cudaFuncSetAttribute(mpc_track_step_kernel<FORM, PP>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); } \
  void step_launch_##name(int grid, int smem, cudaStream_t st, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg, const StepArgs& a) { \
    mpc_track_step_kernel<FORM, PP><<<grid, 32, smem, st>>>(p, s, cfg, a);                                                   \
  }

// 0..8: shared parameters (the launch's Params); 9..17: the same variants with per-problem parameters
#if MPC_TU == 0
SOLVE_TU(0, false, 256, 1, FORM_SHORT)
#elif MPC_TU == 1
SOLVE_TU(1, false, 256, 1, FORM_GENERAL)
#elif MPC_TU == 2
SOLVE_TU(2, false, 128, 2, FORM_GENERAL)
#elif MPC_TU == 3
ROLLOUT_TU(short, false, FORM_SHORT)
#elif MPC_TU == 4
ROLLOUT_TU(general, false, FORM_GENERAL)
#elif MPC_TU == 5
SOLVE_TU(3, false, 256, 1, FORM_PAIR)
#elif MPC_TU == 6
ROLLOUT_TU(pair, false, FORM_PAIR)
#elif MPC_TU == 7
SOLVE_REG_TU(4, false, MPC_REG_MAXT, MPC_REG_STATE, 2)
#elif MPC_TU == 8
SOLVE_REG_TU(5, false, 256, MPC_REG_STATE, 1)
#elif MPC_TU == 9
SOLVE_TU(pp0, true, 256, 1, FORM_SHORT)
#elif MPC_TU == 10
SOLVE_TU(pp1, true, 256, 1, FORM_GENERAL)
#elif MPC_TU == 11
SOLVE_TU(pp2, true, 128, 2, FORM_GENERAL)
#elif MPC_TU == 12
ROLLOUT_TU(pp_short, true, FORM_SHORT)
#elif MPC_TU == 13
ROLLOUT_TU(pp_general, true, FORM_GENERAL)
#elif MPC_TU == 14
SOLVE_TU(pp3, true, 256, 1, FORM_PAIR)
#elif MPC_TU == 15
ROLLOUT_TU(pp_pair, true, FORM_PAIR)
#elif MPC_TU == 16
SOLVE_REG_TU(pp4, true, MPC_REG_MAXT, MPC_REG_STATE, 2)
#elif MPC_TU == 17
SOLVE_REG_TU(pp5, true, 256, MPC_REG_STATE, 1)
#else
#error "MPC_TU must be 0..17"
#endif
