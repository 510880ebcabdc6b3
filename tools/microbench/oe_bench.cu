// Microbenchmark of the odd-even block solve (mpc_oe.h) in isolation: cycles of the forward sweep, the stage-parallel
// diagonal step, the backward sweep and the factorisation, for W independent one-warp problems per SM.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o oe_bench oe_bench.cu && ./oe_bench [N]
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include "../../rrt_mpc_b200/csrc/mpc_exec.cuh"
using namespace mpc;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); exit(1);} } while (0)

__device__ void fill(const View& w, const OEView& oe, int lane) {
  const int N = w.N;
  for (int j = lane; j < oe.J; j += 32) {
    double* s = oe.sinv + OE_SYM * j;
    for (int r = 0; r < 6; ++r) for (int c = 0; c <= r; ++c) s[MPC_SP(r, c)] = r == c ? 4.0 + (j % 3) : 0.05 * ((r + c + j) % 5);
    s[21] = 0.0;
  }
  for (int o = lane; o < oe_nodd(N); o += 32) {
    double* s = oe.dinv + OE_SYM * o;
    for (int r = 0; r < 6; ++r) for (int c = 0; c <= r; ++c) s[MPC_SP(r, c)] = r == c ? 0.3 : 0.01 * ((r + c + o) % 5);
    s[21] = 0.0;
  }
  for (int i = lane; i < oe.J - 1; i += 32) {
    double* g = (i < oe.jm ? oe.gt + OE_G * i : oe.gb + OE_G * (i - oe.jm));
    for (int t = 0; t < OE_G; ++t) g[t] = 0.02 * ((t + i) % 7) - 0.05;
  }
  for (int k = lane; k <= N + 1; k += 32) { double* x = w.nx(k); for (int t = 0; t < 6; ++t) x[t] = k <= N ? 1.0 + 0.01 * ((k + t) % 9) : 0.0; }
}
// ---- variants of the forward sweep (timing experiments) ----
// V1: 6 lanes per half, the new vector is exchanged with shuffles (the store for the diagonal step is off the critical path)
__device__ __forceinline__ void fwd_shfl6(int lane, const View& w, const OEView& oe) {
  const bool act = lane < 12; const bool bottom = (lane / 6) & 1; const int r = lane % 6; const int base = bottom ? 6 : 0;
  const OEHalf h = oe_half(w, oe, bottom);
  const int cnt = h.cnt, cmax = oe.jm > oe.nb ? oe.jm : oe.nb;
  const int xs = h.xstep * 8;
  const unsigned xlast = smem_u32(h.xlast) + 8 * r;
  unsigned xrow = smem_u32(h.x0) + xs, gp = smem_u32(h.g0) + 48 * r;
  double a[6], gA[6], gB[6], nbA, nbB, y;
  lds_row(smem_u32(h.x0), a);
  double ymid = lds_f64(xlast);
  lds_row(gp, gA); nbA = lds_f64(cnt == 1 ? xlast : xrow + 8 * r);
  for (int i = 1; i <= cmax; i += 2) {
    lds_row(gp + 288, gB); nbB = lds_f64(i + 1 == cnt ? xlast : xrow + xs + 8 * r);
    y = oe_row_dot(gA, nbA, a);
    ymid = (i == cnt) ? y : ymid;
    sts_f64_if(act && i < cnt, xrow + 8 * r, y);
#pragma unroll
    for (int c = 0; c < 6; ++c) a[c] = __shfl_sync(0xffffffffu, y, base + c);
    if (i + 1 > cmax) break;
    lds_row(gp + 576, gA); nbA = lds_f64(i + 2 == cnt ? xlast : xrow + 2 * xs + 8 * r);
    y = oe_row_dot(gB, nbB, a);
    ymid = (i + 1 == cnt) ? y : ymid;
    sts_f64_if(act && i + 1 < cnt, xrow + xs + 8 * r, y);
#pragma unroll
    for (int c = 0; c < 6; ++c) a[c] = __shfl_sync(0xffffffffu, y, base + c);
    gp += 576; xrow += 2 * xs;
  }
  const double yo = __shfl_sync(0xffffffffu, ymid, bottom ? lane - 6 : (lane + 6) & 31);
  double* mrow = w.nx(2 * oe.jm);
  if (lane < 6) mrow[r] = ymid + yo;
  __syncwarp();
}
// V3: as V1 but inside the 12-lane divergent region of the shipped sweeps (shuffles over the 12-lane mask, no barrier at all)
__device__ __forceinline__ void fwd_shfl6_region(int lane, const View& w, const OEView& oe) {
  if (lane < 12) {
    const bool bottom = lane >= 6; const int r = bottom ? lane - 6 : lane; const int base = bottom ? 6 : 0;
    const OEHalf h = oe_half(w, oe, bottom);
    const int cnt = h.cnt, cmax = oe.jm > oe.nb ? oe.jm : oe.nb;
    const int xs = h.xstep * 8;
    const unsigned xlast = smem_u32(h.xlast) + 8 * r;
    unsigned xrow = smem_u32(h.x0) + xs, gp = smem_u32(h.g0) + 48 * r;
    double a[6], gA[6], gB[6], nbA, nbB, y;
    lds_row(smem_u32(h.x0), a);
    double ymid = lds_f64(xlast);
    lds_row(gp, gA); nbA = lds_f64(cnt == 1 ? xlast : xrow + 8 * r);
    for (int i = 1; i <= cmax; i += 2) {
      lds_row(gp + 288, gB); nbB = lds_f64(i + 1 == cnt ? xlast : xrow + xs + 8 * r);
      y = oe_row_dot(gA, nbA, a);
      ymid = (i == cnt) ? y : ymid;
      sts_f64_if(i < cnt, xrow + 8 * r, y);
#pragma unroll
      for (int c = 0; c < 6; ++c) a[c] = __shfl_sync(0xfffu, y, base + c);
      if (i + 1 > cmax) break;
      lds_row(gp + 576, gA); nbA = lds_f64(i + 2 == cnt ? xlast : xrow + 2 * xs + 8 * r);
      y = oe_row_dot(gB, nbB, a);
      ymid = (i + 1 == cnt) ? y : ymid;
      sts_f64_if(i + 1 < cnt, xrow + xs + 8 * r, y);
#pragma unroll
      for (int c = 0; c < 6; ++c) a[c] = __shfl_sync(0xfffu, y, base + c);
      gp += 576; xrow += 2 * xs;
    }
    const double yo = __shfl_sync(0xfffu, ymid, bottom ? lane - 6 : lane + 6);
    double* mrow = w.nx(2 * oe.jm);
    if (lane < 6) mrow[r] = ymid + yo;
  }
  __syncwarp();
}
// V2: 2 lanes per half, 3 rows each (18 fmas), three values exchanged by shuffle
__device__ __forceinline__ void fwd_shfl2(int lane, const View& w, const OEView& oe) {
  const bool act = lane < 4; const bool bottom = (lane >> 1) & 1; const int q = lane & 1;     // rows 3q .. 3q+2
  const OEHalf h = oe_half(w, oe, bottom);
  const int cnt = h.cnt, cmax = oe.jm > oe.nb ? oe.jm : oe.nb;
  const int xs = h.xstep * 8;
  const unsigned xlast = smem_u32(h.xlast) + 24 * q;
  unsigned xrow = smem_u32(h.x0) + xs, gp = smem_u32(h.g0) + 144 * q;
  double a[6], g[18], nb[3], y[3], ymid[3];
  lds_row(smem_u32(h.x0), a);
  for (int t = 0; t < 3; ++t) ymid[t] = lds_f64(xlast + 8 * t);
  for (int i = 1; i <= cmax; ++i) {
    lds_row(gp, g); lds_row(gp + 48, g + 6); lds_row(gp + 96, g + 12);
    const unsigned nr = (i == cnt ? xlast : xrow + 24 * q);
    for (int t = 0; t < 3; ++t) nb[t] = lds_f64(nr + 8 * t);
#pragma unroll
    for (int t = 0; t < 3; ++t) y[t] = oe_row_dot(g + 6 * t, nb[t], a);
#pragma unroll
    for (int t = 0; t < 3; ++t) { ymid[t] = (i == cnt) ? y[t] : ymid[t]; sts_f64_if(act && i < cnt, xrow + 24 * q + 8 * t, y[t]); }
#pragma unroll
    for (int t = 0; t < 3; ++t) { const double o = __shfl_xor_sync(0xffffffffu, y[t], 1); a[3 * q + t] = y[t]; a[3 * (1 - q) + t] = o; }
    gp += 288; xrow += xs;
  }
  if (lane < 2) { double* mrow = w.nx(2 * oe.jm); for (int t = 0; t < 3; ++t) mrow[3 * q + t] = ymid[t]; }
  __syncwarp();
}
template <int VAR>
__global__ void bench_var(int N, int F, int reps, long long* cyc, double* sink) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int fpad, xpad; layout_pads(N, fpad, xpad);
  View w{smem + (size_t)warp * F, N, fpad, xpad};
  const OEView oe = oe_view(w);
  fill(w, oe, lane);
  __syncwarp();
  long long tf = 0;
  for (int r = 0; r < reps; ++r) {
    long long t0 = clock64();
    if (VAR == 0) oe_forward_lanes(lane, [&] { return sweep_lane(lane, w, oe); }, oe); else if (VAR == 1) fwd_shfl6(lane, w, oe); else if (VAR == 3) fwd_shfl6_region(lane, w, oe); else fwd_shfl2(lane, w, oe);
    __syncwarp();
    tf += clock64() - t0;
    for (int k = lane; k <= N; k += 32) { double* x = w.nx(k); for (int t = 0; t < 6; ++t) x[t] = 1.0 + 0.01 * ((k + t + r) % 9); }
    __syncwarp();
  }
  if (lane == 0 && blockIdx.x == 0 && warp == 0) cyc[0] = tf / reps;
  if (lane == 0) sink[blockIdx.x * 32 + warp] = w.nx(0)[0] + oe.sinv[0];
}
__global__ void bench(int N, int F, int reps, long long* cyc, double* sink) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int fpad, xpad; layout_pads(N, fpad, xpad);
  View w{smem + (size_t)warp * F, N, fpad, xpad};
  const OEView oe = oe_view(w);
  fill(w, oe, lane);
  __syncwarp();
  long long tf = 0, td = 0, tb = 0, tfac = 0;
  for (int r = 0; r < reps; ++r) {
    long long t0 = clock64();
    oe_forward_lanes(lane, [&] { return sweep_lane(lane, w, oe); }, oe);
    __syncwarp();
    long long t1 = clock64();
    for (int k = 2 * lane; k <= N; k += 64) oe_diag_stage(w, oe, k);
    __syncwarp();
    long long t2 = clock64();
    oe_backward_lanes(lane, [&] { return sweep_lane(lane, w, oe); }, oe);
    __syncwarp();
    long long t3 = clock64();
    tf += t1 - t0; td += t2 - t1; tb += t3 - t2;
    for (int k = lane; k <= N; k += 32) { double* x = w.nx(k); for (int t = 0; t < 6; ++t) x[t] = 1.0 + 0.01 * ((k + t + r) % 9); }   // keep the numbers bounded
    __syncwarp();
  }
  {
    fill(w, oe, lane);
    __syncwarp();
    long long t0 = clock64();
    double U[21], Uo[21];
    for (int t = 0; t < 21; ++t) U[t] = 0.0;
    if (lane < 2) oe_factor_half(oe_half(w, oe, lane == 1), U);
    __syncwarp();
    for (int t = 0; t < 21; ++t) Uo[t] = __shfl_sync(0xffffffffu, U[t], 1);
    if (lane == 0) oe_factor_middle(oe, U, Uo);
    __syncwarp();
    tfac = clock64() - t0;
  }
  if (lane == 0 && blockIdx.x == 0 && warp == 0) { cyc[0] = tf / reps; cyc[1] = td / reps; cyc[2] = tb / reps; cyc[3] = tfac; }
  if (lane == 0) sink[blockIdx.x * 32 + warp] = w.nx(0)[0] + oe.sinv[0];
}
int main(int argc, char** argv) {
  int N = argc > 1 ? atoi(argv[1]) : 50;
  int F = footprint(N);
  long long* cyc; double* sink;
  CK(cudaMalloc(&cyc, 64)); CK(cudaMalloc(&sink, 148 * 32 * 8));
  CK(cudaFuncSetAttribute(bench, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  int maxw = (227 * 1024) / (F * 8);
  int ws[] = {1, 4, 5, 6, 8};
  for (int wi = 0; wi < 5; ++wi) {
    int W = ws[wi]; if (W > maxw) continue;
    bench<<<148, 32 * W, W * F * 8>>>(N, F, 50, cyc, sink);
    CK(cudaDeviceSynchronize());
    long long h[4]; CK(cudaMemcpy(h, cyc, 32, cudaMemcpyDeviceToHost));
    int steps = oe_mid(N);
    printf("N=%d warps/SM=%d: forward+middle %lld (%.0f/step), diagonal %lld, backward %lld (%.0f/step), sequential factor %lld cycles\n",
           N, W, h[0], (double)h[0] / steps, h[1], h[2], (double)h[2] / steps, h[3]);
  }
  CK(cudaFuncSetAttribute(bench_var<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  CK(cudaFuncSetAttribute(bench_var<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  CK(cudaFuncSetAttribute(bench_var<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  CK(cudaFuncSetAttribute(bench_var<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  for (int var = 0; var < 4; ++var)
    for (int wi = 0; wi < 5; ++wi) {
      int W = ws[wi]; if (W > maxw) continue;
      if (var == 0) bench_var<0><<<148, 32 * W, W * F * 8>>>(N, F, 50, cyc, sink);
      else if (var == 1) bench_var<1><<<148, 32 * W, W * F * 8>>>(N, F, 50, cyc, sink);
      else if (var == 2) bench_var<2><<<148, 32 * W, W * F * 8>>>(N, F, 50, cyc, sink);
      else bench_var<3><<<148, 32 * W, W * F * 8>>>(N, F, 50, cyc, sink);
      CK(cudaDeviceSynchronize());
      long long h[1]; CK(cudaMemcpy(h, cyc, 8, cudaMemcpyDeviceToHost));
      printf("N=%d warps/SM=%d forward variant %d (0 shipped: smem exchange in a 12-lane region, 1 shuffle x6 lanes all lanes converged, 2 shuffle 2 lanes x 3 rows, 3 shuffle x6 lanes in the 12-lane region): %lld cycles (%.0f/step)\n", N, W, var, h[0], (double)h[0] / oe_mid(N));
    }
  return 0;
}
