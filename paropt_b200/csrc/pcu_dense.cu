// pcu_dense.cu -- device side of pcu_dense.cuh: a single-CTA kernel that runs the
// small dense algebra of the default iteration's KKT solve between the Gram pass and
// the one pass that applies the step, so that the chain  DiagRhsF -> Gram -> dense ->
// Pass2SVF  needs no host round trip (LU of G and Ce, SMW coefficients, dense
// residuals, the refinement in the column space of [A|Z]).
//
// The flat work buffer (<= 5k doubles) is staged in shared memory by all threads, warp
// 0 runs the lane-parallel algorithm of pcu_dense.cuh on it (matrices of at most
// 32 x 32), all threads write the result region back.
//
#include <stdio.h>
#include <stdlib.h>

#include "pcu_dense.cuh"

#define PCU_DENSE_THREADS 128

__global__ void __launch_bounds__(PCU_DENSE_THREADS, 1)
    pcu_dense_kernel(double *buf, const DenseOff o, const double *Sin, long long *tick) {
  extern __shared__ double2 dense_smem2[];
  double *w = reinterpret_cast<double *>(dense_smem2);
  double *scratch = w + o.total;
  const int tid = threadIdx.x;
  if (tick && tid == 0) tick[0] = clock64();
  // the inputs only (the rest is produced here)
  for (int i = tid; i < o.S; i += PCU_DENSE_THREADS) w[i] = buf[i];
  const int nS = o.ld * o.ld;
  for (int i = tid; i < nS; i += PCU_DENSE_THREADS) w[o.S + i] = Sin[i];
  __syncthreads();
  if (tick && tid == 0) tick[1] = clock64();
  if (tid < 32) pcu_dense_solve(w, o, scratch, tick);
  __syncthreads();
  if (tick && tid == 0) tick[4] = clock64();
  for (int i = o.S + tid; i < o.total; i += PCU_DENSE_THREADS) buf[i] = w[i];
  if (tick && tid == 0) tick[5] = clock64();
}

// Enqueues pcu_dense_solve on `stream`.  buf: device work buffer (layout `o`, inputs
// in place); Sin: Gram result.
int pcu_dense_enqueue(cudaStream_t stream, double *buf, const DenseOff &o, const double *Sin) {
  const size_t smem = sizeof(double) * (size_t)(o.total + PCU_DENSE_SCRATCH(o.c, o.q));
  if (smem > 48 * 1024) {
    static bool raised[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !raised[dev]) {
      if (cudaFuncSetAttribute(pcu_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               96 * 1024) != cudaSuccess)
        return 1;
      if (dev >= 0 && dev < 64) raised[dev] = true;
    }
    if (smem > 96 * 1024) return 1;
  }
  static long long *ticks = nullptr;
  static int tick_calls = 0;
  const bool profile = getenv("PCU_DENSE_TICKS") != nullptr;
  if (profile && !ticks) cudaMalloc(&ticks, 8 * sizeof(long long));
  pcu_dense_kernel<<<1, PCU_DENSE_THREADS, smem, stream>>>(buf, o, Sin,
                                                           profile ? ticks : nullptr);
  if (profile && ++tick_calls % 20 < 1) {
    cudaStreamSynchronize(stream);
    long long t[8];
    cudaMemcpy(t, ticks, sizeof(t), cudaMemcpyDeviceToHost);
    fprintf(stderr, "dense kernel (c=%d q=%d) cycles: stage-in %lld, setup %lld, step %lld, "
            "refinement %lld, stage-out %lld, total %lld\n", o.c, o.q, t[1] - t[0], t[2] - t[1],
            t[3] - t[2], t[4] - t[3], t[5] - t[4], t[5] - t[0]);
  }
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

// The same solve on the host (the KKT solve's host route: PCU_NO_CHAIN, several GPUs).
void pcu_dense_host(double *w, const DenseOff &o, const double *Sin) {
  double scratch[PCU_DENSE_SCRATCH(PCU_DENSE_MAXM / 2, PCU_DENSE_MAXM / 2) + 8 * PCU_DENSE_MAXM];
  for (int i = 0; i < o.ld * o.ld; i++) w[o.S + i] = Sin[i];
  pcu_dense_solve(w, o, scratch);
}
