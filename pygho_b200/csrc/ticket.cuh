// Deterministic in-kernel grid reductions shared by the fused BatchNorm kernels (fused_mlp.cu)
// and the GEMM with a statistics epilogue (linear_stats.cu).
#pragma once
#include <cuda_runtime.h>
#include <math.h>

namespace pgh {

// Two-level ticketed combine.  Every CTA of the launch has written W floats (W % 4 == 0) to
// part[blockIdx.x * W ..]; exactly one CTA returns true, with fin[0..W) (shared memory, double)
// holding the sum over all CTAs added in a fixed order.  tickets[0..1+ngroups) must be zero on
// entry and are zero again on exit (self-resetting: the buffer is reused by the next launch).
// The combining CTA issues its loads 8 partials at a time (128-bit each) before adding them in
// order: the tail costs a few L2 round trips, not one per partial.
__device__ inline bool ticketed_combine(const float* part, float* part2, int W, int blocks, int grp,
                                 int ngroups, int* tickets, double* fin) {
  __shared__ int s_last;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
  const int g = blockIdx.x / grp;
  const int g_lo = g * grp;
  const int g_n = min(grp, blocks - g_lo);
  const int W4 = W >> 2;
  constexpr int kInFlight = 8;
  if (blocks == 1) {
    // a single CTA (the graph-level and node-level layers of small batches): its own partial,
    // no fence, no ticket -- the whole tail is one barrier and one L2 round trip
    __syncthreads();
    for (int e = tid; e < W4; e += nt) {
      const float4 v = __ldcg(reinterpret_cast<const float4*>(part) + e);
      fin[4 * e] = (double)v.x; fin[4 * e + 1] = (double)v.y; fin[4 * e + 2] = (double)v.z; fin[4 * e + 3] = (double)v.w;
    }
    __syncthreads();
    return true;
  }
  __threadfence();                       // release: this CTA's partial is visible before its ticket
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(tickets + 1 + g, 1) == g_n - 1);
  __syncthreads();
  if (!s_last) return false;
  if (ngroups == 1) {
    // one group: its last CTA is the last CTA -- sum the partials straight into fin
    for (int e = tid; e < W4; e += nt) {
      double ax = 0.0, ay = 0.0, az = 0.0, aw = 0.0;
      const float4* p = reinterpret_cast<const float4*>(part) + e;
      for (int b0 = 0; b0 < g_n; b0 += kInFlight) {
        float4 v[kInFlight];
#pragma unroll
        for (int u = 0; u < kInFlight; ++u) v[u] = __ldcg(p + (size_t)min(b0 + u, g_n - 1) * W4);
#pragma unroll
        for (int u = 0; u < kInFlight; ++u)
          if (b0 + u < g_n) { ax += (double)v[u].x; ay += (double)v[u].y; az += (double)v[u].z; aw += (double)v[u].w; }
      }
      fin[4 * e] = ax; fin[4 * e + 1] = ay; fin[4 * e + 2] = az; fin[4 * e + 3] = aw;
    }
    if (tid == 0) tickets[1] = 0;
    __syncthreads();
    return true;
  }
  // acquire side: the partials are read with ld.global.cg (L2, never a stale L1 line) after the
  // barrier that follows the ticket -- the pattern of CUDA's threadFenceReduction sample
  for (int e = tid; e < W4; e += nt) {
    double ax = 0.0, ay = 0.0, az = 0.0, aw = 0.0;
    const float4* p = reinterpret_cast<const float4*>(part + (size_t)g_lo * W) + e;
    for (int b0 = 0; b0 < g_n; b0 += kInFlight) {
      float4 v[kInFlight];
#pragma unroll
      for (int u = 0; u < kInFlight; ++u) v[u] = __ldcg(p + (size_t)min(b0 + u, g_n - 1) * W4);
#pragma unroll
      for (int u = 0; u < kInFlight; ++u)
        if (b0 + u < g_n) { ax += (double)v[u].x; ay += (double)v[u].y; az += (double)v[u].z; aw += (double)v[u].w; }
    }
    reinterpret_cast<float4*>(part2 + (size_t)g * W)[e] = make_float4((float)ax, (float)ay, (float)az, (float)aw);
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    tickets[1 + g] = 0;
    s_last = (atomicAdd(tickets, 1) == ngroups - 1);
  }
  __syncthreads();
  if (!s_last) return false;
  for (int e = tid; e < W4; e += nt) {
    double ax = 0.0, ay = 0.0, az = 0.0, aw = 0.0;
    const float4* p = reinterpret_cast<const float4*>(part2) + e;
    for (int b0 = 0; b0 < ngroups; b0 += kInFlight) {
      float4 v[kInFlight];
#pragma unroll
      for (int u = 0; u < kInFlight; ++u) v[u] = __ldcg(p + (size_t)min(b0 + u, ngroups - 1) * W4);
#pragma unroll
      for (int u = 0; u < kInFlight; ++u)
        if (b0 + u < ngroups) { ax += (double)v[u].x; ay += (double)v[u].y; az += (double)v[u].z; aw += (double)v[u].w; }
    }
    fin[4 * e] = ax; fin[4 * e + 1] = ay; fin[4 * e + 2] = az; fin[4 * e + 3] = aw;
  }
  if (tid == 0) tickets[0] = 0;
  __syncthreads();
  return true;
}


// Per-channel epilogue of a BatchNorm statistics reduction, run by the CTA that won the ticket:
// fin[c] = sum (y - shift), fin[C + c] = sum (y - shift)^2 over n rows.
//   local_out == NULL : mean, rstd (+ running statistics with the unbiased variance; with n == 0
//                       mean = 0 and rstd = 1/sqrt(eps), and the running statistics keep their
//                       values: an empty batch is not evidence of mean 0 and variance 0)
//   local_out != NULL : the rank-local (mean, M2, count) rows for cross-rank merging (SyncBN)
// shift may be NULL (= 0).  nbt: BatchNorm1d.num_batches_tracked (int64) or NULL.
__device__ inline void bn_finalize_stats(const double* fin, int C, double n,
                                         const float* __restrict__ shift, float eps, float momentum,
                                         float* __restrict__ mean, float* __restrict__ rstd,
                                         float* __restrict__ running_mean,
                                         float* __restrict__ running_var,
                                         float* __restrict__ local_out, long long* __restrict__ nbt) {
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
  if (tid == 0 && nbt) nbt[0] += 1;
  for (int c = tid; c < C; c += nt) {
    const double sc = fin[c], qc = fin[C + c];
    const double ms = n > 0.0 ? sc / n : 0.0;              // mean of (y - shift)
    const double m = n > 0.0 ? ms + (shift ? (double)shift[c] : 0.0) : 0.0;
    double m2 = qc - sc * ms;                               // sum of squared deviations
    if (m2 < 0.0) m2 = 0.0;
    if (local_out) {
      local_out[c] = (float)m;
      local_out[C + c] = (float)m2;
      local_out[2 * C + c] = (float)n;
      continue;
    }
    const double var = n > 0.0 ? m2 / n : 0.0;              // biased variance
    mean[c] = (float)m;
    rstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean && n > 0.0) {
      const double unbiased = n > 1.0 ? m2 / (n - 1.0) : var;
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)m;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
  }
}

}  // namespace pgh
