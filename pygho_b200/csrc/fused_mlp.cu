// Fused BatchNorm(training) + activation around the tuplewise Linear layers.
//
// The reference's MLP block is Linear -> BatchNorm1d over ALL tuples of the batch -> SiLU
// (honn/utils.py:46-61, 85-142).  With stock ATen kernels one block costs 5 full passes over
// the (tuples x channels) activation forward and 7 backward (plus a separate column reduce for
// the Linear bias gradient).  These kernels do it in 3 + 5 passes, all HBM-streaming:
//
//   forward   stats(y) -> mean, rstd            (1 read)
//             z = act(gamma * (y - mean) * rstd + beta)          (1 read, 1 write)
//   backward  reduce: sum dyh, sum dyh*xh  with dyh = dz * act'(yh) recomputed   (2 reads)
//             dy = gamma*rstd*(dyh - mean(dyh) - xh*mean(dyh*xh)), column sums of dy (2 reads, 1 write)
//
// Thread layout everywhere: a thread owns 4 consecutive channels (one 128-bit lane of the
// row) and walks rows with stride, so every warp request is a contiguous 512 B piece of a row
// and per-channel accumulators live in registers.  Partial sums go to a workspace and are
// combined IN THE SAME LAUNCH by a two-level "last CTA done" ticket: the last CTA of every group
// of 16 adds that group's partials in block order, the last group adds the group sums in group
// order and runs the per-channel epilogue.  Who combines depends on timing, WHAT is added in
// which order does not: deterministic, no floating-point atomics, no second launch (round 1
// used a separate *_final kernel per reduction: 51 tiny launches per SSWL+ step).
//
// Optional device-side row count (`rows_dev`): the tensors may be padded to a fixed capacity so
// that a whole training step can be replayed as ONE CUDA graph for batches of different sizes
// (pygho_b200/static.py).  Rows >= *rows_dev are excluded from every statistic, their forward
// output is 0 and their gradient is 0.
//
// Optional cross-rank statistics (SyncBN, SURVEY.md Q11): `stats` can emit the rank-local
// (mean, M2, count) triple instead of finishing; after an all-gather `sync_finalize` merges the
// ranks with Chan's formula in rank order (bitwise identical on every rank); the backward
// `reduce` emits the local sums, which are all-reduced before `apply`.
#include <math.h>

#include "common.cuh"
#include "ticket.cuh"

namespace pgh {

constexpr int kBnThreads = 256;

// run-time tuning (pgh_set_tuning): [2] partial-reduction CTAs per SM (default 4), [3] rows in
// flight per thread in the backward kernels (2 or 4), [4] 1 = the apply passes walk the rows in
// the opposite direction of the reduce pass before them (the tail of that pass is still in the
// 126 MB L2), [5] elements in flight per thread of the forward apply (1, 2 or 4; default 2).
// Sweep on B200 (profiles/r1_bn_sweep.txt): 2 rows in flight and 4 CTAs/SM are best, the
// reverse walk buys nothing (the L2 does not keep the tail of a streaming pass)
static int bn_tune(int key, int dflt) { return g_tune[key] > 0 ? g_tune[key] : dflt; }

constexpr int kBnMaxGroups = 63;   // ticket words per launch: 1 + groups <= 64

struct BnGeom {
  int c4;        // float4 columns per row
  int ty;        // row lanes per block
  int blocks;
  long long rows_per_block;
  int grp;       // partial CTAs per first-level group
  int ngroups;
  size_t smem;   // dynamic shared memory of the reduction kernels
};

static BnGeom bn_geom(int64_t rows, int64_t C) {
  BnGeom g;
  g.c4 = (int)(C / 4);
  g.ty = kBnThreads / g.c4;
  if (g.ty < 1) g.ty = 1;
  const long long max_blocks = (long long)kSMs * bn_tune(2, 4);
  long long rpb = (rows + max_blocks - 1) / max_blocks;
  const long long min_rows = 8LL * g.ty;
  if (rpb < min_rows) rpb = min_rows;
  rpb = (rpb + g.ty - 1) / g.ty * g.ty;
  g.rows_per_block = rpb;
  g.blocks = (int)((rows + rpb - 1) / rpb);
  g.grp = 16;
  while ((g.blocks + g.grp - 1) / g.grp > kBnMaxGroups) g.grp *= 2;
  g.ngroups = (g.blocks + g.grp - 1) / g.grp;
  const size_t red = (size_t)g.c4 * g.ty * 2 * sizeof(float4);
  const size_t fin = (size_t)2 * C * sizeof(double);
  g.smem = red > fin ? red : fin;
  return g;
}

__device__ __forceinline__ long long valid_rows(long long rows, const int* __restrict__ rows_dev) {
  if (!rows_dev) return rows;
  const long long v = (long long)__ldg(rows_dev);
  return v < rows ? (v < 0 ? 0 : v) : rows;
}

template <int ACT>
__device__ __forceinline__ float act_grad(float x) {
  if (ACT == 1) {
    const float s = 1.f / (1.f + __expf(-x));
    return s * (1.f + x * (1.f - s));
  }
  if (ACT == 2) return x > 0.f ? 1.f : 0.f;
  return 1.f;
}

// block-level reduction over the ty row lanes of two float4 accumulators; result valid for ty==0
__device__ __forceinline__ void reduce_rows(float4& a, float4& b, float4* sm, int c4, int ty_n) {
  const int tx = threadIdx.x, ty = threadIdx.y;
  if (ty_n == 1) return;
  sm[(ty * c4 + tx) * 2] = a;
  sm[(ty * c4 + tx) * 2 + 1] = b;
  __syncthreads();
  if (ty == 0) {
    for (int t = 1; t < ty_n; ++t) {
      const float4 x = sm[(t * c4 + tx) * 2], y = sm[(t * c4 + tx) * 2 + 1];
      a.x += x.x; a.y += x.y; a.z += x.z; a.w += x.w;
      b.x += y.x; b.y += y.y; b.z += y.z; b.w += y.w;
    }
  }
}

// ---- forward statistics: shifted sums (shift = row 0) to avoid cancellation -------------
// local_out != NULL (SyncBN): emit the rank-local (mean, M2, count) rows instead of finishing.
__global__ void __launch_bounds__(kBnThreads, 4) bn_stats_kernel(const float* __restrict__ y, long long rows_cap, int C,
                                const int* __restrict__ rows_dev, long long rows_per_block,
                                float* __restrict__ part, float* __restrict__ part2, int blocks,
                                int grp, int ngroups, int* __restrict__ tickets, float eps,
                                float momentum, float* __restrict__ mean, float* __restrict__ rstd,
                                float* __restrict__ running_mean, float* __restrict__ running_var,
                                float* __restrict__ local_out, long long* __restrict__ nbt) {
  pdl_enter();
  extern __shared__ float4 sm[];
  const long long rows = valid_rows(rows_cap, rows_dev);
  const int tx = threadIdx.x, c4 = blockDim.x, ty_n = blockDim.y;
  const float4 shift = __ldg(reinterpret_cast<const float4*>(y) + tx);
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  const long long r1 = min(rows, r0 + rows_per_block);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
  const float4* base = reinterpret_cast<const float4*>(y) + tx;
#pragma unroll 4
  for (long long r = r0 + threadIdx.y; r < r1; r += ty_n) {
    const float4 v = __ldg(base + r * c4);
    const float dx = v.x - shift.x, dy = v.y - shift.y, dz = v.z - shift.z, dw = v.w - shift.w;
    s.x += dx; s.y += dy; s.z += dz; s.w += dw;
    q.x = fmaf(dx, dx, q.x); q.y = fmaf(dy, dy, q.y); q.z = fmaf(dz, dz, q.z); q.w = fmaf(dw, dw, q.w);
  }
  reduce_rows(s, q, sm, c4, ty_n);
  if (threadIdx.y == 0) {
    float4* p = reinterpret_cast<float4*>(part + (size_t)blockIdx.x * 2 * C);
    p[tx] = s;
    p[c4 + tx] = q;
  }
  double* fin = reinterpret_cast<double*>(sm);
  if (!ticketed_combine(part, part2, 2 * C, blocks, grp, ngroups, tickets, fin)) return;
  bn_finalize_stats(fin, C, (double)rows, y, eps, momentum, mean, rstd, running_mean, running_var,
                    local_out, nbt);
}

// SyncBN: merge the (mean, M2, count) triples of `world` ranks (gathered: (world, 3, C)) with
// Chan's pairwise formula in rank order; every rank computes the same bits.
__global__ void bn_sync_finalize_kernel(const float* __restrict__ gathered, int world, int C,
                                        float eps, float momentum, float* __restrict__ mean,
                                        float* __restrict__ rstd, float* __restrict__ running_mean,
                                        float* __restrict__ running_var, float* __restrict__ inv_n) {
  pdl_enter();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double n = 0.0, m = 0.0, m2 = 0.0;
  for (int r = 0; r < world; ++r) {
    const float* g = gathered + (size_t)r * 3 * C;
    const double nb = (double)g[2 * C + c];
    if (nb <= 0.0) continue;
    const double mb = (double)g[c], m2b = (double)g[C + c];
    const double tot = n + nb, delta = mb - m;
    m += delta * (nb / tot);
    m2 += m2b + delta * delta * (n * nb / tot);
    n = tot;
  }
  const double var = n > 0.0 ? m2 / n : 0.0;
  mean[c] = (float)m;
  rstd[c] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean) {
    const double unbiased = n > 1.0 ? m2 / (n - 1.0) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)m;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
  if (c == 0 && inv_n) inv_n[0] = n > 0.0 ? (float)(1.0 / n) : 0.f;
}

// ---- forward apply ------------------------------------------------------------------------
template <int ACT, int UN>
__global__ void bn_act_fwd_kernel(const float4* __restrict__ y, const float4* __restrict__ mean,
                                  const float4* __restrict__ rstd, const float4* __restrict__ gamma,
                                  const float4* __restrict__ beta, long long n4_cap, int c4,
                                  const int* __restrict__ rows_dev,
                                  const float4* __restrict__ residual, float4* __restrict__ z) {
  pdl_enter();
  const long long n4 = valid_rows(n4_cap / c4, rows_dev) * c4;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < n4; i0 += stride * UN) {
    float4 v[UN], res[UN];
    long long idx[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      idx[u] = min(i0 + u * stride, n4 - 1);                 // clamped: loads are unconditional
      v[u] = __ldg(y + idx[u]);
      if (residual) res[u] = __ldg(residual + idx[u]);
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      if (i0 + u * stride >= n4) break;
      const int c = (int)(idx[u] % c4);
      const float4 m = __ldg(mean + c), r = __ldg(rstd + c);
      const float4 g = gamma ? __ldg(gamma + c) : make_float4(1.f, 1.f, 1.f, 1.f);
      const float4 b = beta ? __ldg(beta + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 o;
      o.x = act_fwd<ACT>(fmaf((v[u].x - m.x) * r.x, g.x, b.x));
      o.y = act_fwd<ACT>(fmaf((v[u].y - m.y) * r.y, g.y, b.y));
      o.z = act_fwd<ACT>(fmaf((v[u].z - m.z) * r.z, g.z, b.z));
      o.w = act_fwd<ACT>(fmaf((v[u].w - m.w) * r.w, g.w, b.w));
      if (residual) { o.x += res[u].x; o.y += res[u].y; o.z += res[u].z; o.w += res[u].w; }
      z[idx[u]] = o;
    }
  }
  // padded rows (static-capacity tensors): defined, finite output
  for (long long i = n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4_cap; i += stride)
    z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// ---- backward reduce: S1 = sum dyh, S2 = sum dyh * xh; epilogue writes dbeta / dgamma --------
template <int ACT, int UN>
__global__ void __launch_bounds__(kBnThreads, 4) bn_act_bwd_reduce_kernel(const float* __restrict__ dz, const float* __restrict__ y,
                                         const float* __restrict__ mean, const float* __restrict__ rstd,
                                         const float* __restrict__ gamma, const float* __restrict__ beta,
                                         long long rows_cap, int C, const int* __restrict__ rows_dev,
                                         long long rows_per_block, float* __restrict__ part,
                                         float* __restrict__ part2, int blocks, int grp, int ngroups,
                                         int* __restrict__ tickets, float* __restrict__ sums,
                                         float* __restrict__ dgamma, float* __restrict__ dbeta,
                                         int accumulate) {
  pdl_enter();
  extern __shared__ float4 sm[];
  const long long rows = valid_rows(rows_cap, rows_dev);
  const int tx = threadIdx.x, c4 = blockDim.x, ty_n = blockDim.y;
  const float4 m = __ldg(reinterpret_cast<const float4*>(mean) + tx);
  const float4 rs = __ldg(reinterpret_cast<const float4*>(rstd) + tx);
  const float4 g = gamma ? __ldg(reinterpret_cast<const float4*>(gamma) + tx) : make_float4(1.f, 1.f, 1.f, 1.f);
  const float4 bt = beta ? __ldg(reinterpret_cast<const float4*>(beta) + tx) : make_float4(0.f, 0.f, 0.f, 0.f);
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  const long long r1 = min(rows, r0 + rows_per_block);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
  const float4* yb = reinterpret_cast<const float4*>(y) + tx;
  const float4* db = reinterpret_cast<const float4*>(dz) + tx;
  for (long long rb = r0 + threadIdx.y; rb < r1; rb += (long long)ty_n * UN) {
    float4 vv[UN], dd[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u) {                 // clamped rows: all 2*UN loads issue together
      const long long r = min(rb + (long long)u * ty_n, r1 - 1);
      vv[u] = __ldg(yb + r * c4);
      dd[u] = __ldg(db + r * c4);
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      if (rb + (long long)u * ty_n >= r1) break;
      const float4 v = vv[u], d = dd[u];
      const float xx = (v.x - m.x) * rs.x, xy = (v.y - m.y) * rs.y, xz = (v.z - m.z) * rs.z, xw = (v.w - m.w) * rs.w;
      const float gx = d.x * act_grad<ACT>(fmaf(xx, g.x, bt.x)), gy = d.y * act_grad<ACT>(fmaf(xy, g.y, bt.y));
      const float gz = d.z * act_grad<ACT>(fmaf(xz, g.z, bt.z)), gw = d.w * act_grad<ACT>(fmaf(xw, g.w, bt.w));
      s.x += gx; s.y += gy; s.z += gz; s.w += gw;
      q.x = fmaf(gx, xx, q.x); q.y = fmaf(gy, xy, q.y); q.z = fmaf(gz, xz, q.z); q.w = fmaf(gw, xw, q.w);
    }
  }
  reduce_rows(s, q, sm, c4, ty_n);
  if (threadIdx.y == 0) {
    float4* p = reinterpret_cast<float4*>(part + (size_t)blockIdx.x * 2 * C);
    p[tx] = s;
    p[c4 + tx] = q;
  }
  double* fin = reinterpret_cast<double*>(sm);
  if (!ticketed_combine(part, part2, 2 * C, blocks, grp, ngroups, tickets, fin)) return;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
  for (int c = tid; c < C; c += nt) {
    const float s1 = (float)fin[c], s2 = (float)fin[C + c];
    sums[c] = s1;
    sums[C + c] = s2;
    if (dbeta) dbeta[c] = accumulate ? dbeta[c] + s1 : s1;
    if (dgamma) dgamma[c] = accumulate ? dgamma[c] + s2 : s2;
  }
}

// ---- backward apply: dy and the column sums of dy (the Linear bias gradient) ------------------
// sums = (S1, S2) over ALL rows of the statistics (all ranks under SyncBN); inv_n = 1 / that
// row count (device scalar) or NULL = 1 / this tensor's valid rows.
template <int ACT, int UN>
__global__ void __launch_bounds__(kBnThreads, 4) bn_act_bwd_apply_kernel(const float* __restrict__ dz, const float* __restrict__ y,
                                        const float* __restrict__ mean, const float* __restrict__ rstd,
                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                        const float* __restrict__ sums, const float* __restrict__ inv_n,
                                        long long rows_cap, int C, const int* __restrict__ rows_dev,
                                        long long rows_per_block, float* __restrict__ dy,
                                        float* __restrict__ part, float* __restrict__ part2,
                                        int blocks, int grp, int ngroups, int* __restrict__ tickets,
                                        float* __restrict__ dbias, int accumulate) {
  pdl_enter();
  extern __shared__ float4 sm[];
  const long long rows = valid_rows(rows_cap, rows_dev);
  const int tx = threadIdx.x, c4 = blockDim.x, ty_n = blockDim.y;
  const float4 m = __ldg(reinterpret_cast<const float4*>(mean) + tx);
  const float4 rs = __ldg(reinterpret_cast<const float4*>(rstd) + tx);
  const float4 g = gamma ? __ldg(reinterpret_cast<const float4*>(gamma) + tx) : make_float4(1.f, 1.f, 1.f, 1.f);
  const float4 bt = beta ? __ldg(reinterpret_cast<const float4*>(beta) + tx) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float in = inv_n ? __ldg(inv_n) : (rows > 0 ? 1.f / (float)rows : 0.f);
  float4 a1 = __ldcg(reinterpret_cast<const float4*>(sums) + tx);
  float4 a2 = __ldcg(reinterpret_cast<const float4*>(sums + C) + tx);
  a1 = make_float4(a1.x * in, a1.y * in, a1.z * in, a1.w * in);
  a2 = make_float4(a2.x * in, a2.y * in, a2.z * in, a2.w * in);
  const float4 sc = make_float4(g.x * rs.x, g.y * rs.y, g.z * rs.z, g.w * rs.w);
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  const long long r1 = min(rows, r0 + rows_per_block);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f), unused = s;
  const float4* yb = reinterpret_cast<const float4*>(y) + tx;
  const float4* db = reinterpret_cast<const float4*>(dz) + tx;
  float4* ob = reinterpret_cast<float4*>(dy) + tx;
  for (long long rb = r0 + threadIdx.y; rb < r1; rb += (long long)ty_n * UN) {
    float4 vv[UN], dd[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const long long r = min(rb + (long long)u * ty_n, r1 - 1);
      vv[u] = __ldg(yb + r * c4);
      dd[u] = __ldg(db + r * c4);
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const long long r = rb + (long long)u * ty_n;
      if (r >= r1) break;
      const float4 v = vv[u], d = dd[u];
      const float xx = (v.x - m.x) * rs.x, xy = (v.y - m.y) * rs.y, xz = (v.z - m.z) * rs.z, xw = (v.w - m.w) * rs.w;
      const float gx = d.x * act_grad<ACT>(fmaf(xx, g.x, bt.x)), gy = d.y * act_grad<ACT>(fmaf(xy, g.y, bt.y));
      const float gz = d.z * act_grad<ACT>(fmaf(xz, g.z, bt.z)), gw = d.w * act_grad<ACT>(fmaf(xw, g.w, bt.w));
      float4 o;
      o.x = sc.x * (gx - a1.x - xx * a2.x);
      o.y = sc.y * (gy - a1.y - xy * a2.y);
      o.z = sc.z * (gz - a1.z - xz * a2.z);
      o.w = sc.w * (gw - a1.w - xw * a2.w);
      ob[r * c4] = o;
      s.x += o.x; s.y += o.y; s.z += o.z; s.w += o.w;
    }
  }
  // padded rows of this CTA's slab: zero gradient
  if (rows < rows_cap) {
    const long long p0 = max(r0, rows), p1 = min(rows_cap, r0 + rows_per_block);
    for (long long r = p0 + threadIdx.y; r < p1; r += ty_n) ob[r * c4] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (!dbias) return;
  reduce_rows(s, unused, sm, c4, ty_n);
  if (threadIdx.y == 0) reinterpret_cast<float4*>(part + (size_t)blockIdx.x * C)[tx] = s;
  double* fin = reinterpret_cast<double*>(sm);
  if (!ticketed_combine(part, part2, C, blocks, grp, ngroups, tickets, fin)) return;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
  for (int c = tid; c < C; c += nt) dbias[c] = accumulate ? dbias[c] + (float)fin[c] : (float)fin[c];
}

// out[e] (+)= sum_k part[k * n4 + e]  (float4 elements): the reduction over the split-K slabs
// of the tall-skinny weight-gradient GEMMs.  Block = 32 elements x 8 slab lanes: lane y adds the
// slabs y, y+8, ... (all loads of a thread in flight at once), then the 8 lanes are added in
// lane order: one L2 round trip, fixed order.
constexpr int kSlabLanes = 8, kSlabMax = 8;    // <= 64 slabs per call
__global__ void sum_slabs_kernel(const float4* __restrict__ part, int slabs, long long n4,
                                 float4* __restrict__ out, int accumulate) {
  pdl_enter();
  __shared__ float4 sm[kSlabLanes][32];
  const long long e = (long long)blockIdx.x * 32 + threadIdx.x;
  const int y = threadIdx.y;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (e < n4) {
    float4 v[kSlabMax];
#pragma unroll
    for (int u = 0; u < kSlabMax; ++u) {
      const int k = y + u * kSlabLanes;
      v[u] = __ldg(part + (size_t)min(k, slabs - 1) * n4 + e);
    }
#pragma unroll
    for (int u = 0; u < kSlabMax; ++u)
      if (y + u * kSlabLanes < slabs) { a.x += v[u].x; a.y += v[u].y; a.z += v[u].z; a.w += v[u].w; }
  }
  sm[y][threadIdx.x] = a;
  __syncthreads();
  if (y == 0 && e < n4) {
    float4 r = accumulate ? out[e] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int t = 0; t < kSlabLanes; ++t) {
      const float4 x = sm[t][threadIdx.x];
      r.x += x.x; r.y += x.y; r.z += x.z; r.w += x.w;
    }
    out[e] = r;
  }
}

// AdamW over ONE flat parameter / gradient / moment buffer (decoupled weight decay, bias
// correction, torch.optim.AdamW's update order).  `step` is a device scalar holding the number of
// updates done so far (float); the caller increments it after the launch, so the step can be
// captured in a CUDA graph.  grad_scale folds the 1 / world_size of the gradient average in.
__global__ void adamw_flat_kernel(float4* __restrict__ p, const float4* __restrict__ g,
                                  float4* __restrict__ m, float4* __restrict__ v, long long n4,
                                  const float* __restrict__ step, float lr, float b1, float b2,
                                  float eps, float wd, float grad_scale) {
  pdl_enter();
  const float t = __ldg(step) + 1.f;
  const float bc1 = 1.f - powf(b1, t), bc2 = 1.f - powf(b2, t);
  const float step_size = lr / bc1, inv_sqrt_bc2 = rsqrtf(bc2), decay = 1.f - lr * wd;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    float4 pp = p[i], gg = g[i], mm = m[i], vv = v[i];
#define PGH_ADAM(X)                                                            \
    {                                                                          \
      const float gr = gg.X * grad_scale;                                      \
      mm.X = b1 * mm.X + (1.f - b1) * gr;                                      \
      vv.X = b2 * vv.X + (1.f - b2) * gr * gr;                                 \
      const float denom = sqrtf(vv.X) * inv_sqrt_bc2 + eps;                    \
      pp.X = pp.X * decay - step_size * (mm.X / denom);                        \
    }
    PGH_ADAM(x) PGH_ADAM(y) PGH_ADAM(z) PGH_ADAM(w)
#undef PGH_ADAM
    p[i] = pp; m[i] = mm; v[i] = vv;
  }
}

static bool bn_ok(int64_t rows, int64_t C) {
  return rows > 0 && C >= 4 && C % 4 == 0 && C / 4 <= kBnThreads;
}

}  // namespace pgh

using namespace pgh;

extern "C" size_t pgh_bn_ws_bytes(int64_t rows, int64_t C) {
  if (!bn_ok(rows, C)) return 256;
  const BnGeom g = bn_geom(rows, C);
  return (size_t)g.blocks * 2 * C * sizeof(float) + 256 + (size_t)g.ngroups * 2 * C * sizeof(float);
}

static float* bn_part2(void* ws, const BnGeom& g, int64_t C) {
  size_t off = ((size_t)g.blocks * 2 * C * sizeof(float) + 255) & ~(size_t)255;
  return reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + off);
}

extern "C" int pgh_bn_stats_f32(const float* y, int64_t rows, int64_t C, const int32_t* rows_dev,
                                float eps, float momentum, float* mean, float* rstd,
                                float* running_mean, float* running_var, float* local_out,
                                int64_t* num_batches_tracked, void* ws, size_t ws_bytes,
                                int32_t* tickets, void* stream) {
  if (!y || !ws || !tickets || (!local_out && (!mean || !rstd))) return arg_error("bn_stats: null pointer");
  if (!bn_ok(rows, C)) return arg_error("bn_stats: need rows > 0, C % 4 == 0, C <= 1024");
  if ((reinterpret_cast<uintptr_t>(y) & 15)) return arg_error("bn_stats: y must be 16-byte aligned");
  const BnGeom g = bn_geom(rows, C);
  if (ws_bytes < pgh_bn_ws_bytes(rows, C)) return arg_error("bn_stats: workspace too small");
  launch_pdl(bn_stats_kernel, dim3(g.blocks), dim3(dim3(g.c4, g.ty)), g.smem, as_stream(stream), 
      y, rows, (int)C, rows_dev, g.rows_per_block, reinterpret_cast<float*>(ws), bn_part2(ws, g, C),
      g.blocks, g.grp, g.ngroups, tickets, eps, momentum, mean, rstd, running_mean, running_var,
      local_out, reinterpret_cast<long long*>(num_batches_tracked));
  return check_launch("bn_stats");
}

extern "C" int pgh_adamw_flat_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                                  int64_t n, const float* step, float lr, float beta1, float beta2,
                                  float eps, float weight_decay, float grad_scale, void* stream) {
  if (!param || !grad || !exp_avg || !exp_avg_sq || !step || n < 0 || (n & 3))
    return arg_error("adamw_flat: arguments (n % 4 == 0)");
  if ((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) |
       reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15)
    return arg_error("adamw_flat: buffers must be 16-byte aligned");
  if (n == 0) return 0;
  const long long n4 = n / 4;
  long long nb = (n4 + 255) / 256;
  if (nb > kSMs * 8) nb = kSMs * 8;
  launch_pdl(adamw_flat_kernel, dim3((unsigned)nb), dim3(256), 0, as_stream(stream), 
      reinterpret_cast<float4*>(param), reinterpret_cast<const float4*>(grad),
      reinterpret_cast<float4*>(exp_avg), reinterpret_cast<float4*>(exp_avg_sq), n4, step, lr, beta1,
      beta2, eps, weight_decay, grad_scale);
  return check_launch("adamw_flat");
}

extern "C" int pgh_sum_slabs_f32(const float* part, int64_t slabs, int64_t n, float* out,
                                 int accumulate, void* stream) {
  if (!part || !out || slabs < 1 || slabs > kSlabLanes * kSlabMax || n < 0 || (n & 3))
    return arg_error("sum_slabs: arguments (1 <= slabs <= 64, n % 4 == 0)");
  if ((reinterpret_cast<uintptr_t>(part) | reinterpret_cast<uintptr_t>(out)) & 15)
    return arg_error("sum_slabs: tensors must be 16-byte aligned");
  if (n == 0) return 0;
  const long long n4 = n / 4;
  launch_pdl(sum_slabs_kernel, dim3(blocks_for(n4, 32)), dim3(dim3(32, kSlabLanes)), 0, as_stream(stream), 
      reinterpret_cast<const float4*>(part), (int)slabs, n4, reinterpret_cast<float4*>(out), accumulate);
  return check_launch("sum_slabs");
}

extern "C" int pgh_bn_sync_finalize_f32(const float* gathered, int64_t world, int64_t C, float eps,
                                        float momentum, float* mean, float* rstd,
                                        float* running_mean, float* running_var, float* inv_n,
                                        void* stream) {
  if (!gathered || !mean || !rstd || world < 1 || C < 1) return arg_error("bn_sync_finalize: arguments");
  launch_pdl(bn_sync_finalize_kernel, dim3(blocks_for(C, 128)), dim3(128), 0, as_stream(stream), 
      gathered, (int)world, (int)C, eps, momentum, mean, rstd, running_mean, running_var, inv_n);
  return check_launch("bn_sync_finalize");
}

extern "C" int pgh_bn_act_res_fwd_f32(const float* y, const float* mean, const float* rstd,
                                      const float* gamma, const float* beta, int64_t rows,
                                      int64_t C, const int32_t* rows_dev, int act,
                                      const float* residual, float* z, void* stream) {
  if (!y || !mean || !rstd || !z) return arg_error("bn_act_fwd: null pointer");
  if (!bn_ok(rows, C)) return arg_error("bn_act_fwd: need rows > 0, C % 4 == 0, C <= 1024");
  if ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(z) |
       reinterpret_cast<uintptr_t>(residual)) & 15)
    return arg_error("bn_act_fwd: tensors must be 16-byte aligned");
  const long long n4 = rows * (C / 4);
  long long nb = (n4 + 255) / 256;
  if (nb > 148 * 16) nb = 148 * 16;
  cudaStream_t s = as_stream(stream);
#define PGH_FWD_U(A, U) launch_pdl(bn_act_fwd_kernel<A, U>, dim3((unsigned)nb), dim3(256), 0, s,                         \
      (const float4*)y, (const float4*)mean, (const float4*)rstd, (const float4*)gamma,             \
      (const float4*)beta, n4, (int)(C / 4), rows_dev, (const float4*)residual, (float4*)z)
#define PGH_FWD(A)                                                                                   \
  do {                                                                                               \
    const int un_ = bn_tune(5, 2);                                                                   \
    if (un_ >= 4) PGH_FWD_U(A, 4); else if (un_ == 2) PGH_FWD_U(A, 2); else PGH_FWD_U(A, 1);        \
  } while (0)
  if (act == 1) PGH_FWD(1); else if (act == 2) PGH_FWD(2); else if (act == 0) PGH_FWD(0);
  else return arg_error("bn_act_fwd: act");
#undef PGH_FWD_U
#undef PGH_FWD
  return check_launch("bn_act_fwd");
}

extern "C" int pgh_bn_act_bwd_reduce_f32(const float* dz, const float* y, const float* mean,
                                         const float* rstd, const float* gamma, const float* beta,
                                         int64_t rows, int64_t C, const int32_t* rows_dev, int act,
                                         float* sums, float* dgamma, float* dbeta, int accumulate,
                                         void* ws, size_t ws_bytes, int32_t* tickets, void* stream) {
  if (!dz || !y || !mean || !rstd || !sums || !ws || !tickets) return arg_error("bn_act_bwd_reduce: null pointer");
  if (!bn_ok(rows, C)) return arg_error("bn_act_bwd_reduce: need rows > 0, C % 4 == 0, C <= 1024");
  if ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(dz)) & 15)
    return arg_error("bn_act_bwd_reduce: tensors must be 16-byte aligned");
  if (act < 0 || act > 2) return arg_error("bn_act_bwd_reduce: act");
  const BnGeom g = bn_geom(rows, C);
  if (ws_bytes < pgh_bn_ws_bytes(rows, C)) return arg_error("bn_act_bwd_reduce: workspace too small");
  cudaStream_t s = as_stream(stream);
  const dim3 blk(g.c4, g.ty);
#define PGH_RED_U(A, U)                                                                              \
  launch_pdl(bn_act_bwd_reduce_kernel<A, U>, dim3(g.blocks), dim3(blk), g.smem, s,                                       \
      dz, y, mean, rstd, gamma, beta, rows, (int)C, rows_dev, g.rows_per_block,                      \
      reinterpret_cast<float*>(ws), bn_part2(ws, g, C), g.blocks, g.grp, g.ngroups, tickets, sums,   \
      dgamma, dbeta, accumulate)
#define PGH_RED(A)                                                                                   \
  do {                                                                                               \
    if (bn_tune(3, 2) >= 4) { PGH_RED_U(A, 4); } else { PGH_RED_U(A, 2); }                           \
  } while (0)
  if (act == 1) { PGH_RED(1); } else if (act == 2) { PGH_RED(2); } else { PGH_RED(0); }
#undef PGH_RED_U
#undef PGH_RED
  return check_launch("bn_act_bwd_reduce");
}

extern "C" int pgh_bn_act_bwd_apply_f32(const float* dz, const float* y, const float* mean,
                                        const float* rstd, const float* gamma, const float* beta,
                                        const float* sums, const float* inv_n, int64_t rows,
                                        int64_t C, const int32_t* rows_dev, int act, float* dy,
                                        float* dbias, int accumulate, void* ws, size_t ws_bytes,
                                        int32_t* tickets, void* stream) {
  if (!dz || !y || !mean || !rstd || !sums || !dy || !ws || !tickets) return arg_error("bn_act_bwd_apply: null pointer");
  if (!bn_ok(rows, C)) return arg_error("bn_act_bwd_apply: need rows > 0, C % 4 == 0, C <= 1024");
  if ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(dz) | reinterpret_cast<uintptr_t>(dy) |
       reinterpret_cast<uintptr_t>(sums)) & 15)
    return arg_error("bn_act_bwd_apply: tensors must be 16-byte aligned");
  if (act < 0 || act > 2) return arg_error("bn_act_bwd_apply: act");
  const BnGeom g = bn_geom(rows, C);
  if (ws_bytes < pgh_bn_ws_bytes(rows, C)) return arg_error("bn_act_bwd_apply: workspace too small");
  cudaStream_t s = as_stream(stream);
  const dim3 blk(g.c4, g.ty);
#define PGH_APP_U(A, U)                                                                              \
  launch_pdl(bn_act_bwd_apply_kernel<A, U>, dim3(g.blocks), dim3(blk), g.smem, s,                                        \
      dz, y, mean, rstd, gamma, beta, sums, inv_n, rows, (int)C, rows_dev, g.rows_per_block, dy,     \
      reinterpret_cast<float*>(ws), bn_part2(ws, g, C), g.blocks, g.grp, g.ngroups, tickets, dbias,  \
      accumulate)
#define PGH_APP(A)                                                                                   \
  do {                                                                                               \
    if (bn_tune(3, 2) >= 4) { PGH_APP_U(A, 4); } else { PGH_APP_U(A, 2); }                           \
  } while (0)
  if (act == 1) { PGH_APP(1); } else if (act == 2) { PGH_APP(2); } else { PGH_APP(0); }
#undef PGH_APP_U
#undef PGH_APP
  return check_launch("bn_act_bwd_apply");
}
