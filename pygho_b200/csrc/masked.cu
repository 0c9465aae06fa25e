// MaskedTensor kernels: 2-FWL contraction (CUDA-core path), masked pooling, masked fill.
//
// Layout is the reference's: (b, n, n, dense) with the dense (channel) axis contiguous
// (backend/MaTensor.py:34-111).  Every kernel maps lanes to channels, so each warp
// request is one contiguous 128 B line.
#include <cooperative_groups.h>
#include <math.h>

#include "common.cuh"

namespace pgh {

// ------------------------------------------------------------------ mamamm, algo 0
// One CTA per (graph b, 32-channel slab).  lane = channel; each warp owns 4x4 output
// tiles (i, k) in registers and walks j.  Exact fp32 (sequential j order).
constexpr int kTI = 4, kTK = 4;

__global__ void __launch_bounds__(256)
mamamm_simt_kernel(const float* __restrict__ A, long long sAi, long long sAj,
                   const float* __restrict__ B, long long sBj, long long sBk,
                   const unsigned char* __restrict__ mask, const int* __restrict__ ext, int n_i,
                   int n_j, int n_k, int dense, float* __restrict__ out) {
  const int b = blockIdx.x;
  // valid extents: operand pads are zero, so the j loop can stop at the valid extent
  const int nj_valid = ext ? min(max(ext[3 * b + 1], 0), n_j) : n_j;
  const int ch = blockIdx.y * 32 + (threadIdx.x & 31);
  const int warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const bool ch_ok = ch < dense;
  const float* Ab = A + (size_t)b * n_i * n_j * dense + ch;
  const float* Bb = B + (size_t)b * n_j * n_k * dense + ch;
  float* Ob = out + (size_t)b * n_i * n_k * dense + ch;
  const unsigned char* Mb = mask + (size_t)b * n_i * n_k;
  const int tiles_i = (n_i + kTI - 1) / kTI, tiles_k = (n_k + kTK - 1) / kTK;
  for (int tile = warp; tile < tiles_i * tiles_k; tile += nwarps) {
    const int i0 = (tile / tiles_k) * kTI, k0 = (tile % tiles_k) * kTK;
    float acc[kTI][kTK];
#pragma unroll
    for (int x = 0; x < kTI; ++x)
#pragma unroll
      for (int y = 0; y < kTK; ++y) acc[x][y] = 0.f;
    if (ch_ok) {
      for (int j = 0; j < nj_valid; ++j) {
        float a[kTI], bb[kTK];
#pragma unroll
        for (int x = 0; x < kTI; ++x)
          a[x] = (i0 + x < n_i) ? __ldg(Ab + ((size_t)(i0 + x) * sAi + (size_t)j * sAj) * dense) : 0.f;
#pragma unroll
        for (int y = 0; y < kTK; ++y)
          bb[y] = (k0 + y < n_k) ? __ldg(Bb + ((size_t)j * sBj + (size_t)(k0 + y) * sBk) * dense) : 0.f;
#pragma unroll
        for (int x = 0; x < kTI; ++x)
#pragma unroll
          for (int y = 0; y < kTK; ++y) acc[x][y] = fmaf(a[x], bb[y], acc[x][y]);
      }
#pragma unroll
      for (int x = 0; x < kTI; ++x)
#pragma unroll
        for (int y = 0; y < kTK; ++y)
          if (i0 + x < n_i && k0 + y < n_k) {
            const size_t o = (size_t)(i0 + x) * n_k + (k0 + y);
            Ob[o * dense] = Mb[o] ? acc[x][y] : 0.f;
          }
    }
  }
}

// ------------------------------------------------------------------ masked pooling
// View (outer, red, inner, dense): reduce the middle extent.  A thread owns 4 channels of one
// (outer, inner) output row and walks the reduced extent 4 rows at a time (4 independent
// 128-bit loads + 4 mask bytes in flight); a warp covers 128 consecutive channels, so every
// request is a contiguous 512 B piece of a row.  HBM bound: one read of the input.
struct PoolView {
  long long outer;
  int red, inner, c4;
};

template <int AGGR>
__global__ void masked_pool_kernel(const float4* __restrict__ data,
                                   const unsigned char* __restrict__ mask, PoolView v,
                                   float4* __restrict__ out, unsigned char* __restrict__ out_mask,
                                   long long total) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int ch = (int)(idx % v.c4);
  const long long rest = idx / v.c4;               // (outer, inner) flattened
  const int in = (int)(rest % v.inner);
  const long long o = rest / v.inner;
  const float init = AGGR == PGH_MAX ? -INFINITY : AGGR == PGH_MIN ? INFINITY : 0.f;
  float4 acc = make_float4(init, init, init, init);
  int cnt = 0;
  const long long base = o * v.red * v.inner + in;  // position of r = 0
  const unsigned char* mp = mask + base;
  const float4* dp = data + base * v.c4 + ch;
  const long long pstep = v.inner, dstep = (long long)v.inner * v.c4;
  auto take = [&](const float4& x) {
    if (AGGR == PGH_MAX) acc = make_float4(fmaxf(acc.x, x.x), fmaxf(acc.y, x.y), fmaxf(acc.z, x.z), fmaxf(acc.w, x.w));
    else if (AGGR == PGH_MIN) acc = make_float4(fminf(acc.x, x.x), fminf(acc.y, x.y), fminf(acc.z, x.z), fminf(acc.w, x.w));
    else acc = make_float4(acc.x + x.x, acc.y + x.y, acc.z + x.z, acc.w + x.w);
  };
  int r = 0;
  for (; r + 4 <= v.red; r += 4) {
    unsigned char m[4];
    float4 x[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) m[u] = __ldg(mp + (r + u) * pstep);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (m[u]) x[u] = __ldg(dp + (r + u) * dstep);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (m[u]) { take(x[u]); ++cnt; }
  }
  for (; r < v.red; ++r)
    if (__ldg(mp + r * pstep)) { take(__ldg(dp + r * dstep)); ++cnt; }
  if (cnt == 0) acc = make_float4(0.f, 0.f, 0.f, 0.f);
  else if (AGGR == PGH_MEAN) {
    const float n = (float)cnt;
    acc = make_float4(acc.x / n, acc.y / n, acc.z / n, acc.w / n);
  }
  if (AGGR == PGH_MAX || AGGR == PGH_MIN) {         // filterinf, MaTensor.py:8-31
    if (isinf(acc.x)) acc.x = 0.f;
    if (isinf(acc.y)) acc.y = 0.f;
    if (isinf(acc.z)) acc.z = 0.f;
    if (isinf(acc.w)) acc.w = 0.f;
  }
  out[idx] = acc;
  if (out_mask && ch == 0) out_mask[rest] = cnt > 0;
}

// Warp-cooperative variant for dense % 128 == 0 (all 32 lanes of a warp share one output row):
// the mask bytes of 32 reduced positions are fetched with ONE load per lane and turned into a
// warp-uniform bit set, so the value loads no longer wait for a mask load each and 8 of them are
// in flight per lane.  Same ascending order of the reduction as the per-thread kernel.
// SPLIT (few output rows, long reduced extent, e.g. pooling both tuple dims of a graph): one
// thread-block CLUSTER of kPoolCluster CTAs x 8 warps per output row; warp s of the cluster takes
// the 32-position chunks s, s + 64, ...; partial results are combined in warp order inside each CTA
// and then in CTA-rank order through distributed shared memory (deterministic, no workspace).
constexpr int kPoolCluster = 8;

template <int AGGR, bool SPLIT>
__global__ void __launch_bounds__(256)
masked_pool_warp_kernel(const float4* __restrict__ data, const unsigned char* __restrict__ mask,
                        PoolView v, float4* __restrict__ out, unsigned char* __restrict__ out_mask,
                        long long warps_total) {
  const long long w = SPLIT ? (long long)(blockIdx.x / kPoolCluster)
                          : ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= warps_total) return;
  const int lane = threadIdx.x & 31;
  const int wid = (int)(threadIdx.x >> 5);
  const int crank = SPLIT ? (int)(blockIdx.x % kPoolCluster) : 0;     // == rank in the cluster (1-D grid)
  const int sub = SPLIT ? crank * 8 + wid : 0;
  constexpr int kStep = SPLIT ? 256 * kPoolCluster : 32;
  const int cg = v.c4 >> 5;
  const int ch = (int)(w % cg) * 32 + lane;
  const long long rest = w / cg;
  const int in = (int)(rest % v.inner);
  const long long o = rest / v.inner;
  const float init = AGGR == PGH_MAX ? -INFINITY : AGGR == PGH_MIN ? INFINITY : 0.f;
  float4 acc = make_float4(init, init, init, init);
  int cnt = 0;
  const long long base = o * v.red * v.inner + in;
  const unsigned char* mp = mask + base;
  const float4* dp = data + base * v.c4 + ch;
  const long long pstep = v.inner, dstep = (long long)v.inner * v.c4;
  auto take = [&](const float4& x) {
    if (AGGR == PGH_MAX) acc = make_float4(fmaxf(acc.x, x.x), fmaxf(acc.y, x.y), fmaxf(acc.z, x.z), fmaxf(acc.w, x.w));
    else if (AGGR == PGH_MIN) acc = make_float4(fminf(acc.x, x.x), fminf(acc.y, x.y), fminf(acc.z, x.z), fminf(acc.w, x.w));
    else acc = make_float4(acc.x + x.x, acc.y + x.y, acc.z + x.z, acc.w + x.w);
  };
  for (int rc = sub * 32; rc < v.red; rc += kStep) {
    const unsigned char m = rc + lane < v.red ? __ldg(mp + (rc + lane) * pstep) : (unsigned char)0;
    unsigned bits = __ballot_sync(0xffffffffu, m != 0);
    cnt += __popc(bits);
    const float4* dq = dp + rc * dstep;
    while (bits) {
      float4 x[8];
      int n = 0;
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (bits) {
          const int r = __ffs(bits) - 1;
          bits &= bits - 1;
          x[u] = __ldg(dq + r * dstep);
          n = u + 1;
        }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (u < n) take(x[u]);
    }
  }
  if (SPLIT) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ float4 part[8][32];
    __shared__ int pcnt[8];
    __shared__ float4 cpart[kPoolCluster][32];   // used in the cluster's rank-0 CTA
    __shared__ int ccnt[kPoolCluster];
    part[wid][lane] = acc;
    if (lane == 0) pcnt[wid] = cnt;
    __syncthreads();
    if (wid == 0) {
      acc = part[0][lane];
      cnt = pcnt[0];
#pragma unroll
      for (int q = 1; q < 8; ++q) { take(part[q][lane]); cnt += pcnt[q]; }
      cluster.map_shared_rank(&cpart[0][0], 0)[crank * 32 + lane] = acc;
      if (lane == 0) cluster.map_shared_rank(&ccnt[0], 0)[crank] = cnt;
    }
    cluster.sync();
    if (crank != 0 || wid != 0) return;
    acc = cpart[0][lane];
    cnt = ccnt[0];
#pragma unroll
    for (int q = 1; q < kPoolCluster; ++q) { take(cpart[q][lane]); cnt += ccnt[q]; }
  }
  if (cnt == 0) acc = make_float4(0.f, 0.f, 0.f, 0.f);
  else if (AGGR == PGH_MEAN) {
    const float n = (float)cnt;
    acc = make_float4(acc.x / n, acc.y / n, acc.z / n, acc.w / n);
  }
  if (AGGR == PGH_MAX || AGGR == PGH_MIN) {
    if (isinf(acc.x)) acc.x = 0.f;
    if (isinf(acc.y)) acc.y = 0.f;
    if (isinf(acc.z)) acc.z = 0.f;
    if (isinf(acc.w)) acc.w = 0.f;
  }
  out[rest * v.c4 + ch] = acc;
  if (out_mask && ch == 0) out_mask[rest] = cnt > 0;
}

// max / min backward: the tie count of one channel, or -1 once a valid entry is the infinite
// extreme (+inf for max, -inf for min).  The forward replaced that inf by 0 (filterinf), and like
// the reference's masked_fill the replaced output passes no gradient, not even to valid zeros.
// The -1 is sticky under pool_cnt_add, the combine of partial counts; weights need a count > 0.
__device__ __forceinline__ int pool_tie(int c, float x, float ov, float pole) {
  return (c < 0 || x == pole) ? -1 : c + (x == ov);
}
__device__ __forceinline__ int pool_cnt_add(int a, int b) { return (a < 0 || b < 0) ? -1 : a + b; }

// Backward, warp-cooperative (dense % 128 == 0): mask bits by ballot, stores never wait for a
// mask load; the tie / valid counts of mean, max and min come from the same bit sets.
template <int AGGR, bool SPLIT>
__global__ void __launch_bounds__(256)
masked_pool_bwd_warp_kernel(const float4* __restrict__ data, const unsigned char* __restrict__ mask,
                            const float4* __restrict__ outp, const float4* __restrict__ g_out,
                            PoolView v, float4* __restrict__ g_data, long long warps_total) {
  const long long w = SPLIT ? (long long)(blockIdx.x / kPoolCluster)
                          : ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= warps_total) return;
  const int lane = threadIdx.x & 31;
  const int wid = (int)(threadIdx.x >> 5);
  const int crank = SPLIT ? (int)(blockIdx.x % kPoolCluster) : 0;     // == rank in the cluster (1-D grid)
  const int sub = SPLIT ? crank * 8 + wid : 0;
  constexpr int kStep = SPLIT ? 256 * kPoolCluster : 32;
  const int cg = v.c4 >> 5;
  const int ch = (int)(w % cg) * 32 + lane;
  const long long rest = w / cg;
  const int in = (int)(rest % v.inner);
  const long long o = rest / v.inner;
  const long long base = o * v.red * v.inner + in;
  const unsigned char* mp = mask + base;
  const float4* dp = data + base * v.c4 + ch;
  float4* gp = g_data + base * v.c4 + ch;
  const long long pstep = v.inner, dstep = (long long)v.inner * v.c4;
  const float4 g = g_out[rest * v.c4 + ch];
  constexpr bool kExt = (AGGR == PGH_MAX || AGGR == PGH_MIN);
  constexpr float kPole = AGGR == PGH_MAX ? INFINITY : -INFINITY;
  const float4 ov = kExt ? outp[rest * v.c4 + ch] : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 wgt = g;
  if (AGGR != PGH_SUM) {
    int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    for (int rc = sub * 32; rc < v.red; rc += kStep) {
      const unsigned char m = rc + lane < v.red ? __ldg(mp + (rc + lane) * pstep) : (unsigned char)0;
      unsigned bits = __ballot_sync(0xffffffffu, m != 0);
      if (!kExt) { c0 += __popc(bits); continue; }
      const float4* dq = dp + rc * dstep;
      while (bits) {
        float4 x[8];
        int n = 0;
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (bits) {
            const int r = __ffs(bits) - 1;
            bits &= bits - 1;
            x[u] = __ldg(dq + r * dstep);
            n = u + 1;
          }
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (u < n) {
            c0 = pool_tie(c0, x[u].x, ov.x, kPole); c1 = pool_tie(c1, x[u].y, ov.y, kPole);
            c2 = pool_tie(c2, x[u].z, ov.z, kPole); c3 = pool_tie(c3, x[u].w, ov.w, kPole);
          }
      }
    }
    if (!kExt) c1 = c2 = c3 = c0;
    if (SPLIT) {
      namespace cg = cooperative_groups;
      cg::cluster_group cluster = cg::this_cluster();
      __shared__ int4 pc[8][32];
      __shared__ int4 cpc[32];                    // this CTA's counts, read by the whole cluster
      pc[wid][lane] = make_int4(c0, c1, c2, c3);
      __syncthreads();
      if (wid == 0) {
        int4 t = make_int4(0, 0, 0, 0);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int4 u = pc[q][lane];
          t = make_int4(pool_cnt_add(t.x, u.x), pool_cnt_add(t.y, u.y), pool_cnt_add(t.z, u.z), pool_cnt_add(t.w, u.w));
        }
        cpc[lane] = t;
      }
      cluster.sync();
      c0 = c1 = c2 = c3 = 0;
#pragma unroll
      for (int q = 0; q < kPoolCluster; ++q) {
        const int4 t = cluster.map_shared_rank(&cpc[0], q)[lane];
        c0 = pool_cnt_add(c0, t.x); c1 = pool_cnt_add(c1, t.y);
        c2 = pool_cnt_add(c2, t.z); c3 = pool_cnt_add(c3, t.w);
      }
      cluster.sync();                              // peers may exit only after everyone has read
    }
    wgt = make_float4(c0 > 0 ? g.x / (float)c0 : 0.f, c1 > 0 ? g.y / (float)c1 : 0.f,
                      c2 > 0 ? g.z / (float)c2 : 0.f, c3 > 0 ? g.w / (float)c3 : 0.f);
  }
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int rc = sub * 32; rc < v.red; rc += kStep) {
    const unsigned char m = rc + lane < v.red ? __ldg(mp + (rc + lane) * pstep) : (unsigned char)0;
    const unsigned bits = __ballot_sync(0xffffffffu, m != 0);
    const int nr = min(32, v.red - rc);
    const float4* dq = dp + rc * dstep;
    float4* gq = gp + rc * dstep;
    if (kExt) {
      for (int r0 = 0; r0 < nr; r0 += 8) {
        float4 x[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (r0 + u < nr && ((bits >> (r0 + u)) & 1u)) x[u] = __ldg(dq + (r0 + u) * dstep);
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (r0 + u < nr) {
            float4 val = zero;
            if ((bits >> (r0 + u)) & 1u)
              val = make_float4(x[u].x == ov.x ? wgt.x : 0.f, x[u].y == ov.y ? wgt.y : 0.f,
                                x[u].z == ov.z ? wgt.z : 0.f, x[u].w == ov.w ? wgt.w : 0.f);
            gq[(r0 + u) * dstep] = val;
          }
      }
    } else {
      for (int r = 0; r < nr; ++r) gq[r * dstep] = ((bits >> r) & 1u) ? wgt : zero;
    }
  }
}

template <int AGGR>
__global__ void masked_pool_bwd_kernel(const float4* __restrict__ data,
                                       const unsigned char* __restrict__ mask,
                                       const float4* __restrict__ outp,
                                       const float4* __restrict__ g_out, PoolView v,
                                       float4* __restrict__ g_data, long long total) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int ch = (int)(idx % v.c4);
  const long long rest = idx / v.c4;
  const int in = (int)(rest % v.inner);
  const long long o = rest / v.inner;
  const long long base = o * v.red * v.inner + in;
  const unsigned char* mp = mask + base;
  const float4* dp = data + base * v.c4 + ch;
  float4* gp = g_data + base * v.c4 + ch;
  const long long pstep = v.inner, dstep = (long long)v.inner * v.c4;
  const float4 g = g_out[idx];
  constexpr bool kExt = (AGGR == PGH_MAX || AGGR == PGH_MIN);
  constexpr float kPole = AGGR == PGH_MAX ? INFINITY : -INFINITY;
  const float4 ov = kExt ? outp[idx] : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 w = g;
  if (AGGR != PGH_SUM) {
    // mean: 1/#valid ; max/min: 1/#ties per channel (torch.amax backward splits evenly), none
    // where a valid entry is the infinite extreme (pool_tie)
    int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    for (int r = 0; r < v.red; ++r) {
      if (!__ldg(mp + r * pstep)) continue;
      if (kExt) {
        const float4 x = __ldg(dp + r * dstep);
        c0 = pool_tie(c0, x.x, ov.x, kPole); c1 = pool_tie(c1, x.y, ov.y, kPole);
        c2 = pool_tie(c2, x.z, ov.z, kPole); c3 = pool_tie(c3, x.w, ov.w, kPole);
      } else {
        ++c0;
      }
    }
    if (!kExt) c1 = c2 = c3 = c0;
    w = make_float4(c0 > 0 ? g.x / (float)c0 : 0.f, c1 > 0 ? g.y / (float)c1 : 0.f,
                    c2 > 0 ? g.z / (float)c2 : 0.f, c3 > 0 ? g.w / (float)c3 : 0.f);
  }
  for (int r = 0; r < v.red; ++r) {
    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
    if (__ldg(mp + r * pstep)) {
      if (kExt) {
        const float4 x = __ldg(dp + r * dstep);
        val = make_float4(x.x == ov.x ? w.x : 0.f, x.y == ov.y ? w.y : 0.f,
                          x.z == ov.z ? w.z : 0.f, x.w == ov.w ? w.w : 0.f);
      } else {
        val = w;
      }
    }
    gp[r * dstep] = val;
  }
}

// SPLIT kernels: one cluster of kPoolCluster CTAs per output row
template <typename... KArgs, typename... Args>
static void pool_cluster_launch(void (*kern)(KArgs...), long long rows, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(rows * kPoolCluster));
  cfg.blockDim = dim3(256);
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = kPoolCluster;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

static int pool_view(int64_t b, int64_t n1, int64_t n2, int64_t dense, int red_dims, PoolView& v) {
  if (dense % 4) return arg_error("masked_pool: dense % 4 != 0");
  v.c4 = (int)(dense / 4);
  if (red_dims == 1) { v.outer = b; v.red = (int)n1; v.inner = (int)n2; }
  else if (red_dims == 2) { v.outer = b * n1; v.red = (int)n2; v.inner = 1; }
  else if (red_dims == 3) { v.outer = b; v.red = (int)(n1 * n2); v.inner = 1; }
  else return arg_error("masked_pool: red_dims");
  return 0;
}

__global__ void masked_fill_kernel(const float* __restrict__ data,
                                   const unsigned char* __restrict__ mask, long long rows,
                                   int dense, float value, float* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * dense) return;
  out[idx] = mask[idx / dense] ? data[idx] : value;
}

// dense % 4 == 0, 16-byte aligned: 128 bits per thread, masked-out rows are not read
__global__ void masked_fill4_kernel(const float4* __restrict__ data,
                                    const unsigned char* __restrict__ mask, long long total4,
                                    int c4, float value, float4* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total4) return;
  out[idx] = __ldg(mask + idx / c4) ? __ldg(data + idx) : make_float4(value, value, value, value);
}

int mamamm_tc_launch(const float* A, int trans_a, const float* B, int trans_b,
                     const unsigned char* mask, const int* ext, int64_t b, int64_t n_i,
                     int64_t n_j, int64_t n_k, int64_t dense, int pipelined, float* out,
                     cudaStream_t s);

// ext[b] = (1 + last row with a valid entry, 1 + last column with a valid entry) of a
// (b, n1, n2) mask; one CTA per graph
__global__ void mask_extents_kernel(const unsigned char* __restrict__ mask, int n1, int n2,
                                    int* __restrict__ ext) {
  __shared__ int rmax, cmax;
  if (threadIdx.x == 0) { rmax = 0; cmax = 0; }
  __syncthreads();
  const unsigned char* m = mask + (size_t)blockIdx.x * n1 * n2;
  int r = 0, c = 0;
  for (int p = threadIdx.x; p < n1 * n2; p += blockDim.x)
    if (m[p]) { r = max(r, p / n2 + 1); c = max(c, p % n2 + 1); }
  atomicMax(&rmax, r);
  atomicMax(&cmax, c);
  __syncthreads();
  if (threadIdx.x == 0) { ext[2 * blockIdx.x] = rmax; ext[2 * blockIdx.x + 1] = cmax; }
}

}  // namespace pgh

using namespace pgh;

extern "C" int pgh_mask_extents(const uint8_t* mask, int64_t b, int64_t n1, int64_t n2,
                                int32_t* ext, void* stream) {
  if (!mask || !ext) return arg_error("mask_extents: null pointer");
  if (b <= 0) return 0;
  mask_extents_kernel<<<(unsigned)b, 256, 0, as_stream(stream)>>>(mask, (int)n1, (int)n2, ext);
  return check_launch("mask_extents");
}

namespace pgh {
int mamamm_smem_launch(const float* A, int trans_a, const float* B, int trans_b,
                       const unsigned char* mask, const int* ext, const int* order, int64_t b,
                       int64_t n_i, int64_t n_j, int64_t n_k, int64_t dense, float* out, cudaStream_t s);
}

extern "C" int pgh_mamamm_f32(const float* A, int trans_a, const float* B, int trans_b,
                              const uint8_t* mask, const int32_t* ext, const int32_t* order,
                              int64_t b, int64_t n_i, int64_t n_j, int64_t n_k, int64_t dense,
                              int algo, float* out, void* stream) {
  if (!A || !B || !mask || !out) return arg_error("mamamm: null pointer");
  if (b < 0 || n_i <= 0 || n_j <= 0 || n_k <= 0 || dense <= 0) return arg_error("mamamm: sizes");
  if (b == 0) return 0;
  cudaStream_t s = as_stream(stream);
  // 4 = exact fp32 from a TMA-fed shared-memory ring (csrc/mamamm_smem.cu); shapes it does not
  // take (dense % 16, more than 512 columns, a stage that does not fit twice) run on algo 0
  if (algo == 4) {
    const int rc = mamamm_smem_launch(A, trans_a, B, trans_b, mask, ext, order, b, n_i, n_j, n_k, dense, out, s);
    if (rc >= 0) return rc;
    algo = 0;
  }
  // 1 = tcgen05, one CTA per (graph, slab); 2 = tcgen05, persistent warp-specialised pipeline
  // (falls back to 1 when two tile stages do not fit in shared memory)
  if (algo == 1 || algo == 2)
    return mamamm_tc_launch(A, trans_a, B, trans_b, mask, ext, b, n_i, n_j, n_k, dense, algo == 2,
                            out, s);
  if (algo != 0) return arg_error("mamamm: algo");
  // A' (b, n_i, n_j): stored (b, n_i, n_j) or, transposed, (b, n_j, n_i)
  const long long sAi = trans_a ? 1 : n_j, sAj = trans_a ? n_i : 1;
  const long long sBj = trans_b ? 1 : n_k, sBk = trans_b ? n_j : 1;
  dim3 grid((unsigned)b, (unsigned)((dense + 31) / 32));
  mamamm_simt_kernel<<<grid, 256, 0, s>>>(A, sAi, sAj, B, sBj, sBk, mask, ext, (int)n_i,
                                          (int)n_j, (int)n_k, (int)dense, out);
  return check_launch("mamamm_simt");
}

extern "C" int pgh_masked_pool_f32(const float* data, const uint8_t* mask, int64_t b, int64_t n1,
                                   int64_t n2, int64_t dense, int red_dims, int aggr, float* out,
                                   uint8_t* out_mask, void* stream) {
  if (!data || !mask || !out) return arg_error("masked_pool: null pointer");
  PoolView v;
  if (int e = pool_view(b, n1, n2, dense, red_dims, v)) return e;
  if ((reinterpret_cast<uintptr_t>(data) | reinterpret_cast<uintptr_t>(out)) & 15)
    return arg_error("masked_pool: tensors must be 16-byte aligned");
  const long long total = v.outer * v.inner * v.c4;
  if (total <= 0) return 0;
  cudaStream_t s = as_stream(stream);
  const unsigned nb = blocks_for(total, 256);
  const bool warp_path = v.c4 % 32 == 0;
  const long long warps = v.outer * v.inner * (v.c4 / 32);
  const unsigned nbw = blocks_for(warps * 32, 256);
  // few output rows with a long reduced extent: one CTA of 8 warps per output row
  const bool split = v.red >= 128 && warps < 8LL * kSMs;
#define PGH_POOL(AG)                                                                                         \
  do {                                                                                                       \
    if (warp_path && split) pool_cluster_launch(masked_pool_warp_kernel<AG, true>, warps, s, (const float4*)data, mask, v, (float4*)out, out_mask, warps); \
    else if (warp_path) masked_pool_warp_kernel<AG, false><<<nbw, 256, 0, s>>>((const float4*)data, mask, v, (float4*)out, out_mask, warps); \
    else masked_pool_kernel<AG><<<nb, 256, 0, s>>>((const float4*)data, mask, v, (float4*)out, out_mask, total);   \
  } while (0)
  switch (aggr) {
    case PGH_SUM: PGH_POOL(PGH_SUM); break;
    case PGH_MEAN: PGH_POOL(PGH_MEAN); break;
    case PGH_MAX: PGH_POOL(PGH_MAX); break;
    case PGH_MIN: PGH_POOL(PGH_MIN); break;
    default: return arg_error("masked_pool: aggr");
  }
#undef PGH_POOL
  return check_launch("masked_pool");
}

extern "C" int pgh_masked_pool_bwd_f32(const float* data, const uint8_t* mask, const float* out,
                                       const float* g_out, int64_t b, int64_t n1, int64_t n2,
                                       int64_t dense, int red_dims, int aggr, float* g_data,
                                       void* stream) {
  if (!data || !mask || !g_out || !g_data) return arg_error("masked_pool_bwd: null pointer");
  if ((aggr == PGH_MAX || aggr == PGH_MIN) && !out) return arg_error("masked_pool_bwd: out needed");
  PoolView v;
  if (int e = pool_view(b, n1, n2, dense, red_dims, v)) return e;
  if ((reinterpret_cast<uintptr_t>(data) | reinterpret_cast<uintptr_t>(g_out) |
       reinterpret_cast<uintptr_t>(g_data) | reinterpret_cast<uintptr_t>(out)) & 15)
    return arg_error("masked_pool_bwd: tensors must be 16-byte aligned");
  const long long total = v.outer * v.inner * v.c4;
  if (total <= 0) return 0;
  cudaStream_t s = as_stream(stream);
  const unsigned nb = blocks_for(total, 256);
  const bool warp_path = v.c4 % 32 == 0;
  const long long warps = v.outer * v.inner * (v.c4 / 32);
  const unsigned nbw = blocks_for(warps * 32, 256);
  // few output rows with a long reduced extent: one CTA of 8 warps per output row
  const bool split = v.red >= 128 && warps < 8LL * kSMs;
#define PGH_POOLB(AG)                                                                                        \
  do {                                                                                                       \
    if (warp_path && split) pool_cluster_launch(masked_pool_bwd_warp_kernel<AG, true>, warps, s, (const float4*)data, mask, (const float4*)out, (const float4*)g_out, v, (float4*)g_data, warps); \
    else if (warp_path) masked_pool_bwd_warp_kernel<AG, false><<<nbw, 256, 0, s>>>((const float4*)data, mask, (const float4*)out, (const float4*)g_out, v, (float4*)g_data, warps); \
    else masked_pool_bwd_kernel<AG><<<nb, 256, 0, s>>>((const float4*)data, mask, (const float4*)out, (const float4*)g_out, v, (float4*)g_data, total); \
  } while (0)
  switch (aggr) {
    case PGH_SUM: PGH_POOLB(PGH_SUM); break;
    case PGH_MEAN: PGH_POOLB(PGH_MEAN); break;
    case PGH_MAX: PGH_POOLB(PGH_MAX); break;
    case PGH_MIN: PGH_POOLB(PGH_MIN); break;
    default: return arg_error("masked_pool_bwd: aggr");
  }
#undef PGH_POOLB
  return check_launch("masked_pool_bwd");
}

extern "C" int pgh_masked_fill_f32(const float* data, const uint8_t* mask, int64_t rows,
                                   int64_t dense, float value, float* out, void* stream) {
  if (!data || !mask || !out) return arg_error("masked_fill: null pointer");
  if (rows * dense <= 0) return 0;
  if (dense % 4 == 0 && !((reinterpret_cast<uintptr_t>(data) | reinterpret_cast<uintptr_t>(out)) & 15))
    masked_fill4_kernel<<<blocks_for(rows * dense / 4, 256), 256, 0, as_stream(stream)>>>(
        (const float4*)data, mask, rows * dense / 4, (int)(dense / 4), value, (float4*)out);
  else
    masked_fill_kernel<<<blocks_for(rows * dense, 256), 256, 0, as_stream(stream)>>>(
        data, mask, rows, (int)dense, value, out);
  return check_launch("masked_fill");
}
