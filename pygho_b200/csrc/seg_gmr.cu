// Fused gather - multiply - segmented reduce kernels (the sparse half of the hot path).
//
// One kernel family serves spspmm forward and backward, spmm, sparse pooling, unpooling
// and their autograd replays: every one of them is
//     out[r,:] = aggr_{t in seg(r)}  A[ia(t),:] * B[ib(t),:]
// over a CSR-by-row plan.  Design (B200): a group of `lpr` lanes owns one output row and
// 4 consecutive floats per lane (128-bit loads, a 512 B row of dense=128 is one fully
// coalesced warp request); the row's slice of the plan is loaded cooperatively (one
// coalesced request per 32 entries) and broadcast with warp shuffles, so the dependent
// chain is rowptr -> plan slice -> values with up to 4 independent value loads in flight
// per lane.  Accumulation is sequential in plan order in registers: deterministic, no
// atomics, one coalesced store per row.  HBM-bound: algorithmic bytes are
// 4*dense*(nA + nB + n_rows) + 4*(2T + n_rows + 1)  (SURVEY.md section 8d).
#include <math.h>
#include <stdarg.h>

#include "common.cuh"

namespace pgh {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

template <int VEC>
__device__ __forceinline__ void ldv(const float* __restrict__ p, float (&r)[VEC]) {
  if constexpr (VEC == 4) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p));
    r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
  } else {
    r[0] = __ldg(p);
  }
}

template <int VEC>
__device__ __forceinline__ void stv(float* __restrict__ p, const float (&r)[VEC]) {
  if constexpr (VEC == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(r[0], r[1], r[2], r[3]);
  } else {
    p[0] = r[0];
  }
}

// Geometry shared by the three kernels: which row / column slice this lane owns.
struct Lane {
  long long row;
  int sub, beg, len, maxlen;
  bool row_ok;
};

__device__ __forceinline__ Lane lane_setup(const int* __restrict__ rowptr, long long n_rows,
                                           int lpr) {
  Lane L;
  const int lane = threadIdx.x & 31;
  const int rpw = 32 / lpr;
  const long long warp = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  L.sub = lane & (lpr - 1);
  L.row = warp * rpw + lane / lpr;
  L.row_ok = L.row < n_rows;
  int beg = 0, end = 0;
  if (L.row_ok) {
    if (rowptr) {
      beg = __ldg(rowptr + L.row);
      end = __ldg(rowptr + L.row + 1);
    } else {
      beg = (int)L.row;
      end = beg + 1;
    }
  }
  L.beg = beg;
  L.len = end - beg;
  L.maxlen = (rpw == 1) ? L.len : __reduce_max_sync(0xffffffffu, L.len);
  return L;
}

constexpr int kUnroll = 4;
constexpr int kThreads = 256;

template <int AGGR, int VEC, bool HAS_B>
__global__ void __launch_bounds__(kThreads)
seg_gmr_kernel(const float* __restrict__ a_val, const int* __restrict__ c,
               const float* __restrict__ a_scale, const float* __restrict__ b_val,
               const int* __restrict__ d, const int* __restrict__ rowptr, long long n_rows,
               int dense, int lda, int ldb, int ldo, int lpr, int accum,
               float* __restrict__ out) {
  pdl_enter();
  const Lane L = lane_setup(rowptr, n_rows, lpr);
  const int colstep = lpr * VEC;
  for (int col0 = 0; col0 < dense; col0 += colstep) {
    const int col = col0 + L.sub * VEC;
    const bool col_ok = col < dense;
    float acc[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v)
      acc[v] = (AGGR == PGH_MAX) ? -INFINITY : (AGGR == PGH_MIN) ? INFINITY : 0.f;
    for (int base = 0; base < L.maxlen; base += lpr) {
      // cooperative, coalesced load of this row's slice of the plan
      const int t = L.beg + base + L.sub;
      int ci = 0, di = 0;
      float sc = 1.f;
      if (base + L.sub < L.len) {
        ci = c ? __ldg(c + t) : t;
        if (HAS_B) di = d ? __ldg(d + t) : t;
        if (a_scale) sc = __ldg(a_scale + ci);
      }
      const int chunk = min(lpr, L.maxlen - base);
#pragma unroll 1
      for (int k = 0; k < chunk; k += kUnroll) {
        int cc[kUnroll], dd[kUnroll];
        float ss[kUnroll];
        bool ok[kUnroll];
        float av[kUnroll][VEC], bv[kUnroll][VEC];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
          const int kk = k + u;
          cc[u] = __shfl_sync(0xffffffffu, ci, kk, lpr);
          dd[u] = HAS_B ? __shfl_sync(0xffffffffu, di, kk, lpr) : 0;
          ss[u] = __shfl_sync(0xffffffffu, sc, kk, lpr);
          ok[u] = col_ok && kk < chunk && (base + kk) < L.len;
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
          if (ok[u]) {
            ldv<VEC>(a_val + (size_t)cc[u] * lda + col, av[u]);
            if (HAS_B) ldv<VEC>(b_val + (size_t)dd[u] * ldb + col, bv[u]);
          }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
          if (ok[u]) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
              float m = __fmul_rn(av[u][v], ss[u]);
              if (HAS_B) m = __fmul_rn(m, bv[u][v]);
              if (AGGR == PGH_MAX) acc[v] = fmaxf(acc[v], m);
              else if (AGGR == PGH_MIN) acc[v] = fminf(acc[v], m);
              else acc[v] = __fadd_rn(acc[v], m);
            }
          }
        }
      }
    }
    if (L.row_ok && col_ok) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        if (L.len == 0) acc[v] = 0.f;
        else if (AGGR == PGH_MEAN) acc[v] = acc[v] / (float)L.len;
      }
      if (accum) {
        float old[VEC];
        ldv<VEC>(out + (size_t)L.row * ldo + col, old);
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[v] = __fadd_rn(old[v], acc[v]);
      }
      stv<VEC>(out + (size_t)L.row * ldo + col, acc);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Lean streaming kernel for dense % 128 == 0 (the benchmark width): a warp owns rw consecutive
// output rows and walks ALL their plan entries as one stream, U entries (2*U row loads of 512 B)
// in flight per lane regardless of row boundaries.  The ZINC-shaped plans have ~2 entries per
// row, so batching loads across rows is what turns a latency-bound kernel (rowptr -> plan ->
// values chain per row) into a bandwidth-bound one.  Row boundaries are warp-uniform (every lane
// handles the same entry, lanes = columns), so the flush of a finished row is a plain uniform
// branch and one coalesced 512 B store.
constexpr int kMaxRW = 16;  // rows per warp upper bound (<= 31: lane i holds rowptr[r0 + i])
// ncu on the first streaming kernel of that design (profiles/r1_seg_gmr_v3_issue.md; archived in
// profiles/probes/seg_gmr_retired_r2.cu.txt): 32.2 M warp instructions per launch = 69 per plan
// entry, i.e. 28.6 us of pure issue time on 148 SMs -- it was as much issue-bound as memory-bound
// (sm__throughput 49 %, DRAM 49 %).  This kernel keeps its work split, load batching and
// sequential reduction order, but everything the inner loop does not need is compiled out or
// hoisted:
//   * a_scale / accumulate / mean are template parameters, not run-time tests per entry;
//   * full groups of U entries run without index clamps or validity tests, the (single)
//     partial group of a warp is a separate, guarded copy of the body;
//   * the row-end test is one compare + one branch per entry; the flush keeps a running output
//     pointer and only tracks row lengths for mean / max / min (empty rows of a sum are 0 anyway);
//   * sum / mean accumulate with one FMA per component (a*b is not rounded separately; max /
//     min keep the separately rounded product because the tie-splitting backward compares it
//     bit for bit with the stored extremum).
template <int AGGR, bool HAS_B, bool HAS_SCALE, bool ACCUM, int U, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
seg_gmr_lean_kernel(const float* __restrict__ a_val, const int* __restrict__ c,
                    const float* __restrict__ a_scale, const float* __restrict__ b_val,
                    const int* __restrict__ d, const int* __restrict__ rowptr,
                    long long n_rows, int dense, int lda, int ldb, int ldo, int rw,
                    const float* __restrict__ acc_src, int lds,
                    const float* __restrict__ acc_src2, int lds2,
                    const float* __restrict__ copy_src, int ldcs, float* __restrict__ copy_dst,
                    int ldcd, float* __restrict__ out) {
  pdl_enter();
  constexpr unsigned kFull = 0xffffffffu;
  constexpr bool kLen = (AGGR != PGH_SUM);          // row lengths matter (mean, empty max/min rows)
  const int lane = threadIdx.x & 31;
  const long long warp = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  const long long r0 = warp * rw;
  if (r0 >= n_rows) return;
  const int nr = (int)min((long long)rw, n_rows - r0);
  int rp = 0;
  if (lane <= nr) rp = rowptr ? __ldg(rowptr + r0 + lane) : (int)(r0 + lane);
  const int e_beg = __shfl_sync(kFull, rp, 0);
  const int e_end = __shfl_sync(kFull, rp, nr);
  const float init = (AGGR == PGH_MAX) ? -INFINITY : (AGGR == PGH_MIN) ? INFINITY : 0.f;
  for (int col = lane * 4; col < dense; col += 128) {
    const float* __restrict__ a_col = a_val + col;
    const float* __restrict__ b_col = HAS_B ? b_val + col : nullptr;
    float* __restrict__ o_ptr = out + (size_t)r0 * ldo + col;      // row being reduced
    float4 acc = make_float4(init, init, init, init);
    int cur = 0;
    int cur_beg = e_beg;
    int cur_end = __shfl_sync(kFull, rp, 1);
#define PGH_FLUSH()                                                                     \
  do {                                                                                  \
    float4 r_ = acc;                                                                    \
    if (kLen) {                                                                         \
      const int len_ = cur_end - cur_beg;                                               \
      cur_beg = cur_end;                                                                \
      if (len_ == 0) r_ = make_float4(0.f, 0.f, 0.f, 0.f);                              \
      else if (AGGR == PGH_MEAN) {                                                      \
        const float n_ = (float)len_;                                                   \
        r_ = make_float4(acc.x / n_, acc.y / n_, acc.z / n_, acc.w / n_);               \
      }                                                                                 \
    }                                                                                   \
    if (ACCUM) {       /* out = acc_src + reduction (acc_src == out: accumulate in place) */ \
      const float4 o_ = *reinterpret_cast<const float4*>(                               \
          acc_src + (size_t)(r0 + cur) * lds + col);                                    \
      r_ = make_float4(__fadd_rn(o_.x, r_.x), __fadd_rn(o_.y, r_.y),                    \
                       __fadd_rn(o_.z, r_.z), __fadd_rn(o_.w, r_.w));                   \
      if (acc_src2) {  /* second addend (warp-uniform): out = (acc_src + red) + acc_src2 */ \
        const float4 p_ = __ldg(reinterpret_cast<const float4*>(                        \
            acc_src2 + (size_t)(r0 + cur) * lds2 + col));                               \
        r_ = make_float4(__fadd_rn(r_.x, p_.x), __fadd_rn(r_.y, p_.y),                  \
                         __fadd_rn(r_.z, p_.z), __fadd_rn(r_.w, p_.w));                 \
      }                                                                                 \
    }                                                                                   \
    *reinterpret_cast<float4*>(o_ptr) = r_;                                             \
    o_ptr += ldo;                                                                       \
    if (copy_src)      /* fused row copy: copy_dst[row] = copy_src[row] (warp-uniform) */  \
      *reinterpret_cast<float4*>(copy_dst + (size_t)(r0 + cur) * ldcd + col) =          \
          __ldg(reinterpret_cast<const float4*>(copy_src + (size_t)(r0 + cur) * ldcs + col)); \
    acc = make_float4(init, init, init, init);                                          \
    ++cur;                                                                              \
    cur_end = __shfl_sync(kFull, rp, cur + 1);      /* source lane wraps mod 32 */      \
  } while (0)
#define PGH_REDUCE(AV, BV, SS)                                                          \
  do {                                                                                  \
    float4 m_ = AV;                                                                     \
    if (HAS_SCALE)                                                                      \
      m_ = make_float4(__fmul_rn(m_.x, SS), __fmul_rn(m_.y, SS), __fmul_rn(m_.z, SS),   \
                       __fmul_rn(m_.w, SS));                                            \
    if (AGGR == PGH_MAX || AGGR == PGH_MIN) {                                           \
      if (HAS_B)                                                                        \
        m_ = make_float4(__fmul_rn(m_.x, BV.x), __fmul_rn(m_.y, BV.y),                  \
                         __fmul_rn(m_.z, BV.z), __fmul_rn(m_.w, BV.w));                 \
      if (AGGR == PGH_MAX)                                                              \
        acc = make_float4(fmaxf(acc.x, m_.x), fmaxf(acc.y, m_.y), fmaxf(acc.z, m_.z),   \
                          fmaxf(acc.w, m_.w));                                          \
      else                                                                              \
        acc = make_float4(fminf(acc.x, m_.x), fminf(acc.y, m_.y), fminf(acc.z, m_.z),   \
                          fminf(acc.w, m_.w));                                          \
    } else if (HAS_B) {                                                                 \
      acc = make_float4(__fmaf_rn(m_.x, BV.x, acc.x), __fmaf_rn(m_.y, BV.y, acc.y),     \
                        __fmaf_rn(m_.z, BV.z, acc.z), __fmaf_rn(m_.w, BV.w, acc.w));    \
    } else {                                                                            \
      acc = make_float4(__fadd_rn(acc.x, m_.x), __fadd_rn(acc.y, m_.y),                 \
                        __fadd_rn(acc.z, m_.z), __fadd_rn(acc.w, m_.w));                \
    }                                                                                   \
  } while (0)
    for (int base = e_beg; base < e_end; base += 32) {
      const int t = base + lane;
      int ci = 0, di = 0;
      float sc = 1.f;
      if (t < e_end) {
        ci = c ? __ldg(c + t) : t;
        if (HAS_B) di = d ? __ldg(d + t) : t;
        if (HAS_SCALE) sc = __ldg(a_scale + ci);
      }
      const int chunk = min(32, e_end - base);
      int k = 0;
#pragma unroll 1
      for (; k + U <= chunk; k += U) {              // full groups: no clamps, no validity tests
        float4 av[U], bv[U];
        float ss[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int cc = __shfl_sync(kFull, ci, k + u);
          av[u] = __ldg(reinterpret_cast<const float4*>(a_col + (size_t)cc * lda));
          if (HAS_B) {
            const int dd = __shfl_sync(kFull, di, k + u);
            bv[u] = __ldg(reinterpret_cast<const float4*>(b_col + (size_t)dd * ldb));
          }
          if (HAS_SCALE) ss[u] = __shfl_sync(kFull, sc, k + u);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int tt = base + k + u;
          if (tt >= cur_end) {
            do PGH_FLUSH(); while (tt >= cur_end);
          }
          PGH_REDUCE(av[u], bv[u], ss[u]);
        }
      }
      if (k < chunk) {                              // the one partial group of this warp
        const int rem = chunk - k;
        float4 av[U], bv[U];
        float ss[U];
#pragma unroll
        for (int u = 0; u < U - 1; ++u) {
          const int kk = min(k + u, chunk - 1);     // clamped: the loads stay unconditional
          const int cc = __shfl_sync(kFull, ci, kk);
          av[u] = __ldg(reinterpret_cast<const float4*>(a_col + (size_t)cc * lda));
          if (HAS_B) {
            const int dd = __shfl_sync(kFull, di, kk);
            bv[u] = __ldg(reinterpret_cast<const float4*>(b_col + (size_t)dd * ldb));
          }
          if (HAS_SCALE) ss[u] = __shfl_sync(kFull, sc, kk);
        }
#pragma unroll
        for (int u = 0; u < U - 1; ++u) {
          if (u < rem) {
            const int tt = base + k + u;
            if (tt >= cur_end) {
              do PGH_FLUSH(); while (tt >= cur_end);
            }
            PGH_REDUCE(av[u], bv[u], ss[u]);
          }
        }
      }
    }
    while (cur < nr) PGH_FLUSH();
#undef PGH_REDUCE
#undef PGH_FLUSH
  }
}

// ---------------------------------------------------------------------------------------
// Ring kernel (dense % 128 == 0, one operand: pooling, unpooling, coalesce): same work split
// and the same sequential reduction order as the lean kernel, but the value rows travel
// global -> shared memory with cp.async (LDGSTS, 16 B per lane = one 512 B row per warp
// instruction) into a per-lane FIFO of NS stages, so the number of rows in flight is bounded by
// shared memory (NS x 512 B per warp) instead of registers.  A lane only ever reads back the
// 16 B it copied itself, so the pipeline needs no barrier at all: cp.async.wait_group is per
// thread.  The plan of the NEXT 32 entries is prefetched into registers while the current 32
// are streamed, which removes the plan-load bubble of the register-staged kernel.
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() {
  asm volatile("cp.async.commit_group;\n" ::: "memory");
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];\n"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(saddr)
               : "memory");
  return v;
}

// b_val, d and ldb are not read: the argument list is that of the row-wise kernel.
template <int AGGR, int NS, int U, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
seg_gmr_ring_kernel(const float* __restrict__ a_val, const int* __restrict__ c,
                    const float* __restrict__ a_scale, const float* __restrict__ b_val,
                    const int* __restrict__ d, const int* __restrict__ rowptr,
                    long long n_rows, int dense, int lda, int ldb, int ldo, int rw, int accum,
                    float* __restrict__ out) {
  pdl_enter();
  static_assert(NS % U == 0 && 32 % U == 0 && NS <= 32, "ring geometry");
  constexpr unsigned kFull = 0xffffffffu;
  constexpr int NG = NS / U;                        // commit groups in flight
  extern __shared__ __align__(16) unsigned char ring_smem[];
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const long long warp = (long long)blockIdx.x * WARPS + wib;
  const long long r0 = warp * rw;
  if (r0 >= n_rows) return;
  const int nr = (int)min((long long)rw, n_rows - r0);
  int rp = 0;
  if (lane <= nr) rp = rowptr ? __ldg(rowptr + r0 + lane) : (int)(r0 + lane);
  const int e_beg = __shfl_sync(kFull, rp, 0);
  const int e_end = __shfl_sync(kFull, rp, nr);
  // stage s of this lane: ring + s * 512
  const uint32_t ring = (uint32_t)__cvta_generic_to_shared(ring_smem) +
                        (uint32_t)((wib * NS) * 32 + lane) * 16u;
  const float init = (AGGR == PGH_MAX) ? -INFINITY : (AGGR == PGH_MIN) ? INFINITY : 0.f;
  for (int col = lane * 4; col < dense; col += 128) {
    const float* __restrict__ a_col = a_val + col;
    float* __restrict__ o_col = out + (size_t)r0 * ldo + col;
    float4 acc = make_float4(init, init, init, init);
    int cur = 0;
    int cur_beg = e_beg;
    int cur_end = __shfl_sync(kFull, rp, 1);
#define PGH_FLUSH()                                                                     \
  do {                                                                                  \
    const int len_ = cur_end - cur_beg;                                                 \
    float4 r_ = acc;                                                                    \
    if (len_ == 0) r_ = make_float4(0.f, 0.f, 0.f, 0.f);                                \
    else if (AGGR == PGH_MEAN) {                                                        \
      const float n_ = (float)len_;                                                     \
      r_ = make_float4(acc.x / n_, acc.y / n_, acc.z / n_, acc.w / n_);                 \
    }                                                                                   \
    if (accum) {                                                                        \
      const float4 o_ = *reinterpret_cast<const float4*>(o_col + (size_t)cur * ldo);    \
      r_ = make_float4(__fadd_rn(o_.x, r_.x), __fadd_rn(o_.y, r_.y),                    \
                       __fadd_rn(o_.z, r_.z), __fadd_rn(o_.w, r_.w));                   \
    }                                                                                   \
    *reinterpret_cast<float4*>(o_col + (size_t)cur * ldo) = r_;                         \
    acc = make_float4(init, init, init, init);                                          \
    ++cur;                                                                              \
    cur_beg = cur_end;                                                                  \
    cur_end = __shfl_sync(kFull, rp, min(cur + 1, 31));                                 \
  } while (0)
    // plan registers: chunk holding the consume pointer (0) and the one after it (1)
    int ci0 = 0, ci1 = 0;
    float sc0 = 1.f, sc1 = 1.f;
#define PGH_LOAD_PLAN(BASE, CI, SC)                                                     \
  do {                                                                                  \
    const int t_ = (BASE) + lane;                                                       \
    CI = 0; SC = 1.f;                                                                   \
    if (t_ < e_end) {                                                                   \
      CI = c ? __ldg(c + t_) : t_;                                                      \
      if (a_scale) SC = __ldg(a_scale + CI);                                            \
    }                                                                                   \
  } while (0)
    PGH_LOAD_PLAN(e_beg, ci0, sc0);
    PGH_LOAD_PLAN(e_beg + 32, ci1, sc1);
    int chunk_base = e_beg;                         // first entry of chunk 0's registers
    int ti = e_beg;                                 // next entry to issue
// issue one commit group: entries ti .. ti+U-1 into the slots they map to
#define PGH_ISSUE()                                                                     \
  do {                                                                                  \
    _Pragma("unroll") for (int u_ = 0; u_ < U; ++u_) {                                  \
      const int t_ = ti + u_;                                                           \
      if (t_ < e_end) {                                                                 \
        const int off_ = t_ - chunk_base;                                               \
        const int cc_ = __shfl_sync(kFull, off_ < 32 ? ci0 : ci1, off_ & 31);           \
        const uint32_t slot_ = ring + (uint32_t)(((t_ - e_beg) % NS) * 512);            \
        cp_async16(slot_, a_col + (size_t)cc_ * lda);                                   \
      }                                                                                 \
    }                                                                                   \
    cp_async_commit();                                                                  \
    ti += U;                                                                            \
  } while (0)
#pragma unroll
    for (int g = 0; g < NG; ++g) PGH_ISSUE();
    for (int tc = e_beg; tc < e_end; tc += U) {
      cp_async_wait<NG - 1>();
      float4 av[U];
      float ss[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int t = min(tc + u, e_end - 1);
        const uint32_t slot = ring + (uint32_t)(((t - e_beg) % NS) * 512);
        av[u] = lds128(slot);
        ss[u] = a_scale ? __shfl_sync(kFull, sc0, (t - chunk_base) & 31) : 1.f;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (tc + u < e_end) {
          const int tt = tc + u;
          while (tt >= cur_end) PGH_FLUSH();
          float4 m = av[u];
          if (a_scale)
            m = make_float4(__fmul_rn(m.x, ss[u]), __fmul_rn(m.y, ss[u]), __fmul_rn(m.z, ss[u]),
                            __fmul_rn(m.w, ss[u]));
          if (AGGR == PGH_MAX)
            acc = make_float4(fmaxf(acc.x, m.x), fmaxf(acc.y, m.y), fmaxf(acc.z, m.z), fmaxf(acc.w, m.w));
          else if (AGGR == PGH_MIN)
            acc = make_float4(fminf(acc.x, m.x), fminf(acc.y, m.y), fminf(acc.z, m.z), fminf(acc.w, m.w));
          else
            acc = make_float4(__fadd_rn(acc.x, m.x), __fadd_rn(acc.y, m.y),
                              __fadd_rn(acc.z, m.z), __fadd_rn(acc.w, m.w));
        }
      }
      // the slots just read are free again: refill them (the LDS results above have been
      // consumed, so the reads completed before these copies are issued)
      PGH_ISSUE();
      if (tc + U - chunk_base >= 32) {              // consume pointer enters the next chunk
        chunk_base += 32;
        ci0 = ci1; sc0 = sc1;
        PGH_LOAD_PLAN(chunk_base + 32, ci1, sc1);
      }
    }
    cp_async_wait<0>();
    while (cur < nr) PGH_FLUSH();
#undef PGH_ISSUE
#undef PGH_LOAD_PLAN
#undef PGH_FLUSH
  }
}

// gscaled[r,:] = grad[r,:] / (#entries of seg(r) whose product equals out[r,:])
template <int VEC, bool HAS_B>
__global__ void __launch_bounds__(kThreads)
seg_tie_kernel(const float* __restrict__ a_val, const int* __restrict__ c,
               const float* __restrict__ b_val, const int* __restrict__ d,
               const int* __restrict__ rowptr, long long n_rows, int dense, int lpr,
               const float* __restrict__ outp, const float* __restrict__ grad,
               float* __restrict__ gscaled) {
  const Lane L = lane_setup(rowptr, n_rows, lpr);
  const int colstep = lpr * VEC;
  for (int col0 = 0; col0 < dense; col0 += colstep) {
    const int col = col0 + L.sub * VEC;
    const bool col_ok = col < dense;
    float ov[VEC], gv[VEC];
    int cnt[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) { ov[v] = 0.f; gv[v] = 0.f; cnt[v] = 0; }
    if (L.row_ok && col_ok) {
      ldv<VEC>(outp + (size_t)L.row * dense + col, ov);
      ldv<VEC>(grad + (size_t)L.row * dense + col, gv);
      // torch's scatter_reduce amax/amin backward also counts the (zero) initial value of
      // the output as a tie when the result is exactly 0, even with include_self=False
      // (FunctionsManual.cpp scatter_reduce_backward: N = (self == result) + ...); the
      // reference inherits that through backend/utils.py:50-55, so it is reproduced here.
#pragma unroll
      for (int v = 0; v < VEC; ++v) cnt[v] = (ov[v] == 0.f) ? 1 : 0;
    }
    for (int base = 0; base < L.maxlen; base += lpr) {
      const int t = L.beg + base + L.sub;
      int ci = 0, di = 0;
      if (base + L.sub < L.len) {
        ci = c ? __ldg(c + t) : t;
        if (HAS_B) di = d ? __ldg(d + t) : t;
      }
      const int chunk = min(lpr, L.maxlen - base);
#pragma unroll 1
      for (int k = 0; k < chunk; ++k) {
        const int cc = __shfl_sync(0xffffffffu, ci, k, lpr);
        const int dd = HAS_B ? __shfl_sync(0xffffffffu, di, k, lpr) : 0;
        if (col_ok && (base + k) < L.len) {
          float av[VEC], bv[VEC];
          ldv<VEC>(a_val + (size_t)cc * dense + col, av);
          if (HAS_B) ldv<VEC>(b_val + (size_t)dd * dense + col, bv);
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            const float m = HAS_B ? __fmul_rn(av[v], bv[v]) : av[v];
            cnt[v] += (m == ov[v]) ? 1 : 0;
          }
        }
      }
    }
    if (L.row_ok && col_ok) {
      float r[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) r[v] = cnt[v] > 0 ? gv[v] / (float)cnt[v] : 0.f;
      stv<VEC>(gscaled + (size_t)L.row * dense + col, r);
    }
  }
}

// g_self[p,:] = sum_{t in seg(p)} [self[p,:]*O(t) == out[row(t),:]] * gscaled[row(t),:] * O(t)
template <int VEC, bool HAS_O>
__global__ void __launch_bounds__(kThreads)
seg_select_bwd_kernel(const float* __restrict__ self_val, const float* __restrict__ other_val,
                      const int* __restrict__ other_idx, const int* __restrict__ row_idx,
                      const int* __restrict__ rowptr, long long n_rows, int dense, int lpr,
                      const float* __restrict__ outp, const float* __restrict__ gscaled,
                      float* __restrict__ g_self) {
  const Lane L = lane_setup(rowptr, n_rows, lpr);
  const int colstep = lpr * VEC;
  for (int col0 = 0; col0 < dense; col0 += colstep) {
    const int col = col0 + L.sub * VEC;
    const bool col_ok = col < dense;
    float sv[VEC], acc[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) { sv[v] = 0.f; acc[v] = 0.f; }
    if (L.row_ok && col_ok) ldv<VEC>(self_val + (size_t)L.row * dense + col, sv);
    for (int base = 0; base < L.maxlen; base += lpr) {
      const int t = L.beg + base + L.sub;
      int ri = 0, oi = 0;
      if (base + L.sub < L.len) {
        ri = row_idx ? __ldg(row_idx + t) : t;
        if (HAS_O) oi = other_idx ? __ldg(other_idx + t) : t;
      }
      const int chunk = min(lpr, L.maxlen - base);
#pragma unroll 1
      for (int k = 0; k < chunk; ++k) {
        const int rr = __shfl_sync(0xffffffffu, ri, k, lpr);
        const int oo = HAS_O ? __shfl_sync(0xffffffffu, oi, k, lpr) : 0;
        if (col_ok && (base + k) < L.len) {
          float ov[VEC], gv[VEC], xv[VEC];
          ldv<VEC>(outp + (size_t)rr * dense + col, ov);
          ldv<VEC>(gscaled + (size_t)rr * dense + col, gv);
          if (HAS_O) ldv<VEC>(other_val + (size_t)oo * dense + col, xv);
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            const float m = HAS_O ? __fmul_rn(sv[v], xv[v]) : sv[v];
            const float w = HAS_O ? __fmul_rn(gv[v], xv[v]) : gv[v];
            acc[v] = __fadd_rn(acc[v], (m == ov[v]) ? w : 0.f);
          }
        }
      }
    }
    if (L.row_ok && col_ok) stv<VEC>(g_self + (size_t)L.row * dense + col, acc);
  }
}

__global__ void inv_count_kernel(const int* __restrict__ rowptr, long long n_rows,
                                 float* __restrict__ inv) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n_rows) {
    const int n = __ldg(rowptr + r + 1) - __ldg(rowptr + r);
    inv[r] = 1.f / (float)max(n, 1);
  }
}

template <int AGGR>
__global__ void seg_reduce_i64_kernel(const long long* __restrict__ val,
                                      const int* __restrict__ perm,
                                      const int* __restrict__ rowptr, long long n_rows,
                                      int dense, long long* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows * dense) return;
  const long long r = i / dense;
  const int col = (int)(i % dense);
  const int beg = rowptr[r], end = rowptr[r + 1];
  long long acc = 0;
  for (int t = beg; t < end; ++t) {
    const long long x = val[(size_t)(perm ? perm[t] : t) * dense + col];
    if (t == beg) acc = x;
    else if (AGGR == PGH_MAX) acc = x > acc ? x : acc;
    else if (AGGR == PGH_MIN) acc = x < acc ? x : acc;
    else acc += x;
  }
  if (AGGR == PGH_MEAN && end > beg) {
    // torch integer "mean" = floor division (backend/utils.py:50-55 via scatter_reduce_)
    const long long n = end - beg;
    long long q = acc / n;
    if ((acc % n != 0) && ((acc < 0) != (n < 0))) --q;
    acc = q;
  }
  out[i] = acc;
}

struct Geometry {
  int vec, lpr;
  unsigned blocks;
};

static Geometry geometry(int64_t n_rows, int64_t dense, bool aligned) {
  Geometry g;
  g.vec = (aligned && dense % 4 == 0) ? 4 : 1;
  const int64_t units = dense / g.vec;
  int lpr = 1;
  while (lpr < 32 && lpr < units) lpr <<= 1;
  g.lpr = lpr;
  const int rows_per_block = (kThreads / 32) * (32 / lpr);
  g.blocks = blocks_for(n_rows, rows_per_block);
  return g;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }


// run-time tuning knobs (pgh_set_tuning): [2, 3, 5] fused BN kernels (fused_mlp.cu), [7] mamamm
// profiling ablations (mamamm_smem.cu), [8] programmatic dependent launch (common.cuh)
int g_tune[16] = {0, 0, 0, 0, 0, 0, 0, 0, /* [8] */ 1, 0, 0, 0, 0, 0, 0, 0};

// single operand (pooling, unpooling, coalesce): the cp.async ring kernel wins
// (profiles/probes/bench_gmr.py.txt) with 8 stages of 2 entries and 4 warps per CTA
template <int AGGR>
static void launch_ring(cudaStream_t s, const float* a_val, const int* c, const float* a_scale,
                        const int* rowptr, int64_t n_rows, int64_t n_entries, int dense, int lda,
                        int ldo, int accum, float* out) {
  constexpr int NS = 8, U = 2, WARPS = 4;
  constexpr int kEntriesPerWarp = 16;               // rows per warp: aim at this many plan entries
  constexpr int smem = WARPS * NS * 512;
  int rw = kEntriesPerWarp;
  if (n_entries > 0 && n_rows > 0) {
    const double avg = (double)n_entries / (double)n_rows;
    rw = (int)((double)kEntriesPerWarp / (avg > 0.5 ? avg : 0.5));
  }
  if (rw < 1) rw = 1;
  if (rw > 31) rw = 31;
  auto kern = seg_gmr_ring_kernel<AGGR, NS, U, WARPS>;
  static bool configured = false;
  if (!configured) {
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    configured = true;
  }
  const unsigned nb = blocks_for(n_rows, WARPS * rw);
  launch_pdl(kern, dim3(nb), dim3(WARPS * 32), smem, s, a_val, c, a_scale, nullptr, nullptr, rowptr,
             n_rows, dense, lda, 0, ldo, rw, accum, out);
}

struct LeanExtra {                       // optional fused epilogue work, all row-aligned with out
  const float* add_src = nullptr;        // out = add_src + reduction (NULL + accum: in place)
  int ld_add = 0;
  const float* add_src2 = nullptr;       // optional second addend (needs add_src or accum)
  int ld_add2 = 0;
  const float* copy_src = nullptr;       // copy_dst[row] = copy_src[row]
  int ld_copy_src = 0;
  float* copy_dst = nullptr;
  int ld_copy_dst = 0;
};

// two operands or a fused epilogue: the lean kernel (half the instructions of the first
// streaming kernel, 54 vs 61 us on the SSWL key, profiles/r1_gmr_ablate.txt) with 4 entries in
// flight at 64 registers (4 CTAs/SM), measured best for the short rows of the SSWL keys
template <int AGGR>
static void launch_lean(cudaStream_t s, const float* a_val, const int* c, const float* a_scale,
                        const float* b_val, const int* d, const int* rowptr, int64_t n_rows,
                        int64_t n_entries, int dense, int lda, int ldb, int ldo, int accum,
                        float* out, const LeanExtra& x) {
  // rows per warp: aim at ~32 plan entries per warp, at least 4 warps' worth of blocks per SM
  int rw = kMaxRW;
  if (n_entries > 0 && n_rows > 0) {
    const double avg = (double)n_entries / (double)n_rows;
    rw = (int)(32.0 / (avg > 0.5 ? avg : 0.5));
    // small problems: keep >= 4 CTAs per SM in the grid rather than long per-warp streams
    const int64_t cap = n_rows / (int64_t)(kSMs * 4 * (kThreads / 32));
    if (rw > cap) rw = (int)cap;
    if (rw < 1) rw = 1;
    if (rw > kMaxRW) rw = kMaxRW;
  }
  const unsigned nb = blocks_for(n_rows, (kThreads / 32) * rw);
  const float* acc_src = x.add_src ? x.add_src : out;
  const int lds = x.add_src ? x.ld_add : ldo;
  const bool acc = accum || x.add_src;
#define PGH_LEAN(B, S, A)                                                                      \
  launch_pdl(seg_gmr_lean_kernel<AGGR, B, S, A, 4, 4>, dim3(nb), dim3(kThreads), 0, s,         \
      a_val, c, a_scale, b_val, d, rowptr, n_rows, dense, lda, ldb, ldo, rw, acc_src, lds,     \
      x.add_src2, x.ld_add2, x.copy_src, x.ld_copy_src, x.copy_dst, x.ld_copy_dst, out)
  const int sel = (b_val ? 4 : 0) | (a_scale ? 2 : 0) | (acc ? 1 : 0);
  switch (sel) {
    case 0: PGH_LEAN(false, false, false); break;
    case 1: PGH_LEAN(false, false, true); break;
    case 2: PGH_LEAN(false, true, false); break;
    case 3: PGH_LEAN(false, true, true); break;
    case 4: PGH_LEAN(true, false, false); break;
    case 5: PGH_LEAN(true, false, true); break;
    case 6: PGH_LEAN(true, true, false); break;
    default: PGH_LEAN(true, true, true); break;
  }
#undef PGH_LEAN
}

// dense % 128 == 0 with 16-byte rows: the ring kernel for one operand, the lean kernel for two
// operands or a fused epilogue; any other width or alignment: the row-wise kernel
template <int AGGR, int VEC>
static int launch_gmr(const Geometry& g, cudaStream_t s, const float* a_val, const int* c,
                      const float* a_scale, const float* b_val, const int* d,
                      const int* rowptr, int64_t n_rows, int64_t n_entries, int dense, int lda,
                      int ldb, int ldo, int accum, float* out, const LeanExtra* extra = nullptr) {
  if (VEC == 4 && dense % 128 == 0) {
    if (b_val || extra) {
      const LeanExtra none;
      launch_lean<AGGR>(s, a_val, c, a_scale, b_val, d, rowptr, n_rows, n_entries, dense, lda, ldb,
                        ldo, accum, out, extra ? *extra : none);
    } else {
      launch_ring<AGGR>(s, a_val, c, a_scale, rowptr, n_rows, n_entries, dense, lda, ldo, accum,
                        out);
    }
    return 0;
  }
  if (extra) return arg_error("seg_gmr_fused: needs dense % 128 == 0 and 16-byte aligned rows");
  if (b_val)
    launch_pdl(seg_gmr_kernel<AGGR, VEC, true>, dim3(g.blocks), dim3(kThreads), 0, s, 
        a_val, c, a_scale, b_val, d, rowptr, n_rows, dense, lda, ldb, ldo, g.lpr, accum, out);
  else
    launch_pdl(seg_gmr_kernel<AGGR, VEC, false>, dim3(g.blocks), dim3(kThreads), 0, s, 
        a_val, c, a_scale, b_val, d, rowptr, n_rows, dense, lda, ldb, ldo, g.lpr, accum, out);
  return 0;
}

}  // namespace pgh

using namespace pgh;

extern "C" const char* pgh_last_error(void) { return pgh::g_err; }
extern "C" int pgh_abi_version(void) { return 4; }

extern "C" int pgh_set_tuning(int key, int value) {
  if (!(key == 2 || key == 3 || key == 5 || key == 7 || key == 8)) return arg_error("set_tuning: key");
  pgh::g_tune[key] = value;
  return 0;
}

extern "C" int pgh_device_info(int32_t* out5) {
  int dev = 0;
  PGH_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp p;
  PGH_CUDA(cudaGetDeviceProperties(&p, dev));
  out5[0] = dev;
  out5[1] = p.multiProcessorCount;
  out5[2] = (int32_t)(p.l2CacheSize >> 10);  // KiB
  out5[3] = p.major;
  out5[4] = p.minor;
  return 0;
}

extern "C" int pgh_seg_gmr_ld_f32(const float* a_val, int64_t lda, const int32_t* c,
                                  const float* a_scale, const float* b_val, int64_t ldb,
                                  const int32_t* d, const int32_t* rowptr, int64_t n_rows,
                                  int64_t n_entries, int64_t dense, int aggr, int accumulate,
                                  float* out, int64_t ldo, void* stream) {
  if (!a_val || !out) return arg_error("seg_gmr: a_val and out are required");
  if (n_rows < 0 || dense <= 0 || dense > (1 << 20)) return arg_error("seg_gmr: sizes");
  if (aggr < 0 || aggr > 3) return arg_error("seg_gmr: aggr");
  if (accumulate && aggr > 1) return arg_error("seg_gmr: accumulate needs sum or mean");
  if (lda < dense || ldo < dense || (b_val && ldb < dense) || lda > 0x7fffffff ||
      ldb > 0x7fffffff || ldo > 0x7fffffff)
    return arg_error("seg_gmr: leading dimensions");
  if (n_rows == 0) return 0;
  const bool al = aligned16(a_val) && aligned16(out) && (!b_val || aligned16(b_val)) &&
                  lda % 4 == 0 && ldo % 4 == 0 && (!b_val || ldb % 4 == 0);
  const Geometry g = geometry(n_rows, dense, al);
  cudaStream_t s = as_stream(stream);
  if (!rowptr) n_entries = n_rows;
  const int la = (int)lda, lb = (int)(b_val ? ldb : dense), lo = (int)ldo;
#define PGH_GMR(AG)                                                                       \
  if (g.vec == 4) launch_gmr<AG, 4>(g, s, a_val, c, a_scale, b_val, d, rowptr, n_rows,   \
                                    n_entries, (int)dense, la, lb, lo, accumulate, out);  \
  else launch_gmr<AG, 1>(g, s, a_val, c, a_scale, b_val, d, rowptr, n_rows, n_entries,   \
                         (int)dense, la, lb, lo, accumulate, out)
  switch (aggr) {
    case PGH_SUM: PGH_GMR(PGH_SUM); break;
    case PGH_MEAN: PGH_GMR(PGH_MEAN); break;
    case PGH_MAX: PGH_GMR(PGH_MAX); break;
    default: PGH_GMR(PGH_MIN); break;
  }
#undef PGH_GMR
  return check_launch("seg_gmr");
}

extern "C" int pgh_seg_gmr_fused_f32(const float* a_val, int64_t lda, const int32_t* c,
                                     const float* a_scale, const float* b_val, int64_t ldb,
                                     const int32_t* d, const int32_t* rowptr, int64_t n_rows,
                                     int64_t n_entries, int64_t dense, int aggr,
                                     const float* add_src, int64_t ld_add, const float* add_src2,
                                     int64_t ld_add2, const float* copy_src,
                                     int64_t ld_copy_src, float* copy_dst, int64_t ld_copy_dst,
                                     float* out, int64_t ldo, void* stream) {
  if (!a_val || !out) return arg_error("seg_gmr_fused: a_val and out are required");
  if (n_rows < 0 || dense <= 0 || dense % 128 != 0) return arg_error("seg_gmr_fused: dense % 128");
  if (aggr < 0 || aggr > 1) return arg_error("seg_gmr_fused: sum or mean only");
  if ((copy_src == nullptr) != (copy_dst == nullptr)) return arg_error("seg_gmr_fused: copy pair");
  if (add_src2 && !add_src) return arg_error("seg_gmr_fused: add_src2 needs add_src");
  if (add_src2 && (ld_add2 < dense || ld_add2 > 0x7fffffff || ld_add2 % 4 ||
                   (reinterpret_cast<uintptr_t>(add_src2) & 15)))
    return arg_error("seg_gmr_fused: add_src2 layout");
  const int64_t lim = 0x7fffffff;
  if (lda < dense || ldo < dense || (b_val && ldb < dense) || lda > lim || ldb > lim || ldo > lim ||
      (add_src && (ld_add < dense || ld_add > lim)) ||
      (copy_src && (ld_copy_src < dense || ld_copy_dst < dense || ld_copy_src > lim ||
                    ld_copy_dst > lim)))
    return arg_error("seg_gmr_fused: leading dimensions");
  if (n_rows == 0) return 0;
  const bool al = aligned16(a_val) && aligned16(out) && (!b_val || aligned16(b_val)) &&
                  lda % 4 == 0 && ldo % 4 == 0 && (!b_val || ldb % 4 == 0) &&
                  (!add_src || (aligned16(add_src) && ld_add % 4 == 0)) &&
                  (!copy_src || (aligned16(copy_src) && aligned16(copy_dst) &&
                                 ld_copy_src % 4 == 0 && ld_copy_dst % 4 == 0));
  if (!al) return arg_error("seg_gmr_fused: rows must be 16-byte aligned");
  const Geometry g = geometry(n_rows, dense, true);
  if (!rowptr) n_entries = n_rows;
  LeanExtra x;
  x.add_src = add_src; x.ld_add = (int)ld_add;
  x.add_src2 = add_src2; x.ld_add2 = (int)ld_add2;
  x.copy_src = copy_src; x.ld_copy_src = (int)ld_copy_src;
  x.copy_dst = copy_dst; x.ld_copy_dst = (int)ld_copy_dst;
  const int la = (int)lda, lb = (int)(b_val ? ldb : dense), lo = (int)ldo;
  int rc;
  if (aggr == PGH_SUM)
    rc = launch_gmr<PGH_SUM, 4>(g, as_stream(stream), a_val, c, a_scale, b_val, d, rowptr, n_rows,
                                n_entries, (int)dense, la, lb, lo, 0, out, &x);
  else
    rc = launch_gmr<PGH_MEAN, 4>(g, as_stream(stream), a_val, c, a_scale, b_val, d, rowptr, n_rows,
                                 n_entries, (int)dense, la, lb, lo, 0, out, &x);
  if (rc) return rc;
  return check_launch("seg_gmr_fused");
}


extern "C" int pgh_seg_gmr_f32(const float* a_val, const int32_t* c, const float* a_scale,
                               const float* b_val, const int32_t* d, const int32_t* rowptr,
                               int64_t n_rows, int64_t n_entries, int64_t dense, int aggr,
                               float* out, void* stream) {
  return pgh_seg_gmr_ld_f32(a_val, dense, c, a_scale, b_val, dense, d, rowptr, n_rows, n_entries,
                            dense, aggr, 0, out, dense, stream);
}

extern "C" int pgh_seg_tie_scale_f32(const float* a_val, const int32_t* c, const float* b_val,
                                     const int32_t* d, const int32_t* rowptr, int64_t n_rows,
                                     int64_t dense, const float* out, const float* grad,
                                     float* gscaled, void* stream) {
  if (!a_val || !out || !grad || !gscaled) return arg_error("seg_tie_scale: null pointer");
  if (n_rows < 0 || dense <= 0) return arg_error("seg_tie_scale: sizes");
  if (n_rows == 0) return 0;
  const bool al = aligned16(a_val) && aligned16(out) && aligned16(grad) && aligned16(gscaled) &&
                  (!b_val || aligned16(b_val));
  const Geometry g = geometry(n_rows, dense, al);
  cudaStream_t s = as_stream(stream);
  const int dn = (int)dense;
  if (g.vec == 4) {
    if (b_val) seg_tie_kernel<4, true><<<g.blocks, kThreads, 0, s>>>(a_val, c, b_val, d, rowptr, n_rows, dn, g.lpr, out, grad, gscaled);
    else seg_tie_kernel<4, false><<<g.blocks, kThreads, 0, s>>>(a_val, c, b_val, d, rowptr, n_rows, dn, g.lpr, out, grad, gscaled);
  } else {
    if (b_val) seg_tie_kernel<1, true><<<g.blocks, kThreads, 0, s>>>(a_val, c, b_val, d, rowptr, n_rows, dn, g.lpr, out, grad, gscaled);
    else seg_tie_kernel<1, false><<<g.blocks, kThreads, 0, s>>>(a_val, c, b_val, d, rowptr, n_rows, dn, g.lpr, out, grad, gscaled);
  }
  return check_launch("seg_tie_scale");
}

extern "C" int pgh_seg_select_bwd_f32(const float* self_val, const float* other_val,
                                      const int32_t* other_idx, const int32_t* row_idx,
                                      const int32_t* rowptr, int64_t n_rows, int64_t dense,
                                      const float* out, const float* gscaled, float* g_self,
                                      void* stream) {
  if (!self_val || !out || !gscaled || !g_self) return arg_error("seg_select_bwd: null pointer");
  if (n_rows < 0 || dense <= 0) return arg_error("seg_select_bwd: sizes");
  if (n_rows == 0) return 0;
  const bool al = aligned16(self_val) && aligned16(out) && aligned16(gscaled) &&
                  aligned16(g_self) && (!other_val || aligned16(other_val));
  const Geometry g = geometry(n_rows, dense, al);
  cudaStream_t s = as_stream(stream);
  const int dn = (int)dense;
  if (g.vec == 4) {
    if (other_val) seg_select_bwd_kernel<4, true><<<g.blocks, kThreads, 0, s>>>(self_val, other_val, other_idx, row_idx, rowptr, n_rows, dn, g.lpr, out, gscaled, g_self);
    else seg_select_bwd_kernel<4, false><<<g.blocks, kThreads, 0, s>>>(self_val, other_val, other_idx, row_idx, rowptr, n_rows, dn, g.lpr, out, gscaled, g_self);
  } else {
    if (other_val) seg_select_bwd_kernel<1, true><<<g.blocks, kThreads, 0, s>>>(self_val, other_val, other_idx, row_idx, rowptr, n_rows, dn, g.lpr, out, gscaled, g_self);
    else seg_select_bwd_kernel<1, false><<<g.blocks, kThreads, 0, s>>>(self_val, other_val, other_idx, row_idx, rowptr, n_rows, dn, g.lpr, out, gscaled, g_self);
  }
  return check_launch("seg_select_bwd");
}

extern "C" int pgh_inv_count_f32(const int32_t* rowptr, int64_t n_rows, float* inv,
                                 void* stream) {
  if (!rowptr || !inv) return arg_error("inv_count: null pointer");
  if (n_rows <= 0) return 0;
  inv_count_kernel<<<blocks_for(n_rows, 256), 256, 0, as_stream(stream)>>>(rowptr, n_rows, inv);
  return check_launch("inv_count");
}

extern "C" int pgh_seg_reduce_i64(const int64_t* val, const int32_t* perm, const int32_t* rowptr,
                                  int64_t n_rows, int64_t dense, int aggr, int64_t* out,
                                  void* stream) {
  if (!val || !rowptr || !out) return arg_error("seg_reduce_i64: null pointer");
  if (n_rows <= 0 || dense <= 0) return 0;
  const unsigned nb = blocks_for(n_rows * dense, 256);
  cudaStream_t s = as_stream(stream);
  const long long* v = reinterpret_cast<const long long*>(val);
  long long* o = reinterpret_cast<long long*>(out);
  switch (aggr) {
    case PGH_SUM: seg_reduce_i64_kernel<PGH_SUM><<<nb, 256, 0, s>>>(v, perm, rowptr, n_rows, (int)dense, o); break;
    case PGH_MEAN: seg_reduce_i64_kernel<PGH_MEAN><<<nb, 256, 0, s>>>(v, perm, rowptr, n_rows, (int)dense, o); break;
    case PGH_MAX: seg_reduce_i64_kernel<PGH_MAX><<<nb, 256, 0, s>>>(v, perm, rowptr, n_rows, (int)dense, o); break;
    case PGH_MIN: seg_reduce_i64_kernel<PGH_MIN><<<nb, 256, 0, s>>>(v, perm, rowptr, n_rows, (int)dense, o); break;
    default: return arg_error("seg_reduce_i64: aggr");
  }
  return check_launch("seg_reduce_i64");
}
