// Linear layer with the BatchNorm statistics in its epilogue (tuplewise MLP, SURVEY.md 8f-2):
//
//   y[r, :] = x[r, :] @ W^T + b                          (reference honn/utils.py:85-142, nn.Linear)
//   mean[c], rstd[c] of y over the valid rows            (the BatchNorm1d that follows it, :46-61)
//
// in ONE pass over x and y: the reference (and round 1) re-read the whole (tuples x channels)
// output just to get its per-channel mean and variance.  Blackwell-native pipeline:
//
//   warp 0   TMA producer: cp.async.bulk.tensor 2-D boxes (32 K-elements x 128 rows, 128-byte
//            swizzle) of x and W into a 5-stage shared-memory ring, completion on mbarriers
//   warp 1   MMA issuer: one thread issues tcgen05.mma.kind::tf32 (M=128, N=128, K=8) from the
//            swizzled K-major tiles into a TMEM accumulator (2 x 128 columns, double-buffered);
//            tcgen05.commit releases ring slots and publishes finished accumulators
//   warps 4-7  epilogue: tcgen05.ld (lane = output row), + bias, 256-bit global stores, and the
//            column sums / sums of squares of the tile: a 31-shuffle transpose-reduce per 32
//            columns leaves lane l with the totals of column l, accumulated in double over all
//            tiles of the persistent CTA
//   end      per-CTA partials -> two-level ticketed combine (ticket.cuh) -> mean / rstd /
//            running statistics (or the rank-local triple for SyncBN) by the last CTA
//
// Eval mode (kEval, pgh_linear_bn_eval_f32): the same producer, MMA issuer and TMEM double
// buffer; the BatchNorm uses its running statistics, so the whole block is one epilogue
//   z[r, c] = act(acc[r, c] * s[c] + t[c]) (+ residual[r, c]),
//   s = gamma * rsqrt(running_var + eps),  t = (bias - running_mean) * s + beta
// with no statistics, no workspace and no combine.  Rows >= rows_dev get 0 (as bn_act_fwd).
//
// TF32 like the reference on a GPU (example/zinc.py:30 set_float32_matmul_precision('high')).
// HBM-bound by design: per 128-row tile 128 x K x 4 B in, 64 KB out; W stays in L2.
// Shapes: N in {128, 256, 384}, K % 32 == 0 (every large Linear of the SSWL+/NGNN/DSSGNN/PPGN/I2
// models: 128 -> 128, 384 -> 128, 384 -> 384, 256 -> 128); anything else is left to cuBLAS by the
// caller.  N = 128 * NT: the W box is loaded as NT sub-tiles of 128 rows, the accumulator is
// 128 x N (double-buffered in TMEM while 2 N <= 512 columns, single-buffered for N = 384: the
// TMA ring keeps filling during the epilogue), N = 384 is issued as a 256- and a 128-column MMA.
#include <cuda.h>

#include "common.cuh"
#include "ticket.cuh"

namespace pgh {

constexpr int kLsBM = 128, kLsBK = 32;
constexpr int kLsTileBytes = kLsBM * kLsBK * 4;            // 16 KB: 128 rows x 32 K-elements
constexpr int kLsThreads = 256;
constexpr int kLsMaxStages = 5;

template <int NT>
struct LsCfg {
  static constexpr int N = 128 * NT;
  static constexpr int kStages = NT == 1 ? 5 : 3;
  static constexpr int kStageBytes = (1 + NT) * kLsTileBytes;
  static constexpr int kAccBufs = (2 * N <= 512) ? 2 : 1;
  static constexpr int kTmemCols = NT == 1 ? 256 : 512;
  static constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + 1024;   // + alignment slack
};

__device__ __forceinline__ uint32_t ls_smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start>>4 [0,14), LBO>>4 [16,30) (=1, unused for swizzled K-major), SBO>>4 [32,46) = 1024 B
// between 8-row groups, version = 1 [46,48), layout_type = 2 (SWIZZLE_128B) [61,64)
__device__ __forceinline__ uint64_t ls_desc_sw128(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}

// kind::tf32 instruction descriptor: D=F32 [4,6)=1, A=TF32 [7,10)=2, B=TF32 [10,13)=2,
// both K-major, N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t ls_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void ls_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

// bounded wait (a lost arrival traps -> reported as a launch error instead of a hang)
__device__ __forceinline__ void ls_mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t spin = 0; spin < (1u << 14); ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity), "r"(1000000u)
        : "memory");
    if (done) return;
  }
  __trap();
}

__device__ __forceinline__ void ls_mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void ls_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void ls_tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                               int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void ls_umma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void ls_umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}

// 32 consecutive accumulator columns of this thread's TMEM lane (= output row)
__device__ __forceinline__ void ls_tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),
        "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]),
        "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]),
        "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void ls_st_global_v8(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]),
               "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}

// Sum over the 32 lanes of 32 per-lane values: afterwards lane l holds in v[0] the total of
// element l.  Recursive halving: 16 + 8 + 4 + 2 + 1 = 31 shuffles (a plain butterfly per
// element would need 160).  Fixed order -> deterministic.
__device__ __forceinline__ float ls_transpose_reduce(float (&v)[32], int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool upper = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < s; ++i) {
      const float send = upper ? v[i] : v[i + s];
      const float keep = upper ? v[i + s] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  return v[0];
}

struct LsBars {
  unsigned long long full[kLsMaxStages], empty[kLsMaxStages], tfull[2], tempty[2];
};

// eval-mode operands (unused by the training instantiation)
struct LsEvalArgs {
  const float* gamma;        // NULL: 1
  const float* beta;         // NULL: 0
  const float* residual;     // NULL: none; else (M, N) row-major, 16-byte aligned
};

// kEval = false: Linear + BatchNorm statistics (training); kEval = true: Linear + BatchNorm with
// running statistics + activation ACT (+ residual) written to y
template <int NT, bool kEval, int ACT>
__global__ void __launch_bounds__(kLsThreads, 1)
linear_stats_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                    const float* __restrict__ bias, long long M, int K, const int* __restrict__ rows_dev,
                    float* __restrict__ y, float* __restrict__ part, float* __restrict__ part2,
                    int grp, int ngroups, int* __restrict__ tickets, float eps, float momentum,
                    float* __restrict__ mean, float* __restrict__ rstd, float* __restrict__ running_mean,
                    float* __restrict__ running_var, float* __restrict__ local_out,
                    long long* __restrict__ nbt, const LsEvalArgs ev) {
  extern __shared__ unsigned char ls_smem_raw[];
  __shared__ LsBars bars;
  __shared__ uint32_t tmem_holder;
  using Cfg = LsCfg<NT>;
  constexpr int kLsBN = Cfg::N, kLsStages = Cfg::kStages, kLsStageBytes = Cfg::kStageBytes;
  constexpr int kLsTmemCols = Cfg::kTmemCols, kBufs = Cfg::kAccBufs;
  __shared__ float s_part[4][2][kLsBN];            // per epilogue warp: column sums / sums of squares
  __shared__ double s_fin[2 * kLsBN];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t ring = (ls_smem_u32(ls_smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B: 1024-B aligned
  // programmatic dependent launch (common.cuh): global memory is first touched after the
  // griddepcontrol.wait that follows the barrier set-up and the TMEM allocation
#ifdef PGH_PDL_EARLY_TRIGGER
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
  const int m_tiles = (int)((M + kLsBM - 1) / kLsBM);
  const int kblocks = K / kLsBK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kLsStages; ++s) {
      ls_mbar_init(ls_smem_u32(&bars.full[s]), 1);
      ls_mbar_init(ls_smem_u32(&bars.empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      ls_mbar_init(ls_smem_u32(&bars.tfull[a]), 1);
      ls_mbar_init(ls_smem_u32(&bars.tempty[a]), 4);     // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     ls_smem_u32(&tmem_holder)),
                 "r"(kLsTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_holder;
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const long long rows_valid = rows_dev ? min(M, (long long)max(__ldg(rows_dev), 0)) : M;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x) {
        const int row0 = tile * kLsBM;
        for (int kb = 0; kb < kblocks; ++kb) {
          ls_mbar_wait(ls_smem_u32(&bars.empty[stage]), phase ^ 1u);
          const uint32_t full = ls_smem_u32(&bars.full[stage]);
          const uint32_t dst = ring + (uint32_t)stage * kLsStageBytes;
          ls_mbar_expect_tx(full, kLsStageBytes);
          ls_tma_load_2d(dst, &map_x, full, kb * kLsBK, row0);
#pragma unroll
          for (int t = 0; t < NT; ++t)
            ls_tma_load_2d(dst + (1 + t) * kLsTileBytes, &map_w, full, kb * kLsBK, t * 128);
          if (++stage == kLsStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      const uint32_t idesc = ls_idesc_tf32(kLsBM, NT == 3 ? 256 : kLsBN);
      const uint32_t idesc_tail = ls_idesc_tf32(kLsBM, 128);          // NT == 3: columns 256..383
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x, ++it) {
        const int buf = kBufs == 2 ? (it & 1) : 0;
        const uint32_t aphase = (uint32_t)(kBufs == 2 ? (it >> 1) : it) & 1u;
        ls_mbar_wait(ls_smem_u32(&bars.tempty[buf]), aphase ^ 1u);   // epilogue drained this buffer
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t acc = tmem_base + (uint32_t)buf * kLsBN;
        for (int kb = 0; kb < kblocks; ++kb) {
          ls_mbar_wait(ls_smem_u32(&bars.full[stage]), phase);       // TMA landed this stage
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a_addr = ring + (uint32_t)stage * kLsStageBytes;
          const uint32_t b_addr = a_addr + kLsTileBytes;
#pragma unroll
          for (int k = 0; k < kLsBK / 8; ++k) {
            ls_umma_tf32(acc, ls_desc_sw128(a_addr + k * 32), ls_desc_sw128(b_addr + k * 32), idesc,
                         (uint32_t)((kb | k) != 0));
            if (NT == 3)      // W rows 256..383 = third 16 KB sub-tile, accumulator columns 256..
              ls_umma_tf32(acc + 256, ls_desc_sw128(a_addr + k * 32),
                           ls_desc_sw128(b_addr + 2 * kLsTileBytes + k * 32), idesc_tail,
                           (uint32_t)((kb | k) != 0));
          }
          ls_umma_commit(ls_smem_u32(&bars.empty[stage]));           // slot free once the MMAs retire
          if (++stage == kLsStages) { stage = 0; phase ^= 1u; }
        }
        ls_umma_commit(ls_smem_u32(&bars.tfull[buf]));               // accumulator complete
      }
    }
  } else if (kEval && warp >= 4) {
    // ===== eval epilogue: TMEM -> scale / shift -> activation (+ residual) -> global =====
    const int q = warp - 4;
    float* s_scale = s_part[0][0];                // the statistics scratch is free in eval mode
    float* s_shift = s_part[0][1];
    // running statistics / parameters are written by earlier kernels (optimizer, load_state_dict
    // copies): read after griddepcontrol.wait
    for (int c = threadIdx.x - 128; c < kLsBN; c += 128) {
      const float sc = (ev.gamma ? __ldg(ev.gamma + c) : 1.f) * rsqrtf(__ldg(running_var + c) + eps);
      s_scale[c] = sc;
      s_shift[c] = fmaf((bias ? __ldg(bias + c) : 0.f) - __ldg(running_mean + c), sc,
                        ev.beta ? __ldg(ev.beta + c) : 0.f);
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");   // the four epilogue warps only
    int it = 0;
    for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x, ++it) {
      const int buf = kBufs == 2 ? (it & 1) : 0;
      const uint32_t aphase = (uint32_t)(kBufs == 2 ? (it >> 1) : it) & 1u;
      ls_mbar_wait(ls_smem_u32(&bars.tfull[buf]), aphase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const long long row = (long long)tile * kLsBM + q * 32 + lane;
      const bool row_ok = row < M, row_valid = row < rows_valid;
      float* yrow = y + (size_t)row * kLsBN;
      const float4* rrow =
          ev.residual ? reinterpret_cast<const float4*>(ev.residual + (size_t)row * kLsBN) : nullptr;
#pragma unroll
      for (int cb = 0; cb < 4 * NT; ++cb) {
        float v[32];
        ls_tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * kLsBN + cb * 32), v);
        if (row_ok) {
          float o[32];
#pragma unroll
          for (int i = 0; i < 32; ++i)
            o[i] = row_valid ? act_fwd<ACT>(fmaf(v[i], s_scale[cb * 32 + i], s_shift[cb * 32 + i])) : 0.f;
          if (ev.residual && row_valid) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 r = __ldg(rrow + cb * 8 + i);
              o[4 * i] += r.x; o[4 * i + 1] += r.y; o[4 * i + 2] += r.z; o[4 * i + 3] += r.w;
            }
          }
#pragma unroll
          for (int i = 0; i < 32; i += 8) ls_st_global_v8(yrow + cb * 32 + i, o + i);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) ls_mbar_arrive(ls_smem_u32(&bars.tempty[buf]));
    }
  } else if (!kEval && warp >= 4) {
    // ===== epilogue: TMEM -> registers -> global, column statistics =====
    const int q = warp - 4;                       // TMEM lane quarter this warp may access
    double acc_s[4 * NT], acc_q[4 * NT];
#pragma unroll
    for (int i = 0; i < 4 * NT; ++i) acc_s[i] = acc_q[i] = 0.0;
    int it = 0;
    for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x, ++it) {
      const int buf = kBufs == 2 ? (it & 1) : 0;
      const uint32_t aphase = (uint32_t)(kBufs == 2 ? (it >> 1) : it) & 1u;
      ls_mbar_wait(ls_smem_u32(&bars.tfull[buf]), aphase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const long long row = (long long)tile * kLsBM + q * 32 + lane;
      const bool row_ok = row < M, row_valid = row < rows_valid;
      float* yrow = y + (size_t)row * kLsBN;
#pragma unroll
      for (int cb = 0; cb < 4 * NT; ++cb) {
        float v[32];
        ls_tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * kLsBN + cb * 32), v);
        if (row_ok) {
          float o[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = v[i] + (bias ? __ldg(bias + cb * 32 + i) : 0.f);
#pragma unroll
          for (int i = 0; i < 32; i += 8) ls_st_global_v8(yrow + cb * 32 + i, o + i);
        }
        float sq[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          if (!row_valid) v[i] = 0.f;             // pad / out-of-range rows: no statistics
          sq[i] = v[i] * v[i];
        }
        acc_s[cb] += (double)ls_transpose_reduce(v, lane);
        acc_q[cb] += (double)ls_transpose_reduce(sq, lane);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) ls_mbar_arrive(ls_smem_u32(&bars.tempty[buf]));
    }
#pragma unroll
    for (int cb = 0; cb < 4 * NT; ++cb) {
      s_part[q][0][cb * 32 + lane] = (float)acc_s[cb];
      s_part[q][1][cb * 32 + lane] = (float)acc_q[cb];
    }
  }

  // ===== all roles converge: per-CTA partial, ticketed combine, statistics =====
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (warp == 2)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kLsTmemCols)
                 : "memory");
  if constexpr (!kEval) {
    for (int t = threadIdx.x; t < 2 * kLsBN; t += kLsThreads) {
      const int which = t / kLsBN, c = t - which * kLsBN;
      const float tot = ((s_part[0][which][c] + s_part[1][which][c]) + s_part[2][which][c]) + s_part[3][which][c];
      part[(size_t)blockIdx.x * 2 * kLsBN + t] = tot;
    }
    if (!ticketed_combine(part, part2, 2 * kLsBN, gridDim.x, grp, ngroups, tickets, s_fin)) return;
    // statistics of (y - bias): shift = bias
    bn_finalize_stats(s_fin, kLsBN, (double)rows_valid, bias, eps, momentum, mean, rstd, running_mean,
                      running_var, local_out, nbt);
  }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// (rows x K) row-major fp32 matrix, box = 32 K-elements (128 B) x 128 rows, 128-byte swizzle;
// rows beyond the tensor are zero-filled by the TMA unit
static bool make_map(CUtensorMap* map, const float* base, int64_t rows, int64_t K) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)K * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)kLsBK, (cuuint32_t)kLsBM};
  const cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int ls_grid(int64_t M) {
  const int64_t tiles = (M + kLsBM - 1) / kLsBM;
  return (int)(tiles < kSMs ? tiles : kSMs);
}

struct LsGeom { int grid, grp, ngroups; };

static LsGeom ls_geom(int64_t M) {
  LsGeom g;
  g.grid = ls_grid(M);
  g.grp = 16;
  g.ngroups = (g.grid + g.grp - 1) / g.grp;
  return g;
}

}  // namespace pgh

using namespace pgh;

extern "C" int pgh_linear_stats_supported(int64_t M, int64_t K, int64_t N) {
  return M > 0 && (N == 128 || N == 256 || N == 384) && K >= kLsBK && K % kLsBK == 0 && K <= 4096;
}

extern "C" size_t pgh_linear_stats_ws_bytes(int64_t M) {
  if (M <= 0) return 256;
  const LsGeom g = ls_geom(M);
  constexpr int kMaxN = 384;
  return ((size_t)g.grid * 2 * kMaxN * sizeof(float) + 255) / 256 * 256 +
         (size_t)g.ngroups * 2 * kMaxN * sizeof(float) + 256;
}

template <int NT, bool kEval, int ACT>
static int ls_launch(const CUtensorMap& map_x, const CUtensorMap& map_w, const float* bias, int64_t M,
                     int64_t K, const int32_t* rows_dev, float* y, const LsGeom& g, void* ws,
                     int32_t* tickets, float eps, float momentum, float* mean, float* rstd,
                     float* running_mean, float* running_var, float* local_out, int64_t* nbt,
                     const LsEvalArgs& ev, cudaStream_t s) {
  using Cfg = LsCfg<NT>;
  static bool attr_set = false;
  if (!attr_set) {
    PGH_CUDA(cudaFuncSetAttribute(linear_stats_kernel<NT, kEval, ACT>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes));
    attr_set = true;
  }
  float* part = nullptr;
  float* part2 = nullptr;
  if (!kEval) {
    part = reinterpret_cast<float*>(ws);
    part2 = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) +
                                     ((size_t)g.grid * 2 * Cfg::N * sizeof(float) + 255) / 256 * 256);
  }
  launch_pdl(linear_stats_kernel<NT, kEval, ACT>, dim3(g.grid), dim3(kLsThreads), Cfg::kSmemBytes, s,
      map_x, map_w, bias, M, (int)K, rows_dev, y, part, part2, g.grp, g.ngroups, tickets, eps, momentum,
      mean, rstd, running_mean, running_var, local_out, reinterpret_cast<long long*>(nbt), ev);
  return check_launch(kEval ? "linear_bn_eval" : "linear_stats");
}

extern "C" int pgh_linear_stats_f32(const float* x, int64_t M, int64_t K, const float* w, int64_t N,
                                    const float* bias, const int32_t* rows_dev, float* y, float eps,
                                    float momentum, float* mean, float* rstd, float* running_mean,
                                    float* running_var, float* local_out, int64_t* num_batches_tracked,
                                    void* ws, size_t ws_bytes, int32_t* tickets, void* stream) {
  if (!x || !w || !y || !ws || !tickets || (!local_out && (!mean || !rstd)))
    return arg_error("linear_stats: null pointer");
  if (!pgh_linear_stats_supported(M, K, N)) return arg_error("linear_stats: need N in {128, 256, 384}, K % 32 == 0");
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w)) & 15)
    return arg_error("linear_stats: x and w must be 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(y) & 31) return arg_error("linear_stats: y must be 32-byte aligned");
  if (ws_bytes < pgh_linear_stats_ws_bytes(M)) return arg_error("linear_stats: workspace too small");
  CUtensorMap map_x, map_w;
  if (!make_map(&map_x, x, M, K) || !make_map(&map_w, w, N, K))
    return arg_error("linear_stats: cuTensorMapEncodeTiled failed");
  const LsGeom g = ls_geom(M);
  cudaStream_t s = as_stream(stream);
#define PGH_LS(NT_) ls_launch<NT_, false, 0>(map_x, map_w, bias, M, K, rows_dev, y, g, ws, tickets, eps, \
                                   momentum, mean, rstd, running_mean, running_var, local_out,          \
                                   num_batches_tracked, LsEvalArgs{}, s)
  if (N == 128) return PGH_LS(1);
  if (N == 256) return PGH_LS(2);
  return PGH_LS(3);
#undef PGH_LS
}

extern "C" int pgh_linear_bn_eval_f32(const float* x, int64_t M, int64_t K, const float* w, int64_t N,
                                      const float* bias, const float* gamma, const float* beta,
                                      const float* running_mean, const float* running_var, float eps,
                                      int act, const float* residual, const int32_t* rows_dev, float* z,
                                      void* stream) {
  if (!x || !w || !running_mean || !running_var || !z) return arg_error("linear_bn_eval: null pointer");
  if (!pgh_linear_stats_supported(M, K, N))
    return arg_error("linear_bn_eval: need N in {128, 256, 384}, K % 32 == 0, K <= 4096");
  if (act < 0 || act > 2) return arg_error("linear_bn_eval: act");
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w) |
       reinterpret_cast<uintptr_t>(residual)) & 15)
    return arg_error("linear_bn_eval: x, w and residual must be 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(z) & 31) return arg_error("linear_bn_eval: z must be 32-byte aligned");
  CUtensorMap map_x, map_w;
  if (!make_map(&map_x, x, M, K) || !make_map(&map_w, w, N, K))
    return arg_error("linear_bn_eval: cuTensorMapEncodeTiled failed");
  const LsGeom g = ls_geom(M);
  const LsEvalArgs ev{gamma, beta, residual};
  cudaStream_t s = as_stream(stream);
  float* rm = const_cast<float*>(running_mean);     // read only: the eval kernel writes no statistics
  float* rv = const_cast<float*>(running_var);
#define PGH_EV(NT_, A_) ls_launch<NT_, true, A_>(map_x, map_w, bias, M, K, rows_dev, z, g, nullptr, nullptr, \
                                                 eps, 0.f, nullptr, nullptr, rm, rv, nullptr, nullptr, ev, s)
#define PGH_EV_ACT(NT_) return act == 1 ? PGH_EV(NT_, 1) : act == 2 ? PGH_EV(NT_, 2) : PGH_EV(NT_, 0)
  if (N == 128) PGH_EV_ACT(1);
  if (N == 256) PGH_EV_ACT(2);
  PGH_EV_ACT(3);
#undef PGH_EV_ACT
#undef PGH_EV
}
