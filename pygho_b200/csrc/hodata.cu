// Batch preparation on the device (SURVEY.md 8f rank 1 + 3): hop-distance matrices of all
// graphs of a batch, the k-hop tuple sets built from them, and the padded dense layouts of
// the MaskedTensor path.  The reference does this on the CPU, node by node in Python
// (hodata/SpTupleSampler.py:91-126), with scipy (hodata/MaTupleSampler.py:11-31) and with
// torch indexing (hodata/MaData.py:26-212).
//
// Integer / byte work, latency- and HBM-bound; nothing here touches tensor cores.
//   graph_dist : one CTA per graph; adjacency as bit rows in shared memory (n x ceil(n/32)
//                words, <= 128 KB for n = 1024); one warp per root node runs the BFS with the
//                visited and frontier sets spread over the lanes (lane w = word w), so one BFS
//                level is |frontier| shared-memory row ORs and no global traffic at all.
//   khop_emit  : one warp per root node compacts its distance row with ballots into the
//                (i, j)-sorted tuple list at the offset given by the scanned row counts.
//   resistance : one CTA per graph (n <= 128); fp64 Gauss-Jordan inversion of the grounded
//                Laplacian in shared memory (<= 132 KiB), the only floating-point kernel here.
//   spd_dense / rd_dense / pad_rows / dense_adj : one thread per output element, coalesced.
#include "common.cuh"

namespace pgh {

constexpr int kDistThreads = 256;
constexpr unsigned kFullMask = 0xffffffffu;

__global__ void __launch_bounds__(kDistThreads)
graph_dist_kernel(const long long* __restrict__ edge_src, const long long* __restrict__ edge_dst,
                  const long long* __restrict__ node_ptr, const long long* __restrict__ edge_ptr,
                  const long long* __restrict__ sq_ptr, int cutoff, int max_nodes,
                  unsigned char* __restrict__ D, int* __restrict__ cnt) {
  extern __shared__ unsigned int adj[];               // adj[t * W + w]: bit s set <=> edge s -> t
  const int g = blockIdx.x;
  const long long n0 = node_ptr[g];
  const int n = (int)(node_ptr[g + 1] - n0);
  if (n <= 0 || n > max_nodes) return;                // host checked max_nodes; stay in bounds
  const int W = (n + 31) >> 5;
  for (int i = threadIdx.x; i < n * W; i += blockDim.x) adj[i] = 0u;
  __syncthreads();
  const long long e0 = edge_ptr[g], e1 = edge_ptr[g + 1];
  for (long long e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
    const long long s = edge_src[e] - n0, t = edge_dst[e] - n0;
    if (s >= 0 && s < n && t >= 0 && t < n)
      atomicOr(&adj[(int)t * W + (int)(s >> 5)], 1u << (int)(s & 31));
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  unsigned char* __restrict__ Dg = D + sq_ptr[g];
  for (int root = warp; root < n; root += nwarps) {
    unsigned char* __restrict__ row = Dg + (size_t)root * n;
    for (int j = lane; j < n; j += 32) row[j] = 255;
    __syncwarp();
    unsigned int visited = (lane == (root >> 5)) ? (1u << (root & 31)) : 0u;
    unsigned int frontier = visited;
    if (lane == 0) row[root] = 0;
    for (int d = 1; d <= cutoff; ++d) {
      unsigned int nxt = 0u;
      for (int s = 0; s < W; ++s) {
        unsigned int fw = __shfl_sync(kFullMask, frontier, s);
        while (fw) {                                   // warp-uniform: fw is a broadcast value
          const int u = (s << 5) + __ffs(fw) - 1;
          fw &= fw - 1;
          if (lane < W) nxt |= adj[u * W + lane];
        }
      }
      nxt &= ~visited;
      if (!__any_sync(kFullMask, nxt != 0u)) break;
      visited |= nxt;
      unsigned int w = nxt;
      while (w) {
        const int b = __ffs(w) - 1;
        w &= w - 1;
        row[(lane << 5) + b] = (unsigned char)d;
      }
      frontier = nxt;
    }
    if (cnt) {
      const int c = __reduce_add_sync(kFullMask, __popc(visited));
      if (lane == 0) cnt[n0 + root] = c;
    }
  }
}

__global__ void __launch_bounds__(256)
khop_emit_kernel(const unsigned char* __restrict__ D, const long long* __restrict__ node_ptr,
                 const long long* __restrict__ sq_ptr, const long long* __restrict__ node_graph,
                 const long long* __restrict__ rowptr, long long n_nodes, long long n_tuples,
                 long long* __restrict__ tupleid, long long* __restrict__ feat) {
  const int lane = threadIdx.x & 31;
  const long long v = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (v >= n_nodes) return;
  const long long g = node_graph[v];
  const long long n0 = node_ptr[g];
  const int n = (int)(node_ptr[g + 1] - n0);
  const unsigned char* __restrict__ row = D + sq_ptr[g] + (size_t)(v - n0) * n;
  long long pos = rowptr[v];
  for (int j0 = 0; j0 < n; j0 += 32) {
    const int j = j0 + lane;
    const int dv = j < n ? (int)row[j] : 255;
    const bool keep = dv != 255;
    const unsigned int bal = __ballot_sync(kFullMask, keep);
    if (keep) {
      const long long p = pos + __popc(bal & ((1u << lane) - 1u));
      if (p < n_tuples) {
        tupleid[p] = v;
        tupleid[n_tuples + p] = n0 + j;
        feat[p] = dv;
      }
    }
    pos += __popc(bal);
  }
}

__global__ void __launch_bounds__(256)
spd_dense_kernel(const unsigned char* __restrict__ D, const long long* __restrict__ node_ptr,
                 const long long* __restrict__ sq_ptr, long long total, int nmax, int clamp,
                 long long fill, long long* __restrict__ out, unsigned char* __restrict__ mask) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int j = (int)(idx % nmax);
  const int i = (int)((idx / nmax) % nmax);
  const long long g = idx / ((long long)nmax * nmax);
  const long long n0 = node_ptr[g];
  const int n = (int)(node_ptr[g + 1] - n0);
  const bool ok = i < n && j < n;
  long long v = fill;
  if (ok) {
    const int dv = (int)D[sq_ptr[g] + (size_t)i * n + j];
    v = dv < clamp ? dv : clamp;
  }
  out[idx] = v;
  mask[idx] = ok ? 1 : 0;
}


// I2Sampler (hodata/SpTupleSampler.py:129-174): for every directed edge (i, j) the nodes within
// `hop` of i or of j, with both distances as feature.  One warp per edge; count pass and emit
// pass share the row walk.  D must hold distances up to hop + 1 (255 beyond).
template <bool EMIT>
__global__ void __launch_bounds__(256)
i2_edge_kernel(const unsigned char* __restrict__ D, const long long* __restrict__ edge_src,
               const long long* __restrict__ edge_dst, const long long* __restrict__ node_ptr,
               const long long* __restrict__ sq_ptr, const long long* __restrict__ node_graph,
               long long n_edges, int hop, int* __restrict__ cnt,
               const long long* __restrict__ rowptr, long long n_tuples,
               long long* __restrict__ tupleid, long long* __restrict__ feat) {
  const int lane = threadIdx.x & 31;
  const long long e = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= n_edges) return;
  const long long i = edge_src[e], j = edge_dst[e];
  const long long g = node_graph[i];
  const long long n0 = node_ptr[g];
  const int n = (int)(node_ptr[g + 1] - n0);
  const unsigned char* __restrict__ ri = D + sq_ptr[g] + (size_t)(i - n0) * n;
  const unsigned char* __restrict__ rj = D + sq_ptr[g] + (size_t)(j - n0) * n;
  long long pos = EMIT ? rowptr[e] : 0;
  int total = 0;
  for (int k0 = 0; k0 < n; k0 += 32) {
    const int k = k0 + lane;
    const int di = k < n ? (int)ri[k] : 255, dj = k < n ? (int)rj[k] : 255;
    const bool keep = di <= hop || dj <= hop;
    const unsigned int bal = __ballot_sync(kFullMask, keep);
    if (EMIT) {
      if (keep) {
        const long long p = pos + __popc(bal & ((1u << lane) - 1u));
        if (p < n_tuples) {
          tupleid[p] = i;
          tupleid[n_tuples + p] = j;
          tupleid[2 * n_tuples + p] = n0 + k;
          feat[2 * p] = di < hop + 1 ? di : hop + 1;
          feat[2 * p + 1] = dj < hop + 1 ? dj : hop + 1;
        }
      }
      pos += __popc(bal);
    } else {
      total += __popc(bal);
    }
  }
  if (!EMIT && lane == 0) cnt[e] = total;
}

// rdsampler (hodata/MaTupleSampler.py:34-57): effective resistance of every node pair,
// R[i, j] = L+[i, i] + L+[j, j] - 2 L+[i, j] with L+ the pseudo-inverse of the Laplacian of the
// simple undirected graph.  One CTA per graph, all in shared memory:
//   adjacency bit set (both directions, duplicates once, no self-loops) -> degrees and connected
//   components (min-label propagation) -> M = L + sum_c (1/n_c) 1_c 1_c^T, which is SPD and has
//   M^-1 = L+ + sum_c (1/n_c) 1_c 1_c^T -> in-place Gauss-Jordan inversion of M in fp64 (no
//   pivoting: SPD) -> R from M^-1, where the 1/n_c terms cancel within a component and are
//   subtracted across components.  Every value is computed from the ordered pair (min, max), so
//   R is bit-symmetric; the diagonal is written as 0.
constexpr int kRdThreads = 256;
constexpr int kRdMaxNodes = 128;

inline size_t rd_smem_bytes(int n) {
  const int W = (n + 31) >> 5;
  return (size_t)n * (n + 1) * sizeof(double)                  // M (n x n) + pivot column
         + (size_t)n * W * sizeof(unsigned int)               // adjacency bits
         + (size_t)2 * n * sizeof(int);                        // component label, component size
}

__global__ void __launch_bounds__(kRdThreads)
resistance_kernel(const long long* __restrict__ edge_src, const long long* __restrict__ edge_dst,
                  const long long* __restrict__ node_ptr, const long long* __restrict__ edge_ptr,
                  const long long* __restrict__ sq_ptr, int max_nodes, float* __restrict__ R) {
  extern __shared__ double rd_smem[];
  const int g = blockIdx.x;
  const long long n0 = node_ptr[g];
  const int n = (int)(node_ptr[g + 1] - n0);
  if (n <= 0 || n > max_nodes) return;                // host checked max_nodes; stay in bounds
  const int W = (n + 31) >> 5;
  const int nn = n * n;
  double* M = rd_smem;                                 // M[i * n + j]
  double* col = M + nn;                                // pivot column of the current step
  unsigned int* adj = reinterpret_cast<unsigned int*>(col + n);   // adj[i * W + w]
  int* label = reinterpret_cast<int*>(adj + n * W);
  int* csize = label + n;

  for (int i = threadIdx.x; i < n * W; i += blockDim.x) adj[i] = 0u;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    label[i] = i;
    csize[i] = 0;
  }
  __syncthreads();
  const long long e0 = edge_ptr[g], e1 = edge_ptr[g + 1];
  for (long long e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
    const long long s = edge_src[e] - n0, t = edge_dst[e] - n0;
    if (s >= 0 && s < n && t >= 0 && t < n && s != t) {
      atomicOr(&adj[(int)s * W + (int)(t >> 5)], 1u << (int)(t & 31));
      atomicOr(&adj[(int)t * W + (int)(s >> 5)], 1u << (int)(s & 31));
    }
  }
  __syncthreads();

  // connected components: every node takes the smallest label of its closed neighbourhood until
  // nothing changes; the fixed point is the smallest node id of the component
  const int v = threadIdx.x;
  while (true) {
    int m = v < n ? label[v] : 0;
    if (v < n)
      for (int w = 0; w < W; ++w)
        for (unsigned int bits = adj[v * W + w]; bits; bits &= bits - 1)
          m = min(m, label[(w << 5) + __ffs(bits) - 1]);
    __syncthreads();
    const bool changed = v < n && m != label[v];
    if (changed) label[v] = m;
    if (!__syncthreads_or(changed)) break;
  }
  if (v < n) atomicAdd(&csize[label[v]], 1);
  __syncthreads();

  for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
    const int i = idx / n, j = idx - i * n;
    double x = 0.0;
    if (i == j) {
      for (int w = 0; w < W; ++w) x += (double)__popc(adj[i * W + w]);
    } else if ((adj[i * W + (j >> 5)] >> (j & 31)) & 1u) {
      x = -1.0;
    }
    if (label[i] == label[j]) x += 1.0 / (double)csize[label[i]];
    M[idx] = x;
  }
  __syncthreads();

  // in-place Gauss-Jordan, one warp per row: after step k, M holds the inverse with respect to
  // pivots 0..k.  Each element sees the same operations in the same order on every launch.
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int k = 0; k < n; ++k) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) col[i] = M[i * n + k];
    __syncthreads();
    const double piv = 1.0 / col[k];
    for (int j = threadIdx.x; j < n; j += blockDim.x) M[k * n + j] = j == k ? piv : M[k * n + j] * piv;
    __syncthreads();
    for (int i = warp; i < n; i += nwarps) {
      if (i == k) continue;
      const double f = col[i];
      for (int j = lane; j < n; j += 32)
        M[i * n + j] = j == k ? -f * piv : M[i * n + j] - f * M[k * n + j];
    }
    __syncthreads();
  }

  float* __restrict__ Rg = R + sq_ptr[g];
  for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
    const int r = idx / n, c = idx - r * n;
    const int i = min(r, c), j = max(r, c);
    float out = 0.0f;
    if (i != j) {
      double x;
      if (label[i] == label[j])
        x = M[i * n + i] + M[j * n + j] - 2.0 * M[i * n + j];
      else
        x = (M[i * n + i] - 1.0 / (double)csize[label[i]]) +
            (M[j * n + j] - 1.0 / (double)csize[label[j]]);
      out = (float)x;
    }
    Rg[idx] = out;
  }
}

__global__ void __launch_bounds__(256)
rd_dense_kernel(const float* __restrict__ R, const long long* __restrict__ node_ptr,
                const long long* __restrict__ sq_ptr, long long total, int nmax, float fill,
                float* __restrict__ out, unsigned char* __restrict__ mask) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int j = (int)(idx % nmax);
  const int i = (int)((idx / nmax) % nmax);
  const long long g = idx / ((long long)nmax * nmax);
  const int n = (int)(node_ptr[g + 1] - node_ptr[g]);
  const bool ok = i < n && j < n;
  out[idx] = ok ? R[sq_ptr[g] + (size_t)i * n + j] : fill;
  mask[idx] = ok ? 1 : 0;
}

template <typename T>
__global__ void __launch_bounds__(256)
pad_rows_kernel(const T* __restrict__ src, const long long* __restrict__ ptr, long long total,
                int nmax, int width, T fill, T* __restrict__ out, unsigned char* __restrict__ mask) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int w = (int)(idx % width);
  const int i = (int)((idx / width) % nmax);
  const long long g = idx / ((long long)width * nmax);
  const long long p0 = ptr[g];
  const bool ok = i < (int)(ptr[g + 1] - p0);
  out[idx] = ok ? src[(p0 + i) * width + w] : fill;
  if (w == 0) mask[idx / width] = ok ? 1 : 0;
}

template <typename T>
__global__ void __launch_bounds__(256)
fill_kernel(T* __restrict__ out, long long n_out, T fill, unsigned char* __restrict__ mask,
            long long n_mask) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n_out) out[idx] = fill;
  if (idx < n_mask) mask[idx] = 0;
}

template <typename T>
__global__ void __launch_bounds__(256)
dense_adj_kernel(const long long* __restrict__ edge_src, const long long* __restrict__ edge_dst,
                 const long long* __restrict__ edge_graph, const long long* __restrict__ node_ptr,
                 const T* __restrict__ attr, long long total, long long n_graphs, int nmax,
                 int width, T* __restrict__ out, unsigned char* __restrict__ mask) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int w = (int)(idx % width);
  const long long e = idx / width;
  const long long g = edge_graph[e];
  if (g < 0 || g >= n_graphs) return;
  const long long off = node_ptr ? node_ptr[g] : 0;
  const long long r = edge_src[e] - off, c = edge_dst[e] - off;
  if (r < 0 || r >= nmax || c < 0 || c >= nmax) return;
  const long long cell = (g * nmax + r) * nmax + c;
  out[cell * width + w] = attr[idx];
  if (w == 0) mask[cell] = 1;
}

}  // namespace pgh

using namespace pgh;

extern "C" int pgh_graph_dist_u8(const int64_t* edge_src, const int64_t* edge_dst,
                                 const int64_t* node_ptr, const int64_t* edge_ptr,
                                 const int64_t* sq_ptr, int64_t n_graphs, int64_t max_nodes,
                                 int cutoff, uint8_t* D, int32_t* cnt, void* stream) {
  if (n_graphs == 0) return 0;
  if (!node_ptr || !edge_ptr || !sq_ptr || !D) return arg_error("graph_dist: null pointer");
  if (n_graphs < 0 || max_nodes < 1 || max_nodes > 1024)
    return arg_error("graph_dist: graphs of 1..1024 nodes are supported");
  if (cutoff < 0 || cutoff > 254) return arg_error("graph_dist: cutoff must be in [0, 254]");
  const size_t smem = (size_t)max_nodes * ((max_nodes + 31) / 32) * sizeof(unsigned int);
  static size_t configured = 48 * 1024;
  if (smem > configured) {
    PGH_CUDA(cudaFuncSetAttribute(graph_dist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
    configured = smem;
  }
  graph_dist_kernel<<<(unsigned)n_graphs, kDistThreads, smem, as_stream(stream)>>>(
      (const long long*)edge_src, (const long long*)edge_dst, (const long long*)node_ptr,
      (const long long*)edge_ptr, (const long long*)sq_ptr, cutoff, (int)max_nodes, D, cnt);
  return check_launch("graph_dist");
}

extern "C" int pgh_khop_emit(const uint8_t* D, const int64_t* node_ptr, const int64_t* sq_ptr,
                             const int64_t* node_graph, const int64_t* rowptr, int64_t n_nodes,
                             int64_t n_tuples, int64_t* tupleid, int64_t* feat, void* stream) {
  if (n_nodes == 0 || n_tuples == 0) return 0;
  if (!D || !node_ptr || !sq_ptr || !node_graph || !rowptr || !tupleid || !feat)
    return arg_error("khop_emit: null pointer");
  khop_emit_kernel<<<blocks_for(n_nodes, 8), 256, 0, as_stream(stream)>>>(
      D, (const long long*)node_ptr, (const long long*)sq_ptr, (const long long*)node_graph,
      (const long long*)rowptr, n_nodes, n_tuples, (long long*)tupleid, (long long*)feat);
  return check_launch("khop_emit");
}


extern "C" int pgh_i2_count(const uint8_t* D, const int64_t* edge_src, const int64_t* edge_dst,
                            const int64_t* node_ptr, const int64_t* sq_ptr,
                            const int64_t* node_graph, int64_t n_edges, int hop, int32_t* cnt,
                            void* stream) {
  if (n_edges == 0) return 0;
  if (!D || !edge_src || !edge_dst || !node_ptr || !sq_ptr || !node_graph || !cnt)
    return arg_error("i2_count: null pointer");
  if (hop < 0 || hop > 253) return arg_error("i2_count: hop must be in [0, 253]");
  i2_edge_kernel<false><<<blocks_for(n_edges, 8), 256, 0, as_stream(stream)>>>(
      D, (const long long*)edge_src, (const long long*)edge_dst, (const long long*)node_ptr,
      (const long long*)sq_ptr, (const long long*)node_graph, n_edges, hop, cnt, nullptr, 0,
      nullptr, nullptr);
  return check_launch("i2_count");
}

extern "C" int pgh_i2_emit(const uint8_t* D, const int64_t* edge_src, const int64_t* edge_dst,
                           const int64_t* node_ptr, const int64_t* sq_ptr,
                           const int64_t* node_graph, const int64_t* rowptr, int64_t n_edges,
                           int64_t n_tuples, int hop, int64_t* tupleid, int64_t* feat,
                           void* stream) {
  if (n_edges == 0 || n_tuples == 0) return 0;
  if (!D || !edge_src || !edge_dst || !node_ptr || !sq_ptr || !node_graph || !rowptr || !tupleid ||
      !feat)
    return arg_error("i2_emit: null pointer");
  if (hop < 0 || hop > 253) return arg_error("i2_emit: hop must be in [0, 253]");
  i2_edge_kernel<true><<<blocks_for(n_edges, 8), 256, 0, as_stream(stream)>>>(
      D, (const long long*)edge_src, (const long long*)edge_dst, (const long long*)node_ptr,
      (const long long*)sq_ptr, (const long long*)node_graph, n_edges, hop, nullptr,
      (const long long*)rowptr, n_tuples, (long long*)tupleid, (long long*)feat);
  return check_launch("i2_emit");
}

extern "C" int pgh_spd_dense_i64(const uint8_t* D, const int64_t* node_ptr, const int64_t* sq_ptr,
                                 int64_t n_graphs, int64_t nmax, int clamp, int64_t fill,
                                 int64_t* out, uint8_t* mask, void* stream) {
  const int64_t total = n_graphs * nmax * nmax;
  if (total == 0) return 0;
  if (!D || !node_ptr || !sq_ptr || !out || !mask) return arg_error("spd_dense: null pointer");
  if (clamp < 0 || clamp > 255) return arg_error("spd_dense: clamp must be in [0, 255]");
  spd_dense_kernel<<<blocks_for(total, 256), 256, 0, as_stream(stream)>>>(
      D, (const long long*)node_ptr, (const long long*)sq_ptr, total, (int)nmax, clamp,
      (long long)fill, (long long*)out, mask);
  return check_launch("spd_dense");
}

extern "C" int pgh_resistance_f32(const int64_t* edge_src, const int64_t* edge_dst,
                                  const int64_t* node_ptr, const int64_t* edge_ptr,
                                  const int64_t* sq_ptr, int64_t n_graphs, int64_t max_nodes,
                                  float* R, void* stream) {
  if (n_graphs == 0) return 0;
  if (!node_ptr || !edge_ptr || !sq_ptr || !R) return arg_error("resistance: null pointer");
  if (n_graphs < 0 || max_nodes < 1 || max_nodes > kRdMaxNodes)
    return arg_error("resistance: graphs of 1..128 nodes are supported");
  const size_t smem = rd_smem_bytes((int)max_nodes);
  static size_t configured = 48 * 1024;
  if (smem > configured) {
    PGH_CUDA(cudaFuncSetAttribute(resistance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
    configured = smem;
  }
  resistance_kernel<<<(unsigned)n_graphs, kRdThreads, smem, as_stream(stream)>>>(
      (const long long*)edge_src, (const long long*)edge_dst, (const long long*)node_ptr,
      (const long long*)edge_ptr, (const long long*)sq_ptr, (int)max_nodes, R);
  return check_launch("resistance");
}

extern "C" int pgh_rd_dense_f32(const float* R, const int64_t* node_ptr, const int64_t* sq_ptr,
                                int64_t n_graphs, int64_t nmax, float fill, float* out,
                                uint8_t* mask, void* stream) {
  const int64_t total = n_graphs * nmax * nmax;
  if (total == 0) return 0;
  if (!R || !node_ptr || !sq_ptr || !out || !mask) return arg_error("rd_dense: null pointer");
  rd_dense_kernel<<<blocks_for(total, 256), 256, 0, as_stream(stream)>>>(
      R, (const long long*)node_ptr, (const long long*)sq_ptr, total, (int)nmax, fill, out, mask);
  return check_launch("rd_dense");
}

extern "C" int pgh_pad_rows(const void* src, const int64_t* ptr, int64_t n_graphs, int64_t nmax,
                            int64_t width, int elem_bytes, uint64_t fill, void* out,
                            uint8_t* mask, void* stream) {
  const int64_t total = n_graphs * nmax * width;
  if (total == 0) return 0;
  if (!src || !ptr || !out || !mask) return arg_error("pad_rows: null pointer");
  cudaStream_t s = as_stream(stream);
  if (elem_bytes == 8)
    pad_rows_kernel<unsigned long long><<<blocks_for(total, 256), 256, 0, s>>>(
        (const unsigned long long*)src, (const long long*)ptr, total, (int)nmax, (int)width,
        (unsigned long long)fill, (unsigned long long*)out, mask);
  else if (elem_bytes == 4)
    pad_rows_kernel<unsigned int><<<blocks_for(total, 256), 256, 0, s>>>(
        (const unsigned int*)src, (const long long*)ptr, total, (int)nmax, (int)width,
        (unsigned int)fill, (unsigned int*)out, mask);
  else
    return arg_error("pad_rows: elem_bytes must be 4 or 8");
  return check_launch("pad_rows");
}

extern "C" int pgh_dense_adj(const int64_t* edge_src, const int64_t* edge_dst,
                             const int64_t* edge_graph, const int64_t* node_ptr,
                             const void* edge_attr, int64_t n_edges, int64_t n_graphs,
                             int64_t nmax, int64_t width, int elem_bytes, uint64_t fill, void* out,
                             uint8_t* mask, void* stream) {
  const int64_t n_mask = n_graphs * nmax * nmax;
  const int64_t n_out = n_mask * width;
  if (n_out == 0) return 0;
  if (!out || !mask) return arg_error("dense_adj: null pointer");
  if (n_edges > 0 && (!edge_src || !edge_dst || !edge_graph || !edge_attr))
    return arg_error("dense_adj: null pointer");
  if (elem_bytes != 4 && elem_bytes != 8) return arg_error("dense_adj: elem_bytes must be 4 or 8");
  cudaStream_t s = as_stream(stream);
  const int64_t total = n_edges * width;
  if (elem_bytes == 8) {
    fill_kernel<unsigned long long><<<blocks_for(n_out, 256), 256, 0, s>>>(
        (unsigned long long*)out, n_out, (unsigned long long)fill, mask, n_mask);
    if (total)
      dense_adj_kernel<unsigned long long><<<blocks_for(total, 256), 256, 0, s>>>(
          (const long long*)edge_src, (const long long*)edge_dst, (const long long*)edge_graph,
          (const long long*)node_ptr, (const unsigned long long*)edge_attr, total, n_graphs,
          (int)nmax, (int)width, (unsigned long long*)out, mask);
  } else {
    fill_kernel<unsigned int><<<blocks_for(n_out, 256), 256, 0, s>>>(
        (unsigned int*)out, n_out, (unsigned int)fill, mask, n_mask);
    if (total)
      dense_adj_kernel<unsigned int><<<blocks_for(total, 256), 256, 0, s>>>(
          (const long long*)edge_src, (const long long*)edge_dst, (const long long*)edge_graph,
          (const long long*)node_ptr, (const unsigned int*)edge_attr, total, n_graphs, (int)nmax,
          (int)width, (unsigned int*)out, mask);
  }
  return check_launch("dense_adj");
}

// ------------------------------------------------------------------ batched device copies
// n independent device -> device copies in ONE launch (the table travels in the kernel
// parameters): a freshly built batch is moved into the static buffers a captured training step
// replays on (pygho_b200/static.py mirror_into: ~60 arrays per batch, each its own copy kernel
// before).  Sizes are multiples of 4 bytes, pointers 4-byte aligned; 16-byte vectors where both
// sides allow it.
namespace pgh {
constexpr int kCopyMax = 64;
constexpr int kCopyChunk = 16384;       // bytes per CTA
struct CopyTable {
  const char* src[kCopyMax];
  char* dst[kCopyMax];
  long long bytes[kCopyMax];
  int first_cta[kCopyMax + 1];
  int n;
};

__global__ void __launch_bounds__(256) multi_copy_kernel(const __grid_constant__ CopyTable tab) {
  int e = 0;
  while (e + 1 < tab.n && (int)blockIdx.x >= tab.first_cta[e + 1]) ++e;
  const long long off = (long long)((int)blockIdx.x - tab.first_cta[e]) * kCopyChunk;
  const long long len = min((long long)kCopyChunk, tab.bytes[e] - off);
  const char* s = tab.src[e] + off;
  char* d = tab.dst[e] + off;
  if (((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d)) & 15) == 0) {
    const long long n16 = len >> 4;
    for (long long i = threadIdx.x; i < n16; i += 256)
      reinterpret_cast<int4*>(d)[i] = reinterpret_cast<const int4*>(s)[i];
    for (long long i = (n16 << 2) + threadIdx.x; i < (len >> 2); i += 256)
      reinterpret_cast<int*>(d)[i] = reinterpret_cast<const int*>(s)[i];
  } else {
    for (long long i = threadIdx.x; i < (len >> 2); i += 256)
      reinterpret_cast<int*>(d)[i] = reinterpret_cast<const int*>(s)[i];
  }
}
}  // namespace pgh

extern "C" int pgh_multi_copy(const void* const* src, void* const* dst, const int64_t* bytes, int n,
                              void* stream) {
  if (n < 0 || (n > 0 && (!src || !dst || !bytes))) return arg_error("multi_copy: arguments");
  cudaStream_t s = as_stream(stream);
  for (int base = 0; base < n; base += pgh::kCopyMax) {
    pgh::CopyTable tab;
    int m = 0, ctas = 0;
    for (int i = base; i < n && m < pgh::kCopyMax; ++i) {
      if (bytes[i] < 0 || (bytes[i] & 3) || ((reinterpret_cast<uintptr_t>(src[i]) | reinterpret_cast<uintptr_t>(dst[i])) & 3))
        return arg_error("multi_copy: sizes and pointers must be multiples of 4 bytes");
      if (bytes[i] == 0) continue;
      if (!src[i] || !dst[i]) return arg_error("multi_copy: null pointer");
      tab.src[m] = static_cast<const char*>(src[i]);
      tab.dst[m] = static_cast<char*>(dst[i]);
      tab.bytes[m] = bytes[i];
      tab.first_cta[m] = ctas;
      ctas += (int)((bytes[i] + pgh::kCopyChunk - 1) / pgh::kCopyChunk);
      ++m;
    }
    if (m == 0) continue;
    tab.first_cta[m] = ctas;
    tab.n = m;
    pgh::multi_copy_kernel<<<ctas, 256, 0, s>>>(tab);
  }
  return check_launch("multi_copy");
}
