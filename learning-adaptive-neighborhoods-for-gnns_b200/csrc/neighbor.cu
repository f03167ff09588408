// k-hop neighbour sampling on the device: what torch_geometric.loader.NeighborLoader does for train_pubmed.py:370-375
// (third-party, CPU; torch_sparse / pyg-lib neighbor_sample).  The sampling rules, the Philox stream and the
// relabelling order are stated in include/dggb.h; tests/neighbor_ref.py restates them as a sequential loop.
//
// One hop, for frontier F (m slots) with fanout k:
//   neighbor_count_kernel   per-slot emission count (the caller scans it in int64 and reads the total)
//   neighbor_sample_kernel  a warp per slot: draws the CSC positions, writes them with the target's local id, and
//                           claims every source not yet in n_id with atomicMin(claim[u], emission index)
//   neighbor_flag_kernel    flags the first emission of each newly discovered source (claim[u] == emission index)
//   neighbor_assign_kernel  after the caller's scan of the flags: local[u] = next id, new_nodes[id] = u
// and once per batch neighbor_edges_kernel (local source ids of every emission) and neighbor_reset_kernel, which puts
// back local / claim for the nodes the batch touched, so the O(N) workspace is filled once per graph, not per batch.
#include <climits>

#include "common.cuh"
#include "philox.cuh"

namespace dggb {

constexpr int kMaxFanout = 1024;      // Floyd's set lives in shared memory, one 4 KB slice per warp
constexpr int kMaxHops = 255;         // the hop index takes the top 8 bits of the second Philox counter word
constexpr int kSampleWarps = 8;

__device__ __forceinline__ long long emission_count(int d, int k, int replace) {
  if (d == 0 || k == 0) return 0;
  if (k < 0 || (!replace && k >= d)) return d;
  return k;
}

// x_i of the contract: lane (i & 3) of philox4x32_7(counter = (t, (hop << 24) | (i >> 2)), key = seed)
__device__ __forceinline__ uint32_t draw_bits(int t, int hop, int i, uint32_t k0, uint32_t k1) {
  const uint4 b = philox4x32_7((uint32_t)t, ((uint32_t)hop << 24) | (uint32_t)(i >> 2), k0, k1);
  const int q = i & 3;
  return q == 0 ? b.x : (q == 1 ? b.y : (q == 2 ? b.z : b.w));
}

// local[seed[t]] = t.  status <- 1 when a seed is out of range or repeated (the first occurrence keeps its id)
__global__ void neighbor_seed_kernel(const int32_t* __restrict__ seeds, int b, int n, int32_t* __restrict__ local,
                                     long long* __restrict__ status) {
  pdl_trigger();
  pdl_wait();
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < b; t += gridDim.x * blockDim.x) {
    const int s = __ldg(seeds + t);
    if (s < 0 || s >= n || atomicCAS(local + s, -1, t) != -1) *status = 1;
  }
}

__global__ void neighbor_count_kernel(const int32_t* __restrict__ colptr, int n, const int32_t* __restrict__ frontier,
                                      int m, int k, int replace, long long* __restrict__ counts) {
  pdl_trigger();
  pdl_wait();
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < m; t += gridDim.x * blockDim.x) {
    const int v = __ldg(frontier + t);
    long long c = 0;
    if (v >= 0 && v < n) c = emission_count(__ldg(colptr + v + 1) - __ldg(colptr + v), k, replace);
    counts[t] = c;
  }
}

__device__ __forceinline__ void emit(long long e, int p, int dst_local, const int32_t* __restrict__ row,
                                     const int32_t* __restrict__ local, int32_t* __restrict__ claim,
                                     int32_t* __restrict__ out_pos, int32_t* __restrict__ out_dst) {
  out_pos[e] = p;
  out_dst[e] = dst_local;
  const int u = __ldg(row + p);
  if (local[u] < 0) atomicMin(claim + u, (int)e);
}

// offsets: inclusive int64 scan of the counts (slot t emits [offsets[t-1], offsets[t]))
__global__ void __launch_bounds__(kSampleWarps * kWarp)
    neighbor_sample_kernel(const int32_t* __restrict__ colptr, const int32_t* __restrict__ row,
                           const int32_t* __restrict__ frontier, int m, int k, int replace, int hop, uint32_t k0,
                           uint32_t k1, int frontier_base, const long long* __restrict__ offsets,
                           const int32_t* __restrict__ local, int32_t* __restrict__ claim,
                           int32_t* __restrict__ out_pos, int32_t* __restrict__ out_dst) {
  __shared__ int s_set[kSampleWarps][kMaxFanout];
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  int* set = s_set[wib];
  for (int t = blockIdx.x * kSampleWarps + wib; t < m; t += gridDim.x * kSampleWarps) {
    const int v = __ldg(frontier + t);
    const int beg = __ldg(colptr + v), d = __ldg(colptr + v + 1) - beg;
    const long long cnt = emission_count(d, k, replace);
    if (cnt == 0) continue;
    const long long o = t == 0 ? 0 : __ldg(offsets + t - 1);
    const int dst_local = frontier_base + t;
    if (k < 0 || (!replace && k >= d)) {                          // every entry, ascending
      for (int i = lane; i < d; i += kWarp) emit(o + i, beg + i, dst_local, row, local, claim, out_pos, out_dst);
    } else if (replace) {                                         // k independent draws, in draw order
      for (int i = lane; i < k; i += kWarp) {
        const uint32_t x = draw_bits(t, hop, i, k0, k1);
        emit(o + i, beg + (int)(((unsigned long long)x * (unsigned)d) >> 32), dst_local, row, local, claim, out_pos,
             out_dst);
      }
    } else {                                                      // Floyd: k distinct positions, then ascending
      // slot i of the set is written and searched by lane (i & 31) only, so the membership test needs no barrier
      for (int i0 = 0; i0 < k; i0 += kWarp) {
        const uint32_t xl = i0 + lane < k ? draw_bits(t, hop, i0 + lane, k0, k1) : 0u;
        const int steps = min(kWarp, k - i0);
        for (int s = 0; s < steps; ++s) {
          const int i = i0 + s, j = d - k + i;
          const uint32_t x = __shfl_sync(0xffffffffu, xl, s);
          const int r = (int)(((unsigned long long)x * (unsigned)(j + 1)) >> 32);
          bool hit = false;
          for (int q = lane; q < i; q += kWarp) hit |= set[q] == r;
          hit = __any_sync(0xffffffffu, hit);
          if (lane == s) set[i] = hit ? j : r;
        }
      }
      __syncwarp();
      for (int q = lane; q < k; q += kWarp) {                     // rank of a distinct value = its sorted slot
        const int val = set[q];
        int rank = 0;
        for (int w = 0; w < k; ++w) rank += set[w] < val;
        emit(o + rank, beg + val, dst_local, row, local, claim, out_pos, out_dst);
      }
      __syncwarp();                                               // the set is reused by the warp's next slot
    }
  }
}

// flags[e] = 1 when emission e is the first of a source not yet in n_id
__global__ void neighbor_flag_kernel(const int32_t* __restrict__ row, const int32_t* __restrict__ pos, int count,
                                     const int32_t* __restrict__ local, const int32_t* __restrict__ claim,
                                     int32_t* __restrict__ flags) {
  pdl_trigger();
  pdl_wait();
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < count; e += gridDim.x * blockDim.x) {
    const int u = __ldg(row + __ldg(pos + e));
    flags[e] = (__ldg(local + u) < 0 && __ldg(claim + u) == e) ? 1 : 0;
  }
}

// scan: inclusive int32 scan of flags.  A flagged emission's source gets local id base + scan[e] - 1
__global__ void neighbor_assign_kernel(const int32_t* __restrict__ row, const int32_t* __restrict__ pos, int count,
                                       const int32_t* __restrict__ flags, const int32_t* __restrict__ scan, int base,
                                       int32_t* __restrict__ local, int32_t* __restrict__ new_nodes) {
  pdl_trigger();
  pdl_wait();
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < count; e += gridDim.x * blockDim.x) {
    if (__ldg(flags + e) == 0) continue;
    const int u = __ldg(row + __ldg(pos + e)), id = __ldg(scan + e) - 1;
    new_nodes[id] = u;
    local[u] = base + id;
  }
}

__global__ void neighbor_edges_kernel(const int32_t* __restrict__ row, const int32_t* __restrict__ pos,
                                      const int32_t* __restrict__ dst, long long count,
                                      const int32_t* __restrict__ local, long long* __restrict__ edge_index) {
  pdl_trigger();
  pdl_wait();
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < count;
       e += (long long)gridDim.x * blockDim.x) {
    edge_index[e] = __ldg(local + __ldg(row + __ldg(pos + e)));
    edge_index[count + e] = __ldg(dst + e);
  }
}

__global__ void neighbor_reset_kernel(const int32_t* __restrict__ nodes, int count, int n, int32_t* __restrict__ local,
                                      int32_t* __restrict__ claim) {
  pdl_trigger();
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const int u = __ldg(nodes + i);
    if (u < 0 || u >= n) continue;
    local[u] = -1;
    claim[u] = INT_MAX;
  }
}

inline int flat_grid(long long count) {
  const long long need = (count + 255) / 256, cap = (long long)kNumSMs * 8;
  return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

}  // namespace dggb
using namespace dggb;

extern "C" int dggb_neighbor_seed(const int32_t* seeds, int32_t num_seeds, int32_t n, int32_t* local,
                                  int64_t* status, void* stream) {
  if (!seeds || !local || !status || num_seeds < 0 || n <= 0) return DGGB_ERR_BAD_ARG;
  cudaStream_t st = as_stream(stream);
  const cudaError_t e = cudaMemsetAsync(status, 0, sizeof(int64_t), st);
  if (e != cudaSuccess) return cuda_status(e);
  if (num_seeds == 0) return DGGB_OK;
  launch_pdl(neighbor_seed_kernel, dim3(flat_grid(num_seeds)), dim3(256), 0, st, seeds, (int)num_seeds, (int)n, local,
             reinterpret_cast<long long*>(status));
  return launch_status();
}

extern "C" int dggb_neighbor_count(const int32_t* colptr, int32_t n, const int32_t* frontier, int32_t m, int32_t k,
                                   int32_t replace, int64_t* counts, void* stream) {
  if (!colptr || !frontier || !counts || n <= 0 || m < 0) return DGGB_ERR_BAD_ARG;
  if (k > kMaxFanout) return DGGB_ERR_BAD_SHAPE;
  if (m == 0) return DGGB_OK;
  launch_pdl(neighbor_count_kernel, dim3(flat_grid(m)), dim3(256), 0, as_stream(stream), colptr, (int)n, frontier,
             (int)m, (int)k, (int)(replace != 0), reinterpret_cast<long long*>(counts));
  return launch_status();
}

extern "C" int dggb_neighbor_sample(const int32_t* colptr, const int32_t* row, const int32_t* frontier, int32_t m,
                                    int32_t k, int32_t replace, int32_t hop, uint64_t seed, int32_t frontier_base,
                                    const int64_t* offsets, const int32_t* local, int32_t* claim, int32_t* out_pos,
                                    int32_t* out_dst, void* stream) {
  if (!colptr || !row || !frontier || !offsets || !local || !claim || !out_pos || !out_dst || m < 0 || hop < 0 ||
      frontier_base < 0)
    return DGGB_ERR_BAD_ARG;
  if (k > kMaxFanout || hop >= kMaxHops) return DGGB_ERR_BAD_SHAPE;
  if (m == 0 || k == 0) return DGGB_OK;
  launch_pdl(neighbor_sample_kernel, dim3(rows_grid(m, kSampleWarps, 4)), dim3(kSampleWarps * kWarp), 0,
             as_stream(stream), colptr, row, frontier, (int)m, (int)k, (int)(replace != 0), (int)hop,
             (uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32), (int)frontier_base,
             reinterpret_cast<const long long*>(offsets), local, claim, out_pos, out_dst);
  return launch_status();
}

extern "C" int dggb_neighbor_flag(const int32_t* row, const int32_t* pos, int32_t count, const int32_t* local,
                                  const int32_t* claim, int32_t* flags, void* stream) {
  if (!row || !pos || !local || !claim || !flags || count < 0) return DGGB_ERR_BAD_ARG;
  if (count == 0) return DGGB_OK;
  launch_pdl(neighbor_flag_kernel, dim3(flat_grid(count)), dim3(256), 0, as_stream(stream), row, pos, (int)count,
             local, claim, flags);
  return launch_status();
}

extern "C" int dggb_neighbor_assign(const int32_t* row, const int32_t* pos, int32_t count, const int32_t* flags,
                                    const int32_t* scan, int32_t base, int32_t* local, int32_t* new_nodes,
                                    void* stream) {
  if (!row || !pos || !flags || !scan || !local || !new_nodes || count < 0 || base < 0) return DGGB_ERR_BAD_ARG;
  if (count == 0) return DGGB_OK;
  launch_pdl(neighbor_assign_kernel, dim3(flat_grid(count)), dim3(256), 0, as_stream(stream), row, pos, (int)count,
             flags, scan, (int)base, local, new_nodes);
  return launch_status();
}

extern "C" int dggb_neighbor_edges(const int32_t* row, const int32_t* pos, const int32_t* dst, int64_t count,
                                   const int32_t* local, int64_t* edge_index, void* stream) {
  if (!row || !pos || !dst || !local || !edge_index || count < 0) return DGGB_ERR_BAD_ARG;
  if (count == 0) return DGGB_OK;
  launch_pdl(neighbor_edges_kernel, dim3(flat_grid(count)), dim3(256), 0, as_stream(stream), row, pos, dst,
             (long long)count, local, reinterpret_cast<long long*>(edge_index));
  return launch_status();
}

extern "C" int dggb_neighbor_reset(const int32_t* nodes, int32_t count, int32_t n, int32_t* local, int32_t* claim,
                                   void* stream) {
  if (!nodes || !local || !claim || count < 0 || n <= 0) return DGGB_ERR_BAD_ARG;
  if (count == 0) return DGGB_OK;
  launch_pdl(neighbor_reset_kernel, dim3(flat_grid(count)), dim3(256), 0, as_stream(stream), nodes, (int)count, (int)n,
             local, claim);
  return launch_status();
}
