// Deterministic multilevel k-way graph partitioning on the device: what METIS does for torch_geometric.loader.ClusterData
// (train_large_graphs.py:402-421; third-party, host cores).  The contract of every phase is stated in include/dggb.h;
// tests/cluster_ref.py restates the phases and the driver (dgg_b200.samplers.partition) in NumPy and the kernels match
// it bit for bit.  Integer arithmetic only, and atomics compute only order-independent results (sums, minima), so the
// partition depends on nothing but the graph and num_parts.
//
//   partition_weights_kernel   per-label summed node weight and smallest member (the anchor)
//   partition_propose_kernel   a warp per node: connection weight per adjacent label in a shared-memory hash table
//                              (rows with more labels than fit are split into passes by label hash), best label
//   partition_admit_kernel     proposals sorted by key (target, gain descending, node id): admitted while the
//                              target's start-of-round weight plus the admitted weight stays <= limit
//   partition_rebalance_kernel the least-loss proposals of each over-full part take the free places in part order
//   contract_keys / heads / fill   coarse entries (cluster pair keys, sorted by the caller, merged per key)
//   partition_bfs_kernel       one block: level-synchronous BFS order of the coarsest graph
//   partition_chunk_kernel / partition_project_kernel
#include <cub/block/block_scan.cuh>

#include "common.cuh"

namespace dggb {

constexpr long long kNoKey = 0x7fffffffffffffffLL;
constexpr int kTableSlots = 1024;        // per warp: 8 KB of (label, weight) slots
constexpr int kProposeWarps = 4;
constexpr int kBfsThreads = 1024;

__host__ __device__ __forceinline__ uint32_t fmix32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x85ebca6bu;
  x ^= x >> 13;
  x *= 0xc2b2ae35u;
  x ^= x >> 16;
  return x;
}

// first index in the sorted keys[0, n) whose value is >= v
__device__ __forceinline__ int lower_bound64(const long long* __restrict__ keys, int n, long long v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(keys + mid) < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void partition_weights_kernel(const int32_t* __restrict__ lab, const int32_t* __restrict__ vw, int n,
                                         int32_t* __restrict__ lw, int32_t* __restrict__ anchor) {
  pdl_trigger();
  pdl_wait();
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) {
    const int l = __ldg(lab + v);
    atomicAdd(lw + l, __ldg(vw + v));
    if (anchor) atomicMin(anchor + l, v);
  }
}

__device__ __forceinline__ bool better(int c, uint32_t h, int bc, uint32_t bh) {
  return c > bc || (c == bc && h > bh);
}

__global__ void __launch_bounds__(kProposeWarps * kWarp)
    partition_propose_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                             const int32_t* __restrict__ ewt, const int32_t* __restrict__ vw,
                             const int32_t* __restrict__ lab, int n, const int32_t* __restrict__ lw,
                             const int32_t* __restrict__ anchor, int limit, int parity, int mode,
                             long long* __restrict__ key) {
  __shared__ int s_key[kProposeWarps][kTableSlots];
  __shared__ int s_val[kProposeWarps][kTableSlots];
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  int* tk = s_key[wib];
  int* tv = s_val[wib];
  for (int v = blockIdx.x * kProposeWarps + wib; v < n; v += gridDim.x * kProposeWarps) {
    const int own = __ldg(lab + v);
    bool active;
    if (mode == 2) {
      active = __ldg(lw + own) > limit && __ldg(anchor + own) != v;
    } else {
      active = (int)(fmix32((uint32_t)v) & 1u) == parity;
      if (mode != 0) active = active && __ldg(anchor + own) != v;
      if (mode == 3) active = active && __ldg(lw + own) > limit;
    }
    if (!active) {
      if (lane == 0) key[v] = kNoKey;
      continue;
    }
    const int beg = __ldg(rowptr + v), end = __ldg(rowptr + v + 1), d = end - beg;
    const long long room = (long long)limit - __ldg(vw + v);
    int own_conn = 0;
    for (int e = beg + lane; e < end; e += kWarp)
      if (__ldg(lab + __ldg(col + e)) == own) own_conn += __ldg(ewt + e);
    own_conn = __reduce_add_sync(0xffffffffu, own_conn);

    int passes = max(1, (d + kTableSlots / 2 - 1) / (kTableSlots / 2));
    int bc = 0, bl = -1;        // best connection and label of this lane (bc = 0: none yet)
    uint32_t bh = 0;
    for (int p = 0; p < passes; ++p) {
      for (int s = lane; s < kTableSlots; s += kWarp) {
        tk[s] = -1;
        tv[s] = 0;
      }
      __syncwarp();
      bool overflow = false;
      for (int e = beg + lane; e < end; e += kWarp) {
        const int l = __ldg(lab + __ldg(col + e));
        if (l == own || (long long)__ldg(lw + l) > room) continue;
        const uint32_t h = fmix32((uint32_t)l);
        if (passes > 1 && (int)((h >> 10) % (uint32_t)passes) != p) continue;
        int slot = (int)(h & (kTableSlots - 1)), probes = 0;
        for (; probes < kTableSlots; ++probes, slot = (slot + 1) & (kTableSlots - 1)) {
          const int prev = atomicCAS(tk + slot, -1, l);
          if (prev == -1 || prev == l) {
            atomicAdd(tv + slot, __ldg(ewt + e));
            break;
          }
        }
        overflow |= probes == kTableSlots;
      }
      __syncwarp();
      if (__any_sync(0xffffffffu, overflow)) {       // too many labels for one table: twice the passes, start again
        passes *= 2;
        p = -1;
        bc = 0;
        bl = -1;
        bh = 0;
        __syncwarp();
        continue;
      }
      for (int s = lane; s < kTableSlots; s += kWarp) {
        const int l = tk[s];
        if (l < 0) continue;
        const uint32_t h = fmix32((uint32_t)l);
        if (better(tv[s], h, bc, bh)) {
          bc = tv[s];
          bh = h;
          bl = l;
        }
      }
      __syncwarp();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int oc = __shfl_xor_sync(0xffffffffu, bc, o), ol = __shfl_xor_sync(0xffffffffu, bl, o);
      const uint32_t oh = __shfl_xor_sync(0xffffffffu, bh, o);
      if (better(oc, oh, bc, bh)) {
        bc = oc;
        bh = oh;
        bl = ol;
      }
    }
    if (lane == 0) {
      const long long gain = (long long)bc - own_conn;
      long long k = kNoKey;
      if (mode == 2)
        k = ((long long)own << 32) | (long long)(uint32_t)(0x7fffffffLL - gain);
      else if (bl >= 0 && (gain > 0 || mode == 3))
        k = ((long long)bl << 32) | (long long)(uint32_t)(0x7fffffffLL - gain);
      key[v] = k;
    }
  }
}

__global__ void partition_admit_kernel(const long long* __restrict__ keys, const long long* __restrict__ order,
                                       const long long* __restrict__ cum, int n, const int32_t* __restrict__ lw,
                                       int limit, int32_t* __restrict__ lab) {
  pdl_trigger();
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const long long k = __ldg(keys + i);
    if (k == kNoKey) continue;
    const int t = (int)(k >> 32);
    const int s = lower_bound64(keys, n, (long long)t << 32);
    const long long seg = __ldg(cum + i) - (s > 0 ? __ldg(cum + s - 1) : 0);
    if ((long long)__ldg(lw + t) + seg <= limit) lab[__ldg(order + i)] = t;
  }
}

__global__ void partition_rebalance_kernel(const long long* __restrict__ keys, const long long* __restrict__ order,
                                           int n, const int32_t* __restrict__ lw, const long long* __restrict__ ex_prefix,
                                           const long long* __restrict__ room_cum, int k, int cap,
                                           int32_t* __restrict__ part) {
  pdl_trigger();
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const long long key = __ldg(keys + i);
    if (key == kNoKey) continue;
    const int p = (int)(key >> 32);
    const int r = i - lower_bound64(keys, n, (long long)p << 32);
    if (r >= __ldg(lw + p) - cap) continue;
    const long long j = __ldg(ex_prefix + p) + r;
    int lo = 0, hi = k;                              // first part q with room_cum[q] > j
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(room_cum + mid) <= j) lo = mid + 1; else hi = mid;
    }
    part[__ldg(order + i)] = lo;
  }
}

// keys[e] = cluster[row] * nc + cluster[col] of entry e, or kNoKey when both ends are in one cluster
__global__ void contract_keys_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int n,
                                     const int32_t* __restrict__ cluster, int nc, long long* __restrict__ keys) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int v = blockIdx.x * wpb + (threadIdx.x >> 5); v < n; v += gridDim.x * wpb) {
    const int cu = __ldg(cluster + v);
    for (int e = __ldg(rowptr + v) + lane; e < __ldg(rowptr + v + 1); e += kWarp) {
      const int cw = __ldg(cluster + __ldg(col + e));
      keys[e] = cu == cw ? kNoKey : (long long)cu * nc + cw;
    }
  }
}

__device__ __forceinline__ bool run_head(const long long* __restrict__ keys, long long i) {
  const long long k = __ldg(keys + i);
  return k != kNoKey && (i == 0 || __ldg(keys + i - 1) != k);
}

__global__ void contract_heads_kernel(const long long* __restrict__ keys, long long nnz, int32_t* __restrict__ heads) {
  pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (long long)gridDim.x * blockDim.x)
    heads[i] = run_head(keys, i) ? 1 : 0;
}

// scan: inclusive int32 scan of the heads; entry j of the coarse graph is the run of keys ending at scan == j + 1
__global__ void contract_fill_kernel(const long long* __restrict__ keys, const long long* __restrict__ idx,
                                     const int32_t* __restrict__ ewt, long long nnz, const int32_t* __restrict__ scan,
                                     int nc, long long* __restrict__ crow, int32_t* __restrict__ ccol,
                                     int32_t* __restrict__ cwt) {
  pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (long long)gridDim.x * blockDim.x) {
    const long long k = __ldg(keys + i);
    if (k == kNoKey) continue;
    const int j = __ldg(scan + i) - 1;
    atomicAdd(cwt + j, __ldg(ewt + __ldg(idx + i)));
    if (run_head(keys, i)) {
      crow[j] = k / nc;
      ccol[j] = (int)(k % nc);
    }
  }
}

// pos[] = -1 and claim[] = 0x7f7f7f7f on entry (the host entry point fills them).  order / pos / claim are written
// by this block while it runs (claim through L2 atomics), so they are read with ld.cg, past the non-coherent L1.
__global__ void __launch_bounds__(kBfsThreads)
    partition_bfs_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int n,
                         int32_t* order, int32_t* pos, int32_t* claim) {
  using Scan = cub::BlockScan<int, kBfsThreads>;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ int s_head, s_tail;
  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x;
  int cursor = 0;                                     // thread 0: no id below it is unvisited
  if (tid == 0) s_tail = 0;
  __syncthreads();
  while (true) {
    const int tail0 = s_tail;
    __syncthreads();
    if (tail0 >= n) break;
    if (tid == 0) {                                   // a new search from the smallest unvisited id
      while (__ldcg(pos + cursor) >= 0) ++cursor;
      order[tail0] = cursor;
      pos[cursor] = tail0;
      s_head = tail0;
      s_tail = tail0 + 1;
    }
    __syncthreads();
    while (true) {
      const int lo = s_head, hi = s_tail;
      __syncthreads();
      if (lo == hi) break;
      for (int i = lo + tid; i < hi; i += kBfsThreads) {          // each new node is claimed by its first parent
        const int f = __ldcg(order + i);
        for (int e = __ldg(rowptr + f); e < __ldg(rowptr + f + 1); ++e) {
          const int u = __ldg(col + e);
          if (__ldcg(pos + u) < 0) atomicMin(claim + u, i);
        }
      }
      __syncthreads();
      int out = hi;
      for (int c = lo; c < hi; c += kBfsThreads) {                // children in (parent position, id) order
        const int i = c + tid;
        int cnt = 0;
        if (i < hi) {
          const int f = __ldcg(order + i);
          for (int e = __ldg(rowptr + f); e < __ldg(rowptr + f + 1); ++e) cnt += __ldcg(claim + __ldg(col + e)) == i;
        }
        int off, total;
        Scan(tmp).ExclusiveSum(cnt, off, total);
        if (i < hi && cnt > 0) {
          const int f = __ldcg(order + i);
          int q = out + off;
          for (int e = __ldg(rowptr + f); e < __ldg(rowptr + f + 1); ++e) {
            const int u = __ldg(col + e);
            if (__ldcg(claim + u) == i) {
              order[q] = u;
              pos[u] = q;
              ++q;
            }
          }
        }
        out += total;
        __syncthreads();
      }
      if (tid == 0) {
        s_head = hi;
        s_tail = out;
      }
      __syncthreads();
    }
  }
}

__global__ void partition_chunk_kernel(const int32_t* __restrict__ order, const long long* __restrict__ prefix, int n,
                                       long long total, int k, int32_t* __restrict__ part) {
  pdl_trigger();
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const long long q = __ldg(prefix + i) * k / total;
    part[__ldg(order + i)] = (int)(q < k - 1 ? q : k - 1);
  }
}

__global__ void partition_project_kernel(const int32_t* __restrict__ map, const int32_t* __restrict__ idx, int n,
                                         int32_t* __restrict__ out) {
  pdl_trigger();
  pdl_wait();
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) out[v] = __ldg(map + __ldg(idx + v));
}

// A ClusterLoader batch: rows node_idx[m] (parent ids of the drawn parts, in draw order) of the permuted parent CSR,
// kept entries = columns inside a drawn part.  A row's entries are sorted by parent id and every part is a contiguous id
// range, so the kept entries of part b are one run, found by binary search; runs are emitted in draw order, which is
// ascending local id.  Drawn part b covers parent ids [start[b], end[b]) and local ids from base[b].
__device__ __forceinline__ int lower_bound32(const int32_t* __restrict__ a, int lo, int hi, int v) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(a + mid) < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

template <bool kFill>
__global__ void cluster_batch_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                     const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                                     const int32_t* __restrict__ base, int nb, const int32_t* __restrict__ node_idx,
                                     int m, int32_t* __restrict__ counts, const int32_t* __restrict__ sub_rowptr,
                                     int32_t* __restrict__ sub_col, int32_t* __restrict__ sub_eid) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int i = blockIdx.x * wpb + (threadIdx.x >> 5); i < m; i += gridDim.x * wpb) {
    const int u = __ldg(node_idx + i);
    const int rb = __ldg(rowptr + u), re = __ldg(rowptr + u + 1);
    int out = kFill ? __ldg(sub_rowptr + i) : 0;
    for (int b0 = 0; b0 < nb; b0 += kWarp) {
      const int b = b0 + lane;
      int lo = 0, hi = 0;
      if (b < nb) {
        lo = lower_bound32(col, rb, re, __ldg(start + b));
        hi = lower_bound32(col, lo, re, __ldg(end + b));
      }
      const int cnt = hi - lo;
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < kWarp; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (kFill && cnt > 0) {
        const int shift = __ldg(base + b) - __ldg(start + b);
        for (int e = lo, q = out + incl - cnt; e < hi; ++e, ++q) {
          sub_col[q] = __ldg(col + e) + shift;
          sub_eid[q] = e;
        }
      }
      out += __shfl_sync(0xffffffffu, incl, kWarp - 1);
    }
    if (!kFill && lane == 0) counts[i] = out;
  }
}

inline int grid_for(long long count) {
  const long long need = (count + 255) / 256, cap = (long long)kNumSMs * 8;
  return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

}  // namespace dggb
using namespace dggb;

extern "C" int dggb_partition_weights(const int32_t* lab, const int32_t* vw, int32_t n, int32_t nlabels, int32_t* lw,
                                      int32_t* anchor, void* stream) {
  if (!lab || !vw || !lw || n <= 0 || nlabels <= 0) return DGGB_ERR_BAD_ARG;
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(lw, 0, (size_t)nlabels * sizeof(int32_t), st);
  if (e == cudaSuccess && anchor) e = cudaMemsetAsync(anchor, 0x7f, (size_t)nlabels * sizeof(int32_t), st);
  if (e != cudaSuccess) return cuda_status(e);
  launch_pdl(partition_weights_kernel, dim3(grid_for(n)), dim3(256), 0, st, lab, vw, (int)n, lw, anchor);
  return launch_status();
}

extern "C" int dggb_partition_propose(const int32_t* rowptr, const int32_t* col, const int32_t* ewt, const int32_t* vw,
                                      const int32_t* lab, int32_t n, const int32_t* lw, const int32_t* anchor,
                                      int32_t limit, int32_t parity, int32_t mode, int64_t* key, void* stream) {
  if (!rowptr || !col || !ewt || !vw || !lab || !lw || !key || n <= 0 || limit < 0 || (parity != 0 && parity != 1))
    return DGGB_ERR_BAD_ARG;
  if (mode < 0 || mode > 3) return DGGB_ERR_UNSUPPORTED;
  if (mode != 0 && !anchor) return DGGB_ERR_BAD_ARG;
  launch_pdl(partition_propose_kernel, dim3(rows_grid(n, kProposeWarps, 8)), dim3(kProposeWarps * kWarp), 0,
             as_stream(stream), rowptr, col, ewt, vw, lab, (int)n, lw, anchor, (int)limit, (int)parity, (int)mode,
             reinterpret_cast<long long*>(key));
  return launch_status();
}

extern "C" int dggb_partition_admit(const int64_t* keys, const int64_t* order, const int64_t* cum, int32_t n,
                                    const int32_t* lw, int32_t limit, int32_t* lab, void* stream) {
  if (!keys || !order || !cum || !lw || !lab || n <= 0) return DGGB_ERR_BAD_ARG;
  launch_pdl(partition_admit_kernel, dim3(grid_for(n)), dim3(256), 0, as_stream(stream),
             reinterpret_cast<const long long*>(keys), reinterpret_cast<const long long*>(order),
             reinterpret_cast<const long long*>(cum), (int)n, lw, (int)limit, lab);
  return launch_status();
}

extern "C" int dggb_partition_rebalance(const int64_t* keys, const int64_t* order, int32_t n, const int32_t* lw,
                                        const int64_t* ex_prefix, const int64_t* room_cum, int32_t k, int32_t cap,
                                        int32_t* part, void* stream) {
  if (!keys || !order || !lw || !ex_prefix || !room_cum || !part || n <= 0 || k <= 0 || cap <= 0)
    return DGGB_ERR_BAD_ARG;
  launch_pdl(partition_rebalance_kernel, dim3(grid_for(n)), dim3(256), 0, as_stream(stream),
             reinterpret_cast<const long long*>(keys), reinterpret_cast<const long long*>(order), (int)n, lw,
             reinterpret_cast<const long long*>(ex_prefix), reinterpret_cast<const long long*>(room_cum), (int)k,
             (int)cap, part);
  return launch_status();
}

extern "C" int dggb_partition_contract_keys(const int32_t* rowptr, const int32_t* col, int32_t n,
                                            const int32_t* cluster, int32_t nc, int64_t* keys, void* stream) {
  if (!rowptr || !col || !cluster || !keys || n <= 0 || nc <= 0) return DGGB_ERR_BAD_ARG;
  launch_pdl(contract_keys_kernel, dim3(rows_grid(n, 8, 8)), dim3(256), 0, as_stream(stream), rowptr, col, (int)n,
             cluster, (int)nc, reinterpret_cast<long long*>(keys));
  return launch_status();
}

extern "C" int dggb_partition_contract_heads(const int64_t* keys, int64_t nnz, int32_t* heads, void* stream) {
  if (!keys || !heads || nnz <= 0) return DGGB_ERR_BAD_ARG;
  launch_pdl(contract_heads_kernel, dim3(grid_for(nnz)), dim3(256), 0, as_stream(stream),
             reinterpret_cast<const long long*>(keys), (long long)nnz, heads);
  return launch_status();
}

extern "C" int dggb_partition_contract_fill(const int64_t* keys, const int64_t* idx, const int32_t* ewt, int64_t nnz,
                                            const int32_t* scan, int32_t nc, int32_t cnnz, int64_t* crow,
                                            int32_t* ccol, int32_t* cwt, void* stream) {
  if (!keys || !idx || !ewt || !scan || !crow || !ccol || !cwt || nnz <= 0 || nc <= 0 || cnnz <= 0)
    return DGGB_ERR_BAD_ARG;
  cudaStream_t st = as_stream(stream);
  const cudaError_t e = cudaMemsetAsync(cwt, 0, (size_t)cnnz * sizeof(int32_t), st);
  if (e != cudaSuccess) return cuda_status(e);
  launch_pdl(contract_fill_kernel, dim3(grid_for(nnz)), dim3(256), 0, st, reinterpret_cast<const long long*>(keys),
             reinterpret_cast<const long long*>(idx), ewt, (long long)nnz, scan, (int)nc,
             reinterpret_cast<long long*>(crow), ccol, cwt);
  return launch_status();
}

extern "C" int dggb_partition_bfs(const int32_t* rowptr, const int32_t* col, int32_t n, int32_t* order, int32_t* pos,
                                  int32_t* claim, void* stream) {
  if (!rowptr || !col || !order || !pos || !claim || n <= 0 || n >= 0x7f7f7f7f) return DGGB_ERR_BAD_ARG;
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(pos, 0xff, (size_t)n * sizeof(int32_t), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(claim, 0x7f, (size_t)n * sizeof(int32_t), st);
  if (e != cudaSuccess) return cuda_status(e);
  launch_pdl(partition_bfs_kernel, dim3(1), dim3(kBfsThreads), 0, st, rowptr, col, (int)n, order, pos, claim);
  return launch_status();
}

extern "C" int dggb_partition_chunk(const int32_t* order, const int64_t* prefix, int32_t n, int64_t total, int32_t k,
                                    int32_t* part, void* stream) {
  if (!order || !prefix || !part || n <= 0 || total <= 0 || k <= 0) return DGGB_ERR_BAD_ARG;
  launch_pdl(partition_chunk_kernel, dim3(grid_for(n)), dim3(256), 0, as_stream(stream), order,
             reinterpret_cast<const long long*>(prefix), (int)n, (long long)total, (int)k, part);
  return launch_status();
}

extern "C" int dggb_partition_project(const int32_t* map, const int32_t* idx, int32_t n, int32_t* out, void* stream) {
  if (!map || !idx || !out || n <= 0) return DGGB_ERR_BAD_ARG;
  launch_pdl(partition_project_kernel, dim3(grid_for(n)), dim3(256), 0, as_stream(stream), map, idx, (int)n, out);
  return launch_status();
}

extern "C" int dggb_cluster_batch_count(const int32_t* rowptr, const int32_t* col, const int32_t* start,
                                        const int32_t* end, int32_t num_drawn, const int32_t* node_idx, int32_t m,
                                        int32_t* counts, void* stream) {
  if (!rowptr || !col || !start || !end || !node_idx || !counts || num_drawn <= 0 || m <= 0) return DGGB_ERR_BAD_ARG;
  launch_pdl(cluster_batch_kernel<false>, dim3(rows_grid(m, 8, 8)), dim3(256), 0, as_stream(stream), rowptr, col, start,
             end, static_cast<const int32_t*>(nullptr), (int)num_drawn, node_idx, (int)m, counts,
             static_cast<const int32_t*>(nullptr), static_cast<int32_t*>(nullptr), static_cast<int32_t*>(nullptr));
  return launch_status();
}

extern "C" int dggb_cluster_batch_fill(const int32_t* rowptr, const int32_t* col, const int32_t* start,
                                       const int32_t* end, const int32_t* base, int32_t num_drawn,
                                       const int32_t* node_idx, int32_t m, const int32_t* sub_rowptr, int32_t* sub_col,
                                       int32_t* sub_eid, void* stream) {
  if (!rowptr || !col || !start || !end || !base || !node_idx || !sub_rowptr || !sub_col || !sub_eid ||
      num_drawn <= 0 || m <= 0)
    return DGGB_ERR_BAD_ARG;
  launch_pdl(cluster_batch_kernel<true>, dim3(rows_grid(m, 8, 8)), dim3(256), 0, as_stream(stream), rowptr, col, start,
             end, base, (int)num_drawn, node_idx, (int)m, static_cast<int32_t*>(nullptr), sub_rowptr, sub_col, sub_eid);
  return launch_status();
}
