// class DGG edge ranker + degree estimator + soft first-k, forward and backward.
// Replaces dgm.py:1781-1810 (gather u,v -> Linear+LeakyReLU -> sum -> sigmoid -> dense N x N scatter ->
// row sum -> Linear(1,1) -> N-long row sort -> tanh first-k -> un-sort scatter -> to_sparse).
//
// Graphs without hub rows (longest row <= 512 entries: Cora, Citeseer, Pubmed): ONE launch per direction, a block
// owning a contiguous range of rows and their edges (dgg_fwd_fused2_kernel; backward dgg_bwd_fused2_kernel, or
// dgg_bwd_fused_kernel for block windows above 6 144 entries).
// Graphs with hub rows: two launches per direction so that a power-law hub cannot serialise a warp:
//   fwd:  edge_score (edge-parallel, perfectly balanced)  ->  row_rank (warp per CSR row)
//   bwd:  row_dk     (warp per CSR row)                    ->  edge_grad (edge-parallel, vector reds)
// Issue/latency-bound at Pubmed size, HBM-bound at scale.  Algorithmic bytes per launch are listed in DESIGN.md.
#include "common.cuh"
#include "edge_common.cuh"
#include <cstdlib>

namespace dggb {

constexpr int kEdgeWarps = 8;  // warps per block

// sum over this lane's chunks of LeakyReLU(y_u - y_v + be); out-of-range chunks contribute exactly 0.
template <int T>
__device__ __forceinline__ float edge_partial(const RowSlice<T>& yu, const RowSlice<T>& yv, const RowSlice<T>& b) {
  float z = 0.f;
#pragma unroll
  for (int t = 0; t < T; ++t) {
    z += leaky(yu.v[t].x - yv.v[t].x + b.v[t].x) + leaky(yu.v[t].y - yv.v[t].y + b.v[t].y) +
         leaky(yu.v[t].z - yv.v[t].z + b.v[t].z) + leaky(yu.v[t].w - yv.v[t].w + b.v[t].w);
  }
  return z;
}

// Branch mask of an entry: [ceil(h / 32)] words, bit c % 32 of word c / 32 set when pre_c = y_u - y_v + be > 0, i.e.
// when LeakyReLU'(pre_c) == 1.  The fused forward writes it so that the fused backward never gathers y again.
// Lane lg's chunk t holds channels 4 (lg + L t) .. +3, all inside word (lg + L t) / 8: for L < 8 the L lanes of a group
// share that word (= L t / 8, the same for every lane), for L >= 8 lanes 8j .. 8j + 7 do (a new word at every t).
__device__ __forceinline__ int branch_word(int lg, int L, int t) { return (L < 8 ? L * t : lg + L * t) >> 3; }

template <int T>
struct BranchBits {
  uint32_t w[T];
};

// edge_partial, and this lane's bits of every chunk t placed in word branch_word(lg, L, t) (chunks at c >= h: 0),
// from one pass over pre_c.  z is summed exactly as edge_partial sums it.
template <int T>
__device__ __forceinline__ float edge_partial_bits(const RowSlice<T>& yu, const RowSlice<T>& yv, const RowSlice<T>& b,
                                                   int lg, int L, BranchBits<T>& bb) {
  float z = 0.f;
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const float px = yu.v[t].x - yv.v[t].x + b.v[t].x, py = yu.v[t].y - yv.v[t].y + b.v[t].y;
    const float pz = yu.v[t].z - yv.v[t].z + b.v[t].z, pw = yu.v[t].w - yv.v[t].w + b.v[t].w;
    z += leaky(px) + leaky(py) + leaky(pz) + leaky(pw);
    const uint32_t nib = (uint32_t)(px > 0.f) | (uint32_t)(py > 0.f) << 1 | (uint32_t)(pz > 0.f) << 2 |
                         (uint32_t)(pw > 0.f) << 3;
    bb.w[t] = nib << ((4 * (lg + L * t)) & 31);
  }
  return z;
}

// The lanes of a word OR their bits and the word's first lane stores it.  Every lane of the warp calls this (the
// word changes at the same t for all of them); `live` gates the stores.
__device__ __forceinline__ void store_branch_word(uint32_t word, int wi, int h, int lg, int L, bool live,
                                                  uint32_t* __restrict__ mrow) {
  for (int o = 1; o < (L < 8 ? L : 8); o <<= 1) word |= __shfl_xor_sync(0xffffffffu, word, o);
  if (live && (lg & 7) == 0 && 32 * wi < h) mrow[wi] = word;
}

template <int T>
__device__ __forceinline__ void store_branch_mask(const BranchBits<T>& bb, int h, int lg, int L, bool live,
                                                  uint32_t* __restrict__ mrow) {
  uint32_t word = 0;
  int wi = branch_word(lg, L, 0);
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int wt = branch_word(lg, L, t);
    if (wt != wi) {
      store_branch_word(word, wi, h, lg, L, live, mrow);
      word = 0;
      wi = wt;
    }
    word |= bb.w[t];
  }
  store_branch_word(word, wi, h, lg, L, live, mrow);
}

// this lane's four bits of every chunk t (bit j: channel 4 (lg + L t) + j), 0 for dead slots and chunks at c >= h
template <int T>
__device__ __forceinline__ void load_branch_mask(uint32_t (&nib)[T], const uint32_t* __restrict__ mrow, int h, int lg,
                                                 int L, bool live) {
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int c = 4 * (lg + L * t);
    nib[t] = (live && c < h) ? (__ldg(mrow + branch_word(lg, L, t)) >> (c & 31)) & 15u : 0u;
  }
}

// d pre of one chunk: dz * LeakyReLU'(pre_c), the same products as dz * leaky_grad(pre_c)
__device__ __forceinline__ float4 branch_scale(uint32_t nib, float dz) {
  const float lo = dz * kLeaky;
  return make_float4((nib & 1u) ? dz : lo, (nib & 2u) ? dz : lo, (nib & 4u) ? dz : lo, (nib & 8u) ? dz : lo);
}

__device__ __forceinline__ float first_k_plus_one(float r, float k) {
  // dgm.py:1801-1804: 1 - 0.5 * (1 + tanh(t - k)), then + 1.0
  const float fk = 1.f - 0.5f * (1.f + tanhf(r - k));
  return fk + 1.f;
}

// ------------------------------------------------------------------------------------------------
// fwd 1/2: R_e = sigmoid(sum_c LeakyReLU(y_u - y_v + be))  [ablation: sigmoid(R_e + noise_e)]
// ------------------------------------------------------------------------------------------------
template <int T>
__global__ void __launch_bounds__(kEdgeWarps* kWarp)
    dgg_edge_score_kernel(const int32_t* __restrict__ erow, const int32_t* __restrict__ col, int nnz, int h, int L,
                          const float* __restrict__ y, const float* __restrict__ be,
                          const float* __restrict__ abl_noise, float* __restrict__ R) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int G = kWarp / L, PER = kWarp / G;  // PER == L
  const int lg = lane % L, grp = lane / L;
  RowSlice<T> bias;
  load_slice<T>(bias, be, h, lg, L);
  const int warps_total = gridDim.x * kEdgeWarps;
  for (int base = (blockIdx.x * kEdgeWarps + (threadIdx.x >> 5)) * kWarp; base < nnz; base += warps_total * kWarp) {
    const int e_l = base + lane;
    const int u_l = (e_l < nnz) ? __ldg(erow + e_l) : 0;
    const int v_l = (e_l < nnz) ? __ldg(col + e_l) : 0;
    float mine = 0.f;
#pragma unroll 4
    for (int it = 0; it < PER; ++it) {
      const int j = grp * PER + it;  // edge slot inside the chunk handled by this group now
      const int u = __shfl_sync(0xffffffffu, u_l, j);
      const int v = __shfl_sync(0xffffffffu, v_l, j);
      RowSlice<T> yu, yv;
      load_slice<T>(yu, y + (size_t)u * h, h, lg, L);
      load_slice<T>(yv, y + (size_t)v * h, h, lg, L);
      const float z = group_sum(edge_partial<T>(yu, yv, bias), L);
      // group grp walks slots [grp*L, grp*L + L) == its own lanes: lane lg keeps iteration lg's result
      if (lg == it) mine = z;
    }
    if (e_l < nnz) {
      float r = sigmoidf_(mine);
      if (abl_noise != nullptr) r = sigmoidf_(r + __ldg(abl_noise + e_l));  // dgm.py:1933-1935
      R[e_l] = r;
    }
  }
}

// 0-based descending rank of element m inside R[beg, beg+deg): ties broken by lower position first.
// All 32 lanes call this together; lanes with m >= deg get garbage they ignore.
//   deg <= 32 : one register per lane + 32 shuffles
//   deg <= kRankCap : the row is staged in this warp's shared-memory slice; every lane then sweeps it with
//                broadcast LDS (independent iterations, throughput- not latency-bound)
//   longer rows: same sweep straight from global/L1
constexpr int kRankCap = 1024;  // floats of shared memory per warp

__device__ __forceinline__ int warp_rank(const float* __restrict__ R, float* srow, bool staged, int beg, int deg,
                                         int m, int lane) {
  const float mine = (m < deg) ? __ldg(R + beg + m) : -INFINITY;
  int cnt = 0;
  if (deg <= kWarp) {
    for (int jj = 0; jj < deg; ++jj) {
      const float rj = __shfl_sync(0xffffffffu, mine, jj);   // m == lane here
      cnt += (rj > mine) || (rj == mine && jj < m);
    }
    return cnt;
  }
  if (staged) {
#pragma unroll 4
    for (int j = 0; j < deg; ++j) {
      const float rj = srow[j];
      cnt += (rj > mine) || (rj == mine && j < m);
    }
  } else {
#pragma unroll 4
    for (int j = 0; j < deg; ++j) {
      const float rj = __ldg(R + beg + j);
      cnt += (rj > mine) || (rj == mine && j < m);
    }
  }
  return cnt;
}

// stage R[beg, beg+deg) into the warp's shared slice (deg <= kRankCap)
__device__ __forceinline__ bool stage_row(const float* __restrict__ R, float* srow, int beg, int deg, int lane) {
  if (deg <= kWarp || deg > kRankCap) return false;
  __syncwarp();
  for (int j = lane; j < deg; j += kWarp) srow[j] = __ldg(R + beg + j);
  __syncwarp();
  return true;
}

// ------------------------------------------------------------------------------------------------
// Hub rows.  The in-row rank is a count (deg^2 compares); a warp owning a 20 k-entry row (real Reddit hubs) would
// run 1.3e7 iterations per lane while the rest of the grid idles.  When the caller passes a scratch list
// (long_ws: [n + 1] int32, long_ws[0] == 0 on entry), the row kernels only compute s / k for rows longer than
// kRankCap, append them to the list, and long_row_rank_kernel spreads their compares over the whole grid:
// one thread per entry, the row swept in shared-memory tiles (20 k entries: 80 blocks x 20 k iterations).
// value modes: 0 out = v * fk(r - k); 1 out = fk(r - k) (k_only); 2 out = v * (fk(r - k) + 1) (class DGG);
// 3 out = r < hard_k ? v : 0 (ablation)
// ------------------------------------------------------------------------------------------------
constexpr int kLongThreads = 256;
constexpr int kLongTile = 2048;

__device__ __forceinline__ float first_k_tanh(float r, float k) { return 1.f - 0.5f * (1.f + tanhf(r - k)); }

__device__ __forceinline__ float ranked_value(int mode, float v, int r, float k, int hard_k) {
  if (mode == 3) return r < hard_k ? v : 0.f;
  const float fk = first_k_tanh((float)r, k);
  return mode == 0 ? v * fk : (mode == 1 ? fk : v * (fk + 1.f));
}

__device__ __forceinline__ void defer_long_row(int32_t* long_ws, int row, int lane) {
  if (lane == 0) long_ws[1 + atomicAdd(long_ws, 1)] = row;
}

__global__ void __launch_bounds__(kLongThreads)
    long_row_rank_kernel(const int32_t* __restrict__ rowptr, const float* __restrict__ R,
                         const float* __restrict__ k_in, int mode, int hard_k, const int32_t* long_ws,
                         int32_t* __restrict__ rank, float* __restrict__ out) {
  pdl_trigger();
  pdl_wait();
  __shared__ float tile[kLongTile];
  const int n_long = long_ws[0];
  for (int q = 0; q < n_long; ++q) {
    const int i = long_ws[1 + q];
    const int beg = __ldg(rowptr + i), deg = __ldg(rowptr + i + 1) - beg;
    const float k = (mode == 3) ? 0.f : k_in[i];
    const int chunks = (deg + kLongThreads - 1) / kLongThreads;
    for (int c = blockIdx.x; c < chunks; c += gridDim.x) {
      const int m = c * kLongThreads + threadIdx.x;
      const float mine = (m < deg) ? R[beg + m] : -INFINITY;
      int cnt = 0;
      for (int j0 = 0; j0 < deg; j0 += kLongTile) {
        const int len = min(kLongTile, deg - j0);
        __syncthreads();
        for (int j = threadIdx.x; j < len; j += kLongThreads) tile[j] = R[beg + j0 + j];
        __syncthreads();
#pragma unroll 8
        for (int j = 0; j < len; ++j) {
          const float rj = tile[j];
          cnt += (rj > mine) || (rj == mine && (j0 + j) < m);
        }
      }
      if (m < deg) {
        rank[beg + m] = cnt;
        out[beg + m] = ranked_value(mode, mine, cnt, k, hard_k);
      }
    }
  }
}

static void launch_long_rows(const int32_t* rowptr, const float* R, const float* k, int mode, int hard_k,
                             const int32_t* long_ws, int32_t* rank, float* out, cudaStream_t st) {
  launch_pdl(long_row_rank_kernel, dim3(kNumSMs * 4), dim3(kLongThreads), 0, st, rowptr, R, k, mode, hard_k, long_ws,
             rank, out);
}

// ------------------------------------------------------------------------------------------------
// fwd 2/2: s_i, k_i = LeakyReLU(w s_i + b), in-row rank, out_e = R_e * (first_k + 1)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kEdgeWarps* kWarp)
    dgg_row_rank_kernel(const int32_t* __restrict__ rowptr, int n, const float* __restrict__ R,
                        const float* __restrict__ deg_w, const float* __restrict__ deg_b, int hard_k,
                        int32_t* __restrict__ rank, float* __restrict__ s_out, float* __restrict__ k_out,
                        float* __restrict__ out, int32_t* long_ws) {
  pdl_trigger();
  pdl_wait();
  __shared__ float srow_all[kEdgeWarps * kRankCap];
  float* srow = srow_all + (threadIdx.x >> 5) * kRankCap;
  const int lane = threadIdx.x & 31;
  const float w = __ldg(deg_w), b = __ldg(deg_b);
  for (int i = blockIdx.x * kEdgeWarps + (threadIdx.x >> 5); i < n; i += gridDim.x * kEdgeWarps) {
    const int beg = __ldg(rowptr + i), end = __ldg(rowptr + i + 1), deg = end - beg;
    float s = 0.f;
    for (int e = beg + lane; e < end; e += kWarp) s += __ldg(R + e);
    s = warp_sum(s);
    const float k = leaky(w * s + b);  // dgm.py:1791-1792
    if (lane == 0) {
      s_out[i] = s;
      k_out[i] = k;
    }
    if (long_ws != nullptr && deg > kRankCap) {   // hub row: ranked by the whole grid afterwards
      defer_long_row(long_ws, i, lane);
      continue;
    }
    const bool staged = stage_row(R, srow, beg, deg, lane);
    for (int mb = 0; mb < deg; mb += kWarp) {
      const int m = mb + lane;
      const int r = warp_rank(R, srow, staged, beg, deg, m, lane);
      if (m < deg) {
        const float val = __ldg(R + beg + m);
        rank[beg + m] = r;
        out[beg + m] = (hard_k >= 0) ? (r < hard_k ? val : 0.f) : val * first_k_plus_one((float)r, k);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// bwd 1/2: d out / d k_i = 0.5 * sum_e g_e R_e sech^2(r_e - k_i)  (SURVEY A.1), chained through the
// degree decoder: ds_i = dk_i * LeakyReLU'(w s_i + b) * w;  d w, d b accumulated per warp.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kEdgeWarps* kWarp)
    dgg_row_dk_kernel(const int32_t* __restrict__ rowptr, int n, const float* __restrict__ R,
                      const int32_t* __restrict__ rank, const float* __restrict__ s_in,
                      const float* __restrict__ k_in, const float* __restrict__ g_out,
                      const float* __restrict__ deg_w, const float* __restrict__ deg_b, float* __restrict__ ds,
                      float* __restrict__ ddeg) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const float w = __ldg(deg_w), b = __ldg(deg_b);
  float dw_acc = 0.f, db_acc = 0.f;
  for (int i = blockIdx.x * kEdgeWarps + (threadIdx.x >> 5); i < n; i += gridDim.x * kEdgeWarps) {
    const int beg = __ldg(rowptr + i), end = __ldg(rowptr + i + 1);
    const float s = __ldg(s_in + i), k = __ldg(k_in + i);
    float dk = 0.f;
    for (int e = beg + lane; e < end; e += kWarp) {
      const float th = tanhf((float)__ldg(rank + e) - k);
      dk += __ldg(g_out + e) * __ldg(R + e) * 0.5f * (1.f - th * th);
    }
    dk = warp_sum(dk);
    const float lr = leaky_grad(w * s + b);
    if (lane == 0) ds[i] = dk * lr * w;
    dw_acc += dk * lr * s;
    db_acc += dk * lr;
  }
  // one pair of atomics per block, not per warp: every warp in the grid targets the same two addresses
  __shared__ float red[2][kEdgeWarps];
  if (lane == 0) {
    red[0][threadIdx.x >> 5] = dw_acc;
    red[1][threadIdx.x >> 5] = db_acc;
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    float t = 0.f;
#pragma unroll
    for (int wv = 0; wv < kEdgeWarps; ++wv) t += red[threadIdx.x][wv];
    atomicAdd(ddeg + threadIdx.x, t);
  }
}

// ------------------------------------------------------------------------------------------------
// bwd 2/2: per edge, recompute z (no E x H tensor is ever stored), then
//   dR = g * (first_k + 1) + ds_u  [hard: g * (rank < hard_k)]   [ablation: *= R2 (1 - R2)]
//   dz = dR * R1 (1 - R1);  d pre_c = dz * LeakyReLU'(pre_c);  dy_u += d pre;  dy_v -= d pre;  dbe += d pre
// ------------------------------------------------------------------------------------------------
template <int T>
__global__ void __launch_bounds__(kEdgeWarps* kWarp)
    dgg_edge_grad_kernel(const int32_t* __restrict__ erow, const int32_t* __restrict__ col, int nnz, int h, int L,
                         const float* __restrict__ y, const float* __restrict__ be,
                         const float* __restrict__ abl_noise, int hard_k, const float* __restrict__ R,
                         const int32_t* __restrict__ rank, const float* __restrict__ k_in,
                         const float* __restrict__ ds, const float* __restrict__ g_out, float* __restrict__ dy,
                         float* __restrict__ dbe) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int G = kWarp / L, PER = kWarp / G;
  const int lg = lane % L, grp = lane / L;
  RowSlice<T> bias, dbe_acc;
  load_slice<T>(bias, be, h, lg, L);
#pragma unroll
  for (int t = 0; t < T; ++t) dbe_acc.v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
  __shared__ float dbe_s[512];   // block-level bias-gradient accumulator (h <= 512)
  for (int c = threadIdx.x; c < h; c += blockDim.x) dbe_s[c] = 0.f;
  __syncthreads();
  const int warps_total = gridDim.x * kEdgeWarps;
  for (int base = (blockIdx.x * kEdgeWarps + (threadIdx.x >> 5)) * kWarp; base < nnz; base += warps_total * kWarp) {
    const int e_l = base + lane;
    const bool ok_l = e_l < nnz;
    const int u_l = ok_l ? __ldg(erow + e_l) : 0;
    const int v_l = ok_l ? __ldg(col + e_l) : 0;
    // per-edge scalar factor dR (everything that does not need the feature rows), one edge per lane
    float dr_l = 0.f;
    if (ok_l) {
      const float g = __ldg(g_out + e_l);
      if (hard_k >= 0) {
        dr_l = (__ldg(rank + e_l) < hard_k) ? g : 0.f;
      } else {
        dr_l = g * first_k_plus_one((float)__ldg(rank + e_l), __ldg(k_in + u_l)) + __ldg(ds + u_l);
      }
      if (abl_noise != nullptr) {
        const float r2 = __ldg(R + e_l);
        dr_l *= r2 * (1.f - r2);  // through the second sigmoid
      }
    }
    int cur_u = -1;
    RowSlice<T> acc;  // running +d pre for the current source row of this group
#pragma unroll
    for (int t = 0; t < T; ++t) acc.v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
    for (int it = 0; it < PER; ++it) {
      const int j = grp * PER + it;
      const int u = __shfl_sync(0xffffffffu, u_l, j);
      const int v = __shfl_sync(0xffffffffu, v_l, j);
      const float dr = __shfl_sync(0xffffffffu, dr_l, j);
      const bool valid = (base + j) < nnz;
      RowSlice<T> yu, yv;
      load_slice<T>(yu, y + (size_t)u * h, h, lg, L, valid);
      load_slice<T>(yv, y + (size_t)v * h, h, lg, L, valid);
      const float z = group_sum(edge_partial<T>(yu, yv, bias), L);
      const float r1 = sigmoidf_(z);
      const float dz = valid ? dr * r1 * (1.f - r1) : 0.f;
      if (u != cur_u) {  // group-uniform branch: flush the finished source row
        if (cur_u >= 0) {
#pragma unroll
          for (int t = 0; t < T; ++t) {
            const int c = 4 * (lg + L * t);
            if (c < h) red_add4(dy + (size_t)cur_u * h + c, acc.v[t]);
            acc.v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        cur_u = u;
      }
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int c = 4 * (lg + L * t);
        float4 d;
        d.x = dz * leaky_grad(yu.v[t].x - yv.v[t].x + bias.v[t].x);
        d.y = dz * leaky_grad(yu.v[t].y - yv.v[t].y + bias.v[t].y);
        d.z = dz * leaky_grad(yu.v[t].z - yv.v[t].z + bias.v[t].z);
        d.w = dz * leaky_grad(yu.v[t].w - yv.v[t].w + bias.v[t].w);
        dbe_acc.v[t].x += d.x; dbe_acc.v[t].y += d.y; dbe_acc.v[t].z += d.z; dbe_acc.v[t].w += d.w;
        if (u != v) {  // a self loop adds +d and -d to the same row: skip both (it still counts for dbe)
          acc.v[t].x += d.x; acc.v[t].y += d.y; acc.v[t].z += d.z; acc.v[t].w += d.w;
          if (valid && c < h) red_add4(dy + (size_t)v * h + c, make_float4(-d.x, -d.y, -d.z, -d.w));
        }
      }
    }
    if (cur_u >= 0) {
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int c = 4 * (lg + L * t);
        if (c < h) red_add4(dy + (size_t)cur_u * h + c, acc.v[t]);
      }
    }
  }
  // flush this warp's bias gradient: combine the G groups first, then one vector red per chunk
#pragma unroll
  for (int t = 0; t < T; ++t) {
    for (int o = L; o < kWarp; o <<= 1) {
      dbe_acc.v[t].x += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].x, o);
      dbe_acc.v[t].y += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].y, o);
      dbe_acc.v[t].z += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].z, o);
      dbe_acc.v[t].w += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].w, o);
    }
    const int c = 4 * (lg + L * t);
    if (grp == 0 && c < h) {
      atomicAdd(&dbe_s[c + 0], dbe_acc.v[t].x);
      atomicAdd(&dbe_s[c + 1], dbe_acc.v[t].y);
      atomicAdd(&dbe_s[c + 2], dbe_acc.v[t].z);
      atomicAdd(&dbe_s[c + 3], dbe_acc.v[t].w);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < h; c += blockDim.x) atomicAdd(dbe + c, dbe_s[c]);
}

// ------------------------------------------------------------------------------------------------
// select_top_k of DGG_LearnableK_debug on CSR rows (dgm.py:1402-1421, A.2): k is an input,
//   fk(r) = 1 - 0.5 * (1 + tanh(r - k_i));  mode 0: out = score * fk (k_times_edge_prob)
// Off-support entries are exact zeros that sort after every positive score, so in-row ranks are exact.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kEdgeWarps* kWarp)
    row_firstk_fwd_kernel(const int32_t* __restrict__ rowptr, int n, const float* __restrict__ score,
                          const float* __restrict__ k_in, int mode, int32_t* __restrict__ rank,
                          float* __restrict__ out, int32_t* long_ws) {
  pdl_trigger();
  pdl_wait();
  __shared__ float srow_all[kEdgeWarps * kRankCap];
  float* srow = srow_all + (threadIdx.x >> 5) * kRankCap;
  const int lane = threadIdx.x & 31;
  for (int i = blockIdx.x * kEdgeWarps + (threadIdx.x >> 5); i < n; i += gridDim.x * kEdgeWarps) {
    const int beg = __ldg(rowptr + i), end = __ldg(rowptr + i + 1), deg = end - beg;
    const float k = __ldg(k_in + i);
    if (long_ws != nullptr && deg > kRankCap) {
      defer_long_row(long_ws, i, lane);
      continue;
    }
    const bool staged = stage_row(score, srow, beg, deg, lane);
    for (int mb = 0; mb < deg; mb += kWarp) {
      const int m = mb + lane;
      const int r = warp_rank(score, srow, staged, beg, deg, m, lane);
      if (m < deg) {
        rank[beg + m] = r;
        const float fk = first_k_tanh((float)r, k);
        out[beg + m] = mode == 1 ? fk : __ldg(score + beg + m) * fk;
      }
    }
  }
}

__global__ void __launch_bounds__(kEdgeWarps* kWarp)
    row_firstk_bwd_kernel(const int32_t* __restrict__ rowptr, int n, const float* __restrict__ score,
                          const float* __restrict__ k_in, int mode, const int32_t* __restrict__ rank,
                          const float* __restrict__ g_out, float* __restrict__ dscore, float* __restrict__ dk) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  for (int i = blockIdx.x * kEdgeWarps + (threadIdx.x >> 5); i < n; i += gridDim.x * kEdgeWarps) {
    const int beg = __ldg(rowptr + i), end = __ldg(rowptr + i + 1);
    const float k = __ldg(k_in + i);
    float acc = 0.f;
    for (int e = beg + lane; e < end; e += kWarp) {
      const float th = tanhf((float)__ldg(rank + e) - k);
      const float g = __ldg(g_out + e);
      dscore[e] = mode == 1 ? 0.f : g * (1.f - 0.5f * (1.f + th));      // k_only: no gradient reaches the scores
      acc += g * (mode == 1 ? 1.f : __ldg(score + e)) * 0.5f * (1.f - th * th);
    }
    acc = warp_sum(acc);
    if (lane == 0) dk[i] = acc;
  }
}

// ------------------------------------------------------------------------------------------------
// Fused kernels for graphs without hub rows (max row length <= kFusedMaxDeg): ONE launch per direction.
// Block b owns the CSR rows that START inside the edge interval [b*epb, (b+1)*epb) -- found from erow in two
// dependent loads, no search -- and therefore the contiguous edge range [rowptr[r0], rowptr[r1]) of at most
// epb + max_deg entries (the block's window).  The forward is always dgg_fwd_fused2_kernel.  The backward is
// dgg_bwd_fused2_kernel when the window holds at most 6 144 entries (two shared-memory floats per entry), and
// dgg_bwd_fused_kernel, which keeps only per-row values in shared memory, for larger windows.
// At Pubmed shape the two-launch path is pure latency (2 x ~12 us for 0.4 MB of edge data); this is one wave of
// blocks with ~4 dependent memory round trips.  R and rank are bit-identical to the two-launch kernels; s, k and
// out differ from them by the summation order of the row sums.
// ------------------------------------------------------------------------------------------------
constexpr int kFusedMaxDeg = 512;
constexpr int kFusedThreads = 256;
constexpr int kFusedRowsCap = 1024;   // rows of ds kept in shared memory (bwd); further rows go through ds_ws

__device__ __forceinline__ void fused_row_range(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ erow,
                                                int n, int nnz, int epb, int* rng) {
  if (threadIdx.x < 2) {
    const long long e = (long long)(blockIdx.x + threadIdx.x) * epb;
    int r;
    if (e >= nnz || (threadIdx.x == 1 && blockIdx.x == gridDim.x - 1)) {
      r = n;                                           // trailing (empty) rows belong to the last block
    } else {
      r = __ldg(erow + e);                             // row holding entry e
      if (__ldg(rowptr + r) < (int)e) ++r;             // it started earlier: the next row is the first one >= e
      else while (r > 0 && __ldg(rowptr + r - 1) == (int)e) --r;   // empty rows that also start at e
    }
    rng[threadIdx.x] = r;
    rng[2 + threadIdx.x] = (r >= n) ? nnz : __ldg(rowptr + r);
  }
  __syncthreads();
}

// LC > 0: lanes per edge and the hidden width (h == 16 * LC, T == 4) are compile-time constants, which folds every
// `chunk < h` guard, the zero fills of out-of-range chunks and the per-chunk address arithmetic (static SASS of the
// runtime-L version: ~270 instructions per edge slot, a third of them guards / CS2R / IMAD).
//
// Backward for windows above 6 144 entries: warp-per-row dk / ds (the first kFusedRowsCap rows' ds in shared memory,
// the rest through ds_ws) -> __syncthreads -> edge-parallel gradients.
template <int T, int LC>
__global__ void __launch_bounds__(kFusedThreads)
    dgg_bwd_fused_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ erow,
                         const int32_t* __restrict__ col, int n, int nnz, int h, int L, int epb,
                         const uint32_t* __restrict__ branch_mask, const float* __restrict__ r1_in,
                         const float* __restrict__ abl_noise, int hard_k, const float* __restrict__ R,
                         const int32_t* __restrict__ rank, const float* __restrict__ s_in,
                         const float* __restrict__ k_in, const float* __restrict__ g_out,
                         const float* __restrict__ deg_w, const float* __restrict__ deg_b, float* ds_ws,
                         float* __restrict__ dy, float* __restrict__ dbe, float* __restrict__ ddeg) {
  pdl_trigger();
  if constexpr (LC > 0) {
    L = LC;
    h = 16 * LC;
  }
  __shared__ float sds[kFusedRowsCap];
  __shared__ float dbe_s[512];           // block-level bias-gradient accumulator (h <= 512)
  __shared__ float red[2][kFusedThreads / kWarp];
  __shared__ int rng[4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int G = kWarp / L, lg = lane % L, grp = lane / L;
  for (int c = threadIdx.x; c < h; c += kFusedThreads) dbe_s[c] = 0.f;
  pdl_wait();
  fused_row_range(rowptr, erow, n, nnz, epb, rng);
  const int r0 = rng[0], r1 = rng[1], eb0 = rng[2], eb1 = rng[3];
  const int nE = eb1 - eb0;
  // ---- phase A: d out / d k_i chained through the degree decoder (soft mode only) ----
  if (hard_k < 0) {
    const float w = __ldg(deg_w), b = __ldg(deg_b);
    float dw_acc = 0.f, db_acc = 0.f;
    const int sub = lane >> 3, sl = lane & 7;
    for (int i0 = r0 + warp * 4; i0 < r1; i0 += (kFusedThreads / kWarp) * 4) {
      const int i = i0 + sub;
      const bool rv = i < r1;
      const int beg = rv ? __ldg(rowptr + i) : 0, end = rv ? __ldg(rowptr + i + 1) : 0;
      const float s = rv ? __ldg(s_in + i) : 0.f, k = rv ? __ldg(k_in + i) : 0.f;
      float dk = 0.f;
      for (int e = beg + sl; e < end; e += 8) {
        const float th = tanhf((float)__ldg(rank + e) - k);
        dk += __ldg(g_out + e) * __ldg(R + e) * 0.5f * (1.f - th * th);
      }
      dk += __shfl_xor_sync(0xffffffffu, dk, 4);
      dk += __shfl_xor_sync(0xffffffffu, dk, 2);
      dk += __shfl_xor_sync(0xffffffffu, dk, 1);
      const float lr = leaky_grad(w * s + b);
      if (rv && sl == 0) {
        const float dsi = dk * lr * w;
        ds_ws[i] = dsi;
        if (i - r0 < kFusedRowsCap) sds[i - r0] = dsi;
        dw_acc += dk * lr * s;
        db_acc += dk * lr;
      }
    }
    dw_acc = warp_sum(dw_acc);
    db_acc = warp_sum(db_acc);
    if (lane == 0) {
      red[0][warp] = dw_acc;
      red[1][warp] = db_acc;
    }
  }
  __syncthreads();
  if (hard_k < 0 && threadIdx.x < 2) {
    float t = 0.f;
#pragma unroll
    for (int wv = 0; wv < kFusedThreads / kWarp; ++wv) t += red[threadIdx.x][wv];
    if (t != 0.f) atomicAdd(ddeg + threadIdx.x, t);
  }
  // ---- phase B: per edge, d pre = dz LeakyReLU'(pre) from the forward's branch mask, scattered ----
  const int W = (h + 31) >> 5;
  RowSlice<T> dbe_acc, acc;
#pragma unroll
  for (int t = 0; t < T; ++t) dbe_acc.v[t] = acc.v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int groups = (kFusedThreads / kWarp) * G;
  const int per = (nE + groups - 1) / groups;
  const int g0 = (warp * G + grp) * per;
  int cur_u = -1;
#pragma unroll 2
  for (int it = 0; it < per; ++it) {
    const int idx = g0 + it;
    const bool valid = idx < nE;
    const int e = eb0 + (valid ? idx : 0);
    const int u = valid ? __ldg(erow + e) : 0, v = valid ? __ldg(col + e) : 0;
    float dr = 0.f;
    if (valid) {
      const float g = __ldg(g_out + e);
      if (hard_k >= 0) {
        dr = (__ldg(rank + e) < hard_k) ? g : 0.f;
      } else {
        const float dsu = (u - r0 < kFusedRowsCap) ? sds[u - r0] : __ldcg(ds_ws + u);
        dr = g * first_k_plus_one((float)__ldg(rank + e), __ldg(k_in + u)) + dsu;
      }
      if (abl_noise != nullptr) {
        const float r2 = __ldg(R + e);
        dr *= r2 * (1.f - r2);  // through the second sigmoid
      }
    }
    uint32_t nib[T];
    load_branch_mask<T>(nib, branch_mask + (size_t)e * W, h, lg, L, valid);
    const float r1e = __ldg(r1_in + e);
    const float dz = valid ? dr * r1e * (1.f - r1e) : 0.f;
    if (valid && u != cur_u) {  // group-uniform branch: flush the finished source row
      if (cur_u >= 0) {
#pragma unroll
        for (int t = 0; t < T; ++t) {
          const int c = 4 * (lg + L * t);
          if (c < h) red_add4(dy + (size_t)cur_u * h + c, acc.v[t]);
          acc.v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      cur_u = u;
    }
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int c = 4 * (lg + L * t);
      const float4 d = branch_scale(nib[t], dz);
      dbe_acc.v[t].x += d.x; dbe_acc.v[t].y += d.y; dbe_acc.v[t].z += d.z; dbe_acc.v[t].w += d.w;
      if (valid && u != v) {  // a self loop adds +d and -d to the same row: skip both (it still counts for dbe)
        acc.v[t].x += d.x; acc.v[t].y += d.y; acc.v[t].z += d.z; acc.v[t].w += d.w;
        if (c < h) red_add4(dy + (size_t)v * h + c, make_float4(-d.x, -d.y, -d.z, -d.w));
      }
    }
  }
  if (cur_u >= 0) {
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int c = 4 * (lg + L * t);
      if (c < h) red_add4(dy + (size_t)cur_u * h + c, acc.v[t]);
    }
  }
#pragma unroll
  for (int t = 0; t < T; ++t) {
    for (int o = L; o < kWarp; o <<= 1) {
      dbe_acc.v[t].x += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].x, o);
      dbe_acc.v[t].y += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].y, o);
      dbe_acc.v[t].z += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].z, o);
      dbe_acc.v[t].w += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].w, o);
    }
    const int c = 4 * (lg + L * t);
    if (grp == 0 && c < h) {
      atomicAdd(&dbe_s[c + 0], dbe_acc.v[t].x);
      atomicAdd(&dbe_s[c + 1], dbe_acc.v[t].y);
      atomicAdd(&dbe_s[c + 2], dbe_acc.v[t].z);
      atomicAdd(&dbe_s[c + 3], dbe_acc.v[t].w);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < h; c += kFusedThreads) atomicAdd(dbe + c, dbe_s[c]);
}

// ------------------------------------------------------------------------------------------------
// Second generation of the fused kernels: the forward for every window, the backward for windows of at most 6 144
// entries (the backward has the contract of dgg_bwd_fused_kernel and its results up to the summation order of the
// row sums).
// Why they are entry-parallel: the ncu source view of the row-parallel design that dgg_bwd_fused_kernel keeps, at
// Pubmed shape (profiles/r02_fused_edge_v2.md), put a third of the stall samples at block barriers (rows dealt to
// 8-lane groups finish at very different times, and rows longer than 32 entries were ranked by the whole block after
// yet another barrier), a quarter behind the per-edge dependent chain "index load -> gather" that every group
// repeated `per` times back to back.  Here
//   * phase 1 walks the block's entries INTERLEAVED over the groups (coalesced index loads) and loads the indices of
//     the next entry while the current entry's rows are in flight: one memory round trip per entry instead of two;
//   * phase 2 is ENTRY-parallel: thread == entry; it sweeps its own row in shared memory, which yields the rank (a
//     count), the row sum s and therefore k in the same loop -- no per-row pass, no long-row pass, one barrier.  The
//     compare work is the same sum of deg^2, but spread evenly (a 171-entry row occupies 171 threads for 171
//     iterations instead of one 8-lane group for 3 600);
//   * backward: entry-parallel as well -- per-entry d out / d k terms into shared memory, each entry's thread sums its
//     row (= dk_i), forms ds_i and its own d z_e; then the scatter phase, which reads each entry's LeakyReLU branch
//     bits from the mask the forward stored (no y gathers: 8 B per entry at h = 64 instead of 2 x 256 B of dependent
//     L2 reads), with the next entry's indices and mask words prefetched.
// ------------------------------------------------------------------------------------------------
template <int T, int LC>
__global__ void __launch_bounds__(kFusedThreads)
    dgg_fwd_fused2_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ erow,
                          const int32_t* __restrict__ col, int n, int nnz, int h, int L, int epb, int cap,
                          const float* __restrict__ y, const float* __restrict__ be,
                          const float* __restrict__ abl_noise, const float* __restrict__ deg_w,
                          const float* __restrict__ deg_b, int hard_k, float* R, int32_t* __restrict__ rank,
                          float* __restrict__ s_out, float* __restrict__ k_out, float* __restrict__ out,
                          uint32_t* __restrict__ branch_mask, float* __restrict__ r1_out, float* zero_ws,
                          long long zero_count) {
  pdl_trigger();
  if constexpr (LC > 0) {
    L = LC;
    h = 16 * LC;
  }
  const int W = (h + 31) >> 5;           // branch-mask words per entry
  extern __shared__ float sR[];          // [cap] scores of this block's entry range
  __shared__ int rng[4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int G = kWarp / L, lg = lane % L, grp = lane / L;
  pdl_wait();
  zero_fill(zero_ws, zero_count);   // the backward's accumulation buffers (dy | dbe | ddeg | ds)
  fused_row_range(rowptr, erow, n, nnz, epb, rng);
  const int r0 = rng[0], r1 = rng[1], eb0 = rng[2], eb1 = rng[3];
  const int nE = eb1 - eb0;
  // ---- phase 1: scores.  entry idx = it * groups + gid ----
  {
    RowSlice<T> bias;
    load_slice<T>(bias, be, h, lg, L);
    const int groups = (kFusedThreads / kWarp) * G;
    const int per = (nE + groups - 1) / groups;
    int idx = warp * G + grp;
    int u_n = 0, v_n = 0;
    if (idx < nE) {
      u_n = __ldg(erow + eb0 + idx);
      v_n = __ldg(col + eb0 + idx);
    }
    for (int it = 0; it < per; ++it, idx += groups) {
      const bool valid = idx < nE;
      const int u = u_n, v = v_n;
      if (idx + groups < nE) {            // next entry's indices travel while this entry's rows do
        u_n = __ldg(erow + eb0 + idx + groups);
        v_n = __ldg(col + eb0 + idx + groups);
      }
      RowSlice<T> yu, yv;
      load_slice<T>(yu, y + (size_t)u * h, h, lg, L, valid);
      load_slice<T>(yv, y + (size_t)v * h, h, lg, L, valid);
      BranchBits<T> bb;   // formed whether or not it is stored: one code path keeps the register count of edge_partial
      const float z = group_sum(edge_partial_bits<T>(yu, yv, bias, lg, L, bb), L);
      if (branch_mask != nullptr) store_branch_mask<T>(bb, h, lg, L, valid, branch_mask + (size_t)(eb0 + idx) * W);
      if (valid && lg == 0) {
        const int e = eb0 + idx;
        float r = sigmoidf_(z);
        if (abl_noise != nullptr) {
          if (r1_out != nullptr) r1_out[e] = r;
          r = sigmoidf_(r + __ldg(abl_noise + e));  // dgm.py:1933-1935
        }
        R[e] = r;
        if (idx < cap) sR[idx] = r;
      }
    }
  }
  __syncthreads();
  // ---- phase 2: thread == entry ----
  const float w = __ldg(deg_w), b = __ldg(deg_b);
  for (int idx = threadIdx.x; idx < nE; idx += kFusedThreads) {
    const int e = eb0 + idx;
    const int u = __ldg(erow + e);
    const int jb = __ldg(rowptr + u) - eb0, je = __ldg(rowptr + u + 1) - eb0;   // the row inside the block's window
    float mine, s = 0.f;
    int cnt = 0;
    if (je <= cap) {
      mine = sR[idx];
#pragma unroll 4
      for (int j = jb; j < je; ++j) {
        const float rj = sR[j];
        s += rj;
        cnt += (rj > mine) || (rj == mine && j < idx);
      }
    } else {                              // beyond the shared-memory window (very large bounded-degree graphs)
      mine = __ldcg(R + e);
#pragma unroll 4
      for (int j = jb; j < je; ++j) {
        const float rj = __ldcg(R + eb0 + j);
        s += rj;
        cnt += (rj > mine) || (rj == mine && j < idx);
      }
    }
    const float k = leaky(w * s + b);  // dgm.py:1791-1792
    rank[e] = cnt;
    out[e] = (hard_k >= 0) ? (cnt < hard_k ? mine : 0.f) : mine * first_k_plus_one((float)cnt, k);
    if (idx == jb) {
      s_out[u] = s;
      k_out[u] = k;
    }
  }
  for (int i = r0 + threadIdx.x; i < r1; i += kFusedThreads) {   // empty rows: s = 0
    if (__ldg(rowptr + i) == __ldg(rowptr + i + 1)) {
      s_out[i] = 0.f;
      k_out[i] = leaky(b);
    }
  }
}

// Keep the minimum of 1 block per SM: with __launch_bounds__(kFusedThreads) alone, ptxas limits <4,4> to 64 registers
// instead of 78 and compiles every instantiation differently.
template <int T, int LC>
__global__ void __launch_bounds__(kFusedThreads, 1)
    dgg_bwd_fused2_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ erow,
                          const int32_t* __restrict__ col, int n, int nnz, int h, int L, int epb, int cap,
                          const uint32_t* __restrict__ branch_mask, const float* __restrict__ r1_in,
                          const float* __restrict__ abl_noise, int hard_k, const float* __restrict__ R,
                          const int32_t* __restrict__ rank, const float* __restrict__ s_in,
                          const float* __restrict__ k_in, const float* __restrict__ g_out,
                          const float* __restrict__ deg_w, const float* __restrict__ deg_b, float* ds_ws,
                          float* __restrict__ dy, float* __restrict__ dbe, float* __restrict__ ddeg) {
  pdl_trigger();
  if constexpr (LC > 0) {
    L = LC;
    h = 16 * LC;
  }
  extern __shared__ float sm2[];         // sT[cap]: d out / d k terms, sDz[cap]: d loss / d z_e   (nE <= cap, host)
  float* sT = sm2;
  float* sDz = sm2 + cap;
  __shared__ float dbe_s[512];           // block-level bias-gradient accumulator (h <= 512)
  __shared__ float red[2][kFusedThreads / kWarp];
  __shared__ int rng[4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int G = kWarp / L, lg = lane % L, grp = lane / L;
  for (int c = threadIdx.x; c < h; c += kFusedThreads) dbe_s[c] = 0.f;
  pdl_wait();
  fused_row_range(rowptr, erow, n, nnz, epb, rng);
  const int eb0 = rng[2], eb1 = rng[3];
  const int nE = eb1 - eb0;
  // ---- phase A: thread == entry.  d out / d k_i = 0.5 sum_e g_e R_e sech^2(r_e - k_i), chained through the degree
  // decoder: ds_i = dk_i LeakyReLU'(w s_i + b) w;  d R_e = g_e (first_k + 1) + ds_i ----
  if (hard_k < 0) {
    for (int idx = threadIdx.x; idx < nE; idx += kFusedThreads) {
      const int e = eb0 + idx;
      const float th = tanhf((float)__ldg(rank + e) - __ldg(k_in + __ldg(erow + e)));
      sT[idx] = __ldg(g_out + e) * __ldg(R + e) * 0.5f * (1.f - th * th);
    }
  }
  __syncthreads();
  {
    const float w = __ldg(deg_w), b = __ldg(deg_b);
    float dw_acc = 0.f, db_acc = 0.f;
    for (int idx = threadIdx.x; idx < nE; idx += kFusedThreads) {
      const int e = eb0 + idx;
      const float g = __ldg(g_out + e);
      float dr;
      if (hard_k >= 0) {
        dr = (__ldg(rank + e) < hard_k) ? g : 0.f;
      } else {
        const int u = __ldg(erow + e);
        const int jb = __ldg(rowptr + u) - eb0, je = __ldg(rowptr + u + 1) - eb0;
        float dk = 0.f;
#pragma unroll 4
        for (int j = jb; j < je; ++j) dk += sT[j];
        const float s = __ldg(s_in + u), k = __ldg(k_in + u);
        const float lr = leaky_grad(w * s + b);
        const float dsi = dk * lr * w;
        if (idx == jb) {                   // once per row
          ds_ws[u] = dsi;
          dw_acc += dk * lr * s;
          db_acc += dk * lr;
        }
        dr = g * first_k_plus_one((float)__ldg(rank + e), k) + dsi;
      }
      if (abl_noise != nullptr) {
        const float r2 = __ldg(R + e);
        dr *= r2 * (1.f - r2);  // through the second sigmoid
      }
      const float r1e = __ldg(r1_in + e);   // the pre-noise sigmoid (R itself without noise)
      sDz[idx] = dr * r1e * (1.f - r1e);
    }
    dw_acc = warp_sum(dw_acc);
    db_acc = warp_sum(db_acc);
    if (lane == 0) {
      red[0][warp] = dw_acc;
      red[1][warp] = db_acc;
    }
  }
  __syncthreads();
  if (hard_k < 0 && threadIdx.x < 2) {
    float t = 0.f;
#pragma unroll
    for (int wv = 0; wv < kFusedThreads / kWarp; ++wv) t += red[threadIdx.x][wv];
    if (t != 0.f) atomicAdd(ddeg + threadIdx.x, t);
  }
  // ---- phase B: per entry, d pre = dz LeakyReLU'(pre) from the forward's branch mask (y is not read), scattered;
  // every group walks a contiguous run (one flush of the source-row accumulator per row change), the indices and mask
  // words of the next entry prefetched ----
  const int W = (h + 31) >> 5;
  RowSlice<T> dbe_acc, acc;
#pragma unroll
  for (int t = 0; t < T; ++t) dbe_acc.v[t] = acc.v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int groups = (kFusedThreads / kWarp) * G;
  const int per = (nE + groups - 1) / groups;
  const int g0 = (warp * G + grp) * per;
  int cur_u = -1;
  int u_n = 0, v_n = 0;
  uint32_t nib_n[T];
  load_branch_mask<T>(nib_n, branch_mask + (size_t)(eb0 + g0) * W, h, lg, L, g0 < nE);
  if (g0 < nE) {
    u_n = __ldg(erow + eb0 + g0);
    v_n = __ldg(col + eb0 + g0);
  }
  for (int it = 0; it < per; ++it) {
    const int idx = g0 + it;
    const bool valid = idx < nE;
    const int u = u_n, v = v_n;
    uint32_t nib[T];
#pragma unroll
    for (int t = 0; t < T; ++t) nib[t] = nib_n[t];
    const bool next = it + 1 < per && idx + 1 < nE;
    if (next) {
      u_n = __ldg(erow + eb0 + idx + 1);
      v_n = __ldg(col + eb0 + idx + 1);
    }
    load_branch_mask<T>(nib_n, branch_mask + (size_t)(eb0 + idx + 1) * W, h, lg, L, next);
    const float dz = valid ? sDz[idx] : 0.f;
    if (valid && u != cur_u) {  // group-uniform branch: flush the finished source row
      if (cur_u >= 0) {
#pragma unroll
        for (int t = 0; t < T; ++t) {
          const int c = 4 * (lg + L * t);
          if (c < h) red_add4(dy + (size_t)cur_u * h + c, acc.v[t]);
          acc.v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      cur_u = u;
    }
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int c = 4 * (lg + L * t);
      const float4 d = branch_scale(nib[t], dz);
      dbe_acc.v[t].x += d.x; dbe_acc.v[t].y += d.y; dbe_acc.v[t].z += d.z; dbe_acc.v[t].w += d.w;
      if (valid && u != v) {  // a self loop adds +d and -d to the same row: skip both (it still counts for dbe)
        acc.v[t].x += d.x; acc.v[t].y += d.y; acc.v[t].z += d.z; acc.v[t].w += d.w;
        if (c < h) red_add4(dy + (size_t)v * h + c, make_float4(-d.x, -d.y, -d.z, -d.w));
      }
    }
  }
  if (cur_u >= 0) {
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int c = 4 * (lg + L * t);
      if (c < h) red_add4(dy + (size_t)cur_u * h + c, acc.v[t]);
    }
  }
#pragma unroll
  for (int t = 0; t < T; ++t) {
    for (int o = L; o < kWarp; o <<= 1) {
      dbe_acc.v[t].x += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].x, o);
      dbe_acc.v[t].y += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].y, o);
      dbe_acc.v[t].z += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].z, o);
      dbe_acc.v[t].w += __shfl_xor_sync(0xffffffffu, dbe_acc.v[t].w, o);
    }
    const int c = 4 * (lg + L * t);
    if (grp == 0 && c < h) {
      atomicAdd(&dbe_s[c + 0], dbe_acc.v[t].x);
      atomicAdd(&dbe_s[c + 1], dbe_acc.v[t].y);
      atomicAdd(&dbe_s[c + 2], dbe_acc.v[t].z);
      atomicAdd(&dbe_s[c + 3], dbe_acc.v[t].w);
    }
  }
  __syncthreads();
  // one 16-byte reduction per four columns: every block of the grid adds into the same h floats at about the same time,
  // and requests on one L2 line serialise (592 blocks x 64 scalar atomics = 38 k requests on two lines)
  if ((h & 3) == 0 && (reinterpret_cast<uintptr_t>(dbe) & 15) == 0) {
    for (int c = 4 * threadIdx.x; c < h; c += 4 * kFusedThreads)
      red_add4(dbe + c, make_float4(dbe_s[c], dbe_s[c + 1], dbe_s[c + 2], dbe_s[c + 3]));
  } else {
    for (int c = threadIdx.x; c < h; c += kFusedThreads) atomicAdd(dbe + c, dbe_s[c]);
  }
}

// grid of the fused kernels: at most one wave (blocks_per_sm from the occupancy calculator), >= 128 edges per block (measured 256 / 128 / 64: forward 16.8 / 14.1 / 14.1 us at Pubmed shape; DGGB_FUSED_EPB overrides)
// The override is read per call, so that one process can run several grids; values below 1 are ignored.
static void fused_grid(int nnz, int blocks_per_sm, int* blocks, int* epb) {
  const char* env = getenv("DGGB_FUSED_EPB");
  const int env_epb = env ? atoi(env) : 0;
  const int min_epb = env_epb >= 1 ? env_epb : 128;
  long long b = ((long long)nnz + min_epb - 1) / min_epb;
  const long long cap = (long long)kNumSMs * (blocks_per_sm < 1 ? 1 : blocks_per_sm);
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  *epb = (int)((nnz + b - 1) / b);
  *blocks = (nnz + *epb - 1) / *epb;
}

// instantiation of the fused kernels for hidden width h: fn(T, LC) with both as std::integral_constant, <4, L> for the
// usual widths h == 16 L (fully specialised), dispatch_T's runtime-L <T, 0> otherwise
template <typename F>
static int dispatch_fused(int h, int L, F&& fn) {
  using I4 = std::integral_constant<int, 4>;
  if (h == 16 * L) {
    switch (L) {
      case 1: return fn(I4{}, std::integral_constant<int, 1>{});
      case 2: return fn(I4{}, std::integral_constant<int, 2>{});
      case 4: return fn(I4{}, std::integral_constant<int, 4>{});
      case 8: return fn(I4{}, std::integral_constant<int, 8>{});
      case 16: return fn(I4{}, std::integral_constant<int, 16>{});
      default: return fn(I4{}, std::integral_constant<int, 32>{});
    }
  }
  return dispatch_T(h, L, [&](auto tc) { return fn(tc, std::integral_constant<int, 0>{}); });
}

// Without an opt-in a block gets at most 48 KB of shared memory, static and dynamic together: the largest score
// windows (12 288 floats in the forward, 2 x 6 144 in the backward) plus the kernels' static arrays exceed it.  The
// opt-in is only requested for large windows, so the small graphs' launches make no extra call.
template <typename K>
static int allow_dynamic_smem(K kern, size_t smem) {
  if (smem <= 40 * 1024) return DGGB_OK;
  return cuda_status(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
}

static int edges_grid(long long nnz, int blocks_per_sm = 8) {
  long long need = (nnz + kEdgeWarps * kWarp - 1) / (kEdgeWarps * kWarp);
  long long cap = (long long)kNumSMs * blocks_per_sm;
  long long g = need < cap ? need : cap;
  return (int)(g < 1 ? 1 : g);
}

}  // namespace dggb

using namespace dggb;

extern "C" int dggb_dgg_edge_fwd(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                                 int32_t nnz, int32_t h, const float* y, const float* be, const float* deg_w,
                                 const float* deg_b, const float* ablation_noise, int32_t hard_k, float* R,
                                 int32_t* rank, float* s, float* k, float* out, int32_t* long_ws, void* stream) {
  // the per-entry arrays may be NULL when there are no entries (an empty tensor has no data pointer)
  if (!rowptr || !y || !be || !deg_w || !deg_b || !s || !k || n < 0 || nnz < 0 || h <= 0 ||
      (nnz > 0 && (!erow || !col || !R || !rank || !out)))
    return DGGB_ERR_BAD_ARG;
  if (h % 4 != 0 || h > 512) return DGGB_ERR_BAD_SHAPE;
  if (n == 0) return DGGB_OK;
  const int L = lanes_per_edge(h);
  int st = DGGB_OK;
  if (nnz > 0) {
    st = dispatch_T(h, L, [&](auto tc) {
      constexpr int T = decltype(tc)::value;
      launch_pdl(dgg_edge_score_kernel<T>, dim3(edges_grid(nnz, resident_blocks(dgg_edge_score_kernel<T>, kEdgeWarps * kWarp))), dim3(kEdgeWarps * kWarp), 0, as_stream(stream), 
          erow, col, nnz, h, L, y, be, ablation_noise, R);
      return launch_status();
    });
    if (st != DGGB_OK) return st;
  }
  launch_pdl(dgg_row_rank_kernel, dim3(rows_grid(n, kEdgeWarps, resident_blocks(dgg_row_rank_kernel, kEdgeWarps * kWarp))), dim3(kEdgeWarps * kWarp), 0, as_stream(stream), 
      rowptr, n, R, deg_w, deg_b, hard_k, rank, s, k, out, long_ws);
  st = launch_status();
  if (st != DGGB_OK || long_ws == nullptr) return st;
  launch_long_rows(rowptr, R, k, hard_k >= 0 ? 3 : 2, hard_k, long_ws, rank, out, as_stream(stream));
  return launch_status();
}

extern "C" int dggb_dgg_edge_bwd(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                                 int32_t nnz, int32_t h, const float* y, const float* be, const float* deg_w,
                                 const float* deg_b, const float* ablation_noise, int32_t hard_k, const float* R,
                                 const int32_t* rank, const float* s, const float* k, const float* g_out,
                                 float* ds_ws, float* dy, float* dbe, float* ddeg, void* stream) {
  if (!rowptr || !y || !be || !deg_w || !deg_b || !s || !k || !ds_ws || !dy || !dbe || !ddeg || n < 0 || nnz < 0 ||
      h <= 0 || (nnz > 0 && (!erow || !col || !R || !rank || !g_out)))
    return DGGB_ERR_BAD_ARG;
  if (h % 4 != 0 || h > 512) return DGGB_ERR_BAD_SHAPE;
  if (n == 0 || nnz == 0) return DGGB_OK;
  const int L = lanes_per_edge(h);
  if (hard_k < 0) {
    launch_pdl(dgg_row_dk_kernel, dim3(rows_grid(n, kEdgeWarps, resident_blocks(dgg_row_dk_kernel, kEdgeWarps * kWarp))), dim3(kEdgeWarps * kWarp), 0, as_stream(stream), 
        rowptr, n, R, rank, s, k, g_out, deg_w, deg_b, ds_ws, ddeg);
    const int st = launch_status();
    if (st != DGGB_OK) return st;
  }
  return dispatch_T(h, L, [&](auto tc) {
    constexpr int T = decltype(tc)::value;
    launch_pdl(dgg_edge_grad_kernel<T>, dim3(edges_grid(nnz, resident_blocks(dgg_edge_grad_kernel<T>, kEdgeWarps * kWarp))), dim3(kEdgeWarps * kWarp), 0, as_stream(stream), 
        erow, col, nnz, h, L, y, be, ablation_noise, hard_k, R, rank, k, ds_ws, g_out, dy, dbe);
    return launch_status();
  });
}

extern "C" int dggb_row_firstk_fwd(const int32_t* rowptr, int32_t n, const float* score, const float* k,
                                   int32_t mode, int32_t* rank, float* out, int32_t* long_ws, void* stream) {
  if (!rowptr || !score || !k || !rank || !out || n < 0) return DGGB_ERR_BAD_ARG;
  if (mode != 0 && mode != 1) return DGGB_ERR_UNSUPPORTED;
  if (n == 0) return DGGB_OK;
  launch_pdl(row_firstk_fwd_kernel,
             dim3(rows_grid(n, kEdgeWarps, resident_blocks(row_firstk_fwd_kernel, kEdgeWarps * kWarp))),
             dim3(kEdgeWarps * kWarp), 0, as_stream(stream), rowptr, n, score, k, mode, rank, out, long_ws);
  const int st = launch_status();
  if (st != DGGB_OK || long_ws == nullptr) return st;
  launch_long_rows(rowptr, score, k, mode, -1, long_ws, rank, out, as_stream(stream));
  return launch_status();
}

extern "C" int dggb_row_firstk_bwd(const int32_t* rowptr, int32_t n, const float* score, const float* k,
                                   int32_t mode, const int32_t* rank, const float* g_out, float* dscore, float* dk,
                                   void* stream) {
  if (!rowptr || !score || !k || !rank || !g_out || !dscore || !dk || n < 0) return DGGB_ERR_BAD_ARG;
  if (mode != 0 && mode != 1) return DGGB_ERR_UNSUPPORTED;
  if (n == 0) return DGGB_OK;
  launch_pdl(row_firstk_bwd_kernel, dim3(rows_grid(n, kEdgeWarps, resident_blocks(row_firstk_bwd_kernel, kEdgeWarps * kWarp))), dim3(kEdgeWarps * kWarp), 0, as_stream(stream), 
      rowptr, n, score, k, mode, rank, g_out, dscore, dk);
  return launch_status();
}

extern "C" int dggb_dgg_edge_fwd_fused_mask(const int32_t* rowptr, const int32_t* erow, const int32_t* col,
                                            int32_t n, int32_t nnz, int32_t max_row_nnz, int32_t h, const float* y,
                                            const float* be, const float* deg_w, const float* deg_b,
                                            const float* ablation_noise, int32_t hard_k, float* R, int32_t* rank,
                                            float* s, float* k, float* out, uint32_t* branch_mask, float* r1,
                                            float* zero_ws, int64_t zero_count, void* stream) {
  if (!rowptr || !erow || !col || !y || !be || !deg_w || !deg_b || !R || !rank || !s || !k || !out || n < 0 ||
      nnz < 0 || h <= 0 || max_row_nnz < 0 || zero_count < 0 ||
      (branch_mask != nullptr && ablation_noise != nullptr && r1 == nullptr))   // the backward would lack r1
    return DGGB_ERR_BAD_ARG;
  if (h % 4 != 0 || h > 512) return DGGB_ERR_BAD_SHAPE;
  if (nnz == 0 || max_row_nnz > kFusedMaxDeg) return DGGB_ERR_UNSUPPORTED;   // use the two-launch entry point
  if (n == 0) return DGGB_OK;
  const int L = lanes_per_edge(h);
  return dispatch_fused(h, L, [&](auto tc, auto lc) {
    auto kern = dgg_fwd_fused2_kernel<decltype(tc)::value, decltype(lc)::value>;
    int occ = 0, blocks, epb;
    // the shared-memory slice depends on epb, which depends on the occupancy: size it for the smallest grid first
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kFusedThreads,
                                                  (size_t)(128 + max_row_nnz) * sizeof(float));
    fused_grid(nnz, occ, &blocks, &epb);
    // shared-memory score window: entries beyond it (bounded-degree graphs with > ~7 M entries make epb large)
    // are re-read from global memory by the rank phase (the `je <= cap` / `idx < cap` guards of the kernel)
    const int cap = min(epb + max_row_nnz, 12288);
    const int st = allow_dynamic_smem(kern, (size_t)cap * sizeof(float));
    if (st != DGGB_OK) return st;
    launch_pdl(kern, dim3(blocks), dim3(kFusedThreads), (size_t)cap * sizeof(float), as_stream(stream), rowptr, erow,
               col, n, nnz, h, L, epb, cap, y, be, ablation_noise, deg_w, deg_b, hard_k, R, rank, s, k, out,
               branch_mask, r1, zero_ws, (long long)zero_count);
    return launch_status();
  });
}

extern "C" int dggb_dgg_edge_bwd_fused_mask(const int32_t* rowptr, const int32_t* erow, const int32_t* col,
                                            int32_t n, int32_t nnz, int32_t max_row_nnz, int32_t h,
                                            const float* deg_w, const float* deg_b, const float* ablation_noise,
                                            int32_t hard_k, const float* R, const int32_t* rank, const float* s,
                                            const float* k, const uint32_t* branch_mask, const float* r1,
                                            const float* g_out, float* ds_ws, float* dy, float* dbe, float* ddeg,
                                            void* stream) {
  if (!rowptr || !erow || !col || !deg_w || !deg_b || !R || !rank || !s || !k || !branch_mask || !g_out || !ds_ws ||
      !dy || !dbe || !ddeg || n < 0 || nnz < 0 || h <= 0 || max_row_nnz < 0 || (ablation_noise && !r1))
    return DGGB_ERR_BAD_ARG;
  if (h % 4 != 0 || h > 512) return DGGB_ERR_BAD_SHAPE;
  if (nnz == 0 || max_row_nnz > kFusedMaxDeg) return DGGB_ERR_UNSUPPORTED;
  if (n == 0) return DGGB_OK;
  const int L = lanes_per_edge(h);
  const float* r1_in = ablation_noise ? r1 : R;   // the pre-noise sigmoid of every entry
  return dispatch_fused(h, L, [&](auto tc, auto lc) {
    constexpr int T = decltype(tc)::value, LC = decltype(lc)::value;
    // second generation: two shared-memory floats per entry of the block's window (epb + max_row_nnz entries), as
    // long as the window its one-wave grid gives fits 48 KB
    auto kern2 = dgg_bwd_fused2_kernel<T, LC>;
    int occ2 = 0, blocks, epb;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, kern2, kFusedThreads,
                                                  (size_t)(128 + max_row_nnz) * 2 * sizeof(float));
    fused_grid(nnz, occ2, &blocks, &epb);
    const int cap = epb + max_row_nnz;
    if (cap <= 6144) {
      const int st = allow_dynamic_smem(kern2, (size_t)cap * 2 * sizeof(float));
      if (st != DGGB_OK) return st;
      launch_pdl(kern2, dim3(blocks), dim3(kFusedThreads), (size_t)cap * 2 * sizeof(float), as_stream(stream),
                 rowptr, erow, col, n, nnz, h, L, epb, cap, branch_mask, r1_in, ablation_noise, hard_k, R, rank, s, k,
                 g_out, deg_w, deg_b, ds_ws, dy, dbe, ddeg);
      return launch_status();
    }
    // larger windows: dgg_bwd_fused_kernel, on the grid of its own occupancy
    auto kern = dgg_bwd_fused_kernel<T, LC>;
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kFusedThreads, 0);
    fused_grid(nnz, occ, &blocks, &epb);
    launch_pdl(kern, dim3(blocks), dim3(kFusedThreads), 0, as_stream(stream), rowptr, erow, col, n, nnz, h, L, epb,
               branch_mask, r1_in, ablation_noise, hard_k, R, rank, s, k, g_out, deg_w, deg_b, ds_ws, dy, dbe, ddeg);
    return launch_status();
  });
}

// The fused entry points without the branch mask.  The forward is the masked one writing no mask.  The backward keeps
// its arguments and its accumulate-into contract but has no mask to read: it runs the two-launch backward, which
// recomputes the pre-activations from y (the dbe flush there uses scalar atomics, so any dbe alignment is fine).
extern "C" int dggb_dgg_edge_fwd_fused(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                                       int32_t nnz, int32_t max_row_nnz, int32_t h, const float* y, const float* be,
                                       const float* deg_w, const float* deg_b, const float* ablation_noise,
                                       int32_t hard_k, float* R, int32_t* rank, float* s, float* k, float* out,
                                       float* zero_ws, int64_t zero_count, void* stream) {
  return dggb_dgg_edge_fwd_fused_mask(rowptr, erow, col, n, nnz, max_row_nnz, h, y, be, deg_w, deg_b, ablation_noise,
                                      hard_k, R, rank, s, k, out, nullptr, nullptr, zero_ws, zero_count, stream);
}

extern "C" int dggb_dgg_edge_bwd_fused(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                                       int32_t nnz, int32_t max_row_nnz, int32_t h, const float* y, const float* be,
                                       const float* deg_w, const float* deg_b, const float* ablation_noise,
                                       int32_t hard_k, const float* R, const int32_t* rank, const float* s,
                                       const float* k, const float* g_out, float* ds_ws, float* dy, float* dbe,
                                       float* ddeg, void* stream) {
  if (!rowptr || !erow || !col || !y || !be || !deg_w || !deg_b || !R || !rank || !s || !k || !g_out || !ds_ws ||
      !dy || !dbe || !ddeg || n < 0 || nnz < 0 || h <= 0 || max_row_nnz < 0)
    return DGGB_ERR_BAD_ARG;
  if (h % 4 != 0 || h > 512) return DGGB_ERR_BAD_SHAPE;
  if (nnz == 0 || max_row_nnz > kFusedMaxDeg) return DGGB_ERR_UNSUPPORTED;
  if (n == 0) return DGGB_OK;
  return dggb_dgg_edge_bwd(rowptr, erow, col, n, nnz, h, y, be, deg_w, deg_b, ablation_noise, hard_k, R, rank, s, k,
                           g_out, ds_ws, dy, dbe, ddeg, stream);
}
