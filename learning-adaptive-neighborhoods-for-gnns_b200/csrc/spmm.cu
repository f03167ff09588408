// CSR SpMM Y = A X (+ optional per-row scale) and its backward (dX = A^T dY via vector reductions,
// dA = SDDMM).  Replaces torch.mm(adj_dense, x) (model.py:594, 67) and PyG DenseGraphConv's adj @ x.
// Warp per row; the 32 lanes split into G groups of L lanes, a group gathers one neighbour row at a
// time with VEC-wide (128-bit when F % 4 == 0) coalesced loads.
// HBM-bound: nnz*(8 + F*4 gathered) + N*F*4 bytes.
#include "common.cuh"
#include <cstdio>
#include <cstdlib>

namespace dggb {

constexpr int kSpmmWarps = 8;

template <int VEC> struct Vec;
template <> struct Vec<4> {
  float4 v;
  __device__ __forceinline__ void zero() { v = make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ void load(const float* p) { v = __ldg(reinterpret_cast<const float4*>(p)); }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = v; }
  __device__ __forceinline__ void fma(float a, const Vec& o) { v.x += a * o.v.x; v.y += a * o.v.y; v.z += a * o.v.z; v.w += a * o.v.w; }
  __device__ __forceinline__ void scale(float a) { v.x *= a; v.y *= a; v.z *= a; v.w *= a; }
  __device__ __forceinline__ float dot(const Vec& o) const { return v.x * o.v.x + v.y * o.v.y + v.z * o.v.z + v.w * o.v.w; }
  __device__ __forceinline__ void xor_add(int o) {
    v.x += __shfl_xor_sync(0xffffffffu, v.x, o); v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
    v.z += __shfl_xor_sync(0xffffffffu, v.z, o); v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
  }
  __device__ __forceinline__ void red(float* p, float a) const { red_add4(p, make_float4(a * v.x, a * v.y, a * v.z, a * v.w)); }
  __device__ __forceinline__ void mul(const Vec& o) { v.x *= o.v.x; v.y *= o.v.y; v.z *= o.v.z; v.w *= o.v.w; }
};
template <> struct Vec<2> {
  float2 v;
  __device__ __forceinline__ void zero() { v = make_float2(0.f, 0.f); }
  __device__ __forceinline__ void load(const float* p) { v = __ldg(reinterpret_cast<const float2*>(p)); }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float2*>(p) = v; }
  __device__ __forceinline__ void fma(float a, const Vec& o) { v.x += a * o.v.x; v.y += a * o.v.y; }
  __device__ __forceinline__ void scale(float a) { v.x *= a; v.y *= a; }
  __device__ __forceinline__ float dot(const Vec& o) const { return v.x * o.v.x + v.y * o.v.y; }
  __device__ __forceinline__ void xor_add(int o) {
    v.x += __shfl_xor_sync(0xffffffffu, v.x, o); v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
  }
  __device__ __forceinline__ void red(float* p, float a) const {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a * v.x), "f"(a * v.y) : "memory");
  }
};
template <> struct Vec<1> {
  float v;
  __device__ __forceinline__ void zero() { v = 0.f; }
  __device__ __forceinline__ void load(const float* p) { v = __ldg(p); }
  __device__ __forceinline__ void store(float* p) const { *p = v; }
  __device__ __forceinline__ void fma(float a, const Vec& o) { v += a * o.v; }
  __device__ __forceinline__ void scale(float a) { v *= a; }
  __device__ __forceinline__ float dot(const Vec& o) const { return v * o.v; }
  __device__ __forceinline__ void xor_add(int o) { v += __shfl_xor_sync(0xffffffffu, v, o); }
  __device__ __forceinline__ void red(float* p, float a) const { atomicAdd(p, a * v); }
};

// Both kernels first pull a 32-entry window of the row's (col, val) pairs into registers with one coalesced
// load per lane and then broadcast them with shuffles: the neighbour-row gathers no longer wait on a dependent
// index load, and several of them are in flight per group (unroll 4).
// (Tried and measured slower at Pubmed shape, model-step graph replay 0.371 -> 0.396 / 0.470 ms: one row per L-lane
// group with the entries read sequentially, with and without a per-warp shared-memory entry window.)
template <int VEC, int T>
__global__ void __launch_bounds__(kSpmmWarps* kWarp)
    spmm_fwd_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                    const float* __restrict__ val, int n, const float* __restrict__ x, int f, int L,
                    const float* __restrict__ row_scale, float* __restrict__ y) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int G = kWarp / L, lg = lane % L, grp = lane / L;
  const int W = VEC * L * T;  // columns covered per pass
  for (int i = blockIdx.x * kSpmmWarps + (threadIdx.x >> 5); i < n; i += gridDim.x * kSpmmWarps) {
    const int beg = __ldg(rowptr + i), end = __ldg(rowptr + i + 1);
    const float rs = row_scale ? __ldg(row_scale + i) : 1.f;
    for (int f0 = 0; f0 < f; f0 += W) {
      Vec<VEC> acc[T];
#pragma unroll
      for (int t = 0; t < T; ++t) acc[t].zero();
      for (int w0 = beg; w0 < end; w0 += kWarp) {
        const int e_l = w0 + lane;
        const int c_l = (e_l < end) ? __ldg(col + e_l) : 0;
        const float a_l = (e_l < end) ? __ldg(val + e_l) : 0.f;
        const int cnt = min(kWarp, end - w0);
#pragma unroll 4
        for (int j0 = 0; j0 < cnt; j0 += G) {
          const int j = j0 + grp;
          const int v = __shfl_sync(0xffffffffu, c_l, j & 31);
          const float a = __shfl_sync(0xffffffffu, a_l, j & 31);   // shuffles stay outside any lane-dependent condition
          const float* xr = x + (size_t)v * f;
#pragma unroll
          for (int t = 0; t < T; ++t) {
            const int c = f0 + VEC * (lg + L * t);
            // groups beyond the row's entries issue no load: their index is 0, and row 0 would be one hot L2 line for
            // every short row of the grid (see gcnii_stack_fwd_kernel)
            if (c < f && j < cnt) {
              Vec<VEC> xv;
              xv.load(xr + c);
              acc[t].fma(a, xv);
            }
          }
        }
      }
#pragma unroll
      for (int t = 0; t < T; ++t) {
        for (int o = L; o < kWarp; o <<= 1) acc[t].xor_add(o);
        const int c = f0 + VEC * (lg + L * t);
        if (grp == 0 && c < f) {
          acc[t].scale(rs);
          acc[t].store(y + (size_t)i * f + c);
        }
      }
    }
  }
}

template <int VEC, int T>
__global__ void __launch_bounds__(kSpmmWarps* kWarp)
    spmm_bwd_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                    const float* __restrict__ val, int n, const float* __restrict__ x, int f, int L,
                    const float* __restrict__ row_scale, const float* __restrict__ dy, float* __restrict__ dval,
                    float* __restrict__ dx) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int G = kWarp / L, lg = lane % L, grp = lane / L;
  const int W = VEC * L * T;
  for (int i = blockIdx.x * kSpmmWarps + (threadIdx.x >> 5); i < n; i += gridDim.x * kSpmmWarps) {
    const int beg = __ldg(rowptr + i), end = __ldg(rowptr + i + 1);
    const float rs = row_scale ? __ldg(row_scale + i) : 1.f;
    for (int f0 = 0; f0 < f; f0 += W) {
      Vec<VEC> g[T];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int c = f0 + VEC * (lg + L * t);
        if (c < f) {
          g[t].load(dy + (size_t)i * f + c);
          g[t].scale(rs);
        } else {
          g[t].zero();
        }
      }
      for (int w0 = beg; w0 < end; w0 += kWarp) {
        const int e_l = w0 + lane;
        const int c_l = (e_l < end) ? __ldg(col + e_l) : 0;
        const float a_l = (e_l < end) ? __ldg(val + e_l) : 0.f;
        const int cnt = min(kWarp, end - w0);
#pragma unroll 2
        for (int j0 = 0; j0 < cnt; j0 += G) {
          const int j = j0 + grp;
          const bool valid = j < cnt;
          const int v = __shfl_sync(0xffffffffu, c_l, j & 31);
          const float a = __shfl_sync(0xffffffffu, a_l, j & 31);
          float dot = 0.f;
#pragma unroll
          for (int t = 0; t < T; ++t) {
            const int c = f0 + VEC * (lg + L * t);
            if (c < f && valid) {
              if (dval) {
                Vec<VEC> xv;
                xv.load(x + (size_t)v * f + c);
                dot += g[t].dot(xv);
              }
              if (dx) g[t].red(dx + (size_t)v * f + c, a);
            }
          }
          if (dval) {
            dot = group_sum(dot, L);
            // the G group leaders hold G consecutive entries of the row: one coalesced store
            if (lg == 0 && valid) dval[w0 + j] = (f0 == 0) ? dot : dval[w0 + j] + dot;
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Edge-parallel SpMM for short-row graphs (citation graphs: ~5 entries per row, F = 64).  The warp-per-row kernels
// above spend most of their ~450 instructions per row on per-row bookkeeping and on the cross-group shuffle
// reduction (profiles/r01_h: 9 M warp instructions for 19.7 k rows, 22 us for 33 MB).  Here a group of L lanes walks
// a contiguous run of kRun entries (CSR order, so consecutive entries share their row), keeps the running row sum in
// registers and flushes it when the row changes: a row that lies entirely inside one run is written with plain
// stores, a row cut by a run boundary is combined with 128-bit vector reductions -- y must therefore be ZEROED by the
// caller.  Perfectly balanced under any degree distribution (a 171-entry hub row is just 22 runs), ~40 instructions
// per entry-group.  Backward: per entry, dval_e = rs_u <dy_u, x_v> and dx_v += a_e rs_u dy_u, no flush logic at all.
// The run length adapts to the graph (1-8 entries) so that small graphs still fill the machine.  Measured inside a
// CUDA graph, F = 64 (scripts/small_micro.py): Pubmed shape forward 9.7 us incl. the zero fill (warp per row: 15.2),
// backward 7.7 us (21.7); Citeseer shape 5.0 us (7.7) and 3.4 us (13.6).
// ------------------------------------------------------------------------------------------------
constexpr int kRunMax = 8;   // entries per run; shorter on small graphs so that every SM gets work

template <int T>
__global__ void __launch_bounds__(kSpmmWarps* kWarp)
    spmm_edge_fwd_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ erow,
                         const int32_t* __restrict__ col, const float* __restrict__ val, long long nnz,
                         const float* __restrict__ x, int f, int L, int kRun, const float* __restrict__ row_scale,
                         float* __restrict__ y) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int G = kWarp / L, lg = lane % L, grp = lane / L;
  const long long groups_total = (long long)gridDim.x * kSpmmWarps * G;
  const long long runs = (nnz + kRun - 1) / kRun;
  for (long long run = ((long long)blockIdx.x * kSpmmWarps + (threadIdx.x >> 5)) * G + grp; run < runs;
       run += groups_total) {
    const long long e0 = run * kRun, e1 = min(nnz, e0 + kRun);
    int cur = -1;
    float4 acc[T];
#pragma unroll
    for (int t = 0; t < T; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    auto flush = [&]() {
      if (cur < 0) return;
      const float rs = row_scale ? __ldg(row_scale + cur) : 1.f;
      const bool whole = __ldg(rowptr + cur) >= e0 && __ldg(rowptr + cur + 1) <= e1;   // nobody else adds to this row
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int c = 4 * (lg + L * t);
        if (c < f) {
          const float4 v = make_float4(rs * acc[t].x, rs * acc[t].y, rs * acc[t].z, rs * acc[t].w);
          if (whole) st4(y + (size_t)cur * f + c, v);
          else red_add4(y + (size_t)cur * f + c, v);
        }
        acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
#pragma unroll 2
    for (long long e = e0; e < e1; ++e) {
      const int u = __ldg(erow + e), v = __ldg(col + e);
      const float a = __ldg(val + e);
      if (u != cur) {          // group-uniform
        flush();
        cur = u;
      }
      const float* xr = x + (size_t)v * f;
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int c = 4 * (lg + L * t);
        if (c < f) {
          const float4 xv = ldg4(xr + c);
          acc[t].x = fmaf(a, xv.x, acc[t].x); acc[t].y = fmaf(a, xv.y, acc[t].y);
          acc[t].z = fmaf(a, xv.z, acc[t].z); acc[t].w = fmaf(a, xv.w, acc[t].w);
        }
      }
    }
    flush();
  }
}

template <int T>
__global__ void __launch_bounds__(kSpmmWarps* kWarp)
    spmm_edge_bwd_kernel(const int32_t* __restrict__ erow, const int32_t* __restrict__ col,
                         const float* __restrict__ val, long long nnz, const float* __restrict__ x, int f, int L,
                         int kRun, const float* __restrict__ row_scale, const float* __restrict__ dy,
                         float* __restrict__ dval, float* __restrict__ dx) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int G = kWarp / L, lg = lane % L, grp = lane / L;
  const long long groups_total = (long long)gridDim.x * kSpmmWarps * G;
  const long long runs = (nnz + kRun - 1) / kRun;
  for (long long run = ((long long)blockIdx.x * kSpmmWarps + (threadIdx.x >> 5)) * G + grp; run < runs;
       run += groups_total) {
    const long long e0 = run * kRun, e1 = min(nnz, e0 + kRun);
    int cur = -1;
    float4 g[T];
#pragma unroll 2
    for (long long e = e0; e < e1; ++e) {
      const int u = __ldg(erow + e), v = __ldg(col + e);
      const float a = __ldg(val + e);
      if (u != cur) {          // group-uniform: this row's (scaled) output gradient stays in registers for its entries
        cur = u;
        const float rs = row_scale ? __ldg(row_scale + u) : 1.f;
#pragma unroll
        for (int t = 0; t < T; ++t) {
          const int c = 4 * (lg + L * t);
          g[t] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (c < f) {
            g[t] = ldg4(dy + (size_t)u * f + c);
            g[t].x *= rs; g[t].y *= rs; g[t].z *= rs; g[t].w *= rs;
          }
        }
      }
      float dot = 0.f;
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int c = 4 * (lg + L * t);
        if (c < f) {
          if (dval) {
            const float4 xv = ldg4(x + (size_t)v * f + c);
            dot += g[t].x * xv.x + g[t].y * xv.y + g[t].z * xv.z + g[t].w * xv.w;
          }
          if (dx) red_add4(dx + (size_t)v * f + c, make_float4(a * g[t].x, a * g[t].y, a * g[t].z, a * g[t].w));
        }
      }
      if (dval) {
        dot = group_sum(dot, L);
        if (lg == 0) dval[e] = dot;
      }
    }
  }
}

// run length: 8 entries when that still gives every SM ~4 blocks of work, shorter on small graphs (Cora: 13 k entries)
static int edge_run_len(long long nnz, int L) {
  const int G = kWarp / L;
  const long long groups_wanted = (long long)kNumSMs * 4 * kSpmmWarps * G;
  long long r = nnz / groups_wanted;
  return (int)(r < 1 ? 1 : (r > kRunMax ? kRunMax : r));
}

static int edge_spmm_grid(long long nnz, int L, int kRun, int blocks_per_sm) {
  const int G = kWarp / L;
  const long long runs = (nnz + kRun - 1) / kRun;
  long long need = (runs + (long long)kSpmmWarps * G - 1) / ((long long)kSpmmWarps * G);
  long long cap = (long long)kNumSMs * (blocks_per_sm < 1 ? 1 : blocks_per_sm);
  long long g = need < cap ? need : cap;
  return (int)(g < 1 ? 1 : g);
}

// ------------------------------------------------------------------------------------------------
// SpMM with the layer's dense part folded in (GCNConv model.py:594-598, GraphConvolution / DenseGraphConvolution
// model.py:32-44, 65-77): per row, in one pass,
//     agg_i = rs_i * sum_e a_e x[col_e]                      (128-bit gathers, as spmm_fwd_kernel)
//     s_i   = c1 * agg_i + c2 * h0_i                         (GCNII initial residual; c2 = 0: none)
//     y_i   = act( theta * (s_i W) + beta * s_i + resid_i )  (W [Fin, Fout] in shared memory; act: identity / ReLU)
// instead of SpMM -> axpby -> cuBLAS mm -> axpby -> add -> relu (six launches and four [N, F] round trips per layer;
// the 64-layer GCNII stack is launch-bound at Citeseer size).  s is written out once (the weight gradient
// dW = theta * s^T dY needs it).  Fin % 4 == 0, Fin <= 128, Fout <= 128.
// Backward: ds_i = theta * (g_i W^T) + beta * g_i (W^T in shared memory), then the SpMM backward with c1 * ds_i:
//     dval_e = rs_i <c1 ds_i, x_col>,  dx_col += a_e rs_i c1 ds_i;   ds is written out (d h0 = c2 ds).
// ------------------------------------------------------------------------------------------------
struct SpmmGemmArgs {
  const int32_t* rowptr;
  const int32_t* col;
  const float* val;
  int n, fin, fout, L;
  const float* x;
  const float* row_scale;
  const float* h0;
  const float* w;        // [fin, fout]
  const float* resid;    // [n, fout] or NULL
  float c1, c2, theta, beta;
  int relu;
  int accum;             // backward: bit 0: dval += (instead of =), bit 1: ds_out += -- layers of a stack that share the
                         // adjacency values / h0 accumulate their gradients in place (autograd would add 64 tensors)
  const float* okeep;    // [n, fout] or NULL: dropout multipliers (0 or 1/(1-p)) applied to the layer OUTPUT in the
                         // epilogue (the next layer's F.dropout(input) and its backward are two launches per layer and
                         // direction otherwise; a per-row product, not a per-entry gather)
};

// RB = rows per warp iteration: the W tile is read from shared memory once per RB rows (RB = 4: large graphs, the
// dense part dominates; RB = 1: small graphs -- every row gets its own warp, the dependent-load latency of the
// aggregation is what a 3 k-node layer costs, measured 25.7 -> see DESIGN.md)

// dense part for RB rows at once: out[r][c] = sum_f S[r][f] * M[f][c];  lane owns columns c = lane + 32 q (q < 4).
// S rows are read as broadcast float4, M as conflict-free scalars: 3 LDS per 8 (RB * 2) FMAs at 64 columns.
template <int Q, int RB>
__device__ __forceinline__ void dense_rows(const float* __restrict__ S, int ld_s, const float* __restrict__ M, int k_dim,
                                           int n_cols, int lane, float (&acc)[RB][Q]) {
#pragma unroll
  for (int r = 0; r < RB; ++r)
#pragma unroll
    for (int q = 0; q < Q; ++q) acc[r][q] = 0.f;
  for (int f = 0; f < k_dim; f += 4) {
    float4 sv[RB];
#pragma unroll
    for (int r = 0; r < RB; ++r) sv[r] = *reinterpret_cast<const float4*>(S + r * ld_s + f);
#pragma unroll
    for (int ff = 0; ff < 4; ++ff) {
      float mv[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int c = lane + 32 * q;
        mv[q] = (c < n_cols) ? M[(f + ff) * n_cols + c] : 0.f;
      }
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        const float sf = ff == 0 ? sv[r].x : (ff == 1 ? sv[r].y : (ff == 2 ? sv[r].z : sv[r].w));
#pragma unroll
        for (int q = 0; q < Q; ++q) acc[r][q] = fmaf(sf, mv[q], acc[r][q]);
      }
    }
  }
}

// Block b owns the kSpmmWarps * RB consecutive rows [r0, r1) and therefore the contiguous entry range
// [rowptr[r0], rowptr[r1]).  Phase 1 (aggregation) is ENTRY-parallel inside the block: groups of L lanes walk runs of
// consecutive entries, keep the running row sum in registers and add it to the row's accumulator in shared memory
// when the row changes (shared-memory atomics: rows are only ever touched by their own block) -- balanced under any
// degree distribution inside the block, no per-row shuffle reduction.  Phase 2 (dense part) is row-parallel: each warp
// takes RB rows out of shared memory.  (r02 measurements of the first version, warp-per-row aggregation: 32 us at
// Pubmed shape against 9.7 + 3.7 us for the entry-parallel SpMM + a library GEMM.)
// rp = the block's slice of rowptr in SHARED memory (rp[j] = rowptr[r0 + j], j <= nr): the search and the row
// boundaries of phase 1 were 4-6 dependent global loads per group on the critical path of a 3 k-node layer
__device__ __forceinline__ int row_of_entry(const int* rp, int nr, int e) {
  int lo = 0, hi = nr - 1;                          // last local row j in [0, nr) with rp[j] <= e
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (rp[mid] <= e) lo = mid; else hi = mid - 1;
  }
  return lo;
}
// W (or any [count] fp32 array) global -> shared, 128-bit when both sides allow
__device__ __forceinline__ void stage_floats(float* dst, const float* __restrict__ src, int count) {
  if ((count & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
    for (int c = threadIdx.x; c < count / 4; c += blockDim.x) reinterpret_cast<float4*>(dst)[c] = ldg4(src + 4 * c);
  } else {
    for (int c = threadIdx.x; c < count; c += blockDim.x) dst[c] = __ldg(src + c);
  }
}

template <int T, int Q, int RB>
__global__ void __launch_bounds__(kSpmmWarps* kWarp)
    spmm_gemm_fwd_kernel(SpmmGemmArgs A, float* __restrict__ y, float* __restrict__ s_out) {
  constexpr int R = kSpmmWarps * RB;
  pdl_trigger();
  extern __shared__ __align__(16) float sm[];
  float* Ws = sm;                                   // [fin][fout]
  float* S = sm + A.fin * A.fout;                   // [R][fin] row accumulators, then s
  int* rp = reinterpret_cast<int*>(S + R * A.fin);  // [R + 1] this block's slice of rowptr
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = A.L, G = kWarp / L, lg = lane % L, grp = lane / L;
  const int r0 = blockIdx.x * R, r1 = min(A.n, r0 + R), nr = r1 - r0;
  for (int c = threadIdx.x; c < R * A.fin; c += blockDim.x) S[c] = 0.f;
  pdl_wait();
  // everything the block needs from global memory besides the gathered rows goes in flight together: W, the rowptr
  // slice, and -- into registers -- the phase-2 operands of this warp's rows (row_scale, h0, resid)
  stage_floats(Ws, A.w, A.fin * A.fout);
  for (int c = threadIdx.x; c <= nr; c += blockDim.x) rp[c] = __ldg(A.rowptr + r0 + c);
  float k1v[RB], h0v[RB][4], rsv[RB][Q];
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    const int i = r0 + warp * RB + r;
    const bool ok = i < A.n;
    k1v[r] = A.c1 * ((A.row_scale && ok) ? __ldg(A.row_scale + i) : 1.f);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = lane + 32 * j;
      h0v[r][j] = (A.h0 && ok && c < A.fin) ? __ldg(A.h0 + (size_t)i * A.fin + c) : 0.f;
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int c = lane + 32 * q;
      rsv[r][q] = (A.resid && ok && c < A.fout) ? __ldg(A.resid + (size_t)i * A.fout + c) : 0.f;
    }
  }
  __syncthreads();
  // ---- phase 1: entry-parallel aggregation into S ----
  {
    const int eb0 = rp[0], eb1 = rp[nr];
    const int nE = eb1 - eb0, groups = kSpmmWarps * G;
    const int per = (nE + groups - 1) / groups;
    const int e_beg = eb0 + (warp * G + grp) * per, e_end = min(eb1, e_beg + per);
    if (e_beg < e_end) {
      int cur = row_of_entry(rp, nr, e_beg);        // local row
      int next_start = rp[cur + 1];
      Vec<4> acc[T];
#pragma unroll
      for (int t = 0; t < T; ++t) acc[t].zero();
      auto flush = [&]() {
#pragma unroll
        for (int t = 0; t < T; ++t) {
          const int c = 4 * (lg + L * t);
          if (c < A.fin) {
            float* d = S + cur * A.fin + c;
            atomicAdd(d + 0, acc[t].v.x); atomicAdd(d + 1, acc[t].v.y);
            atomicAdd(d + 2, acc[t].v.z); atomicAdd(d + 3, acc[t].v.w);
          }
          acc[t].zero();
        }
      };
#pragma unroll 2
      for (int e = e_beg; e < e_end; ++e) {
        while (e >= next_start) {                   // group-uniform: the run crossed into the next (non-empty) row
          flush();
          ++cur;
          next_start = rp[cur + 1];
        }
        const int v = __ldg(A.col + e);
        const float a = __ldg(A.val + e);
        const float* xr = A.x + (size_t)v * A.fin;
#pragma unroll
        for (int t = 0; t < T; ++t) {
          const int c = 4 * (lg + L * t);
          if (c < A.fin) {
            Vec<4> xv;
            xv.load(xr + c);
            acc[t].fma(a, xv);
          }
        }
      }
      flush();
    }
  }
  __syncthreads();
  // ---- phase 2: s = c1 rs agg + c2 h0 (in place), y = act(theta s W + beta s + resid), RB rows per warp ----
  // s_out receives theta * s: its only consumer is the weight gradient dW = theta s^T dY
  float* srows = S + warp * RB * A.fin;
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    const int i = r0 + warp * RB + r;
    if (i >= A.n) break;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = lane + 32 * j;
      if (c < A.fin) {
        const float v = fmaf(A.c2, h0v[r][j], k1v[r] * srows[r * A.fin + c]);
        srows[r * A.fin + c] = v;
        if (s_out) s_out[(size_t)i * A.fin + c] = A.theta * v;
      }
    }
  }
  __syncwarp();
  float d[RB][Q];
  dense_rows<Q, RB>(srows, A.fin, Ws, A.fin, A.fout, lane, d);
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    const int i = r0 + warp * RB + r;
    if (i >= A.n) break;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int c = lane + 32 * q;
      if (c < A.fout) {
        float v = A.theta * d[r][q];
        if (A.beta != 0.f) v = fmaf(A.beta, srows[r * A.fin + c], v);      // fout == fin (checked on the host)
        v += rsv[r][q];
        if (A.relu) v = fmaxf(v, 0.f);
        if (A.okeep) v *= __ldg(A.okeep + (size_t)i * A.fout + c);
        y[(size_t)i * A.fout + c] = v;
      }
    }
  }
}

// Small graphs (one row per warp): the entry-parallel aggregation above combines the partial rows with shared-memory
// float atomics (a CAS loop each) and two block barriers -- at Citeseer size (3 327 rows, ~4 entries per row) the ncu
// source view charged 27 % of the instructions and 30 % of the stall samples to those atomics and another 24 % of the
// samples to the barrier behind them (17 us per layer).  Here lane == column: the warp walks its row's entries, every
// neighbour row is one or two coalesced 128-byte loads, eight entries in flight, the sum lands in the registers of the
// lanes that own the columns -- no reduction, no atomics, no barrier besides the one behind the W staging.
template <int Q>
__global__ void __launch_bounds__(kSpmmWarps* kWarp)
    spmm_gemm_fwd_row_kernel(SpmmGemmArgs A, float* __restrict__ y, float* __restrict__ s_out) {
  pdl_trigger();
  extern __shared__ __align__(16) float sm[];
  float* Ws = sm;                                   // [fin][fout]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* srow = sm + A.fin * A.fout + warp * A.fin; // this warp's row of s
  const int i = blockIdx.x * kSpmmWarps + warp;
  const bool ok = i < A.n;
  pdl_wait();
  stage_floats(Ws, A.w, A.fin * A.fout);
  const int beg = ok ? __ldg(A.rowptr + i) : 0, end = ok ? __ldg(A.rowptr + i + 1) : 0;
  const float k1 = A.c1 * ((A.row_scale && ok) ? __ldg(A.row_scale + i) : 1.f);
  float h0v[4], rsv[Q], acc[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = lane + 32 * j;
    h0v[j] = (A.h0 && ok && c < A.fin) ? __ldg(A.h0 + (size_t)i * A.fin + c) : 0.f;
    acc[j] = 0.f;
  }
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const int c = lane + 32 * q;
    rsv[q] = (A.resid && ok && c < A.fout) ? __ldg(A.resid + (size_t)i * A.fout + c) : 0.f;
  }
  const int nj = (A.fin + 31) >> 5;
  for (int e0 = beg; e0 < end; e0 += kWarp) {
    const int e = e0 + lane;
    const int c_l = (e < end) ? __ldg(A.col + e) : 0;
    const float a_l = (e < end) ? __ldg(A.val + e) : 0.f;
    const int cnt = min(kWarp, end - e0);
    for (int k0 = 0; k0 < cnt; k0 += 8) {
      float xv[8][4];
      float av[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {                 // slots beyond the row issue no load (see gcnii_stack_fwd_kernel:
        const int v = __shfl_sync(0xffffffffu, c_l, (k0 + k) & 31);   // a shared dummy row is one hot L2 line for the grid)
        const bool live = k0 + k < cnt;
        av[k] = live ? __shfl_sync(0xffffffffu, a_l, (k0 + k) & 31) : 0.f;
        const float* xr = A.x + (size_t)(live ? v : 0) * A.fin;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = lane + 32 * j;
          xv[k][j] = (live && j < nj && c < A.fin) ? __ldg(xr + c) : 0.f;
        }
      }
#pragma unroll
      for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j] = fmaf(av[k], xv[k][j], acc[j]);
    }
  }
  // s = c1 rs agg + c2 h0;  s_out receives theta * s (see spmm_gemm_fwd_kernel)
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = lane + 32 * j;
    if (c < A.fin) {
      const float v = fmaf(A.c2, h0v[j], k1 * acc[j]);
      srow[c] = v;
      if (s_out && ok) s_out[(size_t)i * A.fin + c] = A.theta * v;
    }
  }
  __syncthreads();                                  // W staged (and this warp's srow written)
  float d[1][Q];
  dense_rows<Q, 1>(srow, A.fin, Ws, A.fin, A.fout, lane, d);
  if (!ok) return;
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const int c = lane + 32 * q;
    if (c < A.fout) {
      float v = A.theta * d[0][q];
      if (A.beta != 0.f) v = fmaf(A.beta, srow[c], v);                     // fout == fin (checked on the host)
      v += rsv[q];
      if (A.relu) v = fmaxf(v, 0.f);
      if (A.okeep) v *= __ldg(A.okeep + (size_t)i * A.fout + c);
      y[(size_t)i * A.fout + c] = v;
    }
  }
}

template <int T, int Q, int RB>
__global__ void __launch_bounds__(kSpmmWarps* kWarp)
    spmm_gemm_bwd_kernel(SpmmGemmArgs A, const float* __restrict__ gy, float* __restrict__ dval,
                         float* __restrict__ dx, float* __restrict__ ds_out, float ds_scale, float* zero_ws,
                         long long zero_count, const float* __restrict__ relu_y, float* __restrict__ gy_masked) {
  constexpr int R = kSpmmWarps * RB;
  pdl_trigger();
  extern __shared__ __align__(16) float sm[];
  // W as it lies in memory ([fin][fout]) with rows padded to fout + 1 floats: lane f reads Wp[f][c] without bank
  // conflicts, and the staging is a straight copy (the transposed copy of the first version -- 32-way conflicting
  // stores plus a division per element -- was 36 % of this kernel's stall samples at Citeseer size)
  float* Wp = sm;
  const int wp = A.fout + 1;
  const int fo4 = (A.fout + 3) & ~3;                        // 16-byte aligned rows
  float* Gs = sm + ((A.fin * wp + 3) & ~3);                 // [R][fo4] rows of gy
  float* DS = Gs + R * fo4;                                 // [R][fin]  ds rows (scaled by c1 rs for phase B)
  int* rp = reinterpret_cast<int*>(DS + R * A.fin);         // [R + 1] this block's slice of rowptr
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = A.L, G = kWarp / L, lg = lane % L, grp = lane / L;
  const int r0 = blockIdx.x * R, r1 = min(A.n, r0 + R), nr = r1 - r0;
  pdl_wait();
  zero_fill(zero_ws, zero_count);       // the split-K buffer of the weight gradient that follows this launch
  if ((A.fout & 3) == 0 && (reinterpret_cast<uintptr_t>(A.w) & 15) == 0) {
    const int per_row = A.fout >> 2;
    for (int c4 = threadIdx.x; c4 < A.fin * per_row; c4 += blockDim.x) {
      const int f = c4 / per_row, o = (c4 - f * per_row) * 4;
      const float4 v = ldg4(A.w + (size_t)f * A.fout + o);
      float* d = Wp + f * wp + o;
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
  } else {
    for (int c = threadIdx.x; c < A.fin * A.fout; c += blockDim.x) {
      const int f = c / A.fout;
      Wp[f * wp + (c - f * A.fout)] = __ldg(A.w + c);
    }
  }
  for (int c = threadIdx.x; c <= nr; c += blockDim.x) rp[c] = __ldg(A.rowptr + r0 + c);
  float k1v[RB];
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    const int i = r0 + warp * RB + r;
    k1v[r] = (i < A.n) ? A.c1 * (A.row_scale ? __ldg(A.row_scale + i) : 1.f) : 0.f;
  }
  for (int c = threadIdx.x; c < R * fo4; c += blockDim.x) {
    const int r = c / fo4, o = c % fo4, i = r0 + r;
    float gv = 0.f;
    if (i < A.n && o < A.fout) {
      gv = __ldg(gy + (size_t)i * A.fout + o);
      // the layer's ReLU backward (threshold on the forward output) folded in; the masked gradient also leaves for
      // the weight gradient dW = (theta s)^T gy that follows
      if (A.okeep) gv *= __ldg(A.okeep + (size_t)i * A.fout + o);        // y = act(z) * keep
      if (relu_y != nullptr && __ldg(relu_y + (size_t)i * A.fout + o) <= 0.f) gv = 0.f;
      if (gy_masked != nullptr) gy_masked[(size_t)i * A.fout + o] = gv;
    }
    Gs[c] = gv;
  }
  __syncthreads();
  const int eb0 = rp[0], eb1 = rp[nr];
  // ---- phase A: ds[r][f] = theta * sum_c g[r][c] Wt[c][f] + beta * g[r][f], RB rows per warp ----
  {
    float* grows = Gs + warp * RB * fo4;
    float d[RB][Q];
#pragma unroll
    for (int r = 0; r < RB; ++r)
#pragma unroll
      for (int q = 0; q < Q; ++q) d[r][q] = 0.f;
    for (int c = 0; c < A.fout; ++c) {                      // d[r][f] = sum_c g[r][c] W[f][c], lane owns f = lane + 32 q
      float wv[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int f = lane + 32 * q;
        wv[q] = (f < A.fin) ? Wp[f * wp + c] : 0.f;
      }
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        const float gv = grows[r * fo4 + c];
#pragma unroll
        for (int q = 0; q < Q; ++q) d[r][q] = fmaf(gv, wv[q], d[r][q]);
      }
    }
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      const int i = r0 + warp * RB + r;
      const float k1 = k1v[r];
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int f = lane + 32 * q;
        if (f < A.fin) {
          float v = A.theta * d[r][q];
          if (A.beta != 0.f) v = fmaf(A.beta, grows[r * fo4 + f], v);
          if (ds_out && i < A.n) {
            float* dst = ds_out + (size_t)i * A.fin + f;
            *dst = (A.accum & 2) ? *dst + ds_scale * v : ds_scale * v;
          }
          DS[(warp * RB + r) * A.fin + f] = k1 * v;
        }
      }
    }
  }
  __syncthreads();
  // ---- phase B: entry-parallel  dval_e = <c1 rs ds_u, x_v>,  dx_v += a_e c1 rs ds_u ----
  const int nE = eb1 - eb0, groups = kSpmmWarps * G;
  const int per = (nE + groups - 1) / groups;
  const int e_beg = eb0 + (warp * G + grp) * per, e_end = min(eb1, e_beg + per);
  if (e_beg < e_end) {
    int cur = row_of_entry(rp, nr, e_beg);          // local row
    int next_start = rp[cur + 1];
    Vec<4> g[T];
    auto load_row = [&]() {
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int c = 4 * (lg + L * t);
        if (c < A.fin) g[t].v = *reinterpret_cast<const float4*>(DS + cur * A.fin + c);
        else g[t].zero();
      }
    };
    load_row();
#pragma unroll 2
    for (int e = e_beg; e < e_end; ++e) {
      if (e >= next_start) {
        while (e >= next_start) {
          ++cur;
          next_start = rp[cur + 1];
        }
        load_row();
      }
      const int v = __ldg(A.col + e);
      const float a = __ldg(A.val + e);
      float dot = 0.f;
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int c = 4 * (lg + L * t);
        if (c < A.fin) {
          if (dval) {
            Vec<4> xv;
            xv.load(A.x + (size_t)v * A.fin + c);
            dot += g[t].dot(xv);
          }
          if (dx) g[t].red(dx + (size_t)v * A.fin + c, a);
        }
      }
      if (dval) {
        dot = group_sum(dot, L);
        if (lg == 0) dval[e] = (A.accum & 1) ? dval[e] + dot : dot;
      }
    }
  }
}

// graphs below this many rows: one row per warp (every row of the layer in flight at once)
constexpr int kSmallGraphRows = 8 * kNumSMs * kSpmmWarps;

static int spmm_gemm_lanes(int fin, int* t_out) {
  const int chunks = fin / 4;
  int L = 1;
  while (L < 32 && 4 * L < chunks) L *= 2;
  int T = (chunks + L - 1) / L;
  *t_out = T > 2 ? 4 : (T >= 2 ? 2 : 1);
  return L;
}

template <typename Fn>
static int dispatch_vec(int f, Fn&& fn) {
  // pick the widest vector the row stride allows, then lanes-per-row L and chunks-per-lane T
  const int vec = (f % 4 == 0) ? 4 : (f % 2 == 0 ? 2 : 1);
  const int chunks = (f + vec - 1) / vec;
  // up to 4 chunks per lane: F = 64 -> 4 lanes per neighbour row, 8 neighbour rows in flight per warp instruction
  // (a 150-entry hub row is 19 iterations instead of 76; the average 6-entry row is one)
  int L = 1;
  while (L < 32 && 4 * L < chunks) L *= 2;
  int T = (chunks + L - 1) / L;
  T = T > 2 ? 4 : (T >= 2 ? 2 : 1);
  if (vec == 4) {
    if (T == 1) return fn(std::integral_constant<int, 4>{}, std::integral_constant<int, 1>{}, L);
    if (T == 2) return fn(std::integral_constant<int, 4>{}, std::integral_constant<int, 2>{}, L);
    return fn(std::integral_constant<int, 4>{}, std::integral_constant<int, 4>{}, L);
  }
  if (vec == 2) {
    if (T == 1) return fn(std::integral_constant<int, 2>{}, std::integral_constant<int, 1>{}, L);
    if (T == 2) return fn(std::integral_constant<int, 2>{}, std::integral_constant<int, 2>{}, L);
    return fn(std::integral_constant<int, 2>{}, std::integral_constant<int, 4>{}, L);
  }
  if (T == 1) return fn(std::integral_constant<int, 1>{}, std::integral_constant<int, 1>{}, L);
  if (T == 2) return fn(std::integral_constant<int, 1>{}, std::integral_constant<int, 2>{}, L);
  return fn(std::integral_constant<int, 1>{}, std::integral_constant<int, 4>{}, L);
}


// ------------------------------------------------------------------------------------------------
// A STACK of GCNII layers in one launch (small graphs).  GCNII_DGG-64 on Citeseer runs 62 identical layers behind its
// last DGG layer -- same adjacency, same h0, 0.85 MB of activations each: per layer the one-launch kernel above costs
// ~13 us of launch + dependent-L2-round-trip latency (rowptr -> entries -> neighbour rows -> W) for ~1 us of work.
// Here the grid is cooperative (every CTA resident), one warp owns ONE row for all layers: its entries (first 32) and
// its h0 row stay in registers, W of layer k + 1 streams into the other half of a shared-memory double buffer
// (cp.async) while layer k computes, and what is left per layer is one gather round trip, the 64 x 64 dense part and a
// grid barrier (atomic counter; neighbour rows of the previous layer are read past L1 with ld.cg).
// y[k] / s_out[k] are the per-layer outputs the backward needs (next input / ReLU mask, theta * s for dW).
// ------------------------------------------------------------------------------------------------
constexpr int kStackMaxLayers = 96;
constexpr int kStackChunks = 16;   // overflow chunks of long rows a CTA spreads over its warps (two per warp)

struct StackArgs {
  const int32_t* rowptr;
  const int32_t* col;
  const float* val;
  int n, f, layers;
  const float* x0;       // [n, f] input of the first layer
  const float* h0;       // [n, f]
  const float* keep;     // [layers, n, f] output dropout multipliers or NULL
  float c1, c2;
  float* y;              // [layers, n, f]
  float* s_out;          // [layers, n, f] (theta * s) or NULL
  unsigned* bar;         // one zeroed counter
  const float* w[kStackMaxLayers];      // [f, f] each
  float theta[kStackMaxLayers];         // beta = 1 - theta
};

__device__ __forceinline__ void cp_async16(float* dst_smem, const float* src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ void stack_grid_barrier(unsigned* bar, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();                       // cumulative: the block's stores (ordered before by bar.sync) become visible
    atomicAdd(bar, 1u);
    unsigned v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
    } while (v < target);
  }
  __syncthreads();
}

#ifdef DGGB_STACK_TRACE
__device__ long long g_stack_trace[2][kStackMaxLayers][8];   // [block 0 | block gridDim/2][layer][t0, t1, t2, t3]
#endif

template <int Q>
#ifndef DGGB_STACK_U
#define DGGB_STACK_U 8
#define DGGB_STACK_MINB 4
#endif
__global__ void __launch_bounds__(kSpmmWarps* kWarp, Q <= 2 ? DGGB_STACK_MINB : 1)      // 4 CTAs per SM: 4 736 rows resident
    gcnii_stack_fwd_kernel(const __grid_constant__ StackArgs A) {
  extern __shared__ __align__(16) float sm[];
  __shared__ int s_beg[kSpmmWarps], s_end[kSpmmWarps];
  const int f = A.f, ff = f * f;
  float* Wbuf = sm;                                   // [2][f][f]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* srow = sm + 2 * ff + warp * f;
  float* ovf = sm + 2 * ff + kSpmmWarps * f;          // [kStackChunks][f] partial sums of spread-out overflow chunks
  const int i = blockIdx.x * kSpmmWarps + warp;
  const bool ok = i < A.n;
  // layer 0's W travels while the row's static data is fetched
  for (int c = threadIdx.x * 4; c < ff; c += blockDim.x * 4) cp_async16(Wbuf + c, A.w[0] + c);
  cp_async_commit();
  const int beg = ok ? __ldg(A.rowptr + i) : 0, end = ok ? __ldg(A.rowptr + i + 1) : 0;
  const int c_l = (beg + lane < end) ? __ldg(A.col + beg + lane) : 0;       // the row's first 32 entries: registers
  const float a_l = (beg + lane < end) ? __ldg(A.val + beg + lane) : 0.f;
  if (lane == 0) {
    s_beg[warp] = beg;
    s_end[warp] = end;
  }
  // Aggregation layout: LPE = f / 4 lanes per entry (one float4 column chunk each), EPS = 32 / LPE entries per step,
  // eight steps in flight: one ROUND = OWN = 8 EPS neighbour rows (16 at f = 64).  (With lane == column and 8 rows in
  // flight a 60-entry row took eight dependent L2 round trips per layer, and every layer of the whole grid waited for
  // that one warp at the barrier: clock64 trace, profiles/r02f_hot_lines.md.)
  constexpr int LPE = 8 * Q, EPS = 32 / LPE, kU = DGGB_STACK_U, OWN = kU * EPS;
  const int sub = lane / LPE, cl = lane % LPE;
  float h0v[Q];
#pragma unroll
  for (int q = 0; q < Q; ++q) h0v[q] = ok ? __ldg(A.h0 + (size_t)i * f + lane + 32 * q) : 0.f;
  __syncthreads();
  // A long row's entries beyond its first round are cut into chunks of OWN entries that the CTA's warps share (chunk c
  // -> warp c % 8; up to kStackChunks per CTA, the rest stays with the owner): a 60-entry row is two rounds of the
  // layer's critical path instead of four.  The table is static over the layers: each warp keeps its (at most two)
  // helper chunks' entries in registers.
  int my_base = 0, my_cov = 0;                        // this row's chunks are ovf[my_base .. my_base + my_cov)
  int hc_len[2] = {0, 0}, hc_col[2] = {0, 0};
  float hc_val[2] = {0.f, 0.f};
  {
    int base = 0;
#pragma unroll
    for (int v = 0; v < kSpmmWarps; ++v) {
      const int dv = s_end[v] - s_beg[v];
      const int nch = dv > OWN ? (dv - OWN + OWN - 1) / OWN : 0;
      const int cov = max(0, min(nch, kStackChunks - base));
      if (v == warp) {
        my_base = base;
        my_cov = cov;
      }
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int c = warp + kSpmmWarps * t;          // the chunk this warp helps with
        if (c >= base && c < base + cov) {
          const int e0 = s_beg[v] + OWN * (1 + c - base);
          hc_len[t] = min(OWN, s_end[v] - e0);
          hc_col[t] = lane < hc_len[t] ? __ldg(A.col + e0 + lane) : 0;
          hc_val[t] = lane < hc_len[t] ? __ldg(A.val + e0 + lane) : 0.f;
        }
      }
      base += cov;
    }
  }
  const int own_cnt = min(end - beg, OWN);
  const int tail_beg = beg + OWN * (1 + my_cov);      // entries nobody helps with (more than kStackChunks chunks per CTA)
  const size_t plane = (size_t)A.n * f;
  for (int k = 0; k < A.layers; ++k) {
    const float* Ws = Wbuf + (k & 1) * ff;
    if (k + 1 < A.layers) {                           // (the other half was last read by layer k - 1's dense part,
      float* Wn = Wbuf + ((k + 1) & 1) * ff;          //  which every warp of the block left before the grid barrier)
      for (int c = threadIdx.x * 4; c < ff; c += blockDim.x * 4) cp_async16(Wn + c, A.w[k + 1] + c);
      cp_async_commit();
    }
    const float* xin = (k == 0) ? A.x0 : A.y + (size_t)(k - 1) * plane;
#ifdef DGGB_STACK_TRACE
    long long t0 = clock64(), t1 = 0, t2 = 0, t3 = 0, ta = 0, tb = 0;
#endif
    // one gather pass over <= 32 entries held by the lanes (cc, aa): rounds of OWN entries, partial sums per entry slot
    auto gather = [&](int cc, float aa, int cnt, float4& acc) {
      for (int k0 = 0; k0 < cnt; k0 += OWN) {
        float4 xv[kU];
        float av[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          // slots beyond the entries issue NO load: pointing them at "row 0, weight 0" made every warp of the grid hit
          // the same two L2 lines ~14 times per layer -- 46 k requests on one line, 12-15 k cycles per round where a
          // round trip is ~1 k (clock64 trace)
          const int j = k0 + u * EPS + sub;
          const int v = __shfl_sync(0xffffffffu, cc, j & 31);
          const float a = __shfl_sync(0xffffffffu, aa, j & 31);
          av[u] = (j < cnt) ? a : 0.f;
          xv[u] = (j < cnt) ? __ldcg(reinterpret_cast<const float4*>(xin + (size_t)v * f) + cl)
                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          acc.x = fmaf(av[u], xv[u].x, acc.x); acc.y = fmaf(av[u], xv[u].y, acc.y);
          acc.z = fmaf(av[u], xv[u].z, acc.z); acc.w = fmaf(av[u], xv[u].w, acc.w);
        }
      }
    };
    auto slot_sum = [&](float4& acc) {                // the EPS entry slots of a step hold partial sums
#pragma unroll
      for (int o = LPE; o < kWarp; o <<= 1) {
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
        acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
      }
    };
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    gather(c_l, a_l, own_cnt, acc);                   // the row's first round
#pragma unroll
    for (int t = 0; t < 2; ++t) {                     // chunks of the CTA's long rows (warp-uniform conditions)
      if (hc_len[t] > 0) {
        float4 acc_o = make_float4(0.f, 0.f, 0.f, 0.f);
        gather(hc_col[t], hc_val[t], hc_len[t], acc_o);
        slot_sum(acc_o);
        if (sub == 0) reinterpret_cast<float4*>(ovf + (size_t)(warp + kSpmmWarps * t) * f)[cl] = acc_o;
      }
    }
    for (int e0 = tail_beg; e0 < end; e0 += kWarp) {  // what is left of a very long row stays with its owner
      const int e = e0 + lane;
      gather((e < end) ? __ldg(A.col + e) : 0, (e < end) ? __ldg(A.val + e) : 0.f, min(kWarp, end - e0), acc);
    }
#ifdef DGGB_STACK_TRACE
    ta = clock64();
#endif
    slot_sum(acc);
    if (sub == 0) reinterpret_cast<float4*>(srow)[cl] = acc;      // the row's own partial sum
#ifdef DGGB_STACK_TRACE
    tb = clock64();
#endif
    if (k + 1 < A.layers) asm volatile("cp.async.wait_group 1;" ::: "memory");   // W of THIS layer has landed
    else cp_async_wait_all();
    __syncthreads();                                  // W, every warp's partial sums and the helpers' chunk sums
    const float theta = A.theta[k], beta = 1.f - theta;
    float sv[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int c = lane + 32 * q;
      float raw = srow[c];
      for (int t = 0; t < my_cov; ++t) raw += ovf[(size_t)(my_base + t) * f + c];
      sv[q] = fmaf(A.c2, h0v[q], A.c1 * raw);
    }
    __syncwarp();
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int c = lane + 32 * q;
      srow[c] = sv[q];
      if (A.s_out && ok) A.s_out[(size_t)k * plane + (size_t)i * f + c] = theta * sv[q];
    }
    __syncwarp();
#ifdef DGGB_STACK_TRACE
    t1 = clock64();
#endif
    float d[1][Q];
    dense_rows<Q, 1>(srow, f, Ws, f, f, lane, d);
    if (ok) {
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int c = lane + 32 * q;
        if (c < f) {
          float v = fmaxf(fmaf(theta, d[0][q], beta * sv[q]), 0.f);
          const size_t o = (size_t)k * plane + (size_t)i * f + c;
          if (A.keep) v *= __ldg(A.keep + o);
          A.y[o] = v;
        }
      }
    }
#ifdef DGGB_STACK_TRACE
    t2 = clock64();
#endif
    if (k + 1 < A.layers) stack_grid_barrier(A.bar, (unsigned)(k + 1) * gridDim.x);
#ifdef DGGB_STACK_TRACE
    t3 = clock64();
    if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x / 2)) {
      long long* t = g_stack_trace[blockIdx.x == 0 ? 0 : 1][k];
      t[0] = t0; t[1] = t1; t[2] = t2; t[3] = t3; t[4] = ta; t[5] = tb;
    }
#endif
  }
}

}  // namespace dggb
using namespace dggb;

extern "C" int dggb_spmm_csr_fwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                                 const float* x, int32_t f, const float* row_scale, float* y, void* stream) {
  if (!rowptr || !col || !val || !x || !y || n < 0 || f <= 0) return DGGB_ERR_BAD_ARG;
  if (n == 0) return DGGB_OK;
  return dispatch_vec(f, [&](auto vc, auto tc, int L) {
    auto kern = spmm_fwd_kernel<decltype(vc)::value, decltype(tc)::value>;
    const int grid = rows_grid(n, kSpmmWarps, resident_blocks(kern, kSpmmWarps * kWarp));
    launch_pdl(kern, dim3(grid), dim3(kSpmmWarps * kWarp), 0,
               as_stream(stream), rowptr, col, val, n, x, f, L, row_scale, y);
    return launch_status();
  });
}

extern "C" int dggb_spmm_csr_bwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                                 const float* x, int32_t f, const float* row_scale, const float* dy, float* dval,
                                 float* dx, void* stream) {
  if (!rowptr || !col || !val || !x || !dy || n < 0 || f <= 0) return DGGB_ERR_BAD_ARG;
  if (n == 0 || (!dval && !dx)) return DGGB_OK;
  return dispatch_vec(f, [&](auto vc, auto tc, int L) {
    auto kern = spmm_bwd_kernel<decltype(vc)::value, decltype(tc)::value>;
    const int grid = rows_grid(n, kSpmmWarps, resident_blocks(kern, kSpmmWarps * kWarp));
    launch_pdl(kern, dim3(grid), dim3(kSpmmWarps * kWarp), 0,
               as_stream(stream), rowptr, col, val, n, x, f, L, row_scale, dy, dval, dx);
    return launch_status();
  });
}

static int spmm_gemm_check(const SpmmGemmArgs& A) {
  if (!A.rowptr || !A.col || !A.val || !A.x || !A.w || A.n < 0 || A.fin <= 0 || A.fout <= 0) return DGGB_ERR_BAD_ARG;
  if (A.fin % 4 != 0 || A.fin > 128 || A.fout > 128 || (A.beta != 0.f && A.fin != A.fout) ||
      ((uintptr_t)A.x % 16) || (A.h0 && ((uintptr_t)A.h0 % 16)))
    return DGGB_ERR_BAD_SHAPE;
  return DGGB_OK;
}

extern "C" int dggb_spmm_gemm_fwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                                  const float* x, int32_t fin, const float* row_scale, const float* h0, float c1,
                                  float c2, const float* w, int32_t fout, float theta, float beta,
                                  const float* resid, int32_t relu, const float* out_keep, float* y, float* s_out,
                                  void* stream) {
  SpmmGemmArgs A{rowptr, col, val, n, fin, fout, 1, x, row_scale, h0, w, resid, c1, c2, theta, beta, relu, 0, out_keep};
  if (out_keep && ((uintptr_t)out_keep % 16)) return DGGB_ERR_BAD_ARG;
  int rc = spmm_gemm_check(A);
  if (rc != DGGB_OK) return rc;
  if (!y || (s_out && ((uintptr_t)s_out % 16))) return DGGB_ERR_BAD_ARG;
  if (n == 0) return DGGB_OK;
  int T = 1;
  A.L = spmm_gemm_lanes(fin, &T);
  const int rb = n >= kSmallGraphRows ? 4 : 1;
  const size_t smem = ((size_t)fin * fout + (size_t)kSpmmWarps * rb * fin + kSpmmWarps * rb + 4) * sizeof(float);
  auto go = [&](auto kern) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e);
    const int grid = (n + kSpmmWarps * rb - 1) / (kSpmmWarps * rb);        // one block per kSpmmWarps * rb rows
    launch_pdl(kern, dim3(grid), dim3(kSpmmWarps * kWarp), smem, as_stream(stream), A, y, s_out);
    return launch_status();
  };
  const int Q = fout <= 32 ? 1 : (fout <= 64 ? 2 : 4);
  // A/B: entry-parallel kernel on small graphs; read per call, so that one process can run both paths
  const bool no_row = getenv("DGGB_SPMM_GEMM_NO_ROW") != nullptr;
  if (rb == 1 && !no_row)
    return Q == 1 ? go(spmm_gemm_fwd_row_kernel<1>) : (Q == 2 ? go(spmm_gemm_fwd_row_kernel<2>) : go(spmm_gemm_fwd_row_kernel<4>));
#define DGGB_SG_Q(T_, R_) (Q == 1 ? go(spmm_gemm_fwd_kernel<T_, 1, R_>) : (Q == 2 ? go(spmm_gemm_fwd_kernel<T_, 2, R_>) : go(spmm_gemm_fwd_kernel<T_, 4, R_>)))
#define DGGB_SG_F(T_) (rb == 4 ? DGGB_SG_Q(T_, 4) : DGGB_SG_Q(T_, 1))
  return T == 1 ? DGGB_SG_F(1) : (T == 2 ? DGGB_SG_F(2) : DGGB_SG_F(4));
#undef DGGB_SG_F
#undef DGGB_SG_Q
}

extern "C" int dggb_spmm_gemm_bwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                                  const float* x, int32_t fin, const float* row_scale, float c1, const float* w,
                                  int32_t fout, float theta, float beta, const float* gy, float* dval, float* dx,
                                  float* ds_out, float ds_scale, float* zero_ws, int64_t zero_count,
                                  const float* relu_y, float* gy_masked, const float* out_keep, int32_t accumulate,
                                  void* stream) {
  SpmmGemmArgs A{rowptr, col, val, n, fin, fout, 1, x, row_scale, nullptr, w, nullptr, c1, 0.f, theta, beta, 0, (int)accumulate, out_keep};
  if (out_keep && ((uintptr_t)out_keep % 16)) return DGGB_ERR_BAD_ARG;
  int rc = spmm_gemm_check(A);
  if (rc != DGGB_OK) return rc;
  if (!gy || (dx && ((uintptr_t)dx % 16)) || zero_count < 0) return DGGB_ERR_BAD_ARG;
  if (n == 0) return DGGB_OK;
  int T = 1;
  A.L = spmm_gemm_lanes(fin, &T);
  const int rb = n >= kSmallGraphRows ? 4 : 1;
  const size_t smem =
      ((size_t)fin * (fout + 1) + 4 + (size_t)kSpmmWarps * rb * (fin + ((fout + 3) & ~3)) + kSpmmWarps * rb + 4) *
      sizeof(float);
  auto go = [&](auto kern) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e);
    const int grid = (n + kSpmmWarps * rb - 1) / (kSpmmWarps * rb);
    launch_pdl(kern, dim3(grid), dim3(kSpmmWarps * kWarp), smem, as_stream(stream), A, gy, dval, dx, ds_out, ds_scale,
               zero_ws, (long long)zero_count, relu_y, gy_masked);
    return launch_status();
  };
  const int Q = fin <= 32 ? 1 : (fin <= 64 ? 2 : 4);
#define DGGB_SG_Q(T_, R_) (Q == 1 ? go(spmm_gemm_bwd_kernel<T_, 1, R_>) : (Q == 2 ? go(spmm_gemm_bwd_kernel<T_, 2, R_>) : go(spmm_gemm_bwd_kernel<T_, 4, R_>)))
#define DGGB_SG_B(T_) (rb == 4 ? DGGB_SG_Q(T_, 4) : DGGB_SG_Q(T_, 1))
  return T == 1 ? DGGB_SG_B(1) : (T == 2 ? DGGB_SG_B(2) : DGGB_SG_B(4));
#undef DGGB_SG_B
#undef DGGB_SG_Q
}

// Edge-parallel variants (F % 4 == 0, F <= 512): y must be zeroed by the caller (rows cut by a run boundary are
// combined with vector reductions); erow = row of every entry (dggb_csr_expand_rows).
extern "C" int dggb_spmm_edge_fwd(const int32_t* rowptr, const int32_t* erow, const int32_t* col, const float* val,
                                  int32_t n, int64_t nnz, const float* x, int32_t f, const float* row_scale,
                                  float* y, void* stream) {
  if (!rowptr || !erow || !col || !val || !x || !y || n < 0 || nnz < 0 || f <= 0) return DGGB_ERR_BAD_ARG;
  if (f % 4 != 0 || f > 512 || ((uintptr_t)x % 16) || ((uintptr_t)y % 16)) return DGGB_ERR_BAD_SHAPE;
  if (nnz == 0) return DGGB_OK;
  int T = 1;
  const int L = spmm_gemm_lanes(f, &T);
  const int run = edge_run_len(nnz, L);
  auto go = [&](auto kern) {
    const int grid = edge_spmm_grid(nnz, L, run, resident_blocks(kern, kSpmmWarps * kWarp));
    launch_pdl(kern, dim3(grid), dim3(kSpmmWarps * kWarp), 0, as_stream(stream), rowptr, erow, col, val,
               (long long)nnz, x, (int)f, L, run, row_scale, y);
    return launch_status();
  };
  return T == 1 ? go(spmm_edge_fwd_kernel<1>) : (T == 2 ? go(spmm_edge_fwd_kernel<2>) : go(spmm_edge_fwd_kernel<4>));
}

extern "C" int dggb_spmm_edge_bwd(const int32_t* erow, const int32_t* col, const float* val, int64_t nnz,
                                  const float* x, int32_t f, const float* row_scale, const float* dy, float* dval,
                                  float* dx, void* stream) {
  if (!erow || !col || !val || !x || !dy || nnz < 0 || f <= 0) return DGGB_ERR_BAD_ARG;
  if (f % 4 != 0 || f > 512 || ((uintptr_t)x % 16) || ((uintptr_t)dy % 16) || (dx && ((uintptr_t)dx % 16)))
    return DGGB_ERR_BAD_SHAPE;
  if (nnz == 0 || (!dval && !dx)) return DGGB_OK;
  int T = 1;
  const int L = spmm_gemm_lanes(f, &T);
  const int run = edge_run_len(nnz, L);
  auto go = [&](auto kern) {
    const int grid = edge_spmm_grid(nnz, L, run, resident_blocks(kern, kSpmmWarps * kWarp));
    launch_pdl(kern, dim3(grid), dim3(kSpmmWarps * kWarp), 0, as_stream(stream), erow, col, val, (long long)nnz, x,
               (int)f, L, run, row_scale, dy, dval, dx);
    return launch_status();
  };
  return T == 1 ? go(spmm_edge_bwd_kernel<1>) : (T == 2 ? go(spmm_edge_bwd_kernel<2>) : go(spmm_edge_bwd_kernel<4>));
}

static int stack_capacity_blocks(int f, size_t* smem_out) {
  const size_t smem = (size_t)(2 * f * f + kSpmmWarps * f + kStackChunks * f) * sizeof(float);
  if (smem_out) *smem_out = smem;
  int occ = 0, dev = 0, sms = kNumSMs;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaError_t e = cudaSuccess;
  auto q = [&](auto kern) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSpmmWarps * kWarp, smem);
  };
  if (f == 32) q(gcnii_stack_fwd_kernel<1>);
  else if (f == 64) q(gcnii_stack_fwd_kernel<2>);
  else if (f == 128) q(gcnii_stack_fwd_kernel<4>);
  else return 0;
  if (e != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return occ * sms;
}

// Largest row count dggb_gcnii_stack_fwd takes for feature width f on this device (one warp per row, all CTAs resident);
// 0: width not supported.
extern "C" int32_t dggb_gcnii_stack_max_rows(int32_t f) { return (int32_t)stack_capacity_blocks((int)f, nullptr) * kSpmmWarps; }

// Forward of `layers` GCNII layers that share the adjacency and h0 (see gcnii_stack_fwd_kernel): y[k] = ReLU(theta_k
// (s_k W_k) + (1 - theta_k) s_k) * keep[k], s_k = c1 (A y[k-1]) + c2 h0, y[-1] = x0.  Returns DGGB_ERR_UNSUPPORTED when
// the grid (one warp per row) cannot be made resident at once or the shape is outside the kernel's range: the caller
// then runs the layers one launch each.
extern "C" int dggb_gcnii_stack_fwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                                    const float* x0, const float* h0, int32_t f, int32_t layers,
                                    const float* const* w_host_ptrs, const float* theta_host, float c1, float c2,
                                    const float* keep, float* y, float* s_out, uint32_t* barrier_zeroed,
                                    void* stream) {
  if (!rowptr || !col || !val || !x0 || !h0 || !w_host_ptrs || !theta_host || !y || !barrier_zeroed || n <= 0 ||
      layers <= 0)
    return DGGB_ERR_BAD_ARG;
  if (layers > kStackMaxLayers || (f != 32 && f != 64 && f != 128)) return DGGB_ERR_UNSUPPORTED;
  StackArgs A{};
  A.rowptr = rowptr; A.col = col; A.val = val; A.n = n; A.f = f; A.layers = layers;
  A.x0 = x0; A.h0 = h0; A.keep = keep; A.c1 = c1; A.c2 = c2; A.y = y; A.s_out = s_out; A.bar = barrier_zeroed;
  for (int k = 0; k < layers; ++k) {
    if (!w_host_ptrs[k] || ((uintptr_t)w_host_ptrs[k] % 16)) return DGGB_ERR_BAD_ARG;
    A.w[k] = w_host_ptrs[k];
    A.theta[k] = theta_host[k];
  }
  size_t smem = 0;
  const int grid = (n + kSpmmWarps - 1) / kSpmmWarps;
  if (stack_capacity_blocks(f, &smem) < grid) return DGGB_ERR_UNSUPPORTED;
  auto go = [&](auto kern) -> int {
    cudaError_t e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kSpmmWarps * kWarp);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = as_stream(stream);
    cudaLaunchAttribute at = {};
    at.id = cudaLaunchAttributeCooperative;           // every CTA resident: the grid barrier cannot deadlock
    at.val.cooperative = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, kern, A);
    if (e != cudaSuccess) return cuda_status(e);
#ifdef DGGB_STACK_TRACE
    static long long host_t[2][kStackMaxLayers][8];
    cudaStreamSynchronize(cfg.stream);
    cudaMemcpyFromSymbol(host_t, g_stack_trace, sizeof(host_t));
    for (int b = 0; b < 2; ++b)
      for (int k = 8; k < 12 && k < layers; ++k)
        printf("blk %s layer %d: loads+fma %lld  reduce+s %lld  readback %lld | dense+store %lld  barrier %lld  (layer %lld)\n",
               b ? "mid" : "0", k, host_t[b][k][4] - host_t[b][k][0], host_t[b][k][5] - host_t[b][k][4],
               host_t[b][k][1] - host_t[b][k][5], host_t[b][k][2] - host_t[b][k][1],
               host_t[b][k][3] - host_t[b][k][2], host_t[b][k][0] - host_t[b][k - 1][0]);
#endif
    return launch_status();
  };
  return f == 32 ? go(gcnii_stack_fwd_kernel<1>) : (f == 64 ? go(gcnii_stack_fwd_kernel<2>) : go(gcnii_stack_fwd_kernel<4>));
}
