// All-pairs DGG scoring + per-row streaming top-K (north-star subsystems 1+2), and the sparse
// recompute backward (subsystem 3).
//
// Replaces the reference's dense pipeline  torch.cdist(z, z) -> exp(-t D) -> log -> + Gumbel ->
// torch.sort(N x N) (dgm.py:275-301)  with one kernel that never materialises N x N:
//
//   S = Z Z^T on the 5th-gen tensor cores (tcgen05.mma kind::tf32, 3xTF32 split => ~fp32 accuracy),
//   operands staged by TMA (128-B swizzle), accumulators double-buffered in TMEM;
//   epilogue (one thread per query row, TMEM lane == row):  d2 = |zi|^2 + |zj|^2 - 2 S,
//   y = -t sqrt(max(d2,0)) [+ G_ij], threshold-pruned insertion into the row's sorted top-Kc list
//   held in shared memory.  Output: idx/val [rows, Kc] sorted descending (rank == position).
//
// Per CTA: 128 query rows x all N columns in tiles of 64.  Warp roles: w0 TMA producer, w1 MMA issuer
// (+ TMEM owner), w2..w5 epilogue.
#include "common.cuh"
#include "tc05.cuh"
#include "philox.cuh"
#include <algorithm>
#include <climits>
#include <cstdlib>

namespace dggb {

// ------------------------------------------------------------------------------------------------
// host: tensor map through the driver entry point (no link-time dependency on libcuda)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

int make_tmap_2d_f32(CUtensorMap* out, const float* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                     uint32_t box_cols) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return DGGB_ERR_CUDA;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * sizeof(float)};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_last_cuda_error = (int)r;
    return DGGB_ERR_CUDA;
  }
  return DGGB_OK;
}

// ------------------------------------------------------------------------------------------------
// pre-pass: z -> (hi, lo) TF32 split + squared norms, padded to a multiple of 128 rows with zeros
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

__global__ void __launch_bounds__(256)
    split_tf32_kernel(const float* __restrict__ z, int n, int npad, int d, int dpad, float* __restrict__ hi,
                      float* __restrict__ lo, float* __restrict__ nrm) {
  const int lane = threadIdx.x & 31;
  for (int i = blockIdx.x * 8 + (threadIdx.x >> 5); i < npad; i += gridDim.x * 8) {
    float acc = 0.f;
    for (int c = lane; c < dpad; c += kWarp) {
      const float v = (i < n && c < d) ? __ldg(z + (size_t)i * d + c) : 0.f;
      const float h = to_tf32(v);
      hi[(size_t)i * dpad + c] = h;
      lo[(size_t)i * dpad + c] = to_tf32(v - h);
      acc += v * v;
    }
    acc = warp_sum(acc);
    if (lane == 0) nrm[i] = acc;
  }
}

// ------------------------------------------------------------------------------------------------
// counter-based Gumbel noise: Philox4x32-7 keyed by the 64-bit seed, counter = (row, col >> 2, 0, 0);
// lane (col & 3) of the 4 outputs belongs to column col.  Any tile regenerates identically (no N x N
// noise tensor in HBM) and a host implementation can materialise the same matrix for small N
// (tests/philox_ref.py).  v = ((x >> 8) + 0.5) * 2^-24 in (0,1);  g = -scale * log(-log1p(-v)).
// ------------------------------------------------------------------------------------------------
// sqrt.approx (MUFU, <= 2 ulp, no slow-path call): the distance already carries ~1e-6 of GEMM rounding
__device__ __forceinline__ float sqrt_fast(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float ex2_fast(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// g = -scale * log(E), E = -log1p(-v) ~ Exp(1), v = ((x >> 8) + 0.5) 2^-24 in (0,1).
// The LARGE Gumbel values (small v, small E) are the ones top-k keeps, so E must be accurate exactly
// there: series for v < 2^-6, fast log otherwise (|dg| <~ 2e-5 either way).
__device__ __forceinline__ float gumbel_from_bits(uint32_t x, float scale) {
  const float v = ((float)(x >> 8) + 0.5f) * 5.9604644775390625e-08f;  // 2^-24
  const float series = v * fmaf(v, fmaf(v, fmaf(v, 0.25f, 0.33333334f), 0.5f), 1.0f);
  const float e = (v < 0.015625f) ? series : -__logf(1.0f - v);
  return -scale * __logf(e);
}

// ------------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------------
constexpr int kBM = 128;  // query rows per CTA (== TMEM lanes)
constexpr int kBN = 64;   // key columns per tile
constexpr int kAPThreads = 192;

constexpr int kQCap = 32;    // per-row candidate queue slots (flushed when >= kQFlush are pending)
constexpr int kQFlush = 16;  // == columns per epilogue chunk, so a chunk can never overflow the queue
constexpr int kChunk = 16;

struct APSmem {  // byte offsets from the 1024-aligned base
  uint32_t a_hi, a_lo, b0, b_stage_bytes, nrm, vals, idx, qv, qi, bars, total;
};

// kb == 0: the k-block-streamed shape (d > 128).  No resident query tile: a stage is ONE 32-feature k-block of both
// operands, [A_hi 128 rows | A_lo 128 rows | B_hi 64 rows | B_lo 64 rows] x 128 B, and the column norms get a ring of
// kNrmSlots slots of their own (a stage is recycled long before the epilogue reads its tile).
constexpr int kNrmSlots = 4;

__host__ __device__ inline APSmem ap_smem_layout(int kb, int split, int stages, int kc) {
  APSmem L;
  const uint32_t a_bytes = kb * kBM * 128;  // [128 rows][128 B] per k-block
  const uint32_t b_bytes = kb == 0 ? (kBM + kBN) * 128 : kb * kBN * 128;
  uint32_t off = 0;
  L.a_hi = off; off += a_bytes;
  L.a_lo = off; off += (split == 3 ? a_bytes : 0);
  L.b0 = off;
  L.b_stage_bytes = b_bytes * (split == 3 ? 2 : 1);
  off += L.b_stage_bytes * stages;
  L.nrm = off; off += (kb == 0 ? kNrmSlots : stages) * kBN * 4;
  L.vals = off; off += kc * kBM * 4;
  L.idx = off; off += kc * kBM * 4;
  L.qv = off; off += kQCap * kBM * 4;
  L.qi = off; off += kQCap * kBM * 4;
  L.bars = off; off += kb == 0 ? 256 : 128;
  L.total = off;
  return L;
}

// ------------------------------------------------------------------------------------------------
// Warp-cooperative merge of one row's pending candidates into its sorted top-Kc list.
// Threads append candidates (score above the row's current K-th value) to a per-row queue with two
// predicated stores -- no per-thread insertion loop, hence no divergence in the streaming loop.  When
// a row has >= kQFlush pending, the whole warp sorts {list (kc) + queue (<= kQCap)} with a bitonic
// network (M slots per lane, shuffles for strides < 32) and writes the best kc back.
// Order: value descending, column ascending among equal values (== stable descending sort).
// ------------------------------------------------------------------------------------------------
struct Cand {
  float v;
  int id;
};
__device__ __forceinline__ bool cand_before(const Cand& a, const Cand& b) {
  return (a.v > b.v) || (a.v == b.v && a.id < b.id);
}

__device__ __forceinline__ Cand cand_shfl_xor(const Cand& c, int j) {
  Cand o;
  o.v = __shfl_xor_sync(0xffffffffu, c.v, j);
  o.id = __shfl_xor_sync(0xffffffffu, c.id, j);
  return o;
}

// M = list slots per lane (1: kc <= 32, 2: kc <= 64).  The list is kept sorted (descending); the queue
// (<= 32 entries, one per lane) is bitonic-sorted ASCENDING so that list ++ queue is a bitonic sequence,
// which log2(#slots) half-cleaner stages then sort -- far fewer exchanges than re-sorting everything.
template <int M>
__device__ __forceinline__ float merge_row(float* Lv, int32_t* Li, const float* Qv, const int32_t* Qi, int kc,
                                           int row_t, int n_q, int lane) {
  constexpr int T = (M == 1) ? 2 : 4;     // total slots per lane, padded to a power of two
  Cand c[T];
#pragma unroll
  for (int m = 0; m < T; ++m) {
    c[m].v = -INFINITY;
    c[m].id = INT_MAX;
  }
#pragma unroll
  for (int m = 0; m < M; ++m) {
    const int slot = lane + 32 * m;
    if (slot < kc) {
      c[m].v = Lv[slot * kBM + row_t];
      const int id = Li[slot * kBM + row_t];
      c[m].id = id < 0 ? INT_MAX : id;    // empty list slot (-inf): sorts after everything
    }
  }
  Cand qd;
  qd.v = lane < n_q ? Qv[lane * kBM + row_t] : -INFINITY;
  qd.id = lane < n_q ? Qi[lane * kBM + row_t] : INT_MAX;
  // sort the queue ascending ("worst first") across the 32 lanes
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const Cand o = cand_shfl_xor(qd, j);
      const bool asc_block = ((lane & k) == 0);
      const bool lower = ((lane & j) == 0);
      const bool keep_worse = (asc_block == lower);
      const bool mine_first = cand_before(qd, o);   // "first" == better
      qd = (mine_first != keep_worse) ? qd : o;
    }
  }
  // slots [0, 32 M) hold the descending list, the LAST 32 slots hold the ascending queue => bitonic
  // (for M == 2 slot block 2 is -inf padding: descending, then flat, then ascending: still bitonic)
  c[T - 1] = qd;
  // bitonic merge (descending): strides >= 32 are in-lane exchanges, 16 ... 1 are shuffles
#pragma unroll
  for (int j = (32 * T) >> 1; j >= 32; j >>= 1) {
#pragma unroll
    for (int m = 0; m < T; ++m) {
      if ((m & (j >> 5)) == 0) {
        const Cand a = c[m], bb = c[m ^ (j >> 5)];
        const bool a_first = cand_before(a, bb);
        c[m] = a_first ? a : bb;
        c[m ^ (j >> 5)] = a_first ? bb : a;
      }
    }
  }
#pragma unroll
  for (int j = 16; j > 0; j >>= 1) {
#pragma unroll
    for (int m = 0; m < T; ++m) {
      const Cand o = cand_shfl_xor(c[m], j);
      const bool lower = ((lane & j) == 0);
      const bool mine_first = cand_before(c[m], o);
      c[m] = (mine_first == lower) ? c[m] : o;
    }
  }
  float kth = -INFINITY;
#pragma unroll
  for (int m = 0; m < M; ++m) {
    const int slot = lane + 32 * m;
    if (slot < kc) {
      Lv[slot * kBM + row_t] = c[m].v;
      Li[slot * kBM + row_t] = (c[m].id == INT_MAX) ? -1 : c[m].id;
    }
    const float cand_kth = __shfl_sync(0xffffffffu, c[m].v, (kc - 1) & 31);
    if (m == ((kc - 1) >> 5)) kth = cand_kth;
  }
  return kth;
}

// NOISE: 0 none, 1 injected tensor, 2 Philox Gumbel(0, noise_scale), 3 none + softmax normaliser (out_rowsum)
// KB = 0: the k-block-streamed instantiation for d > 128 (kblocks = dpad / 32 k-blocks, given at run time).  The query
// tile is loaded again with every key tile, one k-block per stage, so shared memory does not depend on d.  A stage is
// released by the MMA commit alone; the column norms travel in their own ring (nfull / nempty, kNrmSlots slots) that
// the epilogue releases.  Everything else, the epilogue included, is the code of the resident-tile instantiations.
template <int KB, int SPLIT, int NOISE>
__global__ void __launch_bounds__(kAPThreads, 1)
    allpairs_topk_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo,
                         const float* __restrict__ nrm, int n, int row_begin, int row_count,
                         const float* __restrict__ t_ptr, const float* __restrict__ noise, long long noise_ld,
                         unsigned long long seed, float noise_scale, int kc, int stages,
                         int32_t* __restrict__ out_idx, float* __restrict__ out_val, float inv_temp,
                         float* __restrict__ out_rowsum, const float* __restrict__ after_val,
                         const int32_t* __restrict__ after_idx, int kblocks) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-B align WITHOUT laundering the pointer through an integer (keeps it a shared-space pointer, so
  // every access below compiles to LDS/STS instead of generic LD/ST)
  uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
  const APSmem L = ap_smem_layout(KB, SPLIT, stages, kc);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* full = bars;            // [stages]  TMA -> MMA/epilogue
  uint64_t* empty = bars + 4;       // [stages]  MMA + 4 epilogue warps -> TMA  (KB = 0: MMA alone)
  uint64_t* tfull = bars + 8;       // [2]       MMA -> epilogue
  uint64_t* tempty = bars + 10;     // [2]       epilogue -> MMA
  uint64_t* afull = bars + 12;      // A tile landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);
  uint64_t* nfull = bars + 14;      // KB = 0: [kNrmSlots]  column norms of a tile landed
  uint64_t* nempty = bars + 18;     // KB = 0: [kNrmSlots]  4 epilogue warps -> TMA

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = (n + kBN - 1) / kBN;
  const int row0 = row_begin + blockIdx.x * kBM;  // first global row of this CTA

  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&tm_hi);
    if (SPLIT == 3) tc::tma_prefetch_desc(&tm_lo);
    for (int s = 0; s < stages; ++s) {
      tc::mbar_init(full + s, 1);
      tc::mbar_init(empty + s, KB == 0 ? 1 : 5);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(tfull + b, 1);
      tc::mbar_init(tempty + b, 4);
    }
    if constexpr (KB == 0) {
      for (int i = 0; i < kNrmSlots; ++i) {
        tc::mbar_init(nfull + i, 1);
        tc::mbar_init(nempty + i, 4);
      }
    } else {
      tc::mbar_init(afull, 1);
    }
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    tc::tmem_alloc(tmem_slot, 2 * kBN);
    tc::tmem_relinquish();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    if constexpr (KB == 0) {
      // (tile, k-block) in order; the stage counter runs over k-blocks across tiles
      if (lane == 0) {
        int s = 0;
        uint32_t ph = 0;
        for (int jt = 0; jt < num_tiles; ++jt) {
          const int ns = jt % kNrmSlots;
          tc::mbar_wait_backoff(nempty + ns, ((jt / kNrmSlots) & 1) ^ 1);
          tc::mbar_arrive_expect_tx(nfull + ns, kBN * 4);
          tc::bulk_load_1d(smem + L.nrm + ns * kBN * 4, nrm + (size_t)jt * kBN, kBN * 4, nfull + ns);
          for (int kb = 0; kb < kblocks; ++kb, (++s == stages) ? (s = 0, ph ^= 1) : 0) {
            tc::mbar_wait_backoff(empty + s, ph ^ 1);
            tc::mbar_arrive_expect_tx(full + s, L.b_stage_bytes);
            uint8_t* st = smem + L.b0 + s * L.b_stage_bytes;       // A_hi | A_lo | B_hi | B_lo
            uint8_t* sb = st + (SPLIT == 3 ? 2 : 1) * kBM * 128;
            for (int half = 0; half < 2; ++half) {
              tc::tma_load_2d(st + half * 64 * 128, &tm_hi, full + s, kb * 32, row0 + half * 64);
              if (SPLIT == 3) tc::tma_load_2d(st + (kBM + half * 64) * 128, &tm_lo, full + s, kb * 32, row0 + half * 64);
            }
            tc::tma_load_2d(sb, &tm_hi, full + s, kb * 32, jt * kBN);
            if (SPLIT == 3) tc::tma_load_2d(sb + kBN * 128, &tm_lo, full + s, kb * 32, jt * kBN);
          }
        }
      }
    } else if (lane == 0) {
      const uint32_t a_bytes = KB * kBM * 128 * (SPLIT == 3 ? 2 : 1);
      tc::mbar_arrive_expect_tx(afull, a_bytes);
      for (int kb = 0; kb < KB; ++kb)
        for (int half = 0; half < 2; ++half) {
          tc::tma_load_2d(smem + L.a_hi + (kb * kBM + half * 64) * 128, &tm_hi, afull, kb * 32, row0 + half * 64);
          if (SPLIT == 3)
            tc::tma_load_2d(smem + L.a_lo + (kb * kBM + half * 64) * 128, &tm_lo, afull, kb * 32, row0 + half * 64);
        }
      int s = 0;
      uint32_t ph = 0;
      for (int jt = 0; jt < num_tiles; ++jt, (++s == stages) ? (s = 0, ph ^= 1) : 0) {
        tc::mbar_wait_backoff(empty + s, ph ^ 1);
        tc::mbar_arrive_expect_tx(full + s, L.b_stage_bytes + kBN * 4);
        uint8_t* bs = smem + L.b0 + s * L.b_stage_bytes;
        for (int kb = 0; kb < KB; ++kb) {
          tc::tma_load_2d(bs + kb * kBN * 128, &tm_hi, full + s, kb * 32, jt * kBN);
          if (SPLIT == 3) tc::tma_load_2d(bs + (KB + kb) * kBN * 128, &tm_lo, full + s, kb * 32, jt * kBN);
        }
        tc::bulk_load_1d(smem + L.nrm + s * kBN * 4, nrm + (size_t)jt * kBN, kBN * 4, full + s);
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if constexpr (KB == 0) {
      if (lane == 0) {
        constexpr uint32_t idesc = tc::idesc_tf32(kBM, kBN);
        int s = 0;
        uint32_t ph = 0;
        for (int jt = 0; jt < num_tiles; ++jt) {
          const int buf = jt & 1;
          const uint32_t bph = (jt >> 1) & 1;
          const uint32_t d_tmem = tmem_base + buf * kBN;
          tc::mbar_wait_backoff(tempty + buf, bph ^ 1);
          uint32_t acc = 0;
          for (int kb = 0; kb < kblocks; ++kb, (++s == stages) ? (s = 0, ph ^= 1) : 0) {
            tc::mbar_wait_backoff(full + s, ph);
            tc::fence_after_sync();
            const uint32_t a_hi = tc::smem_u32(smem + L.b0 + s * L.b_stage_bytes);
            const uint32_t a_lo = a_hi + kBM * 128;
            const uint32_t b_hi = a_hi + (SPLIT == 3 ? 2 : 1) * kBM * 128;
            const uint32_t b_lo = b_hi + kBN * 128;
#pragma unroll
            for (int sp = 0; sp < SPLIT; ++sp) {
              const uint32_t a = (sp == 2) ? a_lo : a_hi;   // hi*hi, hi*lo, lo*hi
              const uint32_t b = (sp == 1) ? b_lo : b_hi;
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                tc::mma_tf32(d_tmem, tc::smem_desc_k128(a + ks * 32), tc::smem_desc_k128(b + ks * 32), idesc, acc);
                acc = 1;
              }
            }
            tc::mma_commit(empty + s);     // stage reusable once this k-block's MMAs retire
          }
          tc::mma_commit(tfull + buf);     // after the tile's last k-block: accumulator ready for the epilogue
        }
      }
    } else if (lane == 0) {
      constexpr uint32_t idesc = tc::idesc_tf32(kBM, kBN);
      tc::mbar_wait_backoff(afull, 0);
      tc::fence_after_sync();
      const uint32_t a_hi = tc::smem_u32(smem + L.a_hi), a_lo = tc::smem_u32(smem + L.a_lo);
      int s = 0;
      uint32_t ph = 0;
      for (int jt = 0; jt < num_tiles; ++jt, (++s == stages) ? (s = 0, ph ^= 1) : 0) {
        const int buf = jt & 1;
        const uint32_t bph = (jt >> 1) & 1;
        tc::mbar_wait_backoff(tempty + buf, bph ^ 1);
        tc::mbar_wait_backoff(full + s, ph);
        tc::fence_after_sync();
        const uint32_t b_hi = tc::smem_u32(smem + L.b0 + s * L.b_stage_bytes);
        const uint32_t b_lo = b_hi + KB * kBN * 128;
        const uint32_t d_tmem = tmem_base + buf * kBN;
        uint32_t acc = 0;
#pragma unroll
        for (int sp = 0; sp < SPLIT; ++sp) {
          const uint32_t a = (sp == 2) ? a_lo : a_hi;   // hi*hi, hi*lo, lo*hi
          const uint32_t b = (sp == 1) ? b_lo : b_hi;
#pragma unroll
          for (int kb = 0; kb < KB; ++kb)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              tc::mma_tf32(d_tmem, tc::smem_desc_k128(a + kb * kBM * 128 + ks * 32),
                           tc::smem_desc_k128(b + kb * kBN * 128 + ks * 32), idesc, acc);
              acc = 1;
            }
        }
        tc::mma_commit(empty + s);     // smem stage reusable once these MMAs retire
        tc::mma_commit(tfull + buf);   // accumulator ready for the epilogue
      }
    }
  } else {
    // ================= epilogue: thread == query row =================
    const int q = warp & 3;                         // TMEM lane quarter this warp may access
    const int row_t = q * 32 + lane;                // row inside the CTA tile
    const int lrow = blockIdx.x * kBM + row_t;      // row inside this launch's row block
    const bool row_ok = lrow < row_count && (row_begin + lrow) < n;
    const float ni = row_ok ? __ldg(nrm + row_begin + lrow) : 0.f;
    const float t = __ldg(t_ptr);
    float* vals = reinterpret_cast<float*>(smem + L.vals);   // [kc][128]
    int32_t* idxs = reinterpret_cast<int32_t*>(smem + L.idx);
    for (int r = 0; r < kc; ++r) {
      vals[r * kBM + row_t] = -INFINITY;
      idxs[r * kBM + row_t] = -1;
    }
    float* qv = reinterpret_cast<float*>(smem + L.qv);       // [kQCap][128]
    int32_t* qi = reinterpret_cast<int32_t*>(smem + L.qi);
    float thr = -INFINITY;   // this row's current K-th best value (stale between merges: only admits extras)
    int qn = 0;              // pending candidates of this row
    float zsum = 0.f;        // sum_j exp(y_ij * inv_temp): the softmax normaliser of the evaluation branch
    const float* nz = (NOISE == 1 && row_ok) ? noise + (size_t)lrow * noise_ld : nullptr;
    const uint32_t key0 = (uint32_t)seed, key1 = (uint32_t)(seed >> 32);
    const bool wide = kc > 32;
    // continuation pass (rows that need more than 64 entries): only entries that sort strictly AFTER
    // (after_val, after_idx) -- the last entry the previous pass returned for this row -- are admitted
    // (an empty last entry, idx -1: the previous pass ran out of columns, so nothing is left to admit)
    const int ubc = (after_idx != nullptr && row_ok) ? __ldg(after_idx + lrow) : -1;
    const float ubv = (after_val != nullptr && row_ok) ? (ubc < 0 ? -INFINITY : __ldg(after_val + lrow)) : INFINITY;
    auto flush = [&](unsigned need) {
      __syncwarp();   // queue entries were written by their owner lanes; the whole warp reads them below
      while (need) {
        const int src = __ffs(need) - 1;
        need &= need - 1;
        const int n_q = __shfl_sync(0xffffffffu, qn, src);
        const float kth = wide ? merge_row<2>(vals, idxs, qv, qi, kc, q * 32 + src, n_q, lane)
                               : merge_row<1>(vals, idxs, qv, qi, kc, q * 32 + src, n_q, lane);
        if (lane == src) {
          thr = kth;
          qn = 0;
        }
      }
      __syncwarp();
    };
    int s = 0;
    uint32_t ph = 0;
    for (int jt = 0; jt < num_tiles; ++jt, (++s == stages) ? (s = 0, ph ^= 1) : 0) {
      const int buf = jt & 1;
      const uint32_t bph = (jt >> 1) & 1;
      // where this tile's column norms are: its key stage, or (KB = 0) its slot of the norm ring
      const int ns = KB == 0 ? jt % kNrmSlots : s;
      uint64_t* nbar_full = KB == 0 ? nfull + ns : full + s;
      uint64_t* nbar_empty = KB == 0 ? nempty + ns : empty + s;
      tc::mbar_wait(nbar_full, KB == 0 ? (uint32_t)(jt / kNrmSlots) & 1 : ph);   // column norms are in smem
      tc::mbar_wait(tfull + buf, bph);  // accumulator ready
      tc::fence_after_sync();
      const float* nj = reinterpret_cast<const float*>(smem + L.nrm + ns * kBN * 4);
      // the tile(s) that contain this CTA's own diagonal take the variant that pins d2(i,i) = 0 exactly
      const bool diag_tile = (jt * kBN < row0 + kBM) && (jt * kBN + kBN > row0);
#pragma unroll 1
      for (int c0 = 0; c0 < kBN; c0 += kChunk) {
        uint32_t r[kChunk];
        tc::tmem_ld_32x16(tmem_base + ((uint32_t)(q * 32) << 16) + buf * kBN + c0, r);
        tc::tmem_ld_wait();
        if (row_ok) {
          const int jbase = jt * kBN + c0;
          auto body = [&](auto diag_c) {
            // phase 1: straight-line scores for the 16 columns of this chunk (no branches => ILP)
            float y[kChunk];
            float njv[kChunk];
#pragma unroll
            for (int c = 0; c < kChunk; c += 4) {
              const float4 v4 = *reinterpret_cast<const float4*>(nj + c0 + c);
              njv[c] = v4.x; njv[c + 1] = v4.y; njv[c + 2] = v4.z; njv[c + 3] = v4.w;
            }
            uint4 bits = make_uint4(0u, 0u, 0u, 0u);
            unsigned pass = 0u;
#pragma unroll
            for (int c = 0; c < kChunk; ++c) {
              const int j = jbase + c;
              float d2 = fmaf(-2.f, __uint_as_float(r[c]), ni + njv[c]);
              if (decltype(diag_c)::value && j == row_begin + lrow) d2 = 0.f;
              float yy = -t * sqrt_fast(fmaxf(d2, 0.f));
              if (NOISE == 1) {
                if (j < n) yy += __ldg(nz + j);
              } else if (NOISE == 2) {
                if ((c & 3) == 0) bits = philox4x32_7((uint32_t)(row_begin + lrow), (uint32_t)(j >> 2), key0, key1);
                const uint32_t b = (c & 3) == 0 ? bits.x : ((c & 3) == 1 ? bits.y : ((c & 3) == 2 ? bits.z : bits.w));
                yy += gumbel_from_bits(b, noise_scale);
              }
              y[c] = yy;
              if (NOISE == 3 && j < n) zsum += __expf(yy * inv_temp);   // evaluation branch only
              pass |= (j < n && yy > thr && (yy < ubv || (yy == ubv && j > ubc))) ? (1u << c) : 0u;
            }
            // phase 2 (rare once the list is warm): append the survivors to this row's queue
            if (pass) {
#pragma unroll
              for (int c = 0; c < kChunk; ++c) {
                if (pass & (1u << c)) {
                  qv[qn * kBM + row_t] = y[c];
                  qi[qn * kBM + row_t] = jbase + c;
                  ++qn;
                }
              }
            }
          };
          if (diag_tile) body(std::true_type{});
          else body(std::false_type{});
        }
        flush(__ballot_sync(0xffffffffu, qn >= kQFlush));
      }
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) {
        tc::mbar_arrive(tempty + buf);
        tc::mbar_arrive(nbar_empty);
      }
    }
    flush(__ballot_sync(0xffffffffu, qn > 0));
    if (out_rowsum != nullptr && row_ok) out_rowsum[lrow] = zsum;
    // ---- write the sorted lists: lanes sweep the list positions of one row at a time ----
    __syncwarp();
    for (int rr = 0; rr < 32; ++rr) {
      const int rt = q * 32 + rr;
      const int lr = blockIdx.x * kBM + rt;
      if (lr < row_count && (row_begin + lr) < n) {
        for (int r = lane; r < kc; r += kWarp) {
          const int32_t id = idxs[r * kBM + rt];
          out_idx[(size_t)lr * kc + r] = id;
          out_val[(size_t)lr * kc + r] = id < 0 ? 0.f : vals[r * kBM + rt];
        }
      }
    }
  }
  __syncwarp();
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc::fence_after_sync();
    tc::tmem_dealloc(tmem_base, 2 * kBN);
  }
}

// ------------------------------------------------------------------------------------------------
// v2 of the kernel above (kc <= 32): the SIMT epilogue is the bound, so it gets TWO warps per scheduler.
//   * the query tile (A operand, hi/lo) lives in TENSOR MEMORY ("TS" MMA): each epilogue thread copies its own
//     row global -> registers -> tcgen05.st once; that frees 64 KB of shared memory ...
//   * ... which pays for a second, independent epilogue group: group g (4 warps) owns TMEM accumulators g and
//     g+2 (double-buffered, so its MMA overlaps its own epilogue) and scores tiles jt = g, g+2, ... into its own
//     per-row list/queue; the two sorted lists of a row are merged once at the end.
//     10 warps: w0 TMA producer, w1 MMA issuer, w2-5 group 0, w6-9 group 1.  TMEM: 4 x 64 + 128 columns.
//   * a key stage is released by the MMA commit alone: the column norms the epilogue reads travel in their own ring of
//     stages + 4 slots (one mbarrier each).  The producer can be at most stages + 4 tiles ahead of the oldest tile an
//     epilogue group still reads (stage <- MMA commit <- accumulator free <- epilogue of four tiles earlier), so a slot
//     needs no "empty" barrier.  (With the norms inside the stage, a group held its stage for the whole scoring of a
//     tile and the next load + MMA for its buffer arrived late: 16 % of the samples sat in that wait.)
// ------------------------------------------------------------------------------------------------
constexpr int kAP2Threads = 320;

struct AP2Smem {
  uint32_t b0, b_stage_bytes, nrm, vals[2], idx[2], qv[2], qi[2], zpart, bars, total;
};
__host__ __device__ inline AP2Smem ap2_smem_layout(int kb, int split, int stages, int kc, int qcap = kQCap) {
  AP2Smem L;
  uint32_t off = 0;
  L.b0 = off;
  L.b_stage_bytes = kb * kBN * 128 * (split == 3 ? 2 : 1);
  off += L.b_stage_bytes * stages;
  L.nrm = off; off += (stages + 4) * kBN * 4;     // column-norm ring, see the kernel's header
  for (int g = 0; g < 2; ++g) {
    L.vals[g] = off; off += kc * kBM * 4;
    L.idx[g] = off; off += kc * kBM * 4;
    L.qv[g] = off; off += qcap * kBM * 4;
    L.qi[g] = off; off += qcap * kBM * 4;
  }
  L.zpart = L.qv[1];                              // group 1's queue is idle when the partial sums are exchanged
  L.bars = off; off += 256;
  L.total = off;
  return L;
}

// CONT: the continuation instantiation (d = 65..128 at 3xTF32, where v1 has no tile shape): rows are written with
// stride out_ld, and when after_val / after_idx are given ([row_count] with stride after_ld) only entries that sort
// strictly after that entry are admitted -- the predicate of v1's continuation pass.  One column part only.
template <int KB, int SPLIT, int NOISE, bool CONT = false>
__global__ void __launch_bounds__(kAP2Threads, 1)
    allpairs_topk2_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo,
                          const float* __restrict__ z_hi, const float* __restrict__ z_lo, int npad, int dpad,
                          const float* __restrict__ nrm, int n, int row_begin, int row_count,
                          const float* __restrict__ t_ptr, const float* __restrict__ noise, long long noise_ld,
                          unsigned long long seed, float noise_scale, int kc, int stages, int qcap, int qflush,
                          int32_t* __restrict__ out_idx, float* __restrict__ out_val, float inv_temp,
                          float* __restrict__ out_rowsum, int no_prefilter, int tiles_per_part,
                          int32_t* __restrict__ part_idx, float* __restrict__ part_val, int out_ld,
                          const float* __restrict__ after_val, const int32_t* __restrict__ after_idx, int after_ld) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
  const AP2Smem L = ap2_smem_layout(KB, SPLIT, stages, kc, qcap);   // queue: qcap >= qflush - 1 + kChunk slots
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* full = bars;            // [stages]  TMA -> MMA / epilogue
  uint64_t* empty = bars + 4;       // [stages]  MMA commit -> TMA (the epilogue never touches a key stage)
  uint64_t* tfull = bars + 8;       // [4]       MMA -> epilogue group (accumulators g and g+2 belong to group g)
  uint64_t* tempty = bars + 12;     // [4]       epilogue group -> MMA
  uint64_t* aready = bars + 16;     // query tile written to TMEM (8 epilogue warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 17);
  uint64_t* nfull = bars + 18;      // [stages + 4 <= 8]  column norms of a tile landed
  const int nslots = stages + 4;
  constexpr uint32_t kTmemCols = 512;   // 4 accumulators x 64 columns + the query tile (hi | lo)
  constexpr uint32_t kAHi = 4 * kBN, kALo = 4 * kBN + KB * 32;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // column parts (gridDim.y > 1): this CTA scores key tiles [tile0, tile0 + num_tiles) and leaves its sorted list in
  // part_idx / part_val [part][row][kc]; allpairs_merge_parts_kernel picks the best kc of a row's parts
  const int tile0 = blockIdx.y * tiles_per_part;
  const int num_tiles = min(tiles_per_part, (n + kBN - 1) / kBN - tile0);
  const int row0 = row_begin + blockIdx.x * kBM;

  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&tm_hi);
    if (SPLIT == 3) tc::tma_prefetch_desc(&tm_lo);
    for (int s = 0; s < stages; ++s) {
      tc::mbar_init(full + s, 1);
      tc::mbar_init(empty + s, 1);
    }
    for (int b = 0; b < 4; ++b) {
      tc::mbar_init(tfull + b, 1);
      tc::mbar_init(tempty + b, 4);
    }
    tc::mbar_init(aready, 8);
    for (int i = 0; i < nslots; ++i) tc::mbar_init(nfull + i, 1);
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    tc::tmem_alloc(tmem_slot, kTmemCols);
    tc::tmem_relinquish();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer: key tiles only =================
    if (lane == 0) {
      int s = 0, ns = 0;
      uint32_t ph = 0;
      for (int jt = 0; jt < num_tiles; ++jt, (++s == stages) ? (s = 0, ph ^= 1) : 0, (++ns == nslots) ? (ns = 0) : 0) {
        tc::mbar_wait_sleep(empty + s, ph ^ 1, 400);
        tc::mbar_arrive_expect_tx(nfull + ns, kBN * 4);
        tc::bulk_load_1d(smem + L.nrm + ns * kBN * 4, nrm + (size_t)(tile0 + jt) * kBN, kBN * 4, nfull + ns);
        tc::mbar_arrive_expect_tx(full + s, L.b_stage_bytes);
        uint8_t* bs = smem + L.b0 + s * L.b_stage_bytes;
        for (int kb = 0; kb < KB; ++kb) {
          tc::tma_load_2d(bs + kb * kBN * 128, &tm_hi, full + s, kb * 32, (tile0 + jt) * kBN);
          if (SPLIT == 3) tc::tma_load_2d(bs + (KB + kb) * kBN * 128, &tm_lo, full + s, kb * 32, (tile0 + jt) * kBN);
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer: A from TMEM, B from shared memory =================
    if (lane == 0) {
      constexpr uint32_t idesc = tc::idesc_tf32(kBM, kBN);
      tc::mbar_wait_backoff(aready, 0);
      tc::fence_after_sync();
      int s = 0;
      uint32_t ph = 0;
      for (int jt = 0; jt < num_tiles; ++jt, (++s == stages) ? (s = 0, ph ^= 1) : 0) {
        const int buf = jt & 3;
        const uint32_t bph = (jt >> 2) & 1;
        tc::mbar_wait_sleep(tempty + buf, bph ^ 1, 200);
        tc::mbar_wait_sleep(full + s, ph, 200);
        tc::fence_after_sync();
        const uint32_t b_hi = tc::smem_u32(smem + L.b0 + s * L.b_stage_bytes);
        const uint32_t b_lo = b_hi + KB * kBN * 128;
        const uint32_t d_tmem = tmem_base + buf * kBN;
        uint32_t acc = 0;
#pragma unroll
        for (int sp = 0; sp < SPLIT; ++sp) {
          const uint32_t a = tmem_base + ((sp == 2) ? kALo : kAHi);   // hi*hi, hi*lo, lo*hi
          const uint32_t b = (sp == 1) ? b_lo : b_hi;
#pragma unroll
          for (int kb = 0; kb < KB; ++kb)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              tc::mma_tf32_ts(d_tmem, a + kb * 32 + ks * 8, tc::smem_desc_k128(b + kb * kBN * 128 + ks * 32), idesc,
                              acc);
              acc = 1;
            }
        }
        tc::mma_commit(empty + s);
        tc::mma_commit(tfull + buf);
      }
    }
  } else {
    // ================= two epilogue groups; thread == query row =================
    const int g = (warp - 2) >> 2;                  // 0: even tiles / accumulator 0, 1: odd tiles / accumulator 1
    const int q = warp & 3;                         // TMEM lane quarter this warp may access
    const int row_t = q * 32 + lane;
    const int lrow = blockIdx.x * kBM + row_t;
    const bool row_ok = lrow < row_count && (row_begin + lrow) < n;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    // ---- stage this thread's query row (group 0: hi part, group 1: lo part) into tensor memory ----
    {
      const int grow = row0 + row_t;
      const float* src = (g == 0 ? z_hi : z_lo) + (size_t)grow * dpad;
      const bool have = grow < npad && (g == 0 || SPLIT == 3);
#pragma unroll
      for (int kb = 0; kb < KB; ++kb) {
        uint32_t r[32];
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          const float4 v = have ? __ldg(reinterpret_cast<const float4*>(src + kb * 32 + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
          r[c] = __float_as_uint(v.x); r[c + 1] = __float_as_uint(v.y);
          r[c + 2] = __float_as_uint(v.z); r[c + 3] = __float_as_uint(v.w);
        }
        if (g == 0 || SPLIT == 3) tc::tmem_st_32x32(tmem_base + lane_addr + (g == 0 ? kAHi : kALo) + kb * 32, r);
      }
      tc::tmem_st_wait();
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(aready);
    }
    const float ni = row_ok ? __ldg(nrm + row_begin + lrow) : 0.f;
    const float t = __ldg(t_ptr);
    float* vals = reinterpret_cast<float*>(smem + L.vals[g]);
    int32_t* idxs = reinterpret_cast<int32_t*>(smem + L.idx[g]);
    float* qv = reinterpret_cast<float*>(smem + L.qv[g]);
    int32_t* qi = reinterpret_cast<int32_t*>(smem + L.qi[g]);
    for (int r = 0; r < kc; ++r) {
      vals[r * kBM + row_t] = -INFINITY;
      idxs[r * kBM + row_t] = -1;
    }
    float thr = -INFINITY;
    int qn = 0;
    float zsum = 0.f;
    const float* nz = (NOISE == 1 && row_ok) ? noise + (size_t)lrow * noise_ld : nullptr;
    const uint32_t key0 = (uint32_t)seed, key1 = (uint32_t)(seed >> 32);
    // candidate pre-filter of the Philox path (see the streaming loop): log2(e) / scale; off for a degenerate scale and,
    // per row, while |thr| is so large that the rounding of base - thr could exceed the filter's margin
    const float pf_k = 1.4426950408889634f / noise_scale;
    const bool pf_scale_ok = NOISE == 2 && noise_scale > 1e-20f && noise_scale < 1e20f && !no_prefilter;
    bool prefilter = pf_scale_ok;
    float ubv = INFINITY;    // CONT: the previous pass's last entry of this row (idx -1: it ran out of columns)
    int ubc = -1;
    if (CONT && after_val != nullptr && row_ok) {
      ubc = __ldg(after_idx + (size_t)lrow * after_ld);
      ubv = ubc < 0 ? -INFINITY : __ldg(after_val + (size_t)lrow * after_ld);
    }
    auto after_bound = [&](float yy, int j) { return !CONT || yy < ubv || (yy == ubv && j > ubc); };
    const int ld = CONT ? out_ld : kc;
    auto flush = [&](unsigned need) {
      __syncwarp();
      while (need) {
        const int src = __ffs(need) - 1;
        need &= need - 1;
        const int n_q = __shfl_sync(0xffffffffu, qn, src);
        const float kth = merge_row<1>(vals, idxs, qv, qi, kc, q * 32 + src, n_q, lane);
        if (lane == src) {
          thr = kth;
          qn = 0;
          prefilter = pf_scale_ok && !(fabsf(kth) > 3e4f * noise_scale && kth > -INFINITY);
        }
      }
      __syncwarp();
    };
    int ns = g;                                  // norm-ring slot of tile jt (== jt % nslots), and its phase
    uint32_t nph = 0;
    int it = 0;
    for (int jt = g; jt < num_tiles; jt += 2, ++it) {
      const int buf = g + 2 * (it & 1);          // == jt & 3
      const uint32_t bph = (it >> 1) & 1;        // == (jt >> 2) & 1
      tc::mbar_wait(nfull + ns, nph);
      tc::mbar_wait(tfull + buf, bph);
      tc::fence_after_sync();
      const float* nj = reinterpret_cast<const float*>(smem + L.nrm + ns * kBN * 4);
      const int col0 = (tile0 + jt) * kBN;
      const bool diag_tile = (col0 < row0 + kBM) && (col0 + kBN > row0);
#pragma unroll 1
      for (int c0 = 0; c0 < kBN; c0 += kChunk) {
        uint32_t r[kChunk];
        tc::tmem_ld_32x16(tmem_base + lane_addr + buf * kBN + c0, r);
        tc::tmem_ld_wait();
        if (row_ok) {
          const int jbase = col0 + c0;
          auto body = [&](auto diag_c) {
            float y[kChunk];
            float njv[kChunk];
#pragma unroll
            for (int c = 0; c < kChunk; c += 4) {
              const float4 v4 = *reinterpret_cast<const float4*>(nj + c0 + c);
              njv[c] = v4.x; njv[c + 1] = v4.y; njv[c + 2] = v4.z; njv[c + 3] = v4.w;
            }
            uint4 bits = make_uint4(0u, 0u, 0u, 0u);
            unsigned pass = 0u;
            if (NOISE == 2 && prefilter) {
              // Philox noise, two steps.  y = base + g > thr needs g > thr - base, and g = -scale log(E) with
              // E = -log1p(-v) >= v, so a candidate must have v < exp((base - thr) / scale): ONE ex2 per score decides
              // (with a 2^-7 relative margin over the rounding of base, thr and the fast logs) whether the two logs of
              // the Gumbel transform are evaluated at all.  Once a row's list is warm that is ~Kc / N of the scores;
              // the survivors take exactly the arithmetic of the one-step path, so the selection is unchanged.
              uint32_t xb[kChunk];
              // thr = -inf (cold list): +inf, every score is a candidate; log2(1 + 2^-7) is the margin
              const float tk = fmaf(-thr, pf_k, 0.011227255f);
#pragma unroll
              for (int c = 0; c < kChunk; ++c) {
                const int j = jbase + c;
                float d2 = fmaf(-2.f, __uint_as_float(r[c]), ni + njv[c]);
                if (decltype(diag_c)::value && j == row_begin + lrow) d2 = 0.f;
                y[c] = -t * sqrt_fast(fmaxf(d2, 0.f));
                if ((c & 3) == 0) bits = philox4x32_7((uint32_t)(row_begin + lrow), (uint32_t)(j >> 2), key0, key1);
                xb[c] = (c & 3) == 0 ? bits.x : ((c & 3) == 1 ? bits.y : ((c & 3) == 2 ? bits.z : bits.w));
                // v floored to 23 bits (<= v): exponent of 1.0 | mantissa, minus 1 -- no integer conversion
                const float vq = __uint_as_float(0x3f800000u | (xb[c] >> 9)) - 1.0f;
                const float u = ex2_fast(fmaf(y[c], pf_k, tk));
                // candidate <=> vq - u < 0: its sign bit is shifted into the mask (one funnel shift; column c ends up
                // at bit kChunk - 1 - c).  A NaN difference may set the bit: the exact test below rejects it.
                pass = __funnelshift_l(__float_as_uint(vq - u), pass, 1);
              }
              if (pass) {
#pragma unroll
                for (int c = 0; c < kChunk; ++c) {
                  if (pass & (1u << (kChunk - 1 - c))) {
                    const float yy = y[c] + gumbel_from_bits(xb[c], noise_scale);
                    if (jbase + c < n && yy > thr && after_bound(yy, jbase + c)) {
                      qv[qn * kBM + row_t] = yy;
                      qi[qn * kBM + row_t] = jbase + c;
                      ++qn;
                    }
                  }
                }
              }
              return;
            }
#pragma unroll
            for (int c = 0; c < kChunk; ++c) {
              const int j = jbase + c;
              float d2 = fmaf(-2.f, __uint_as_float(r[c]), ni + njv[c]);
              if (decltype(diag_c)::value && j == row_begin + lrow) d2 = 0.f;
              float yy = -t * sqrt_fast(fmaxf(d2, 0.f));
              if (NOISE == 1) {
                if (j < n) yy += __ldg(nz + j);
              } else if (NOISE == 2) {
                if ((c & 3) == 0) bits = philox4x32_7((uint32_t)(row_begin + lrow), (uint32_t)(j >> 2), key0, key1);
                const uint32_t b = (c & 3) == 0 ? bits.x : ((c & 3) == 1 ? bits.y : ((c & 3) == 2 ? bits.z : bits.w));
                yy += gumbel_from_bits(b, noise_scale);
              }
              y[c] = yy;
              if (NOISE == 3 && j < n) zsum += __expf(yy * inv_temp);   // evaluation branch only
              pass |= (j < n && yy > thr && after_bound(yy, j)) ? (1u << c) : 0u;
            }
            if (pass) {
#pragma unroll
              for (int c = 0; c < kChunk; ++c) {
                if (pass & (1u << c)) {
                  qv[qn * kBM + row_t] = y[c];
                  qi[qn * kBM + row_t] = jbase + c;
                  ++qn;
                }
              }
            }
          };
          if (diag_tile) body(std::true_type{});
          else body(std::false_type{});
        }
        flush(__ballot_sync(0xffffffffu, qn >= qflush));
      }
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(tempty + buf);
      ns += 2;
      if (ns >= nslots) { ns -= nslots; nph ^= 1; }
    }
    flush(__ballot_sync(0xffffffffu, qn > 0));
    // ---- merge the two groups' lists (named barrier over the 8 epilogue warps), group 0 writes out ----
    float* zpart = reinterpret_cast<float*>(smem + L.zpart);
    if (g == 1) zpart[row_t] = zsum;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (g == 0) {
      float* vals1 = reinterpret_cast<float*>(smem + L.vals[1]);
      int32_t* idxs1 = reinterpret_cast<int32_t*>(smem + L.idx[1]);
      for (int rr = 0; rr < 32; ++rr) {
        const int rt = q * 32 + rr;
        const int lr = blockIdx.x * kBM + rt;
        if (!(lr < row_count && (row_begin + lr) < n)) continue;   // warp-uniform
        merge_row<1>(vals, idxs, vals1, idxs1, kc, rt, kc, lane);
        __syncwarp();
        if (gridDim.y > 1) {
          const size_t o = ((size_t)blockIdx.y * row_count + lr) * kc;
          for (int r = lane; r < kc; r += kWarp) {
            part_idx[o + r] = idxs[r * kBM + rt];
            part_val[o + r] = vals[r * kBM + rt];       // -inf where the slot is unused (idx -1)
          }
          continue;
        }
        for (int r = lane; r < kc; r += kWarp) {
          const int32_t id = idxs[r * kBM + rt];
          out_idx[(size_t)lr * ld + r] = id;
          out_val[(size_t)lr * ld + r] = id < 0 ? 0.f : vals[r * kBM + rt];
        }
      }
      if (out_rowsum != nullptr && row_ok) out_rowsum[lrow] = zsum + zpart[row_t];
    }
  }
  __syncwarp();
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc::fence_after_sync();
    tc::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// Column parts -> one list.  A row block x all columns is the natural work unit, but a row-sharded rank holds few row
// blocks (Reddit shape on 8 GPUs: 228 on 148 SMs = 1.54 waves, i.e. two).  The host then cuts the column range into S
// parts (grid.y) so that ceil(blocks S / SMs) / S comes closer to blocks / SMs, and this kernel picks the best kc of a
// row's S sorted part lists: one warp per row, rank by counting over the <= 8 x 32 candidates (value descending, column
// ascending among equal values: the order of the single-part kernel, so the result is identical).
// ------------------------------------------------------------------------------------------------
constexpr int kMergeWarps = 8;
constexpr int kMaxParts = 8;
__global__ void __launch_bounds__(kMergeWarps* kWarp)
    allpairs_merge_parts_kernel(const int32_t* __restrict__ part_idx, const float* __restrict__ part_val, int parts,
                                int row_count, int rows_valid, int kc, int32_t* __restrict__ out_idx,
                                float* __restrict__ out_val) {
  __shared__ float sv[kMergeWarps][kMaxParts * 32];
  __shared__ int32_t si[kMergeWarps][kMaxParts * 32];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = parts * kc;
  for (int lr = blockIdx.x * kMergeWarps + w; lr < rows_valid; lr += gridDim.x * kMergeWarps) {
    int valid = 0;
    for (int i = lane; i < total; i += kWarp) {
      const int pt = i / kc, r = i - pt * kc;
      const size_t o = ((size_t)pt * row_count + lr) * kc + r;
      const int32_t id = __ldg(part_idx + o);
      si[w][i] = id;
      sv[w][i] = __ldg(part_val + o);
      valid += id >= 0;
    }
    valid = __reduce_add_sync(0xffffffffu, valid);
    __syncwarp();
    for (int i = lane; i < total; i += kWarp) {
      const int32_t id = si[w][i];
      if (id < 0) continue;
      const float v = sv[w][i];
      int rank = 0;
      for (int j = 0; j < total; ++j) {
        const int32_t idj = si[w][j];
        const float vj = sv[w][j];
        rank += (idj >= 0 && (vj > v || (vj == v && idj < id))) ? 1 : 0;
      }
      if (rank < kc) {
        out_idx[(size_t)lr * kc + rank] = id;
        out_val[(size_t)lr * kc + rank] = v;
      }
    }
    for (int r = valid + lane; r < kc; r += kWarp) {
      out_idx[(size_t)lr * kc + r] = -1;
      out_val[(size_t)lr * kc + r] = 0.f;
    }
    __syncwarp();
  }
}

// sparse recompute backward: for every selected pair (i, j) with upstream gy = dL/dy_ij,
//   y = -t |z_i - z_j|  =>  dt += -D gy ;  g = -t gy / D ;  dz_i += g (z_i - z_j) ;  dz_j -= g (z_i - z_j)
// (zero gradient at D == 0, like torch.cdist's backward).  O(rows * Kc * d), no N^2 work.
// ------------------------------------------------------------------------------------------------
constexpr int kPairWarps = 8;

// V features per lane: 4 (one float4, d % 4 == 0) or 1 (any d)
template <int V>
__device__ __forceinline__ void ldg_v(float (&r)[V], const float* p) {
  if constexpr (V == 4) {
    const float4 f = ldg4(p);
    r[0] = f.x; r[1] = f.y; r[2] = f.z; r[3] = f.w;
  } else {
    r[0] = __ldg(p);
  }
}
template <int V>
__device__ __forceinline__ void red_add_v(float* p, const float (&r)[V], float sign) {
  if constexpr (V == 4) red_add4(p, make_float4(sign * r[0], sign * r[1], sign * r[2], sign * r[3]));
  else atomicAdd(p, sign * r[0]);
}

template <int V>
__global__ void __launch_bounds__(kPairWarps* kWarp)
    allpairs_pair_grad_kernel(const float* __restrict__ z, int n, int d, int L, int row_begin, int row_count,
                              const int32_t* __restrict__ idx, const float* __restrict__ gy, int kc,
                              const float* __restrict__ t_ptr, float* __restrict__ dz, float* __restrict__ dt) {
  const int lane = threadIdx.x & 31;
  const int G = kWarp / L, lg = lane % L, grp = lane / L;
  const float t = __ldg(t_ptr);
  float dt_acc = 0.f;
  for (int lr = blockIdx.x * kPairWarps + (threadIdx.x >> 5); lr < row_count; lr += gridDim.x * kPairWarps) {
    const int i = row_begin + lr;
    if (i >= n) continue;
    const float* zi = z + (size_t)i * d;
    for (int c0 = 0; c0 < d; c0 += V * L) {   // feature chunks of V*L columns
      const int c = c0 + V * lg;
      const bool cok = c < d;
      float a[V], acc[V];
#pragma unroll
      for (int v = 0; v < V; ++v) a[v] = acc[v] = 0.f;
      if (cok) ldg_v<V>(a, zi + c);
      for (int r0 = 0; r0 < kc; r0 += G) {
        const int r = r0 + grp;
        const int j = (r < kc) ? __ldg(idx + (size_t)lr * kc + r) : -1;
        const float g_up = (j >= 0) ? __ldg(gy + (size_t)lr * kc + r) : 0.f;
        // full squared distance needs every chunk: recompute it over all of d (d is small)
        float dist2 = 0.f;
        if (j >= 0)
          for (int cc = V * lg; cc < d; cc += V * L) {
            float p[V], qv[V];
            ldg_v<V>(p, zi + cc);
            ldg_v<V>(qv, z + (size_t)j * d + cc);
            float s = (p[0] - qv[0]) * (p[0] - qv[0]);
#pragma unroll
            for (int v = 1; v < V; ++v) s += (p[v] - qv[v]) * (p[v] - qv[v]);
            dist2 += s;
          }
        dist2 = group_sum(dist2, L);
        const float dist = sqrtf(dist2);
        if (c0 == 0 && lg == 0) dt_acc += -dist * g_up;
        const float g = (dist > 0.f) ? (-t * g_up / dist) : 0.f;
        if (j >= 0 && cok && g != 0.f) {
          float b[V];
          ldg_v<V>(b, z + (size_t)j * d + c);
#pragma unroll
          for (int v = 0; v < V; ++v) {
            b[v] = g * (a[v] - b[v]);
            acc[v] += b[v];
          }
          red_add_v<V>(dz + (size_t)j * d + c, b, -1.f);
        }
      }
      for (int o = L; o < kWarp; o <<= 1)
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] += __shfl_xor_sync(0xffffffffu, acc[v], o);
      if (grp == 0 && cok) red_add_v<V>(dz + (size_t)i * d + c, acc, 1.f);
    }
  }
  dt_acc = warp_sum(dt_acc);
  if (lane == 0 && dt_acc != 0.f) atomicAdd(dt, dt_acc);
}

}  // namespace dggb
using namespace dggb;

// Column parts for the two-group kernel: S in [1, 8] minimising ceil(blocks S / SMs) / S (waves of full-length work),
// each part at least 64 key tiles long.  Every part warms up its own lists (Kc ln(N_part / Kc) insertions per row and
// part instead of Kc ln(N / Kc) per row), measured at 11-14 % of a full-length block per extra part (Reddit shape,
// gpurun_out/ap_prefilter_ab4.txt: 228 blocks in 5 parts = 1.6 instead of 2 waves ran 23.1 instead of 20.3 ms), so
// parts only pay where the row blocks leave SMs idle in EVERY wave (fewer blocks than SMs), not for a ragged last wave.
static int ap_choose_parts(int row_count, int n, int kc) {
  if (kc > 32 || row_count <= 0) return 1;
  if (const char* e = getenv("DGGB_AP_PARTS")) {
    const int v = atoi(e);
    if (v >= 1 && v <= kMaxParts) return std::min(v, std::max(1, ((n + kBN - 1) / kBN) / 8));
  }
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int blocks = (row_count + kBM - 1) / kBM, tiles = (n + kBN - 1) / kBN;
  int best = 1;
  double best_cost = 1e30;
  for (int sp = 1; sp <= kMaxParts; ++sp) {
    if (sp > 1 && tiles / sp < 64) break;
    const double cost = (double)((blocks * sp + sms - 1) / sms) / sp * (1.0 + 0.12 * (sp - 1));
    if (cost < best_cost - 1e-9) {
      best_cost = cost;
      best = sp;
    }
  }
  return best;
}

static int64_t ap_base_workspace(int32_t n, int32_t d) {
  const int64_t npad = ((int64_t)n + 127) / 128 * 128;
  int64_t dpad = ((int64_t)d + 31) / 32 * 32;
  if (dpad == 96) dpad = 128;   // k-blocks come in 1, 2 or 4 (zero-padded columns)
  return npad * dpad * 4 * 2 + npad * 4;
}

extern "C" int64_t dggb_allpairs_workspace_bytes_rows(int32_t n, int32_t d, int32_t row_count, int32_t kc) {
  if (n < 0 || d <= 0 || row_count < 0 || kc <= 0) return DGGB_ERR_BAD_ARG;
  const int parts = d > 128 ? 1 : ap_choose_parts(row_count, n, kc);   // the streamed shape runs unsplit
  return ap_base_workspace(n, d) + (parts > 1 ? (int64_t)parts * row_count * kc * 8 : 0);
}

extern "C" int64_t dggb_allpairs_workspace_bytes(int32_t n, int32_t d) {
  if (n < 0 || d <= 0) return DGGB_ERR_BAD_ARG;
  return ap_base_workspace(n, d);
}

extern "C" int dggb_allpairs_topk_fwd(const float* z, int32_t n, int32_t d, int32_t row_begin, int32_t row_count,
                                      const float* t, const float* noise, int64_t noise_ld, uint64_t seed,
                                      float noise_scale, int32_t kc, int32_t precision, void* workspace,
                                      int64_t workspace_bytes, int32_t* out_idx, float* out_val, float inv_temp,
                                      float* out_rowsum, void* stream) {
  return dggb_allpairs_topk_after_fwd(z, n, d, row_begin, row_count, t, noise, noise_ld, seed, noise_scale, kc,
                                      precision, workspace, workspace_bytes, nullptr, nullptr, out_idx, out_val,
                                      inv_temp, out_rowsum, stream);
}

extern "C" int dggb_allpairs_topk_after_fwd(const float* z, int32_t n, int32_t d, int32_t row_begin,
                                            int32_t row_count, const float* t, const float* noise, int64_t noise_ld,
                                            uint64_t seed, float noise_scale, int32_t kc, int32_t precision,
                                            void* workspace, int64_t workspace_bytes, const float* after_val,
                                            const int32_t* after_idx, int32_t* out_idx, float* out_val,
                                            float inv_temp, float* out_rowsum, void* stream) {
  if ((after_val == nullptr) != (after_idx == nullptr)) return DGGB_ERR_BAD_ARG;
  if (!z || !t || !workspace || !out_idx || !out_val || n <= 0 || d <= 0 || row_begin < 0 || row_count < 0 || kc <= 0)
    return DGGB_ERR_BAD_ARG;
  if (kc > 64) return DGGB_ERR_BAD_SHAPE;
  if (precision != 1 && precision != 3) return DGGB_ERR_UNSUPPORTED;
  if (workspace_bytes < dggb_allpairs_workspace_bytes(n, d)) return DGGB_ERR_WORKSPACE;
  if (row_count == 0) return DGGB_OK;
  const int npad = (n + 127) / 128 * 128;
  int dpad = (d + 31) / 32 * 32;
  if (dpad == 96) dpad = 128;
  float* hi = reinterpret_cast<float*>(workspace);
  float* lo = hi + (size_t)npad * dpad;
  float* nrm = lo + (size_t)npad * dpad;
  cudaStream_t st = as_stream(stream);
  split_tf32_kernel<<<rows_grid(npad, 8, 8), 256, 0, st>>>(z, n, npad, d, dpad, hi, lo, nrm);
  int rc = launch_status();
  if (rc != DGGB_OK) return rc;

  CUtensorMap tm_hi, tm_lo;
  rc = make_tmap_2d_f32(&tm_hi, hi, npad, dpad, 64, 32);
  if (rc != DGGB_OK) return rc;
  rc = make_tmap_2d_f32(&tm_lo, lo, npad, dpad, 64, 32);
  if (rc != DGGB_OK) return rc;

  const int kb = dpad / 32;
  // d > 128: no kernel has room for the whole query tile, so v1's k-block-streamed instantiation (KB = 0) runs the call,
  // unsplit, whatever DGGB_AP_V1 / DGGB_AP_PARTS say
  const bool streamed = kb > 4;
  // ---- v2 (two epilogue groups, A in TMEM) whenever the second list/queue set fits: kc <= 32 ----
  const int nmode2 = noise ? 1 : (noise_scale != 0.f ? 2 : (out_rowsum ? 3 : 0));
  if (out_rowsum && nmode2 != 3) return DGGB_ERR_UNSUPPORTED;
  // measured (scripts/ap_micro.py, N = 37 888, Gpairs/s, v1 -> v2): no noise 352 -> 377, Philox 215 -> 284
  const bool want_v2 = !getenv("DGGB_AP_V1");
  // d = 128 at 3xTF32 (the reference's default dgm_dim): a key stage is 64 KB, so the per-row queues shrink to 16
  // slots (flushed whenever anything is pending) to keep two stages + both groups' lists under 227 KB
  const bool big = (kb == 4 && precision == 3);
  const int qcap = big ? kChunk : kQCap, qflush = big ? 1 : kQFlush;
  if (!streamed && kc <= 32 && (want_v2 || big) && after_val == nullptr) {
    int st2 = 4;
    AP2Smem L2 = ap2_smem_layout(kb, precision, st2, kc, qcap);
    while (st2 > 2 && L2.total + 1024 > 227 * 1024) L2 = ap2_smem_layout(kb, precision, --st2, kc, qcap);
    if (L2.total + 1024 <= 227 * 1024) {
      const size_t smem2 = L2.total + 1024;
      const int grid2 = (row_count + kBM - 1) / kBM;
      const int no_pf = getenv("DGGB_AP_NO_PREFILTER") ? 1 : 0;     // A/B switch: one-step Philox scoring
      // column parts when the row blocks fill the SMs badly and the caller's workspace has room for the part lists
      int parts = (nmode2 == 3) ? 1 : ap_choose_parts(row_count, n, kc);
      const int64_t base_ws = ap_base_workspace(n, d);
      if (parts > 1 && workspace_bytes < base_ws + (int64_t)parts * row_count * kc * 8) parts = 1;
      const int total_tiles = (n + kBN - 1) / kBN;
      const int tpp = (total_tiles + parts - 1) / parts;
      parts = (total_tiles + tpp - 1) / tpp;                        // no empty part
      int32_t* part_idx = reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(workspace) + base_ws);
      float* part_val = reinterpret_cast<float*>(part_idx + (size_t)parts * row_count * kc);
      const dim3 grid2d(grid2, parts);
#define DGGB_AP2_LAUNCH1(KB_, SP_, NM_)                                                                           \
  do {                                                                                                            \
    cudaError_t e = cudaFuncSetAttribute(allpairs_topk2_kernel<KB_, SP_, NM_>,                                    \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);                \
    if (e != cudaSuccess) return cuda_status(e);                                                                  \
    allpairs_topk2_kernel<KB_, SP_, NM_><<<grid2d, kAP2Threads, smem2, st>>>(                                     \
        tm_hi, tm_lo, hi, lo, npad, dpad, nrm, n, row_begin, row_count, t, noise, (long long)noise_ld,            \
        (unsigned long long)seed, noise_scale, kc, st2, qcap, qflush, out_idx, out_val, inv_temp, out_rowsum,     \
        no_pf, tpp, part_idx, part_val, kc, nullptr, nullptr, 0);                                                 \
  } while (0)
#define DGGB_AP2_LAUNCH(KB_, SP_)                                                                                 \
  do {                                                                                                            \
    if (nmode2 == 0) DGGB_AP2_LAUNCH1(KB_, SP_, 0);                                                               \
    else if (nmode2 == 1) DGGB_AP2_LAUNCH1(KB_, SP_, 1);                                                          \
    else if (nmode2 == 2) DGGB_AP2_LAUNCH1(KB_, SP_, 2);                                                          \
    else DGGB_AP2_LAUNCH1(KB_, SP_, 3);                                                                           \
  } while (0)
      if (kb == 1 && precision == 3) DGGB_AP2_LAUNCH(1, 3);
      else if (kb == 1) DGGB_AP2_LAUNCH(1, 1);
      else if (kb == 2 && precision == 3) DGGB_AP2_LAUNCH(2, 3);
      else if (kb == 2) DGGB_AP2_LAUNCH(2, 1);
      else if (kb == 4 && precision == 3) DGGB_AP2_LAUNCH(4, 3);
      else if (kb == 4) DGGB_AP2_LAUNCH(4, 1);
      else return DGGB_ERR_BAD_SHAPE;
#undef DGGB_AP2_LAUNCH
#undef DGGB_AP2_LAUNCH1
      if (parts > 1) {
        rc = launch_status();
        if (rc != DGGB_OK) return rc;
        allpairs_merge_parts_kernel<<<std::min((row_count + kMergeWarps - 1) / kMergeWarps, 148 * 8), kMergeWarps * kWarp,
                                      0, st>>>(part_idx, part_val, parts, row_count,
                                               std::min(row_count, n - row_begin), kc, out_idx, out_val);
      }
      return launch_status();
    }
  }
  // the same tile shape beyond one plain v2 call (kc 33..64, continuation passes): v1 has no instantiation for it, so
  // the continuation instantiation of v2 runs it, kc > 32 as two passes whose second admits only what sorts after
  // the first pass's last entry of the row (ranks 32..kc-1)
  if (big) {
    const int no_pf = getenv("DGGB_AP_NO_PREFILTER") ? 1 : 0;
    auto cont_pass = [&](int kcp, int32_t* oi, float* ov, const float* av, const int32_t* ai, int ald,
                         float* rs) -> int {
      int st2 = 4;
      AP2Smem L2 = ap2_smem_layout(kb, precision, st2, kcp, qcap);
      while (st2 > 2 && L2.total + 1024 > 227 * 1024) L2 = ap2_smem_layout(kb, precision, --st2, kcp, qcap);
      if (L2.total + 1024 > 227 * 1024) return DGGB_ERR_BAD_SHAPE;
      const size_t smem2 = L2.total + 1024;
      const dim3 grid2d((row_count + kBM - 1) / kBM, 1);
      const int tpp = (n + kBN - 1) / kBN;
#define DGGB_AP2C_LAUNCH1(NM_)                                                                                    \
  do {                                                                                                            \
    cudaError_t e = cudaFuncSetAttribute(allpairs_topk2_kernel<4, 3, NM_, true>,                                  \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);                \
    if (e != cudaSuccess) return cuda_status(e);                                                                  \
    allpairs_topk2_kernel<4, 3, NM_, true><<<grid2d, kAP2Threads, smem2, st>>>(                                   \
        tm_hi, tm_lo, hi, lo, npad, dpad, nrm, n, row_begin, row_count, t, noise, (long long)noise_ld,            \
        (unsigned long long)seed, noise_scale, kcp, st2, qcap, qflush, oi, ov, inv_temp, rs, no_pf, tpp, nullptr, \
        nullptr, kc, av, ai, ald);                                                                                \
  } while (0)
      if (nmode2 == 0) DGGB_AP2C_LAUNCH1(0);
      else if (nmode2 == 1) DGGB_AP2C_LAUNCH1(1);
      else if (nmode2 == 2) DGGB_AP2C_LAUNCH1(2);
      else DGGB_AP2C_LAUNCH1(3);
#undef DGGB_AP2C_LAUNCH1
      return launch_status();
    };
    if (kc <= 32) return cont_pass(kc, out_idx, out_val, after_val, after_idx, 1, out_rowsum);
    rc = cont_pass(32, out_idx, out_val, after_val, after_idx, 1, out_rowsum);
    if (rc != DGGB_OK) return rc;
    return cont_pass(kc - 32, out_idx + 32, out_val + 32, out_val + 31, out_idx + 31, kc, nullptr);
  }
  const int kbt = streamed ? 0 : kb;   // template KB
  int stages = 4;
  APSmem L = ap_smem_layout(kbt, precision, stages, kc);
  while (stages > 2 && L.total + 1024 > 227 * 1024) L = ap_smem_layout(kbt, precision, --stages, kc);
  if (L.total + 1024 > 227 * 1024) return DGGB_ERR_BAD_SHAPE;
  const size_t smem_bytes = L.total + 1024;
  const int grid = (row_count + kBM - 1) / kBM;

  // noise mode: injected tensor if given, else Philox when noise_scale != 0, else none
  const int nmode = noise ? 1 : (noise_scale != 0.f ? 2 : (out_rowsum ? 3 : 0));
  if (out_rowsum && nmode != 3) return DGGB_ERR_UNSUPPORTED;   // the normaliser is an evaluation (no-noise) feature
#define DGGB_AP_LAUNCH1(KB_, SP_, NM_)                                                                            \
  do {                                                                                                            \
    cudaError_t e = cudaFuncSetAttribute(allpairs_topk_kernel<KB_, SP_, NM_>,                                     \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);           \
    if (e != cudaSuccess) return cuda_status(e);                                                                  \
    allpairs_topk_kernel<KB_, SP_, NM_><<<grid, kAPThreads, smem_bytes, st>>>(                                    \
        tm_hi, tm_lo, nrm, n, row_begin, row_count, t, noise, (long long)noise_ld, (unsigned long long)seed,      \
        noise_scale, kc, stages, out_idx, out_val, inv_temp, out_rowsum, after_val, after_idx, kb);               \
  } while (0)
#define DGGB_AP_LAUNCH(KB_, SP_)                                                                                  \
  do {                                                                                                            \
    if (nmode == 0) DGGB_AP_LAUNCH1(KB_, SP_, 0);                                                                 \
    else if (nmode == 1) DGGB_AP_LAUNCH1(KB_, SP_, 1);                                                            \
    else if (nmode == 2) DGGB_AP_LAUNCH1(KB_, SP_, 2);                                                            \
    else DGGB_AP_LAUNCH1(KB_, SP_, 3);                                                                            \
  } while (0)

  if (streamed && precision == 3) DGGB_AP_LAUNCH(0, 3);
  else if (streamed) DGGB_AP_LAUNCH(0, 1);
  else if (kb == 1 && precision == 3) DGGB_AP_LAUNCH(1, 3);
  else if (kb == 1) DGGB_AP_LAUNCH(1, 1);
  else if (kb == 2 && precision == 3) DGGB_AP_LAUNCH(2, 3);
  else if (kb == 2) DGGB_AP_LAUNCH(2, 1);
  else if (kb == 4 && precision == 1) DGGB_AP_LAUNCH(4, 1);
  else return DGGB_ERR_BAD_SHAPE;
#undef DGGB_AP_LAUNCH
#undef DGGB_AP_LAUNCH1
  return launch_status();
}

extern "C" int dggb_allpairs_pair_bwd(const float* z, int32_t n, int32_t d, int32_t row_begin, int32_t row_count,
                                      const int32_t* idx, const float* gy, int32_t kc, const float* t, float* dz,
                                      float* dt, void* stream) {
  if (!z || !idx || !gy || !t || !dz || !dt || n <= 0 || d <= 0 || row_count < 0 || kc <= 0) return DGGB_ERR_BAD_ARG;
  if (row_count == 0) return DGGB_OK;
  const dim3 grid(rows_grid(row_count, kPairWarps, 8));
  if (d % 4 == 0)   // one float4 per lane
    allpairs_pair_grad_kernel<4><<<grid, kPairWarps * kWarp, 0, as_stream(stream)>>>(
        z, n, d, pow2_floor32(d / 4), row_begin, row_count, idx, gy, kc, t, dz, dt);
  else              // rows of z are not 16-byte aligned: one float per lane
    allpairs_pair_grad_kernel<1><<<grid, kPairWarps * kWarp, 0, as_stream(stream)>>>(
        z, n, d, pow2_floor32(d), row_begin, row_count, idx, gy, kc, t, dz, dt);
  return launch_status();
}
