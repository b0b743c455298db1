// Cosine top-k search between two embedding sets (DESIGN.md 4.7): for every query row the k keys of highest (or lowest) cosine
// similarity, without ever writing the [Nq][Nk] similarity matrix.
//
//   1. topk_normalize_kernel: unit bf16 copies and fp32 inverse norms of both sets (workspace).  HBM-bound.
//   2. topk_search_kernel: persistent tcgen05 GEMM over (query tile, key range) items.  The 128-row query tile stays in shared memory for the
//      whole item while 256-key tiles stream through the TMA ring; the 128 x 256 fp32 scores land in one of two TMEM accumulators.  The
//      epilogue (4 warps, TMEM lane = query row) keeps a running list of the C = 2k best (score, key) pairs per row in shared memory: a
//      32-column chunk whose maximum does not beat the row's admission threshold (its C-th best so far) costs one tcgen05.ld share and a
//      max tree; the rare survivor is insertion-sorted.  At the end of the item the list goes to the workspace.
//   3. topk_merge_kernel: per query row (one warp), merge the lists of its key ranges, re-score the C candidates in fp32 from the
//      original inputs, and keep the best k.
//
// Ordering: scores are compared after the sign flip of largest = false (s' = -s), equal scores go to the lower key index, NaN is never
// admitted.  Every partial list is the exact top-C of its key range under that strict order, so the merged top-C -- and therefore the
// result -- does not depend on how the key range was split; every pair's bf16 score comes out of the same MMA shape and K order.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace psvae {

constexpr int TK_BM = 128;                       // query rows per tile: one TMEM lane each
constexpr int TK_BN = 256;                       // keys per tile: UMMA N, one 256-column accumulator
constexpr int TK_BK = 64;                        // k-block: 64 bf16 = one 128-byte swizzled row
constexpr int TK_MAX_K = 16, TK_MAX_C = 2 * TK_MAX_K, TK_MAX_DIM = 512;
constexpr int TK_EPI_WARPS = 4;
constexpr int TK_THREADS = 32 * (2 + TK_EPI_WARPS);
constexpr int TK_QBLOCK_BYTES = TK_BM * TK_BK * 2;     // 16 KB per k-block of the resident query tile
constexpr int TK_STAGE_BYTES = TK_BN * TK_BK * 2;      // 32 KB per ring stage (256 keys x 64)
constexpr int TK_MAX_STAGES = 8;
constexpr int TK_SMEM_MAX = 227 * 1024;
constexpr int TK_BAR_BYTES = 1024;

struct TopkShape {
  int64_t nk;              // keys of this call
  int64_t q_row0, k_row0;  // global index of the first query / key row (exclude-self compares these)
  int32_t kb;              // k-blocks of the contraction: ceil(dim / 64) (the TMA zero-fills the K tail)
  int32_t C;               // candidates kept per row
  int32_t m_tiles, k_tiles, splits, tiles_per_split;
  int32_t stages;
  int32_t exclude_self;
  uint32_t list_off, q_off, ring_off;   // shared-memory offsets (bytes, from the 1024-aligned base)
  int2* part;              // [splits][m_tiles * 128][C] (score bits, local key index; -1 = empty)
};

// ---- 1. normalisation: u = bf16(x / max(||x||, 1e-8)), inv = 1 / max(||x||, 1e-8); one warp per row ----
template <typename T>
__global__ void __launch_bounds__(256) topk_normalize_kernel(const T* __restrict__ x, int64_t rows, int dim, bf16* __restrict__ u,
                                                              float* __restrict__ inv) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += nw) {
    const T* xr = x + r * dim;
    float v[TK_MAX_DIM / 32];
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < TK_MAX_DIM / 32; ++i) {
      const int d = lane + 32 * i;
      v[i] = d < dim ? to_f32(xr[d]) : 0.f;
      ss = fmaf(v[i], v[i], ss);
    }
    ss = __shfl_sync(0xffffffffu, warp_sum(ss), 0);
    const float nrm = sqrtf(ss);
    const float iv = isnan(nrm) ? nrm : 1.f / fmaxf(nrm, 1e-8f);      // a NaN row stays NaN (fmaxf would drop it)
    bf16* ur = u + r * dim;
#pragma unroll
    for (int i = 0; i < TK_MAX_DIM / 32; ++i) {
      const int d = lane + 32 * i;
      if (d < dim) ur[d] = __float2bfloat16_rn(v[i] * iv);
    }
    if (lane == 0) inv[r] = iv;
  }
}

// ---- 2. search ----
template <bool LARGEST>
__global__ void __launch_bounds__(TK_THREADS, 1)
topk_search_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k, TopkShape s) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  uint64_t* full_bar = bars;                          // [TK_MAX_STAGES] TMA -> MMA
  uint64_t* empty_bar = bars + TK_MAX_STAGES;         // [TK_MAX_STAGES] MMA -> TMA
  uint64_t* tfull_bar = bars + 2 * TK_MAX_STAGES;     // [2] MMA -> epilogue
  uint64_t* tempty_bar = tfull_bar + 2;               // [2] epilogue -> MMA
  uint64_t* q_full = tempty_bar + 2;                  // query tile landed
  uint64_t* q_empty = q_full + 1;                     // the item's last MMA has read the query tile
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(q_empty + 1);
  uint8_t* const sq = smem + s.q_off;
  uint8_t* const ring = smem + s.ring_off;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tma_q);
    ptx::prefetch_tensormap(&tma_k);
    for (int i = 0; i < TK_MAX_STAGES; ++i) {
      ptx::mbar_init(&full_bar[i], 1);
      ptx::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tfull_bar[i], 1);
      ptx::mbar_init(&tempty_bar[i], TK_EPI_WARPS);
    }
    ptx::mbar_init(q_full, 1);
    ptx::mbar_init(q_empty, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 2 * TK_BN);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t items = (int64_t)s.m_tiles * s.splits;     // item t: query tile t % m_tiles, key range t / m_tiles
  if (warp == 0) {
    // ============================ TMA producer ============================
    int stage = 0;
    uint32_t phase = 0, n = 0;
    for (int64_t t = blockIdx.x; t < items; t += gridDim.x, ++n) {
      const int32_t m = (int32_t)(t % s.m_tiles), sp = (int32_t)(t / s.m_tiles);
      const int32_t kt0 = sp * s.tiles_per_split, kt1 = min(s.k_tiles, kt0 + s.tiles_per_split);
      ptx::mbar_wait(q_empty, (n & 1) ^ 1, 40);
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(q_full, (uint32_t)(s.kb * TK_QBLOCK_BYTES));
        for (int b = 0; b < s.kb; ++b) ptx::tma_load_2d(sq + b * TK_QBLOCK_BYTES, &tma_q, q_full, b * TK_BK, m * TK_BM);
      }
      __syncwarp();
      for (int32_t kt = kt0; kt < kt1; ++kt) {
        for (int b = 0; b < s.kb; ++b) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1, 41);
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(&full_bar[stage], TK_STAGE_BYTES);
            ptx::tma_load_2d(ring + stage * TK_STAGE_BYTES, &tma_k, &full_bar[stage], b * TK_BK, kt * TK_BN);
          }
          __syncwarp();
          if (++stage == s.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ============================ MMA issuer ==============================
    const uint32_t idesc = ptx::make_idesc_bf16(TK_BM, TK_BN, 0, 0);
    const uint64_t dq0 = ptx::make_smem_desc_sw128(ptx::smem_u32(sq), 16, 8 * 128);
    const uint64_t dk0 = ptx::make_smem_desc_sw128(ptx::smem_u32(ring), 16, 8 * 128);
    int stage = 0;
    uint32_t phase = 0, n = 0;
    int64_t it = 0;
    for (int64_t t = blockIdx.x; t < items; t += gridDim.x, ++n) {
      const int32_t sp = (int32_t)(t / s.m_tiles);
      const int32_t kt0 = sp * s.tiles_per_split, kt1 = min(s.k_tiles, kt0 + s.tiles_per_split);
      ptx::mbar_wait(q_full, n & 1, 42);
      ptx::tc_fence_after();
      for (int32_t kt = kt0; kt < kt1; ++kt, ++it) {
        const int acc = (int)(it & 1);
        ptx::mbar_wait(&tempty_bar[acc], (uint32_t)((it >> 1) & 1) ^ 1, 43);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * TK_BN);
        for (int b = 0; b < s.kb; ++b) {
          ptx::mbar_wait(&full_bar[stage], phase, 44);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
#pragma unroll
            for (int kk = 0; kk < TK_BK / 16; ++kk) {
              const uint64_t da = dq0 + (uint64_t)((uint32_t)(b * TK_QBLOCK_BYTES + kk * 32) >> 4);
              const uint64_t db = dk0 + (uint64_t)((uint32_t)(stage * TK_STAGE_BYTES + kk * 32) >> 4);
              ptx::umma_f16(tmem_d, da, db, idesc, (b > 0 || kk > 0) ? 1u : 0u);
            }
            ptx::umma_commit(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == s.stages) { stage = 0; phase ^= 1; }
        }
        if (ptx::elect_one()) ptx::umma_commit(&tfull_bar[acc]);
        __syncwarp();
      }
      if (ptx::elect_one()) ptx::umma_commit(q_empty);
      __syncwarp();
    }
  } else {
    // ============================ epilogue: running top-C per query row ============================
    const int quarter = warp & 3;                      // TMEM lane quarter this warp may read
    const int r = quarter * 32 + lane;                 // row of the query tile
    float* const ls = reinterpret_cast<float*>(smem + s.list_off);        // [C][128] scores, best first
    int* const li = reinterpret_cast<int*>(ls + s.C * TK_BM);              // [C][128] local key indices
    const int C = s.C;
    for (int c = 0; c < C; ++c) { ls[c * TK_BM + r] = -INFINITY; li[c * TK_BM + r] = -1; }
    float thr = -INFINITY;                             // admission threshold: the C-th best score so far
    int64_t it = 0;
    for (int64_t t = blockIdx.x; t < items; t += gridDim.x) {
      const int32_t m = (int32_t)(t % s.m_tiles), sp = (int32_t)(t / s.m_tiles);
      const int32_t kt0 = sp * s.tiles_per_split, kt1 = min(s.k_tiles, kt0 + s.tiles_per_split);
      const int64_t q_lo = s.q_row0 + (int64_t)m * TK_BM;
      const int64_t qg = q_lo + r;                     // global index of this lane's query
      for (int32_t kt = kt0; kt < kt1; ++kt, ++it) {
        const int acc = (int)(it & 1);
        ptx::mbar_wait(&tfull_bar[acc], (uint32_t)((it >> 1) & 1), 45);
        ptx::tc_fence_after();
        const int64_t kbase = (int64_t)kt * TK_BN;
        const int64_t k_lo = s.k_row0 + kbase;
        // columns past the last key, or the diagonal of a self-search, are masked (rare tiles only)
        const bool masked = kbase + TK_BN > s.nk || (s.exclude_self && q_lo < k_lo + TK_BN && k_lo < q_lo + TK_BM);
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * TK_BN);
        auto chunk = [&](const uint32_t (&u)[32], int64_t col0) {
          float v[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = LARGEST ? __uint_as_float(u[i]) : -__uint_as_float(u[i]);
          if (masked) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int64_t j = col0 + i;
              if (j >= s.nk || (s.exclude_self && s.k_row0 + j == qg)) v[i] = __int_as_float(0x7fc00000);
            }
          }
          float mx[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) mx[i] = fmaxf(v[i], v[i + 16]);      // fmaxf drops NaN: a NaN score is never admitted
#pragma unroll
          for (int w = 8; w >= 1; w >>= 1) {
#pragma unroll
            for (int i = 0; i < w; ++i) mx[i] = fmaxf(mx[i], mx[i + w]);
          }
          if (mx[0] > thr) {
            // columns in increasing key order: an equal score already in the list has the lower index, so admission is strict
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (v[i] > thr) {
                int p = C - 1;
                while (p > 0) {
                  const float prev = ls[(p - 1) * TK_BM + r];
                  if (!(v[i] > prev)) break;
                  ls[p * TK_BM + r] = prev;
                  li[p * TK_BM + r] = li[(p - 1) * TK_BM + r];
                  --p;
                }
                ls[p * TK_BM + r] = v[i];
                li[p * TK_BM + r] = (int)(col0 + i);
                thr = ls[(C - 1) * TK_BM + r];
              }
            }
          }
        };
#pragma unroll 1
        for (int ch = 0; ch < TK_BN / 32; ch += 2) {
          uint32_t a[32], b[32];
          ptx::tmem_ld_32x32_issue(taddr + (uint32_t)(ch * 32), a);
          ptx::tmem_ld_32x32_issue(taddr + (uint32_t)(ch * 32 + 32), b);
          ptx::tmem_ld_wait(a);
          ptx::tmem_ld_wait(b);
          chunk(a, kbase + ch * 32);
          chunk(b, kbase + ch * 32 + 32);
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tempty_bar[acc]);
      }
      // the item's list -> workspace; start the next item empty
      int2* dst = s.part + (((int64_t)sp * s.m_tiles + m) * TK_BM + r) * C;
      for (int c = 0; c < C; ++c) {
        dst[c] = make_int2(__float_as_int(ls[c * TK_BM + r]), li[c * TK_BM + r]);
        ls[c * TK_BM + r] = -INFINITY;
        li[c * TK_BM + r] = -1;
      }
      thr = -INFINITY;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 2 * TK_BN);
  }
}

// ---- 3. merge + fp32 re-rank + final selection; one warp per query row ----
// (s, i) ranks before (t, j): a valid entry before an empty one (-1), then a number before NaN, then the higher score, then the lower index
__device__ __forceinline__ bool topk_better(float s, int i, float t, int j) {
  if (i < 0) return false;
  if (j < 0) return true;
  const bool ns = isnan(s), nt = isnan(t);
  if (ns != nt) return nt;
  if (!ns && s != t) return s > t;
  return i < j;
}

template <typename TQ, typename TK, bool LARGEST>
__global__ void __launch_bounds__(256) topk_merge_kernel(const int2* __restrict__ part, int64_t part_rows, int splits, int C, int k,
                                                          const TQ* __restrict__ q, const TK* __restrict__ keys, const float* __restrict__ invq,
                                                          const float* __restrict__ invk, int64_t nq, int dim, int64_t k_row0,
                                                          float* __restrict__ out_sim, int64_t* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < nq; row += nw) {
    // (a) lane c <- the c-th best of the bf16 selection over all key ranges
    int ci = -1;
    if (splits == 1) {
      if (lane < C) ci = part[row * C + lane].y;          // already in order
    } else {
      float ps = INFINITY;            // the previous winner: every later one ranks below it
      int pi = -1;
      const int total = splits * C;
      for (int c = 0; c < C; ++c) {
        float bs = -INFINITY;
        int bi = -1;
        for (int e = lane; e < total; e += 32) {
          const int sp = e / C, j = e - sp * C;
          const int2 v = part[((int64_t)sp * part_rows + row) * C + j];
          const float sv = __int_as_float(v.x);
          if (v.y < 0 || !(sv < ps || (sv == ps && v.y > pi))) continue;
          if (topk_better(sv, v.y, bs, bi)) { bs = sv; bi = v.y; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float os = __shfl_xor_sync(0xffffffffu, bs, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (topk_better(os, oi, bs, bi)) { bs = os; bi = oi; }
        }
        if (bi < 0) break;
        if (lane == c) ci = bi;
        ps = bs;
        pi = bi;
      }
    }
    // (b) fp32 re-score from the original inputs: lane-strided products, one fixed butterfly, lane 0's sum
    float qv[TK_MAX_DIM / 32];
    const float iq = invq[row];
#pragma unroll
    for (int i = 0; i < TK_MAX_DIM / 32; ++i) {
      const int d = lane + 32 * i;
      qv[i] = d < dim ? to_f32(q[row * dim + d]) * iq : 0.f;
    }
    float fs = __int_as_float(0x7fc00000);
    for (int c = 0; c < C; ++c) {
      const int j = __shfl_sync(0xffffffffu, ci, c);
      if (j < 0) break;
      const TK* xr = keys + (int64_t)j * dim;
      float a = 0.f;
#pragma unroll
      for (int i = 0; i < TK_MAX_DIM / 32; ++i) {
        const int d = lane + 32 * i;
        if (d < dim) a = fmaf(qv[i], to_f32(xr[d]), a);
      }
      const float sc = __shfl_sync(0xffffffffu, warp_sum(a), 0) * invk[j];
      if (lane == c) fs = LARGEST ? sc : -sc;
    }
    // (c) the best k of the C by the ordering rule
    bool taken = false;
    for (int rk = 0; rk < k; ++rk) {
      float bs = fs;
      int bi = (ci >= 0 && !taken) ? ci : -1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float os = __shfl_xor_sync(0xffffffffu, bs, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (topk_better(os, oi, bs, bi)) { bs = os; bi = oi; }
      }
      if (lane == 0) {
        out_sim[row * k + rk] = bi >= 0 ? (LARGEST ? bs : -bs) : __int_as_float(0x7fc00000);
        out_idx[row * k + rk] = bi >= 0 ? k_row0 + bi : -1;
      }
      if (bi >= 0 && ci == bi) taken = true;
    }
  }
}

}  // namespace psvae
