// tcgen05 GEMM engine for sm_100a:  C[M,N] = A[M,K] * B[N,K]^T  through a fused epilogue (DESIGN.md 4.1, 4.4).
//
//   * persistent, one CTA per SM, static round-robin tile schedule (n fastest: CTAs sharing a row tile run together), tiles walked
//     incrementally (TileWalk: no divisions in the loop);
//   * warp-specialised: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (one elected thread issues tcgen05.mma),
//     warps 2.. = epilogue: 16 warps for BN = 256, 8 for narrower tiles (tc_epi_warps);
//   * CG = 2: a CTA pair (cluster of 2, tcgen05 cta_group::2) works on one 256 x BN tile -- each CTA stages its own 128 rows of A and
//     half of the B tile, the leader issues UMMA 256 x BN x 16; CG = 1: one CTA, 128 x BN tiles (BN = 64 / 128, or M <= 128);
//   * operands bf16, staged by TMA (cp.async.bulk.tensor, 128B swizzle) through a ring of mbarrier stages (depth = what fits next to the
//     epilogue staging: 5 at BN = 256 / CG = 2); fp32 accumulators live in TMEM, double-buffered (2 x BN columns), so the epilogue of tile
//     i overlaps the MMAs of tile i+1.  EG2: two epilogue groups on alternate tiles for the thin (K <= 128) layers;
//   * both operands may be K-major (row-major [rows][K]) or MN-major (stored [K][rows]): dgrad consumes W as stored and wgrad contracts
//     over the batch, so no transposed copies exist anywhere;
//   * split-K (wgrad: K = batch): every split tile adds its block into the zeroed gradient with a TMA reduce-add (deterministic mode:
//     [splits][M][N] slots through a 3-D store map + an ordered reduce);
//   * grouped (block-diagonal) launches for the two encoders' layers; MULTI: one launch for a whole list of wgrad problems;
//   * epilogue: TMEM -> registers (tcgen05.ld, lane = row) -> functor in packed fp32 pairs -> round to the output type -> block staged in a
//     per-warp swizzled shared-memory buffer -> ONE TMA store per 32 x 64 block (coalesced, clipped at the matrix edge by the hardware;
//     a row-per-lane st.global cost 32 L1 wavefronts per instruction and made the first version LSU-bound).  The auxiliary tile of EpiMse
//     (the reconstruction target) comes in the same way by TMA load.  Bias-gradient column sums (kColSum) are read back out of the staged
//     block and kept in registers across the CTA's tiles.  kLat: the fused encoder head (EpiLatent).
//
// Tile: (128 x CG) x BN x 64 (UMMA K = 16).
#pragma once
#include <cuda.h>

#include <algorithm>

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"
#include "epilogue.cuh"
#include "philox.cuh"
#include "ptx.cuh"

namespace psvae {

constexpr int TC_BM = 128, TC_BK = 64, TC_UMMA_K = 16;
// epilogue warps: 4 TMEM lane quarters x (BN / kColsPerWarp) column groups.  BN = 256 runs 16 of them (4 per SM sub-partition): with 8 the
// epilogue was latency-bound (2 warps per scheduler, ~8 cycles per instruction) and set the tile time of every K <= 512 GEMM.
constexpr int tc_epi_warps(int bn) { return bn == 256 ? 16 : 8; }
constexpr int TC_MAX_EPI_WARPS = 16;
constexpr int TC_BAR_BYTES = 1024;
constexpr int TC_SMEM_MAX = 227 * 1024;
constexpr int TC_MAX_STAGES = 12;          // barrier slots of the operand ring

// Shared-memory plan of one instantiation.  Per epilogue warp: the staged output block (32 rows x 32 cols of TOut: 2 KB bf16 / 4 KB fp32)
// followed by the auxiliary block (Epi::kAuxBytes: 2 KB bf16 activation tile, 4 KB fp32 target tile); the operand ring gets the rest.
// CG = 2: a CTA pair (cluster of 2, tcgen05 cta_group::2) works on one 256 x BN tile: each CTA stages its own 128 rows of A and its
// half of the B tile (BN/2 rows), so the operand bytes per SM and per FLOP drop by a third and the ring gets 6 stages instead of 4.
// kLat: the fused encoder-head kernel (EpiLatent, option "fused_head"): see the kLat branches of gemm_tc_kernel
template <class Epi, class = void> struct epi_latent { static constexpr bool value = false; };
template <class Epi> struct epi_latent<Epi, std::void_t<decltype(Epi::kLatent)>> { static constexpr bool value = Epi::kLatent; };
constexpr int TC_LAT_L = 64;                     // latent width the fused head is written for
constexpr int TC_LAT_WARP_BYTES = 13 * 1024;     // per epilogue warp: mu block / Philox scratch 4 KB | log_sigma 4 KB | z 2 KB | sigma eps / 2 2 KB | logit exchange 1 KB

// EG2 ("two epilogue groups", BN = 256 only): the 16 epilogue warps form two groups of 8 that take ALTERNATE tiles -- group g owns the
// accumulator buffer g -- each warp draining 128 columns instead of 64.  While one group stages and stores its tile the other group's
// tcgen05.ld stream keeps the TMEM read port busy: for the thin (K <= 128) layers, which are bound by the accumulator drain
// (profiles/r01_epilogue_phase_trace_v16.txt: 3.4 k of 4.9 k cycles per tile in the drain, 0.8-1.6 k in staging + store with the port idle).
template <int BN, class Epi, int CG = 1, bool EG2 = false> struct TcCfg {
  static_assert(!EG2 || (BN == 256 && Epi::kAuxBytes == 0 && !Epi::kSplit), "EG2: 16 epilogue warps, no auxiliary tile, no split-K");
  static constexpr int kEpiWarps = tc_epi_warps(BN);
  static constexpr int kThreads = 32 * (2 + kEpiWarps);
  static constexpr int kColsPerWarp = EG2 ? BN / (kEpiWarps / 8) : BN / (kEpiWarps / 4);
  static constexpr bool kLat = epi_latent<Epi>::value;
  static_assert(!kLat || (BN == 128 && CG == 1 && !EG2), "fused head: 128-column tiles on one CTA");
  static constexpr int kABytes = TC_BM * TC_BK * 2;
  static constexpr int kBBytes = kLat ? TC_LAT_L * TC_BK * 2 : (BN / CG) * TC_BK * 2;      // kLat: one group's 64 weight rows per k-block
  static constexpr int kStageBytes = kABytes + kBBytes;
  // staged output block of one epilogue warp: 32 rows x 128 bytes (fp32: 32 columns; bf16: 64 columns = two tcgen05.ld chunks per
  // fence / TMA store) -- except BN = 64 with bf16 output, where a warp owns only 32 columns (32 rows x 64 bytes)
  static constexpr bool kWide = sizeof(typename Epi::TOut) == 2 && BN >= 128;
  static constexpr int kBlockCols = kWide ? 64 : 32;
  static constexpr int kOutBytes = 32 * kBlockCols * (int)sizeof(typename Epi::TOut);
  static constexpr int kOutBufs = EG2 ? 2 : 1;      // EG2: a warp stages two 64-column blocks per tile back to back -- two buffers, so the second does not wait
                                                     // for the first one's TMA store (K <= 128: the ring needs no depth, the 64 KB are free)
  static constexpr int kEpiWarpBytes = kLat ? TC_LAT_WARP_BYTES : kOutBufs * kOutBytes + Epi::kAuxBytes;
  static constexpr int kEpiBytes = kEpiWarps * kEpiWarpBytes;
  static constexpr int kTmemCols = 2 * BN;     // power of two >= 32 for BN in {64,128,256}
  // layout: [barriers][epilogue staging][operand ring]
  static constexpr int kBarOff = 0;
  static constexpr int kOpOff = TC_BAR_BYTES + kEpiBytes;
  static constexpr int kEpiOff = TC_BAR_BYTES;
  static_assert(kOpOff % 1024 == 0, "operand tiles need 1024-byte alignment");
  static constexpr int kOpBudget = TC_SMEM_MAX - 1024 /*align slack*/ - kOpOff;
  static constexpr int kMaxStages = CG == 2 ? 8 : (BN == 256 ? 4 : (BN == 128 ? 6 : 8));
  static constexpr int kFit = kOpBudget / kStageBytes;          // stages that fit
  static constexpr int kStages = kFit < kMaxStages ? kFit : kMaxStages;
  static_assert(kStages >= 2, "operand ring too shallow");
  static constexpr int kSmemBytes = kOpOff + kStages * kStageBytes + 1024 /*align slack*/;
};

// host-side description of a grouped launch (see TcShape::groups)
struct TcGroup {
  int groups = 1;
  int grp_n = 0, grp_k = 0;
  int64_t out_group_stride = 0;      // elements between the groups' output buffers; 0: column ranges of one [M][groups * grp_n] buffer
};

struct TcShape {
  int64_t M;        // rows of C
  int32_t N;        // cols of C
  int64_t K;
  int32_t splits;   // split-K factor (>= 1)
  uint32_t a_lbo, a_sbo, b_lbo, b_sbo;   // UMMA smem-descriptor strides (bytes)
  int32_t stages;   // depth of the operand ring actually used (<= the compiled kStages; option "tc_max_stages")
  int32_t rev_splits;   // MULTI: walk the batch ranges from the end (the rows the backward pass wrote last are the ones still in L2)
  unsigned long long* trace;   // profiling (option "tc_trace_ptr"): per CTA 16 cycle counters -- see tools/tc_trace.py; nullptr = off
  // grouped (block-diagonal) launch: `groups` independent GEMMs laid side by side.  A is [M][groups * grp_k] (group g owns the k range
  // [g * grp_k, (g+1) * grp_k)), C is [M][groups * grp_n]; B stacks the groups' weights along its row dimension: K-major B
  // [groups * grp_n][grp_k] (forward Linear) or MN-major B [groups * grp_k][grp_n] (dgrad).  K above is grp_k.  out3d: the groups' outputs
  // are separate [M][grp_n] buffers a fixed stride apart (third coordinate of the output map) instead of column ranges of one buffer.
  int32_t groups, grp_n, grp_k, out3d;
};

// MULTI ("merged wgrad"): ONE persistent launch works through a list of wgrad problems dW_p[M_p][N_p] += dY_p^T act_p that share the contraction
// length K (the batch rows) and the split factor.  Every (problem, tile, k-split) item costs the same number of k-blocks; the static
// round-robin schedule hands ~12 of them to each CTA pair, so every epilogue but the last overlaps the next item's mainloop and the
// per-launch fixed cost (pipeline fill, one exposed accumulator drain + reduce-add, teardown: ~8 us of a 20-35 us wgrad launch,
// tools/wgrad_probe.py) is paid once per step instead of once per layer.  The problems' tensor maps travel in kernel-parameter space.
constexpr int TC_MAX_PROBLEMS = 20;
struct TcMulti {
  CUtensorMap ta[TC_MAX_PROBLEMS], tb[TC_MAX_PROBLEMS], tout[TC_MAX_PROBLEMS];
  int64_t M[TC_MAX_PROBLEMS];
  int32_t N[TC_MAX_PROBLEMS];
  int32_t m_tiles[TC_MAX_PROBLEMS], n_tiles[TC_MAX_PROBLEMS];
  int32_t tile_begin[TC_MAX_PROBLEMS + 1];      // prefix sums of m_tiles * n_tiles * splits
  int32_t count;
};

// byte offset of 16-byte chunk j of row r inside a staged 32-row block whose rows are ROWB bytes (TMA swizzle = ROWB)
template <int ROWB> __device__ __forceinline__ uint32_t swz_off(int r, int j) {
  if constexpr (ROWB == 128) return (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4));       // SWIZZLE_128B: addr[4:6] ^= addr[7:9]
  else return (uint32_t)(r * 64 + ((j ^ ((r >> 1) & 3)) << 4));                      // SWIZZLE_64B:  addr[4:5] ^= addr[7:8]
}

template <int BN, bool A_MN, bool B_MN, class Epi, int CG, bool EG2 = false, bool MULTI = false>
__device__ __forceinline__ void gemm_tc_body(const CUtensorMap& tma_a, const CUtensorMap& tma_b, const CUtensorMap& tma_out, const CUtensorMap& tma_aux,
                                             const TcMulti* mp, TcShape s, Epi epi) {
  using Cfg = TcCfg<BN, Epi, CG, EG2>;
  static_assert(!MULTI || (A_MN && B_MN && Epi::kSplit && Epi::kAuxBytes == 0 && !EG2), "MULTI: the plain wgrad form");
  using TOut = typename Epi::TOut;
  constexpr int STAGES = TC_MAX_STAGES;                    // barrier slots; s.stages of them are in use
  constexpr int EPI_WARPS = Cfg::kEpiWarps;
  constexpr int TM = TC_BM * CG;                           // rows of one (cluster) tile
  constexpr bool WIDE = Cfg::kWide;
  constexpr int ROWB = Cfg::kBlockCols * (int)sizeof(TOut);   // bytes per staged row: 128, or 64 (bf16 at BN = 64)
  constexpr bool kAux = Epi::kAuxBytes > 0;
  constexpr bool kLat = Cfg::kLat;
  static_assert(!kLat || (!A_MN && !B_MN), "fused head: both operands K-major");
  static_assert(Epi::kAuxBytes == 0 || Epi::kAuxBytes == 2048 || Epi::kAuxBytes == 4096, "aux block: 32x32 bf16 or fp32");
  static_assert(!(Epi::kColSum && sizeof(TOut) != 2), "column sums are read back from a bf16 block");
  extern __shared__ uint8_t smem_raw[];
  // 128B-swizzled tiles need 1024-byte alignment
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kBarOff);
  uint64_t* full_bar = bars;                 // [STAGES]  TMA -> MMA
  uint64_t* empty_bar = bars + STAGES;       // [STAGES]  MMA -> TMA
  uint64_t* tfull_bar = bars + 2 * STAGES;   // [2]       MMA -> epilogue
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;  // [2]   epilogue -> MMA
  uint64_t* aux_bar = bars + 2 * STAGES + 4;     // [EPI_WARPS] aux tile landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4 + EPI_WARPS);
  uint8_t* const sring = smem + Cfg::kOpOff;                                       // operand ring
  float* red_smem = reinterpret_cast<float*>(tmem_slot + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (s.trace != nullptr && threadIdx.x == 0) s.trace[(size_t)blockIdx.x * 16 + 12] = ptx::globaltimer_ns();      // kernel entry
  const uint32_t cta_rank = CG == 2 ? ptx::cluster_ctarank() : 0u;    // rank inside the CTA pair (cluster dims (2,1,1))
  constexpr uint32_t lead_rank = 0u;                                   // cluster rank of the pair's leader
  const bool leader = cta_rank == 0;
  const int64_t work_id = CG == 2 ? (int64_t)(blockIdx.x >> 1) : (int64_t)blockIdx.x;
  const int64_t work_stride = CG == 2 ? (int64_t)(gridDim.x >> 1) : (int64_t)gridDim.x;

  if (warp == 0 && lane == 0) {
    if constexpr (!MULTI) {
      ptx::prefetch_tensormap(&tma_a);
      ptx::prefetch_tensormap(&tma_b);
      ptx::prefetch_tensormap(&tma_out);
    }
    if constexpr (kAux) ptx::prefetch_tensormap(&tma_aux);
    for (int i = 0; i < STAGES; ++i) {
      ptx::mbar_init(&full_bar[i], 1);
      ptx::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tfull_bar[i], 1);
      ptx::mbar_init(&tempty_bar[i], (EG2 ? EPI_WARPS / 2 : EPI_WARPS) * CG);      // CG = 2: the peer's epilogue warps arrive remotely on the leader's barrier; EG2: buffer i belongs to epilogue group i
    }
    for (int i = 0; i < EPI_WARPS; ++i) ptx::mbar_init(&aux_bar[i], 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (CG == 2) {
      ptx::tmem_alloc_cg2(tmem_slot, Cfg::kTmemCols);
      ptx::tmem_relinquish_cg2();
    } else {
      ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync();             // the peer's barriers must be initialised before anything signals them
  else __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above (barrier init, TMEM allocation, descriptor prefetch) overlapped the previous kernel's tail; its results
  // may only be touched from here on.  The successor may be scheduled once every CTA has passed this point.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  const int64_t m_tiles = (s.M + TM - 1) / TM;
  const int64_t n_tiles = (s.N + BN - 1) / BN;
  const int64_t kb_total = (s.K + TC_BK - 1) / TC_BK;
  const int64_t kb_per_split = (kb_total + s.splits - 1) / s.splits;
  const int64_t num_tiles = MULTI ? (int64_t)mp->tile_begin[mp->count] : m_tiles * n_tiles * s.splits;
  // MULTI: global item index -> (problem, tile inside the problem); n fastest, then m, then the k-split (as below)
  auto item_problem = [&](int64_t t) {
    int p = 0;
    while (p + 1 < mp->count && (int32_t)t >= mp->tile_begin[p + 1]) ++p;
    return p;
  };
  // tile order: n fastest -- the CTAs that share an A (row) tile run at the same time, so its second..n-th reads hit L2 instead of HBM;
  // with gridDim.x a multiple of n_tiles every CTA keeps one n_t for all of its tiles
  // (32-bit arithmetic: a 64-bit division here cost 7 % of the epilogue warps' issue slots)
  const uint32_t m_tiles32 = (uint32_t)m_tiles, n_tiles32 = (uint32_t)n_tiles;
  auto tile_m = [&](int64_t t) {
    if constexpr (MULTI) {
      const int p = item_problem(t);
      const uint32_t l = (uint32_t)t - (uint32_t)mp->tile_begin[p];
      return (int64_t)((l / (uint32_t)mp->n_tiles[p]) % (uint32_t)mp->m_tiles[p]);
    } else {
      const uint32_t m = ((uint32_t)t / n_tiles32) % m_tiles32;
      return (int64_t)m;
    }
  };
  auto tile_n = [&](int64_t t) {
    if constexpr (MULTI) {
      const int p = item_problem(t);
      return (int64_t)(((uint32_t)t - (uint32_t)mp->tile_begin[p]) % (uint32_t)mp->n_tiles[p]);
    } else {
      return (int64_t)((uint32_t)t % n_tiles32);
    }
  };
  auto tile_sp = [&](int64_t t) {
    if constexpr (MULTI) {
      const int p = item_problem(t);
      const uint32_t v = ((uint32_t)t - (uint32_t)mp->tile_begin[p]) / ((uint32_t)mp->n_tiles[p] * (uint32_t)mp->m_tiles[p]);
      return (int64_t)(s.rev_splits ? (uint32_t)s.splits - 1u - v : v);      // reduce-add: any order of the batch ranges gives the same sum
    } else {
      const uint32_t sp = (uint32_t)t / (n_tiles32 * m_tiles32);
      return (int64_t)sp;
    }
  };

  auto tile_g = [&](int64_t n_t) { return s.groups > 1 ? (int32_t)(((uint32_t)n_t * (uint32_t)BN) / (uint32_t)s.grp_n) : 0; };
  // (n, m, split) of the tiles work_id, work_id + work_stride, ...: advanced incrementally -- the three divisions per tile and role were 7 % of
  // the warp instructions of the thin layers (ncu, profiles/r02_ncu_epilogue_inst_mix.txt).  MULTI keeps the problem-list lookup above.
  struct TileWalk {
    uint32_t n, m, sp, dn, dm, dsp, nt, mt;
    __device__ __forceinline__ void init(uint32_t t0, uint32_t stride, uint32_t n_tiles_, uint32_t m_tiles_) {
      nt = n_tiles_; mt = m_tiles_;
      n = t0 % nt;
      const uint32_t q = t0 / nt;
      m = q % mt; sp = q / mt;
      dn = stride % nt;
      const uint32_t dq = stride / nt;
      dm = dq % mt; dsp = dq / mt;
    }
    __device__ __forceinline__ void next() {
      n += dn;
      uint32_t carry = 0;
      if (n >= nt) { n -= nt; carry = 1; }
      m += dm + carry;
      sp += dsp;
      if (m >= mt) { m -= mt; ++sp; }
    }
  };
  TileWalk walk;
  if constexpr (!MULTI) walk.init((uint32_t)work_id, (uint32_t)work_stride, n_tiles32, m_tiles32);

  float red = 0.f;
  float lat_kl = 0.f, lat_nll = 0.f, lat_acc = 0.f;      // kLat: this thread's share of the KL sum, the NLL sum and the correct-prediction count
  // profiling: cycles this warp spent inside a class of barrier waits (accumulated per warp, written by lane 0 at the end)
  const bool tracing = s.trace != nullptr;
  long long tw0 = 0, tw1 = 0, tw2 = 0;
  const long long t_begin = tracing ? clock64() : 0;
  const unsigned long long g_begin = tracing ? ptx::globaltimer_ns() : 0ull;
  auto twait = [&](uint64_t* bar, uint32_t parity, int tag, long long& acc_cycles) {
    if (tracing) {
      const long long t0 = clock64();
      ptx::mbar_wait(bar, parity, tag);
      acc_cycles += clock64() - t0;
    } else {
      ptx::mbar_wait(bar, parity, tag);
    }
  };

  if (warp == 0) {
    // ============================ TMA producer ============================
    // warp-uniform loop; the TMA instructions of one k-block are issued by one elected lane
    {
      const CUtensorMap* pa = &tma_a;        // MULTI: the current item's problem maps
      const CUtensorMap* pb = &tma_b;
      // issue (load into sa / sb) or prefetch-to-L2 (null destination with want_* set) the operand boxes of k-block kb of a tile
      auto fetch = [&](int64_t m_t, int64_t n_t, int64_t kb, uint8_t* sa, uint8_t* sb, uint64_t* bar, bool want_a, bool want_b) {
        const int32_t g = tile_g(n_t);
        const int32_t k_el = (int32_t)(kb * TC_BK) + g * s.grp_k;                        // A: group g owns columns [g * grp_k, (g+1) * grp_k)
        const int32_t k_el_b = (int32_t)(kb * TC_BK) + (B_MN ? g * s.grp_k : 0);         // B stacked along k (MN-major) or along n (K-major)
        // CG = 2: the bytes of BOTH CTAs are counted on the leader's barrier (only the leader issues MMAs)
        const uint32_t bar_addr = (CG == 2 && bar) ? ptx::mapa_u32(ptx::smem_u32(bar), lead_rank) : 0u;
        const int32_t a_row = (int32_t)(m_t * TM) + (int32_t)cta_rank * TC_BM;          // this CTA's 128 rows of the tile
        const int32_t b_row = (int32_t)(n_t * BN) + (int32_t)cta_rank * (BN / CG) - (B_MN ? g * s.grp_n : 0);   // this CTA's share of the B tile
        auto ld = [&](void* d, const CUtensorMap* m, int32_t c0, int32_t c1) {
          if constexpr (CG == 2) ptx::tma_load_2d_cg2(d, m, bar_addr, c0, c1);
          else ptx::tma_load_2d(d, m, bar, c0, c1);
        };
        if (want_a) {
          if constexpr (!A_MN) {
            if (sa) ld(sa, pa, k_el, a_row);
            else ptx::tma_prefetch_2d(pa, k_el, a_row);
          } else {
#pragma unroll
            for (int j = 0; j < TC_BM / 64; ++j) {
              if (sa) ld(sa + j * (64 * TC_BK * 2), pa, a_row + j * 64, k_el);
              else ptx::tma_prefetch_2d(pa, a_row + j * 64, k_el);
            }
          }
        }
        int32_t kb_b = k_el_b, row_b = b_row;
        if constexpr (kLat) {
          // two groups concatenated along K: the second half of the k-blocks belongs to log_sigma; a group's 64 weight rows are rows
          // [64 g, 64 g + 64) of the stacked [2L][H] weight matrix and its k range restarts at 0
          const int32_t kbg = (int32_t)(kb_total >> 1), gg = (int32_t)kb >= kbg ? 1 : 0;
          kb_b = ((int32_t)kb - gg * kbg) * TC_BK;
          row_b = gg * TC_LAT_L;
        }
        if (want_b) {
          if constexpr (!B_MN) {
            if (sb) ld(sb, pb, kb_b, row_b);
            else ptx::tma_prefetch_2d(pb, kb_b, row_b);
          } else {
#pragma unroll
            for (int j = 0; j < (BN / CG) / 64; ++j) {
              if (sb) ld(sb + j * (64 * TC_BK * 2), pb, b_row + j * 64, k_el_b);
              else ptx::tma_prefetch_2d(pb, b_row + j * 64, k_el_b);
            }
          }
        }
      };
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t tile = work_id; tile < num_tiles; tile += work_stride, walk.next()) {
        const int64_t m_t = MULTI ? tile_m(tile) : (int64_t)walk.m, n_t = MULTI ? tile_n(tile) : (int64_t)walk.n,
                      sp = MULTI ? tile_sp(tile) : (int64_t)walk.sp;
        const int64_t kb0 = sp * kb_per_split, kb1 = min(kb_total, kb0 + kb_per_split);
        if constexpr (MULTI) {
          const int p = item_problem(tile);
          pa = &mp->ta[p];
          pb = &mp->tb[p];
        }
        for (int64_t kb = kb0; kb < kb1; ++kb) {
          twait(&empty_bar[stage], phase ^ 1, 1, tw0);
          if (ptx::elect_one()) {
            if (leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes * CG);
            uint8_t* const st_base = sring + stage * Cfg::kStageBytes;
            fetch(m_t, n_t, kb, st_base, st_base + Cfg::kABytes, &full_bar[stage], true, true);
          }
          __syncwarp();
          if (++stage == s.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ============================ MMA issuer ==============================
    // The whole warp walks the loop (warp-uniform control flow and operands); only the tcgen05 instructions are predicated on one
    // elected lane.  Descriptors are a precomputed base + a stage / k-slice offset in the 14-bit address field.
    if (leader) {
      const uint32_t idesc = ptx::make_idesc_bf16(TM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      constexpr uint32_t a_kstep = A_MN ? TC_UMMA_K * 128 : TC_UMMA_K * 2;   // bytes to the next K=16 slice
      constexpr uint32_t b_kstep = B_MN ? TC_UMMA_K * 128 : TC_UMMA_K * 2;
      const uint64_t da0 = ptx::make_smem_desc_sw128(ptx::smem_u32(sring), s.a_lbo, s.a_sbo);
      const uint64_t db0 = ptx::make_smem_desc_sw128(ptx::smem_u32(sring) + Cfg::kABytes, s.b_lbo, s.b_sbo);
      int stage = 0;
      uint32_t phase = 0;
      int64_t it = 0;
      for (int64_t tile = work_id; tile < num_tiles; tile += work_stride, ++it, walk.next()) {
        const int64_t sp = MULTI ? tile_sp(tile) : (int64_t)walk.sp;
        const int64_t kb0 = sp * kb_per_split, kb1 = min(kb_total, kb0 + kb_per_split);
        const int acc = (int)(it & 1);
        const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
        twait(&tempty_bar[acc], acc_phase ^ 1, 2, tw1);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        for (int64_t kb = kb0; kb < kb1; ++kb) {
          twait(&full_bar[stage], phase, 3, tw0);
          ptx::tc_fence_after();
          const uint64_t soff = (uint64_t)((uint32_t)(stage * Cfg::kStageBytes) >> 4);
          const uint64_t boff = soff;
          if (ptx::elect_one()) {
            if constexpr (kLat) {
              // accumulator columns [mu 0-63 | ls 0-63]: group gg's 64 weight rows are ONE 64-column MMA per k-step (every MMA re-reads its
              // 4 KB A slice from shared memory whatever its N: two 32-column MMAs per step made this kernel MMA-issue-bound -- 66 cycles per
              // MMA, 34 k of its 54 k cycles, profiles/r02_step_trace_v22.txt); the epilogue warp reads mu and log_sigma of its 32 latent
              // dims with two tcgen05.ld 64 columns apart
              const int64_t kbg = kb_total >> 1;
              const uint32_t gg = kb >= kbg ? 1u : 0u;
              const bool first_kb = (kb == 0 || kb == kbg);
              const uint32_t idesc_lat = ptx::make_idesc_bf16(TM, TC_LAT_L, 0, 0);
#pragma unroll
              for (int kk = 0; kk < TC_BK / TC_UMMA_K; ++kk) {
                const uint64_t da = da0 + soff + (uint64_t)((kk * a_kstep) >> 4);
                const uint64_t db = db0 + boff + (uint64_t)((kk * b_kstep) >> 4);
                ptx::umma_f16(tmem_d + gg * (uint32_t)TC_LAT_L, da, db, idesc_lat, (first_kb && kk == 0) ? 0u : 1u);
              }
            } else {
#pragma unroll
            for (int kk = 0; kk < TC_BK / TC_UMMA_K; ++kk) {
              const uint64_t da = da0 + soff + (uint64_t)((kk * a_kstep) >> 4);
              const uint64_t db = db0 + boff + (uint64_t)((kk * b_kstep) >> 4);
              const uint32_t accum = (kb > kb0 || kk > 0) ? 1u : 0u;
              if constexpr (CG == 2) ptx::umma_f16_cg2(tmem_d, da, db, idesc, accum);
              else ptx::umma_f16(tmem_d, da, db, idesc, accum);
            }
            }
            // smem slot free (in both CTAs of a pair) once these MMAs retire
            if constexpr (CG == 2) ptx::umma_commit_cg2_mc(&empty_bar[stage], (uint16_t)3);
            else ptx::umma_commit(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == s.stages) { stage = 0; phase ^= 1; }
        }
        if (ptx::elect_one()) {                   // accumulator complete (also for an empty K range: the epilogue then sees zeros)
          if constexpr (CG == 2) ptx::umma_commit_cg2_mc(&tfull_bar[acc], (uint16_t)(3u << lead_rank));
          else ptx::umma_commit(&tfull_bar[acc]);
        }
        __syncwarp();
      }
    }
  } else {
    // ============================ epilogue ================================
    const int ew = warp - 2;                 // 0..EPI_WARPS-1
    const int quarter = warp & 3;            // TMEM lane quarter this warp may touch (warp id % 4)
    const int half = EG2 ? (ew >> 2) & 1 : ew >> 2;      // which column group of the BN columns
    const int egrp = ew >> 3;                // EG2: this warp's epilogue group (= the accumulator buffer it drains)
    constexpr int COLS_PER_WARP = Cfg::kColsPerWarp;
    constexpr int CH = COLS_PER_WARP / 32;   // 32-column blocks per tile for this warp
    uint8_t* const obuf0 = smem + Cfg::kEpiOff + ew * Cfg::kEpiWarpBytes;   // staged output block(s)
    const uint32_t obuf0_s = ptx::smem_u32(obuf0);
    uint8_t* abuf = obuf0 + Cfg::kOutBufs * Cfg::kOutBytes;                  // staged auxiliary block
    uint32_t aux_phase = 0;
    const bool do_store = epi.out != nullptr;
    float cs_acc[CH][2];                     // kColSum: this lane's two columns of every block of the current N tile
#pragma unroll
    for (int c = 0; c < CH; ++c) cs_acc[c][0] = cs_acc[c][1] = 0.f;
    int64_t cs_nt = -1;
    auto cs_flush = [&]() {
      if constexpr (Epi::kColSum) {
        if (cs_nt >= 0 && (WIDE || lane < 16)) {
#pragma unroll
          for (int c = 0; c < (WIDE ? CH / 2 : CH); ++c) {
            const int col = (int)(cs_nt * BN) + half * COLS_PER_WARP + c * Cfg::kBlockCols + 2 * lane;
            if (col + 1 < s.N) {
              if (epi.colsum_atomic) {          // fast mode: straight into the (zeroed) bias gradient
                atomicAdd(epi.colsum + col, cs_acc[c][0]);
                atomicAdd(epi.colsum + col + 1, cs_acc[c][1]);
              } else {                          // deterministic mode: one partial row per (CTA, row quarter)
                // the slot is private to this warp and zeroed before the launch; += because a CTA can come back to an N tile
                float2* p = reinterpret_cast<float2*>(epi.colsum + ((int64_t)blockIdx.x * 4 + quarter) * s.N + col);
                float2 o = *p;
                o.x += cs_acc[c][0]; o.y += cs_acc[c][1];
                *p = o;
              }
            }
          }
        }
#pragma unroll
        for (int c = 0; c < CH; ++c) cs_acc[c][0] = cs_acc[c][1] = 0.f;
      }
    };
    int64_t it = 0;
    for (int64_t tile = work_id; tile < num_tiles; tile += work_stride, ++it, walk.next()) {
      const int64_t m_t = MULTI ? tile_m(tile) : (int64_t)walk.m, n_t = MULTI ? tile_n(tile) : (int64_t)walk.n,
                      sp = MULTI ? tile_sp(tile) : (int64_t)walk.sp;
      const int64_t kb0 = sp * kb_per_split, kb1 = min(kb_total, kb0 + kb_per_split);
      const int acc = (int)(it & 1);
      if constexpr (EG2) {
        if (acc != egrp) continue;           // the other group's tile
      }
      const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
      const int32_t row_base = (int32_t)(m_t * TM) + (int32_t)cta_rank * TC_BM + quarter * 32;
      const int64_t row = (int64_t)row_base + lane;
      int64_t pM = s.M;                       // this item's output extent and map (MULTI: its problem's)
      int pN = s.N;
      const CUtensorMap* pout = &tma_out;
      if constexpr (MULTI) {
        const int p = item_problem(tile);
        pM = mp->M[p];
        pN = mp->N[p];
        pout = &mp->tout[p];
      }
      const bool valid = row < pM;
      const int col_base = (int)(n_t * BN) + half * COLS_PER_WARP;
      if constexpr (kLat) {
        // ---- fused encoder head: this warp owns rows [row_base, +32) and latent dims [32 half, 32 half + 32): accumulator columns
        //      [32 half, +32) hold their mu, columns [64 + 32 half, +32) their log_sigma
        static_assert(sizeof(decltype(*epi.z)) == 2, "fused head: bf16 z");
        uint8_t* const st_mu = obuf0;                                  // 32 x 32 fp32 (128-byte swizzled rows); first: Philox scratch [8][32] float4
        uint8_t* const st_ls = obuf0 + 4096;
        uint8_t* const st_z = obuf0 + 8192;                            // 32 x 32 bf16 (64-byte swizzled rows)
        uint8_t* const st_hs = obuf0 + 10240;
        float* const xch = reinterpret_cast<float*>(obuf0 + 12288);    // [2 parities][32 lanes][4] partial logits for the sibling warp
        const float* const xch_sib = reinterpret_cast<const float*>(smem + Cfg::kEpiOff + (ew ^ 4) * Cfg::kEpiWarpBytes + 12288);
        const int lat0 = half * 32;
        twait(&tfull_bar[acc], acc_phase, 4, tw0);
        ptx::tc_fence_after();
        uint32_t r_mu[32], r_ls[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + half * 32);
        ptx::tmem_ld_32x32_issue(taddr, r_mu);
        ptx::tmem_ld_32x32_issue(taddr + TC_LAT_L, r_ls);
        float mu_v[32], ls_v[32];
        load_vec<32>(epi.bias + lat0, mu_v);                           // biases, fetched while the TMEM reads are in flight
        load_vec<32>(epi.bias + epi.L + lat0, ls_v);
        ptx::tmem_ld_wait(r_mu);
        ptx::tmem_ld_wait(r_ls);
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          mu_v[i] += __uint_as_float(r_mu[i]);
          ls_v[i] += __uint_as_float(r_ls[i]);
        }
        // the accumulator buffer is free again: everything this warp needs is in registers
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tempty_bar[acc]);
        // noise: injected, or the counter-based generator (rolled loop: the scratch block keeps the code small, see langevin.cuh)
        if (lane == 0) ptx::bulk_wait_read0();                         // the previous tile's TMA stores have finished reading this warp's blocks
        __syncwarp();
        float e[32];
        if (epi.eps) {
          if (valid) {
            load_vec<32>(epi.eps + row * epi.L + lat0, e);
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) e[i] = 0.f;
          }
        } else {
          float4* const scratch = reinterpret_cast<float4*>(st_mu);
          const uint64_t q0 = (uint64_t)epi.first_quad + (((uint64_t)row * (uint64_t)epi.L + (uint64_t)lat0) >> 2);
#pragma unroll 2
          for (int q = 0; q < 8; ++q) scratch[q * 32 + lane] = philox_normal4(q0 + (uint64_t)q, epi.seed, epi.rng_offset());
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 t = scratch[q * 32 + lane];
            e[4 * q] = t.x; e[4 * q + 1] = t.y; e[4 * q + 2] = t.z; e[4 * q + 3] = t.w;
          }
          __syncwarp();                                                // every lane holds its normals before the block becomes the mu staging block
        }
        // mu / log_sigma blocks (fp32)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          *reinterpret_cast<float4*>(st_mu + swz_off<128>(lane, j)) = make_float4(mu_v[j * 4], mu_v[j * 4 + 1], mu_v[j * 4 + 2], mu_v[j * 4 + 3]);
          *reinterpret_cast<float4*>(st_ls + swz_off<128>(lane, j)) = make_float4(ls_v[j * 4], ls_v[j * 4 + 1], ls_v[j * 4 + 2], ls_v[j * 4 + 3]);
        }
        // reparameterisation (model.py:56-57), sigma eps / 2 for the backward pass, KL partial (lightning.py:115-117)
        float klv = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float zz[8], hh[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float m = mu_v[j * 8 + i], l = ls_v[j * 8 + i], ee = e[j * 8 + i];
            const float sigma = expf(0.5f * l);
            zz[i] = fmaf(sigma, ee, m);
            hh[i] = 0.5f * sigma * ee;
            klv += 1.f + l - m * m - sigma * sigma;
          }
          uint4 uz, uh;
          uz.x = pack_bf16x2(zz[0], zz[1]); uz.y = pack_bf16x2(zz[2], zz[3]); uz.z = pack_bf16x2(zz[4], zz[5]); uz.w = pack_bf16x2(zz[6], zz[7]);
          uh.x = pack_bf16x2(hh[0], hh[1]); uh.y = pack_bf16x2(hh[2], hh[3]); uh.z = pack_bf16x2(hh[4], hh[5]); uh.w = pack_bf16x2(hh[6], hh[7]);
          *reinterpret_cast<uint4*>(st_z + swz_off<64>(lane, j)) = uz;
          *reinterpret_cast<uint4*>(st_hs + swz_off<64>(lane, j)) = uh;
        }
        if (valid) lat_kl += klv;
        // linear-head classifier on mu (lightning.py:73-83): this warp's 32 dims give partial logits; the sibling warp (same rows, the
        // other 32 dims) supplies the rest through shared memory
        if (epi.nc > 0) {
          float lp[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            if (cc < epi.nc) {
              const float* wrow = epi.clf_w + (int64_t)cc * epi.L + lat0;
#pragma unroll
              for (int i = 0; i < 32; ++i) lp[cc] = fmaf(mu_v[i], __ldg(wrow + i), lp[cc]);
            }
          }
          *reinterpret_cast<float4*>(xch + acc * 128 + lane * 4) = make_float4(lp[0], lp[1], lp[2], lp[3]);
          asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory");        // the two warps of this lane quarter
          const float4 o = *reinterpret_cast<const float4*>(xch_sib + acc * 128 + lane * 4);
          float logit[4] = {lp[0] + o.x, lp[1] + o.y, lp[2] + o.z, lp[3] + o.w};
          if (half == 0 && valid) {
            const int64_t ty = epi.y[row];
            const int tgt = (ty < 0 || ty >= (int64_t)epi.nc) ? -1 : (int)ty;
            float mx = -INFINITY, lt = (tgt < 0) ? __int_as_float(0x7fc00000) : 0.f;      // label out of range: NaN loss (see ce_kernel)
            int arg = 0;
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              if (cc < epi.nc) {
                logit[cc] += __ldg(epi.clf_b + cc);
                if (logit[cc] > mx) { mx = logit[cc]; arg = cc; }      // first maximum, like torch.argmax
                if (cc == tgt) lt = logit[cc];
              }
            }
            float se = 0.f;
#pragma unroll
            for (int cc = 0; cc < 4; ++cc)
              if (cc < epi.nc) se += expf(logit[cc] - mx);
            const float lse = logf(se);
            lat_nll += -(lt - mx - lse);
            lat_acc += (arg == tgt) ? 1.f : 0.f;
            if (epi.g_rows) {
              float g[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
              for (int cc = 0; cc < 4; ++cc)
                if (cc < epi.nc) g[cc] = (expf(logit[cc] - mx - lse) - (cc == tgt ? 1.f : 0.f)) * epi.gscale;
              *reinterpret_cast<float4*>(epi.g_rows + row * 8) = make_float4(g[0], g[1], g[2], g[3]);
              *reinterpret_cast<float4*>(epi.g_rows + row * 8 + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          ptx::tma_store_3d(&tma_out, st_mu, lat0, row_base, 0);
          ptx::tma_store_3d(&tma_out, st_ls, lat0, row_base, 1);
          ptx::tma_store_3d(&tma_aux, st_z, lat0, row_base, 0);
          ptx::tma_store_3d(&tma_aux, st_hs, lat0, row_base, 1);
          ptx::bulk_commit();
        }
        continue;
      }
      if constexpr (Epi::kColSum) {
        if (n_t != cs_nt) { cs_flush(); cs_nt = n_t; }
      }
      if constexpr (kAux) {                  // fetch the first auxiliary block while the MMAs of this tile are still running
        if (col_base < pN && lane == 0) {
          ptx::mbar_arrive_expect_tx(&aux_bar[ew], Epi::kAuxBytes);
          ptx::tma_load_2d(abuf, &tma_aux, &aux_bar[ew], col_base, row_base);
        }
        // and pull this warp's auxiliary blocks of the CTA's NEXT tile into L2 (they stream from HBM otherwise)
        const int64_t nxt = tile + work_stride;
        if (nxt < num_tiles && lane < CH) {
          const int32_t nrow = (int32_t)(tile_m(nxt) * TM) + (int32_t)cta_rank * TC_BM + quarter * 32;
          const int ncol = (int)(tile_n(nxt) * BN) + half * COLS_PER_WARP + lane * 32;
          if (ncol < pN) ptx::tma_prefetch_2d(&tma_aux, ncol, nrow);
        }
      }
      uint32_t pre[CH];                      // per-block words the functor wants early (EpiActGrad: the ReLU bit masks)
#pragma unroll
      for (int c = 0; c < CH; ++c) pre[c] = (col_base + c * 32 < pN) ? epi.tc_pre(row, col_base + c * 32, valid) : 0u;
      twait(&tfull_bar[acc], acc_phase, 4, tw0);
      ptx::tc_fence_after();
      const bool zero_acc = kb0 >= kb1;
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const int col_in_tile = half * COLS_PER_WARP + c * 32;
        const int col = col_base + c * 32;
        if (col >= pN) continue;            // warp-uniform
        uint32_t acc_r[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + col_in_tile);
        ptx::tmem_ld_32x32_issue(taddr, acc_r);
        float bv[32];                        // the block's bias values: loaded while the TMEM read is in flight
        if constexpr (Epi::kBias) {
          if (epi.bias && col + 32 <= pN) {
            load_vec<32>(epi.bias + col, bv);
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) bv[i] = (epi.bias && col + i < pN) ? __ldg(epi.bias + col + i) : 0.f;
          }
        }
        ptx::tmem_ld_wait(acc_r);
        if (zero_acc) {                      // empty K range (warp-uniform; a per-element select cost 32 instructions per block)
#pragma unroll
          for (int i = 0; i < 32; ++i) acc_r[i] = 0u;
        }
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          v[i] = __uint_as_float(acc_r[i]);
          v[i + 1] = __uint_as_float(acc_r[i + 1]);
          if constexpr (Epi::kBias) ptx::add2(v[i], v[i + 1], bv[i], bv[i + 1]);
        }
        float aux[32];
        if constexpr (kAux) {
          twait(&aux_bar[ew], aux_phase, 5, tw1);
          aux_phase ^= 1;
          if constexpr (Epi::kAuxBytes == 2048) {          // bf16 tile, 64-byte rows
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 u = *reinterpret_cast<const uint4*>(abuf + swz_off<64>(lane, j));
              const uint32_t wv[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                aux[j * 8 + 2 * q] = __uint_as_float(wv[q] << 16);
                aux[j * 8 + 2 * q + 1] = __uint_as_float(wv[q] & 0xFFFF0000u);
              }
            }
          } else {                                         // fp32 tile, 128-byte rows
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 u = *reinterpret_cast<const float4*>(abuf + swz_off<128>(lane, j));
              aux[j * 4] = u.x; aux[j * 4 + 1] = u.y; aux[j * 4 + 2] = u.z; aux[j * 4 + 3] = u.w;
            }
          }
        }
        epi.tc_transform(row, col, pN, valid, v, aux, pre[c], red);
        if constexpr (kAux) {
          // The staged auxiliary block may be overwritten by the next TMA load only once every lane HOLDS its values: issuing the loads from
          // shared memory is not enough (the last 16-byte chunk of a row was occasionally still in the LSU queue when the next block landed --
          // 32 x 4 wrong targets in one tile of a cold run).  `red` depends on every auxiliary value a lane uses, so pinning it here keeps the
          // consuming FMAs -- which cannot issue before their operands have arrived -- ahead of the TMA instruction in program order.
          static_assert(Epi::kReduce, "the release of the auxiliary block is ordered through the functor's reduction value");
          asm volatile("" ::"f"(red) : "memory");
          __syncwarp();
          if (col + 32 < pN && c + 1 < CH && lane == 0) {
            ptx::mbar_arrive_expect_tx(&aux_bar[ew], Epi::kAuxBytes);
            ptx::tma_load_2d(abuf, &tma_aux, &aux_bar[ew], col + 32, row_base);
          }
        }
        if (do_store) {
          if constexpr (Epi::kColSum) {      // rows past M must not reach the column sums
            if (!valid) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = 0.f;
            }
          }
          // WIDE (bf16, BN >= 128): two consecutive 32-column chunks share one 32 x 128-byte block, one fence and one TMA store
          uint8_t* const obuf = obuf0 + (Cfg::kOutBufs == 2 ? ((WIDE ? (c >> 1) : c) & 1) * Cfg::kOutBytes : 0);
          const uint32_t obuf_s = obuf0_s + (Cfg::kOutBufs == 2 ? ((WIDE ? (c >> 1) : c) & 1) * Cfg::kOutBytes : 0);
          const int part = WIDE ? (c & 1) : 0;
          const bool opens = !WIDE || part == 0;
          const bool closes = !WIDE || part == 1 || col + 32 >= pN || c + 1 == CH;
          if (opens) {          // the TMA store that last used this staging block must have finished reading it
            if (lane == 0) {
              if constexpr (Cfg::kOutBufs == 2) ptx::bulk_wait_read1();      // two blocks alternate: only the store before the last one must be done
              else ptx::bulk_wait_read0();
            }
            __syncwarp();
          }
          if constexpr (sizeof(TOut) == 2) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 u;
              if constexpr (Epi::kReluPack) {          // the functor left the pre-activation: clamp while packing
                u.x = ptx::pack_bf16x2_relu(v[j * 8 + 0], v[j * 8 + 1]);
                u.y = ptx::pack_bf16x2_relu(v[j * 8 + 2], v[j * 8 + 3]);
                u.z = ptx::pack_bf16x2_relu(v[j * 8 + 4], v[j * 8 + 5]);
                u.w = ptx::pack_bf16x2_relu(v[j * 8 + 6], v[j * 8 + 7]);
              } else {
                u.x = pack_bf16x2(v[j * 8 + 0], v[j * 8 + 1]);
                u.y = pack_bf16x2(v[j * 8 + 2], v[j * 8 + 3]);
                u.z = pack_bf16x2(v[j * 8 + 4], v[j * 8 + 5]);
                u.w = pack_bf16x2(v[j * 8 + 6], v[j * 8 + 7]);
              }
              if constexpr (WIDE) ptx::sts128(obuf_s + swz_off<128>(lane, part * 4 + j), u.x, u.y, u.z, u.w);
              else ptx::sts128(obuf_s + swz_off<64>(lane, j), u.x, u.y, u.z, u.w);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              ptx::sts128(obuf_s + swz_off<128>(lane, j), __float_as_uint(v[j * 4]), __float_as_uint(v[j * 4 + 1]), __float_as_uint(v[j * 4 + 2]),
                          __float_as_uint(v[j * 4 + 3]));
          }
          if (closes) {
            ptx::fence_proxy_async_smem();     // generic-proxy writes -> visible to the TMA (async proxy)
            __syncwarp();
            if constexpr (Epi::kColSum) {
              float s0 = 0.f, s1 = 0.f;
              if constexpr (WIDE) {
                // lane l owns columns 2l, 2l+1 of the 64-column block (a half-filled block adds stale-but-unused columns: see flush guard)
                const bool have = part == 1 || lane < 16;
#pragma unroll
                for (int r = 0; r < 32; ++r) {
                  const uint32_t u = ptx::lds32(obuf_s + swz_off<128>(r, lane >> 2) + (lane & 3) * 4);
                  ptx::add2(s0, s1, __uint_as_float(u << 16), __uint_as_float(u & 0xFFFF0000u));
                }
                if (have) { cs_acc[c >> 1][0] += s0; cs_acc[c >> 1][1] += s1; }
              } else {
                // lanes 0-15 walk the even rows, 16-31 the odd rows; lane (l & 15) owns columns 2w, 2w+1 of the block
                const int hw = lane >> 4, w = lane & 15;
#pragma unroll
                for (int rr = 0; rr < 16; ++rr) {
                  const int r = 2 * rr + hw;
                  const uint32_t u = ptx::lds32(obuf_s + swz_off<64>(r, w >> 2) + (w & 3) * 4);
                  ptx::add2(s0, s1, __uint_as_float(u << 16), __uint_as_float(u & 0xFFFF0000u));
                }
                s0 += __shfl_xor_sync(0xffffffffu, s0, 16);
                s1 += __shfl_xor_sync(0xffffffffu, s1, 16);
                cs_acc[c][0] += s0;
                cs_acc[c][1] += s1;
              }
            }
            if (lane == 0) {
              const int bcol = WIDE ? col - part * 32 : col;
              if constexpr (Epi::kSplit) {
                if (epi.reduce_add) ptx::tma_reduce_add_2d(pout, obuf, bcol, row_base);
                else ptx::tma_store_3d(pout, obuf, bcol, row_base, (int32_t)sp);
              } else if (s.out3d) {
                const int32_t g = tile_g(n_t);
                ptx::tma_store_3d(pout, obuf, bcol - g * s.grp_n, row_base, g);
              } else {
                ptx::tma_store_2d(pout, obuf, bcol, row_base);
              }
              ptx::bulk_commit();
            }
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (CG == 2) ptx::mbar_arrive_cluster(ptx::mapa_u32(ptx::smem_u32(&tempty_bar[acc]), lead_rank));
        else ptx::mbar_arrive(&tempty_bar[acc]);
      }
    }
    cs_flush();
    if (lane == 0) ptx::bulk_wait_all();     // shared memory must outlive the last store's read
  }

  // ============================ teardown ==================================
  if (tracing && lane == 0) {
    unsigned long long* t = s.trace + (size_t)blockIdx.x * 16;
    const long long total = clock64() - t_begin;
    if (warp == 0) { t[0] = (unsigned long long)total; t[1] = (unsigned long long)tw0; t[2] = (unsigned long long)tw1; }            // producer: total, wait empty, wait bempty
    if (warp == 1) { t[3] = (unsigned long long)total; t[4] = (unsigned long long)tw0; t[5] = (unsigned long long)tw1; t[6] = (unsigned long long)tw2; }   // MMA: total, wait full, wait tempty, wait bfull
    if (warp == 2) { t[7] = (unsigned long long)total; t[8] = (unsigned long long)tw0; t[9] = (unsigned long long)tw1; }            // epilogue warp 0: total, wait tfull, wait aux
    if (warp == 5) { t[10] = (unsigned long long)total; t[11] = (unsigned long long)tw0; }
    if (warp == 0) t[13] = g_begin;                                                   // role loops start (ns)
    if (warp == 2) t[14] = ptx::globaltimer_ns();                                     // epilogue warp 0 done (ns)
  }
  ptx::tc_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync();     // neither CTA may retire while the pair's MMAs / multicast commits can still touch it
  else __syncthreads();
  if constexpr (kLat) {
    // one (KL sum, NLL sum, correct count) record per CTA, summed in a fixed order (warps, then the three values one after the other)
    float* const outs[3] = {epi.kl_part, epi.nll_part, epi.acc_part};
    const float vals[3] = {lat_kl, lat_nll, lat_acc};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float ws = warp_sum(vals[k]);
      if (lane == 0) red_smem[warp] = ws;
      __syncthreads();
      if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < Cfg::kThreads / 32; ++w) t += red_smem[w];
        if (outs[k]) outs[k][blockIdx.x] = t;
      }
      __syncthreads();
    }
  }
  if constexpr (Epi::kReduce) {
    const float ws = warp_sum(red);
    if (lane == 0) red_smem[warp] = ws;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int w = 0; w < Cfg::kThreads / 32; ++w) t += red_smem[w];
      epi.red_out[blockIdx.x] = t;
    }
  }
  if (warp == 1) {
    __syncwarp();
    ptx::tc_fence_after();
    if constexpr (CG == 2) ptx::tmem_dealloc_cg2(tmem_base, Cfg::kTmemCols);
    else ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
    if (tracing && lane == 0) s.trace[(size_t)blockIdx.x * 16 + 15] = ptx::globaltimer_ns();     // kernel exit
  }
}

template <int BN, bool A_MN, bool B_MN, class Epi, int CG, bool EG2 = false>
__global__ void __launch_bounds__(32 * (2 + tc_epi_warps(BN)), 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const __grid_constant__ CUtensorMap tma_out,
               const __grid_constant__ CUtensorMap tma_aux, TcShape s, Epi epi) {
  gemm_tc_body<BN, A_MN, B_MN, Epi, CG, EG2, false>(tma_a, tma_b, tma_out, tma_aux, nullptr, s, epi);
}

// the merged wgrad launch (MULTI): the problem list, tensor maps included, is one __grid_constant__ kernel parameter
template <int BN, class Epi, int CG>
__global__ void __launch_bounds__(32 * (2 + tc_epi_warps(BN)), 1)
gemm_tc_multi_kernel(const __grid_constant__ TcMulti mp, TcShape s, Epi epi) {
  gemm_tc_body<BN, true, true, Epi, CG, false, true>(mp.ta[0], mp.tb[0], mp.tout[0], mp.ta[0], &mp, s, epi);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct TcOperand {
  const void* ptr;   // bf16
  int64_t rows;      // M (A) or N (B)
  int64_t ld;        // K-major: elements between rows;  MN-major: elements between consecutive k
  bool mn_major;
};

// Encodes (and caches by value) the 2D tensor map of one operand.  Returns 0, or < 0 with the error text set.
int tc_tensor_map(const TcOperand& op, int64_t K, int box_rows, CUtensorMap* out);
// Tensor map of an epilogue block: [32 rows][32 cols] of a row-major [rows][cols] (x splits) matrix of 2- or 4-byte elements.
int tc_block_map(const void* ptr, int elem_bytes, int64_t rows, int64_t cols, int64_t ld, int64_t splits, int64_t split_stride, CUtensorMap* out,
                 int box_cols = 32);
int tc_grid_size();       // number of SMs of the current device (persistent grid)
int tc_device_check();    // 0 when the current device is sm_100
void count_launch();

// UMMA smem-descriptor strides of one staged operand tile (see the canonical layouts in ptx.cuh)
static inline void tc_desc_strides(bool mn_major, uint32_t* lbo, uint32_t* sbo) {
  if (!mn_major) { *lbo = 16; *sbo = 8 * 128; }                 // K-major SW128: 8-row groups 1024 B apart; LBO unused
  else { *lbo = TC_BK * 128; *sbo = 8 * 128; }                  // MN-major SW128: next 64-wide MN block / next 8 k
}

static inline int tc_pick_bn(int N) {
  if (N % 256 == 0) return 256;
  if (N % 128 == 0) return 128;
  return 64;
}
// Tile width for an [M, N] output that is not split and not grouped.  N = 256 is ONE tile column: on CTA pairs the launch takes
// ceil(M / 256 / pairs) rounds -- 3.46 -> 4 at M = 65,536 on 74 pairs (86 % full).  The same output as 128 x 128 one-CTA tiles takes
// 6.92 -> 7 rounds of quarter-size tiles (99 % full), which wins when the tile time is the epilogue's (option "tc_bn_rounds").
int tc_bn_rounds();
int tc_two_cta();
static inline int tc_pick_bn_mn(int64_t M, int N, int force_bn) {
  if (force_bn) return force_bn;
  const int bn = tc_pick_bn(N);
  if (bn == 256 && N == 256 && tc_bn_rounds() && tc_two_cta() && M > TC_BM) {
    const int64_t g = tc_grid_size(), pairs = g / 2;
    const int64_t t256 = ceil_div64(M, 2 * TC_BM), t128 = ceil_div64(M, TC_BM) * 2;
    const double e256 = (double)t256 / (double)(ceil_div64(t256, pairs) * pairs), e128 = (double)t128 / (double)(ceil_div64(t128, g) * g);
    if (e256 < 0.9 && e128 > e256 + 0.08) return 128;
  }
  return bn;
}
// CTAs a launch uses (= rows / 4 of the kColSum partial buffer, = slots of a kReduce epilogue)
int tc_two_cta();         // option "tc_two_cta": use CTA pairs (cta_group::2) where the shape allows
int tc_max_stages();      // option "tc_max_stages": cap of the operand ring depth (0 = none)
unsigned long long* tc_trace_ptr();   // option "tc_trace_ptr": device buffer of gridDim.x * 16 counters, or nullptr
int tc_epi_groups_max_k();
int tc_wgrad_splits();           // option "wgrad_splits" (experiments): batch ranges per tile of the merged wgrad, 0 = chosen by gemm_tc_launch_multi_wgrad
int tc_epi_groups();      // option "tc_epi_groups": K <= 128 forward / dgrad launches with BN = 256 run two epilogue groups on alternate tiles (EG2)
// does this shape run as CTA pairs?  (BN = 256 tiles and more than one 128-row block of M)
static inline bool tc_use_pair(int64_t M, int N, int force_bn = 0) {
  const int bn = tc_pick_bn_mn(M, N, force_bn);
  return tc_two_cta() && bn == 256 && M > TC_BM;
}
// the CTAs a launch uses
static inline int64_t tc_ctas(int64_t M, int N, int splits, int force_bn = 0) {
  const int bn = tc_pick_bn_mn(M, N, force_bn);
  const int cg = tc_use_pair(M, N, force_bn) ? 2 : 1;
  int64_t tiles = ceil_div64(M, TC_BM * cg) * ceil_div64(N, bn) * (splits < 1 ? 1 : splits);
  const int64_t g = tc_grid_size() / cg;
  return (tiles < g ? tiles : g) * cg;
}

template <class Epi, class = void> struct epi_aux_ptr {
  static const void* get(const Epi&) { return nullptr; }
  static int64_t ld(const Epi&) { return 0; }
};
template <class Epi> struct epi_aux_ptr<Epi, std::enable_if_t<(Epi::kAuxBytes > 0)>> {
  static const void* get(const Epi& e) { return e.aux_ptr(); }
  static int64_t ld(const Epi& e) { return e.aux_ld(); }
};
template <class Epi, class = void> struct epi_split_stride {
  static int64_t get(const Epi&) { return 0; }
  static bool reduce(const Epi&) { return false; }
};
template <class Epi> struct epi_split_stride<Epi, std::enable_if_t<Epi::kSplit>> {
  static int64_t get(const Epi& e) { return e.split_stride; }
  static bool reduce(const Epi& e) { return e.reduce_add != 0; }
};
template <class Epi, class = void> struct epi_cs_atomic { static bool get(const Epi&) { return false; } };
template <class Epi> struct epi_cs_atomic<Epi, std::enable_if_t<Epi::kColSum>> { static bool get(const Epi& e) { return e.colsum_atomic != 0; } };

template <int BN, bool A_MN, bool B_MN, class Epi, int CG = 1, bool EG2 = false>
int gemm_tc_launch_bn(const TcOperand& A, const TcOperand& B, int64_t M, int N, int64_t K, int splits, const Epi& epi, cudaStream_t st,
                      const TcGroup& grp = TcGroup()) {
  using Cfg = TcCfg<BN, Epi, CG, EG2>;
  using TOut = typename Epi::TOut;
  CUtensorMap ta, tb, tout, taux;
  // grouped: K is one group's contraction length; A spans all groups' k ranges, an MN-major B all groups' k rows
  PSVAE_TRY(tc_tensor_map(A, K * grp.groups, A_MN ? TC_BK : TC_BM, &ta));
  PSVAE_TRY(tc_tensor_map(B, B_MN ? K * grp.groups : K, B_MN ? TC_BK : BN / CG, &tb));
  TcShape s;
  s.M = M; s.N = N; s.K = K; s.splits = splits < 1 ? 1 : splits;
  tc_desc_strides(A_MN, &s.a_lbo, &s.a_sbo);
  tc_desc_strides(B_MN, &s.b_lbo, &s.b_sbo);
  s.stages = Cfg::kStages;
  s.rev_splits = 0;
  if (tc_max_stages() >= 2 && tc_max_stages() < s.stages) s.stages = tc_max_stages();
  s.trace = tc_trace_ptr();
  s.groups = grp.groups; s.grp_n = grp.grp_n; s.grp_k = grp.grp_k;
  s.out3d = (grp.groups > 1 && grp.out_group_stride != 0) ? 1 : 0;
  if (epi.out) {
    const bool split_slots = Epi::kSplit && !epi_split_stride<Epi>::reduce(epi);
    if (s.out3d) PSVAE_TRY(tc_block_map(epi.out, (int)sizeof(TOut), M, grp.grp_n, epi.ldo, grp.groups, grp.out_group_stride, &tout, Cfg::kBlockCols));
    else PSVAE_TRY(tc_block_map(epi.out, (int)sizeof(TOut), M, N, epi.ldo, split_slots ? s.splits : 0, epi_split_stride<Epi>::get(epi), &tout,
                                Cfg::kBlockCols));
  } else {
    tout = ta;   // never dereferenced: the kernel skips the store
  }
  if constexpr (Epi::kAuxBytes > 0) {
    PSVAE_TRY(tc_block_map(epi_aux_ptr<Epi>::get(epi), Epi::kAuxBytes == 2048 ? 2 : 4, M, N, epi_aux_ptr<Epi>::ld(epi), 0, 0, &taux));
  } else {
    taux = ta;
  }
  auto kern = gemm_tc_kernel<BN, A_MN, B_MN, Epi, CG, EG2>;
  static unsigned long long attr_mask = 0;   // per instantiation, one bit per device
  int dev = 0;
  PSVAE_CUDA(cudaGetDevice(&dev));
  if (!(attr_mask >> (dev & 63) & 1ull)) {
    PSVAE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_mask |= 1ull << (dev & 63);
  }
  const int64_t n_tiles = ceil_div64(N, BN);
  const int64_t tiles = ceil_div64(M, TC_BM * CG) * n_tiles * s.splits;
  int grid = tc_grid_size() / CG;            // CG = 2: one CTA pair per tile
  const int64_t cs_rows = (tiles < grid ? tiles : (int64_t)grid) * CG * 4;     // = 4 * tc_ctas(): what the caller's ordered reduce reads
  if (tiles < grid) grid = (int)tiles;
  grid *= CG;
  if (grid < 1) return 0;
  if constexpr (Epi::kColSum) {
    // every (CTA, row-quarter) writes only the columns of the N tiles it saw: the rest of the partial buffer must read as zero
    if (!epi_cs_atomic<Epi>::get(epi)) PSVAE_CUDA(cudaMemsetAsync(epi.colsum, 0, (size_t)cs_rows * (size_t)N * sizeof(float), st));
  }
  {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(Cfg::kThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    if constexpr (CG == 2) {
      at[na].id = cudaLaunchAttributeClusterDimension;
      at[na].val.clusterDim.x = 2; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
      ++na;
    }
    if (pdl_enabled()) {
      at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[na].val.programmaticStreamSerializationAllowed = 1;
      ++na;
    }
    cfg.attrs = at;
    cfg.numAttrs = na;
    PSVAE_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tout, taux, s, epi));
  }
  count_launch();
  PSVAE_LAUNCH_CHECK("gemm_tc_kernel");
  return 0;
}

// Fused encoder head (EpiLatent): he [M][2H] bf16 (mu half | sigma half), Wstack [2L][H] bf16 (W_mu rows, then W_sigma rows).  One CTA per
// 128-row tile; outputs through 3D maps (slice 0 / 1 = mu / log_sigma, z / sigma eps / 2).  Returns the CTAs launched in *ctas.
template <typename TZ, bool DEV_OFF>
int gemm_tc_launch_latent(const void* he, int64_t ldhe, const void* Wstack, int H, int64_t M, const EpiLatent<TZ, DEV_OFF>& epi, float* mu, float* ls, TZ* z,
                          TZ* hs, cudaStream_t st, int* ctas) {
  using Epi = EpiLatent<TZ, DEV_OFF>;
  constexpr int BN = 128;
  using Cfg = TcCfg<BN, Epi, 1>;
  const int Lz = TC_LAT_L;
  if (epi.L != Lz || H % TC_BK != 0 || epi.nc > 4 || ls <= mu || hs <= z) { set_error("fused head: needs latent_dim 64, hidden_dim %% 64 == 0, <= 4 classes"); return -2; }
  CUtensorMap ta, tb, tout, taux;
  TcOperand a{he, M, ldhe, false};
  TcOperand b{Wstack, (int64_t)2 * Lz, (int64_t)H, false};
  PSVAE_TRY(tc_tensor_map(a, (int64_t)2 * H, TC_BM, &ta));
  PSVAE_TRY(tc_tensor_map(b, (int64_t)H, Lz, &tb));
  PSVAE_TRY(tc_block_map(mu, 4, M, Lz, Lz, 2, (int64_t)(ls - mu), &tout, 32));
  PSVAE_TRY(tc_block_map(z, (int)sizeof(TZ), M, Lz, Lz, 2, (int64_t)(hs - z), &taux, 32));
  TcShape s;
  memset(&s, 0, sizeof(s));
  s.M = M; s.N = BN; s.K = (int64_t)2 * H; s.splits = 1;
  tc_desc_strides(false, &s.a_lbo, &s.a_sbo);
  tc_desc_strides(false, &s.b_lbo, &s.b_sbo);
  s.stages = Cfg::kStages;
  if (tc_max_stages() >= 2 && tc_max_stages() < s.stages) s.stages = tc_max_stages();
  s.trace = tc_trace_ptr();
  s.groups = 1;
  auto kern = gemm_tc_kernel<BN, false, false, Epi, 1, false>;
  static unsigned long long attr_mask = 0;
  int dev = 0;
  PSVAE_CUDA(cudaGetDevice(&dev));
  if (!(attr_mask >> (dev & 63) & 1ull)) {
    PSVAE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_mask |= 1ull << (dev & 63);
  }
  const int64_t tiles = ceil_div64(M, TC_BM);
  int grid = tc_grid_size();
  if (tiles < grid) grid = (int)tiles;
  if (grid < 1) return 0;
  if (ctas) *ctas = grid;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(Cfg::kThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  int na = 0;
  if (pdl_enabled()) {
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = at;
  cfg.numAttrs = na;
  PSVAE_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tout, taux, s, epi));
  count_launch();
  PSVAE_LAUNCH_CHECK("gemm_tc_kernel<EpiLatent>");
  return 0;
}

// One wgrad problem of the merged launch: out[M][N] (fp32, accumulated by TMA reduce-add) += dY[rows][M]^T * act[rows][N]
struct TcWgradProblem {
  const void* dY; int64_t ldy;
  const void* act; int64_t lda;
  float* out; int64_t ldo;
  int M, N;
};

// All of a step's wgrads in ONE persistent launch (see TcMulti).  256 x 256 tiles on CTA pairs for every problem: a problem narrower than the
// tile (the 64-wide latent layers) reads only its valid columns (TMA zero-fills the rest without DRAM traffic) -- these launches are bound by
// streaming the batch, not by the MMAs.
static inline int gemm_tc_launch_multi_wgrad(const TcWgradProblem* probs, int count, int64_t rows, cudaStream_t st, int rev_splits = 0) {
  using Epi = EpiStore;
  constexpr int BN = 256, CG = 2;
  using Cfg = TcCfg<BN, Epi, CG>;
  if (count <= 0) return 0;
  if (count > TC_MAX_PROBLEMS) { set_error("merged wgrad: %d problems, at most %d", count, TC_MAX_PROBLEMS); return -2; }
  static thread_local TcMulti mp;      // 8 KB: not on the stack of every caller
  memset(&mp, 0, sizeof(mp));
  int64_t tiles = 0;
  for (int p = 0; p < count; ++p) {
    const TcWgradProblem& q = probs[p];
    if (q.M % 8 != 0 || q.N % 8 != 0) { set_error("merged wgrad: M=%d, N=%d must be multiples of 8", q.M, q.N); return -2; }
    TcOperand a{q.dY, (int64_t)q.M, q.ldy, true};
    TcOperand b{q.act, (int64_t)q.N, q.lda, true};
    PSVAE_TRY(tc_tensor_map(a, rows, TC_BK, &mp.ta[p]));
    PSVAE_TRY(tc_tensor_map(b, rows, TC_BK, &mp.tb[p]));
    PSVAE_TRY(tc_block_map(q.out, 4, q.M, q.N, q.ldo, 0, 0, &mp.tout[p], Cfg::kBlockCols));
    mp.M[p] = q.M; mp.N[p] = q.N;
    mp.m_tiles[p] = (int32_t)ceil_div64(q.M, TC_BM * CG);
    mp.n_tiles[p] = (int32_t)ceil_div64(q.N, BN);
    tiles += (int64_t)mp.m_tiles[p] * mp.n_tiles[p];
  }
  // Split factor.  Items (tile x batch range) are dealt round-robin to the CTA pairs, so the launch takes ceil(items / pairs) rounds: S is chosen so
  // that tiles * S fills a whole number of rounds (r * pairs) from below -- e.g. 24 tiles on 74 pairs: S = 6 gives 144 items = 1.95 rounds
  // (97 % full), S = 7 gives 168 = 2.27 -> 3 rounds (76 %).  Few, long ranges also mean few reduce-adds per tile.  Measured on the headline
  // shape (ms/step): S = 6 0.643-0.655, S = 3 / 9 / 12 0.647-0.651, S = 7 0.669, S = 10 0.663, S = 40 (the old "12 items per pair") 0.673
  // (profiles/r02_ab_runs.txt).  At least two rounds, so that thin and full-width tiles mix on every pair; at least 8 k-blocks per range.
  const int pairs = tc_grid_size() / CG;
  const int64_t kb = ceil_div64(rows, TC_BK);
  int64_t S = 1;
  {
    const int64_t r0 = std::max<int64_t>(2, ceil_div64(tiles, pairs));
    double best = -1.0;
    for (int64_t r = r0; r < r0 + 4; ++r) {
      int64_t cand = (r * pairs) / tiles;
      if (cand < 1) cand = 1;
      if (cand > kb / 8) cand = std::max<int64_t>(1, kb / 8);
      const int64_t items = tiles * cand;
      const double eff = (double)items / (double)(ceil_div64(items, pairs) * pairs);
      if (eff > best + 1e-9) { best = eff; S = cand; }
    }
  }
  if (tc_wgrad_splits() > 0) S = tc_wgrad_splits();
  if (S > kb) S = kb;
  const int64_t per = ceil_div64(kb, S);
  S = ceil_div64(kb, per);
  int32_t begin = 0;
  for (int p = 0; p < count; ++p) {
    mp.tile_begin[p] = begin;
    begin += (int32_t)(mp.m_tiles[p] * mp.n_tiles[p] * S);
  }
  mp.tile_begin[count] = begin;
  mp.count = count;
  TcShape s;
  memset(&s, 0, sizeof(s));
  s.M = probs[0].M; s.N = probs[0].N; s.K = rows; s.splits = (int32_t)S;
  s.rev_splits = rev_splits;
  tc_desc_strides(true, &s.a_lbo, &s.a_sbo);
  tc_desc_strides(true, &s.b_lbo, &s.b_sbo);
  s.stages = Cfg::kStages;
  if (tc_max_stages() >= 2 && tc_max_stages() < s.stages) s.stages = tc_max_stages();
  s.trace = tc_trace_ptr();
  s.groups = 1;
  EpiStore epi{probs[0].out, probs[0].ldo, 0, 1.f, 0.f, nullptr, 1};
  auto kern = gemm_tc_multi_kernel<BN, Epi, CG>;
  static unsigned long long attr_mask = 0;
  int dev = 0;
  PSVAE_CUDA(cudaGetDevice(&dev));
  if (!(attr_mask >> (dev & 63) & 1ull)) {
    PSVAE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_mask |= 1ull << (dev & 63);
  }
  int grid = pairs;
  if (begin < grid) grid = begin;
  grid *= CG;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(Cfg::kThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  int na = 0;
  at[na].id = cudaLaunchAttributeClusterDimension;
  at[na].val.clusterDim.x = 2; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
  ++na;
  if (pdl_enabled()) {
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = at;
  cfg.numAttrs = na;
  PSVAE_CUDA(cudaLaunchKernelEx(&cfg, kern, mp, s, epi));
  count_launch();
  PSVAE_LAUNCH_CHECK("gemm_tc_multi_kernel");
  return 0;
}

// thin layers (K <= 128) on BN = 256 tiles take the two-epilogue-group kernel (EG2), everything else the plain one
template <int BN, bool A_MN, bool B_MN, class Epi, int CG>
int gemm_tc_launch_pick(const TcOperand& A, const TcOperand& B, int64_t M, int N, int64_t K, int splits, const Epi& epi, cudaStream_t st,
                        const TcGroup& grp = TcGroup()) {
  if constexpr (BN == 256 && !A_MN && !Epi::kSplit && Epi::kAuxBytes == 0) {
    // two epilogue groups on alternate tiles keep the TMEM read port busy through the store phase
    // (not with the ordered column-sum partials of deterministic mode: both groups' warps of a lane quarter would share one partial slot)
    bool ordered_colsum = false;
    if constexpr (Epi::kColSum) ordered_colsum = !epi_cs_atomic<Epi>::get(epi);
    if (tc_epi_groups() && K <= tc_epi_groups_max_k() && !ordered_colsum)
      return gemm_tc_launch_bn<BN, A_MN, B_MN, Epi, CG, true>(A, B, M, N, K, splits, epi, st, grp);
  }
  return gemm_tc_launch_bn<BN, A_MN, B_MN, Epi, CG, false>(A, B, M, N, K, splits, epi, st, grp);
}

// can the tcgen05 epilogue produce the column sums of an [M, N] bf16 output?  (pairs of columns: N even; N % 8 is required anyway)
static inline bool tc_colsum_ok(int N) { return N % 2 == 0; }

// N = all groups' columns, K = one group's contraction length (grp.groups == 1: the plain GEMM)
template <bool A_MN, bool B_MN, class Epi>
int gemm_tc_launch(const TcOperand& A, const TcOperand& B, int64_t M, int N, int64_t K, int splits, const Epi& epi, cudaStream_t st, int force_bn = 0,
                   const TcGroup& grp = TcGroup()) {
  if (N % 8 != 0) { set_error("gemm_tc: N=%d must be a multiple of 8", N); return -2; }
  const int bn = (grp.groups > 1 || splits > 1 || A_MN) ? (force_bn ? force_bn : tc_pick_bn(grp.groups > 1 ? grp.grp_n : N))      // a tile never straddles two groups
                                                        : tc_pick_bn_mn(M, N, force_bn);
  if (grp.groups > 1 && (A_MN || splits > 1 || grp.grp_n % bn != 0 || grp.grp_k % TC_BK != 0 || N != grp.groups * grp.grp_n)) {
    set_error("gemm_tc: grouped launch needs K-major A, no split-K, grp_n %% %d == 0 and grp_k %% %d == 0", bn, TC_BK);
    return -2;
  }
  switch (bn) {
    case 256:
      if (tc_use_pair(M, N, bn)) return gemm_tc_launch_pick<256, A_MN, B_MN, Epi, 2>(A, B, M, N, K, splits, epi, st, grp);
      return gemm_tc_launch_pick<256, A_MN, B_MN, Epi, 1>(A, B, M, N, K, splits, epi, st, grp);
    case 128: return gemm_tc_launch_pick<128, A_MN, B_MN, Epi, 1>(A, B, M, N, K, splits, epi, st, grp);
    case 64: return gemm_tc_launch_pick<64, A_MN, B_MN, Epi, 1>(A, B, M, N, K, splits, epi, st, grp);
  }
  set_error("gemm_tc: unsupported BN=%d", bn);
  return -2;
}

}  // namespace psvae
