// Classifier-guided Langevin dynamics in latent space: the loop of ps_vae/inference.py:77-103,
//   z <- z + 0.5 s^2 * grad_z[ log p(y|z) - 0.5 |z|^2 ] + s * noise_weight * N(0, I),
// with the gradient in closed form through the LatentClassifier chain (latent_classifier.py:58-70;
// SURVEY 3.4) instead of autograd, all `num_steps` steps inside ONE launch: a CTA keeps a tile of 32
// samples (z, activations, classifier weights) in shared memory for the whole loop, the noise comes from
// the counter-based generator (philox.cuh), and nothing goes back to the host between steps (the
// reference does a D2H copy of z and two .item() syncs per step, SURVEY F12).
//
// The analysis variant of the same loop (analysis/sample_gender_transformation.py:61-99) is covered by three more arguments:
// `prior_weight` scales the log p(z) term (the script's PRIOR_WEIGHT; inference.py has 1), `threshold` > 0 stops a sample after the update
// of the first step whose p(y|z) exceeded it (the script's per-sample `break`), and `stop_step` / `last_prob` report, per sample, the step
// at which that happened (num_steps if never) and the classifier probability of its last evaluated step.  A stopped sample keeps its z.
//
// Both kernels come in two instances: ROW_TARGETS = false takes one target for the whole batch (LangevinClf::targets), ROW_TARGETS = true
// gives every row its own (LangevinRows): read from a device array, or drawn in the kernel from a target mix.  A row of the per-row instance
// runs the same floating-point operations in the same order as the shared-target instance does with that row's target, so the two agree
// bit for bit.
#pragma once
#include "common.cuh"
#include "epilogue.cuh"
#include "philox.cuh"

namespace psvae {

constexpr int LG_TILE = 32;      // samples per CTA
constexpr int LG_THREADS = 256;  // 8 warps; lane = sample, warp = output-feature lane
constexpr int LG_MAXC = 16;      // classes per head (padded row length in smem)
constexpr int CLF_LG_MAXC = 8;   // fast path: classes summed over the targeted heads
constexpr int LG_MAX_MIX = 64;   // entries of a target mix (PSVAE_MAX_TARGET_MIX)

struct LangevinClf {
  int L, n_trunk, hidden, act, n_heads;
  int head_classes[4];
  int targets[4];                 // -1: head not named by the target dict -> skipped.  Per-row instances: >= 0 marks a head some row can name
  int64_t g_trunk_w[4], g_trunk_b[4], g_head_w[4], g_head_b[4];   // offsets into the flat parameter buffer
  int s_trunk_w[4], s_trunk_b[4], s_head_w[4], s_head_b[4];       // offsets (floats) into the smem weight area
  int w_floats;                   // size of the smem weight area
};

__device__ __forceinline__ float lg_act(int act, float u) {
  switch (act) {
    case ACT_RELU: return fmaxf(u, 0.f);
    case ACT_TANH: return tanhf(u);
    case ACT_SIGMOID: return 1.f / (1.f + expf(-u));
    case ACT_LEAKY: return u > 0.f ? u : 0.01f * u;
  }
  return u;
}
__device__ __forceinline__ float lg_act_grad(int act, float a) {
  switch (act) {
    case ACT_RELU: return a > 0.f ? 1.f : 0.f;
    case ACT_TANH: return 1.f - a * a;
    case ACT_SIGMOID: return a * (1.f - a);
    case ACT_LEAKY: return a > 0.f ? 1.f : 0.01f;
  }
  return 1.f;
}

// Per-row targets.  A row's targets are packed one byte per head: byte h = class + 1, 0 = head h left out for this row.
struct LangevinRows {
  const int32_t* targets;         // device int32 [n_heads][rows] (class, or -1: head left out), or NULL: draw from the mix
  int32_t* targets_out;           // mix: the drawn targets, same layout
  uint64_t mix_offset;            // Philox offset of the draw: offset0 + num_steps + 1 (no z0 or noise draw uses it)
  int n_mix;
  uint32_t mix[LG_MAX_MIX];       // packed targets of entry k
  uint32_t thr[LG_MAX_MIX - 1];   // a row takes the first entry k < n_mix - 1 with u < thr[k], else the last
};

// The packed targets of row r (global row row0 + r).  A device target outside [-1, classes) or a row that names no head sets `bad` and returns
// class 0 of every head the instance staged, so that the row computes NaN from its NaN z without an out-of-range class index.
__device__ __forceinline__ uint32_t lg_row_targets(const LangevinClf& c, const LangevinRows& rt, int64_t rows, int64_t r, int64_t row0, uint64_t seed,
                                                   bool store, bool& bad) {
  uint32_t p = 0;
  bad = false;
  if (rt.targets) {
    for (int h = 0; h < c.n_heads; ++h) {
      const int t = rt.targets[(int64_t)h * rows + r];
      bad |= t < -1 || t >= c.head_classes[h];
      p |= (uint32_t)((t + 1) & 0xFF) << (8 * h);
    }
    bad |= p == 0;
  } else {
    // word row0 + r of the uint32 stream at offset mix_offset: the layout of psvae_philox_uint32 (oracle/philox_ref.philox_uint32)
    const uint64_t g = (uint64_t)(row0 + r);
    const uint4 w = philox4x32_10((uint32_t)(g >> 2), (uint32_t)(g >> 34), (uint32_t)rt.mix_offset, (uint32_t)(rt.mix_offset >> 32), (uint32_t)seed,
                                  (uint32_t)(seed >> 32));
    const uint32_t u = (g & 3) == 0 ? w.x : (g & 3) == 1 ? w.y : (g & 3) == 2 ? w.z : w.w;
    int k = 0;
    while (k < rt.n_mix - 1 && u >= rt.thr[k]) ++k;
    p = rt.mix[k];
    if (store)
      for (int h = 0; h < c.n_heads; ++h) rt.targets_out[(int64_t)h * rows + r] = (int)((p >> (8 * h)) & 0xFF) - 1;
  }
  if (bad) {
    p = 0;
    for (int h = 0; h < c.n_heads; ++h)
      if (c.targets[h] >= 0) p |= 1u << (8 * h);
  }
  return p;
}

// Target of head h: the shared one, or from the row's packed targets (-1: left out)
template <bool ROW_TARGETS>
__device__ __forceinline__ int lg_target(const LangevinClf& c, uint32_t tp, int h) {
  if constexpr (ROW_TARGETS) return (int)((tp >> (8 * h)) & 0xFF) - 1;
  else return c.targets[h];
}

static inline size_t langevin_smem_bytes(const LangevinClf& c, bool row_targets = false) {
  const int ldz = c.L + 1, ldh = c.hidden + 1;
  size_t f = (size_t)c.w_floats + (size_t)LG_TILE * ldz                // weights, z
             + (size_t)c.n_trunk * LG_TILE * ldh                       // trunk activations
             + 2 * (size_t)LG_TILE * (c.hidden > c.L ? ldh : ldz)      // gradient ping-pong
             + (size_t)4 * LG_TILE * (LG_MAXC + 1)                     // logits / dlogits per head
             + (row_targets ? (size_t)2 * LG_TILE : 0);                // per-row instance: packed targets, bad-row flags
  return f * sizeof(float);
}

template <bool ROW_TARGETS>
__global__ void __launch_bounds__(LG_THREADS) langevin_kernel(LangevinClf c, const float* __restrict__ params, float* __restrict__ z_io,
                                                              int64_t rows, float step_size, int num_steps, float noise_weight, uint64_t seed,
                                                              uint64_t offset0, int64_t row0, int init_from_philox, const float* __restrict__ noise,
                                                              float* __restrict__ history, float* __restrict__ stats, float prior_weight, float threshold,
                                                              int32_t* __restrict__ stop_step, float* __restrict__ last_prob,
                                                              const __grid_constant__ LangevinRows rt) {
  PSVAE_GRID_DEP();
  extern __shared__ float lg_smem[];
  __shared__ int lg_done[LG_TILE], lg_hit[LG_TILE];      // per sample: stopped (threshold reached at an earlier step) / reaches it at this step
  __shared__ int lg_stop[LG_TILE];
  __shared__ float lg_prob[LG_TILE];
  const int L = c.L, H = c.hidden;
  const int ldz = L + 1, ldh = H + 1, ldd = (H > L ? ldh : ldz), ldc = LG_MAXC + 1;
  float* W = lg_smem;
  float* zs = W + c.w_floats;
  float* acts = zs + LG_TILE * ldz;
  float* d0 = acts + c.n_trunk * LG_TILE * ldh;
  float* d1 = d0 + LG_TILE * ldd;
  float* lgt = d1 + LG_TILE * ldd;
  uint32_t* tgt_s = reinterpret_cast<uint32_t*>(lgt + 4 * LG_TILE * ldc);   // per-row instance: packed targets of the tile's rows
  int* bad_s = reinterpret_cast<int*>(tgt_s + LG_TILE);

  const int tid = threadIdx.x, s = tid & 31, g = tid >> 5;
  const int64_t tile_row0 = (int64_t)blockIdx.x * LG_TILE;
  const int64_t row = tile_row0 + s;
  const bool live = row < rows;
  uint32_t tp = 0;                                   // per-row instance: the packed targets of this lane's sample
  if constexpr (ROW_TARGETS) {
    if (tid < LG_TILE) {
      bool bad = false;
      tgt_s[tid] = tile_row0 + tid < rows ? lg_row_targets(c, rt, rows, tile_row0 + tid, row0, seed, true, bad) : 0u;
      bad_s[tid] = bad;
    }
    __syncthreads();
    tp = tgt_s[s];
  }

  // stage classifier weights once
  for (int j = 0; j < c.n_trunk; ++j) {
    const int K = j == 0 ? L : H;
    for (int i = tid; i < H * K; i += LG_THREADS) W[c.s_trunk_w[j] + i] = params[c.g_trunk_w[j] + i];
    for (int i = tid; i < H; i += LG_THREADS) W[c.s_trunk_b[j] + i] = params[c.g_trunk_b[j] + i];
  }
  const int Kf = c.n_trunk ? H : L;
  for (int h = 0; h < c.n_heads; ++h) {
    for (int i = tid; i < c.head_classes[h] * Kf; i += LG_THREADS) W[c.s_head_w[h] + i] = params[c.g_head_w[h] + i];
    for (int i = tid; i < c.head_classes[h]; i += LG_THREADS) W[c.s_head_b[h] + i] = params[c.g_head_b[h] + i];
  }
  // z tile
  const int quads = LG_TILE * (L >> 2);
  for (int q = tid; q < quads; q += LG_THREADS) {
    const int qs = q / (L >> 2), qk = (q % (L >> 2)) << 2;
    const int64_t r = tile_row0 + qs;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < rows) {
      if (init_from_philox) {
        const float4 t = philox_normal4((uint64_t)((row0 + r) * L + qk) >> 2, seed, offset0);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
        load_vec<4>(z_io + r * L + qk, v);
      }
      if constexpr (ROW_TARGETS) {
        if (bad_s[qs]) v[0] = v[1] = v[2] = v[3] = __int_as_float(0x7fffffff);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) zs[qs * ldz + qk + j] = v[j];
  }
  if (tid < LG_TILE) { lg_done[tid] = 0; lg_hit[tid] = 0; lg_stop[tid] = num_steps; lg_prob[tid] = 0.f; }
  __syncthreads();

  const float half_s2 = 0.5f * step_size * step_size;
  const float nscale = step_size * noise_weight;

  for (int step = 0; step < num_steps; ++step) {
    // 1. trunk forward
    for (int j = 0; j < c.n_trunk; ++j) {
      const float* in = j == 0 ? zs : acts + (j - 1) * LG_TILE * ldh;
      const int ldi = j == 0 ? ldz : ldh, K = j == 0 ? L : H;
      float* out = acts + j * LG_TILE * ldh;
      const float* Wj = W + c.s_trunk_w[j];
      const float* bj = W + c.s_trunk_b[j];
      for (int o = g; o < H; o += 8) {
        float a = bj[o];
        const float* w = Wj + o * K;
        const float* x = in + s * ldi;
#pragma unroll 4
        for (int k = 0; k < K; ++k) a = fmaf(x[k], w[k], a);
        out[s * ldh + o] = lg_act(c.act, a);
      }
      __syncthreads();
    }
    // 2. heads
    const float* feat = c.n_trunk ? acts + (c.n_trunk - 1) * LG_TILE * ldh : zs;
    const int ldf = c.n_trunk ? ldh : ldz;
    for (int h = 0; h < c.n_heads; ++h) {
      if (c.targets[h] < 0) continue;
      const float* Wh = W + c.s_head_w[h];
      const float* bh = W + c.s_head_b[h];
      for (int o = g; o < c.head_classes[h]; o += 8) {
        float a = bh[o];
        const float* w = Wh + o * Kf;
        const float* x = feat + s * ldf;
#pragma unroll 4
        for (int k = 0; k < Kf; ++k) a = fmaf(x[k], w[k], a);
        lgt[(h * LG_TILE + s) * ldc + o] = a;
      }
    }
    __syncthreads();
    // 3. softmax -> d log p(y|z) / d logits = onehot(target) - softmax   (warp 0: one sample per lane)
    if (g == 0) {
      float lp_y = 0.f;
      for (int h = 0; h < c.n_heads; ++h) {
        if (c.targets[h] < 0) continue;
        if constexpr (ROW_TARGETS) {
          if (lg_target<true>(c, tp, h) < 0) continue;
        }
        float* lg = lgt + (h * LG_TILE + s) * ldc;
        const int C = c.head_classes[h];
        float mx = lg[0];
        for (int k = 1; k < C; ++k) mx = fmaxf(mx, lg[k]);
        float se = 0.f;
        for (int k = 0; k < C; ++k) se += expf(lg[k] - mx);
        const float lse = logf(se);
        lp_y += lg[lg_target<ROW_TARGETS>(c, tp, h)] - mx - lse;
        for (int k = 0; k < C; ++k) lg[k] = (k == lg_target<ROW_TARGETS>(c, tp, h) ? 1.f : 0.f) - expf(lg[k] - mx - lse);
      }
      if constexpr (ROW_TARGETS) {
        if (bad_s[s]) lp_y = __int_as_float(0x7fffffff);   // a ReLU / sigmoid trunk can map a NaN z to finite logits
      }
      if (!lg_done[s]) {
        const float p = expf(lp_y);
        lg_prob[s] = p;
        if (threshold > 0.f && p > threshold) { lg_hit[s] = 1; lg_stop[s] = step; }
      }
      if (stats) {
        float lp_z = 0.f;
        for (int k = 0; k < L; ++k) lp_z = fmaf(zs[s * ldz + k], zs[s * ldz + k], lp_z);
        lp_z *= -0.5f;
        const float a = warp_sum(live ? lp_y + lp_z : 0.f);
        const float b = warp_sum(live ? expf(lp_y) : 0.f);
        if (s == 0) {
          atomicAdd(stats + 2 * step, a);
          atomicAdd(stats + 2 * step + 1, b);
        }
      }
    }
    __syncthreads();
    // 4. gradient w.r.t. the head input
    float* dcur = d0;
    float* dnext = d1;
    for (int k = g; k < Kf; k += 8) {
      float a = 0.f;
      for (int h = 0; h < c.n_heads; ++h) {
        if (c.targets[h] < 0) continue;
        if constexpr (ROW_TARGETS) {
          if (lg_target<true>(c, tp, h) < 0) continue;
        }
        const float* Wh = W + c.s_head_w[h];
        const float* dl = lgt + (h * LG_TILE + s) * ldc;
        for (int o = 0; o < c.head_classes[h]; ++o) a = fmaf(dl[o], Wh[o * Kf + k], a);
      }
      if (c.n_trunk) a *= lg_act_grad(c.act, feat[s * ldf + k]);
      dcur[s * ldd + k] = a;
    }
    __syncthreads();
    // 5. trunk backward
    for (int j = c.n_trunk - 1; j >= 0; --j) {
      const int K = j == 0 ? L : H;
      const float* Wj = W + c.s_trunk_w[j];
      const float* prev = j == 0 ? nullptr : acts + (j - 1) * LG_TILE * ldh;
      for (int k = g; k < K; k += 8) {
        float a = 0.f;
        const float* d = dcur + s * ldd;
#pragma unroll 4
        for (int o = 0; o < H; ++o) a = fmaf(d[o], Wj[o * K + k], a);
        if (prev) a *= lg_act_grad(c.act, prev[s * ldh + k]);
        dnext[s * ldd + k] = a;
      }
      __syncthreads();
      float* t = dcur; dcur = dnext; dnext = t;
    }
    // 6. Langevin update (thread = 4 consecutive latent dims = one Philox block)
    for (int q = tid; q < quads; q += LG_THREADS) {
      const int qs = q / (L >> 2), qk = (q % (L >> 2)) << 2;
      const int64_t r = tile_row0 + qs;
      if (r >= rows) continue;
      if (lg_done[qs]) {                     // a stopped sample keeps its z (the history repeats it)
        if (history) {
          float zk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) zk[j] = zs[qs * ldz + qk + j];
          store_vec<4>(history + ((int64_t)step * rows + r) * L + qk, zk);
        }
        continue;
      }
      float nz[4] = {0.f, 0.f, 0.f, 0.f};
      if (noise) {
        load_vec<4>(noise + ((int64_t)step * rows + r) * L + qk, nz);
      } else if (nscale != 0.f) {
        const float4 t = philox_normal4((uint64_t)((row0 + r) * L + qk) >> 2, seed, offset0 + 1 + (uint64_t)step);
        nz[0] = t.x; nz[1] = t.y; nz[2] = t.z; nz[3] = t.w;
      }
      float zn[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float zv = zs[qs * ldz + qk + j];
        const float grad = dcur[qs * ldd + qk + j] - prior_weight * zv;
        zn[j] = zv + half_s2 * grad + nscale * nz[j];
        zs[qs * ldz + qk + j] = zn[j];
      }
      if (history) store_vec<4>(history + ((int64_t)step * rows + r) * L + qk, zn);
    }
    __syncthreads();
    if (tid < LG_TILE && lg_hit[tid]) { lg_done[tid] = 1; lg_hit[tid] = 0; }
    const int all_done = __syncthreads_and(tid >= LG_TILE || lg_done[tid] || tile_row0 + tid >= rows);
    if (all_done && !history && !stats) break;
  }
  if (tid < LG_TILE && tile_row0 + tid < rows) {
    if (stop_step) stop_step[tile_row0 + tid] = lg_stop[tid];
    if (last_prob) last_prob[tile_row0 + tid] = lg_prob[tid];
  }

  for (int q = tid; q < quads; q += LG_THREADS) {
    const int qs = q / (L >> 2), qk = (q % (L >> 2)) << 2;
    const int64_t r = tile_row0 + qs;
    if (r >= rows) continue;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = zs[qs * ldz + qk + j];
    store_vec<4>(z_io + r * L + qk, v);
  }
}

}  // namespace psvae

namespace psvae {

// ------------------------------------------------------------------------------------------------
// Fast path: linear heads directly on z (no trunk -- the reference's default LatentClassifier(num_layers=1)), latent_dim in {16,32,64}.
// ONE THREAD PER SAMPLE: z lives in registers for all steps, the head weights are broadcast reads from shared memory, the noise comes
// from the same counter-based generator with the same counters as the generic kernel (so both produce the same z up to fp32 summation
// order).  No __syncthreads and no shared-memory traffic for z inside the loop: the step is pure ALU/SFU work (Philox + Box-Muller).
// The generator runs in a ROLLED loop (two Philox blocks per trip) that parks the step's L normals in the thread's own column of a
// shared-memory buffer; the fully unrolled form (L/4 inlined copies of Philox + Box-Muller per step, > 50 KB of code) ran out of
// instruction cache -- the same "no_instruction" stall ncu showed on the train step's classifier pass.
// ------------------------------------------------------------------------------------------------
constexpr int LGF_THREADS = 128;

// Per-row instance: the block stages every head some row can name; a thread skips, in every loop over classes, the heads its row leaves out
// (skipped, not multiplied by a zero coefficient, which could turn a -0 gradient into +0).
template <int L, bool ROW_TARGETS>
__global__ void __launch_bounds__(LGF_THREADS) langevin_fast_kernel(LangevinClf c, const float* __restrict__ params, float* __restrict__ z_io, int64_t rows,
                                                                    float step_size, int num_steps, float noise_weight, uint64_t seed, uint64_t offset0,
                                                                    int64_t row0, int init_from_philox, const float* __restrict__ noise,
                                                                    float* __restrict__ history, float* __restrict__ stats, float prior_weight, float threshold,
                                                                    int32_t* __restrict__ stop_step, float* __restrict__ last_prob,
                                                                    const __grid_constant__ LangevinRows rt) {
  PSVAE_GRID_DEP();
  __shared__ __align__(16) float W[CLF_LG_MAXC * L];
  __shared__ float bias[CLF_LG_MAXC];
  __shared__ int cls_head[CLF_LG_MAXC];
  __shared__ float4 nz_s[L / 4][LGF_THREADS];            // this thread's normals of the current step: column threadIdx.x (conflict-free 16-byte accesses)
  // flatten the targeted heads' rows: class index cc -> (head, class)
  int n_cls = 0;
  for (int h = 0; h < c.n_heads; ++h) {
    if (c.targets[h] < 0) continue;
    for (int i = threadIdx.x; i < c.head_classes[h] * L; i += LGF_THREADS) W[n_cls * L + i] = params[c.g_head_w[h] + i];
    if ((int)threadIdx.x < c.head_classes[h]) {
      bias[n_cls + threadIdx.x] = params[c.g_head_b[h] + threadIdx.x];
      cls_head[n_cls + threadIdx.x] = h;
    }
    n_cls += c.head_classes[h];
  }
  __syncthreads();
  const int64_t r = (int64_t)blockIdx.x * LGF_THREADS + threadIdx.x;
  const bool live = r < rows;
  const int64_t rr = live ? r : rows - 1;                 // dead lanes shadow the last row (no stores) so that warp-collectives stay converged
  const uint64_t q0 = (uint64_t)((row0 + rr) * L) >> 2;   // first Philox block of this row
  uint32_t tp = 0, cmask = 0;           // per-row instance: this row's packed targets, and the staged classes cc of the heads it names
  bool bad = false;
  if constexpr (ROW_TARGETS) {
    tp = lg_row_targets(c, rt, rows, rr, row0, seed, live, bad);
    int base = 0;
    for (int h = 0; h < c.n_heads; ++h) {
      if (c.targets[h] < 0) continue;
      if ((tp >> (8 * h)) & 0xFF) cmask |= ((1u << c.head_classes[h]) - 1u) << base;
      base += c.head_classes[h];
    }
  }
  float z[L];
  auto draw = [&](uint64_t offset) {
#pragma unroll 2
    for (int q = 0; q < L / 4; ++q) nz_s[q][threadIdx.x] = philox_normal4(q0 + q, seed, offset);
  };
  if (init_from_philox) {
    draw(offset0);
#pragma unroll
    for (int q = 0; q < L / 4; ++q) {
      const float4 t = nz_s[q][threadIdx.x];
      z[4 * q] = t.x; z[4 * q + 1] = t.y; z[4 * q + 2] = t.z; z[4 * q + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int q = 0; q < L / 4; ++q) {
      const float4 t = *reinterpret_cast<const float4*>(z_io + rr * L + 4 * q);
      z[4 * q] = t.x; z[4 * q + 1] = t.y; z[4 * q + 2] = t.z; z[4 * q + 3] = t.w;
    }
  }
  if (ROW_TARGETS && bad) {
#pragma unroll
    for (int k = 0; k < L; ++k) z[k] = __int_as_float(0x7fffffff);
  }
  const float half_s2 = 0.5f * step_size * step_size;
  const float nscale = step_size * noise_weight;
  bool active = true;                    // false once p(y|z) has exceeded the threshold (this sample's z is final)
  int stop = num_steps;
  float prob = 0.f;
  for (int step = 0; step < num_steps; ++step) {
    if (!history && !stats && !__any_sync(0xffffffffu, active && live)) break;      // the whole warp has stopped
    // logits of the targeted heads
    float coef[CLF_LG_MAXC];
#pragma unroll
    for (int cc = 0; cc < CLF_LG_MAXC; ++cc) {
      float a = 0.f;
      if (cc < n_cls && (!ROW_TARGETS || ((cmask >> cc) & 1u))) {
        a = bias[cc];
#pragma unroll
        for (int k = 0; k < L; k += 4) {
          const float4 w = *reinterpret_cast<const float4*>(&W[cc * L + k]);
          a = fmaf(z[k], w.x, a); a = fmaf(z[k + 1], w.y, a); a = fmaf(z[k + 2], w.z, a); a = fmaf(z[k + 3], w.w, a);
        }
      }
      coef[cc] = a;
    }
    // per head: coef <- onehot(target) - softmax ; lp_y += log p(target)
    float lp_y = 0.f;
    {
      int base = 0;
      for (int h = 0; h < c.n_heads; ++h) {
        if (c.targets[h] < 0) continue;
        const int C = c.head_classes[h];
        if constexpr (ROW_TARGETS) {
          if (lg_target<true>(c, tp, h) < 0) { base += C; continue; }
        }
        float mx = -INFINITY;
#pragma unroll
        for (int cc = 0; cc < CLF_LG_MAXC; ++cc)
          if (cc >= base && cc < base + C) mx = fmaxf(mx, coef[cc]);
        float se = 0.f;
#pragma unroll
        for (int cc = 0; cc < CLF_LG_MAXC; ++cc)
          if (cc >= base && cc < base + C) se += expf(coef[cc] - mx);
        const float lse = logf(se);
#pragma unroll
        for (int cc = 0; cc < CLF_LG_MAXC; ++cc)
          if (cc >= base && cc < base + C) {
            const float lp = coef[cc] - mx - lse;
            const bool tgt = (cc - base) == lg_target<ROW_TARGETS>(c, tp, h);
            if (tgt) lp_y += lp;
            coef[cc] = (tgt ? 1.f : 0.f) - expf(lp);
          }
        base += C;
      }
    }
    if (stats) {
      float lp_z = 0.f;
#pragma unroll
      for (int k = 0; k < L; ++k) lp_z = fmaf(z[k], z[k], lp_z);
      lp_z *= -0.5f;
      const float a = warp_sum(live ? lp_y + lp_z : 0.f);
      const float b = warp_sum(live ? expf(lp_y) : 0.f);
      if ((threadIdx.x & 31) == 0) {
        atomicAdd(stats + 2 * step, a);
        atomicAdd(stats + 2 * step + 1, b);
      }
    }
    bool hit = false;
    if (active) {
      prob = expf(lp_y);
      hit = threshold > 0.f && prob > threshold;
    }
    // z <- z + 0.5 s^2 (W^T coef - prior_weight z) + s * noise_weight * N(0, I)
    if (!noise && nscale != 0.f) draw(offset0 + 1 + (uint64_t)step);
#pragma unroll
    for (int q = 0; q < L / 4; ++q) {
      float nz[4];
      {
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (noise) t = *reinterpret_cast<const float4*>(noise + ((int64_t)step * rows + rr) * L + 4 * q);
        else if (nscale != 0.f) t = nz_s[q][threadIdx.x];
        nz[0] = t.x; nz[1] = t.y; nz[2] = t.z; nz[3] = t.w;
      }
      float g[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int cc = 0; cc < CLF_LG_MAXC; ++cc)
        if (cc < n_cls && (!ROW_TARGETS || ((cmask >> cc) & 1u))) {
          const float4 w = *reinterpret_cast<const float4*>(&W[cc * L + 4 * q]);
          g[0] = fmaf(coef[cc], w.x, g[0]); g[1] = fmaf(coef[cc], w.y, g[1]); g[2] = fmaf(coef[cc], w.z, g[2]); g[3] = fmaf(coef[cc], w.w, g[3]);
        }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float zv = z[4 * q + j];
        if (active) z[4 * q + j] = zv + half_s2 * (g[j] - prior_weight * zv) + nscale * nz[j];
      }
      if (history && live)
        *reinterpret_cast<float4*>(history + ((int64_t)step * rows + r) * L + 4 * q) = make_float4(z[4 * q], z[4 * q + 1], z[4 * q + 2], z[4 * q + 3]);
    }
    if (hit) { active = false; stop = step; }
  }
  if (live) {
    if (stop_step) stop_step[r] = stop;
    if (last_prob) last_prob[r] = prob;
#pragma unroll
    for (int q = 0; q < L / 4; ++q)
      *reinterpret_cast<float4*>(z_io + r * L + 4 * q) = make_float4(z[4 * q], z[4 * q + 1], z[4 * q + 2], z[4 * q + 3]);
  }
}

}  // namespace psvae
