// Fused GEMM epilogues shared by the fp32 CUDA-core engine (sgemm.cuh) and the tcgen05 engine (gemm_tc.cuh).
//
// They implement, in the producing kernel, the element-wise tail of each reference op:
//   EpiBiasAct   nn.Linear bias + ReLU (model.py:14-36) / classifier activations (latent_classifier.py:18-23)
//   EpiMse       mse_loss(x_hat, x)/10 and its gradient 2(x_hat-x)/(B*D*10) (lightning.py:113, SURVEY 3.5)
//   EpiActGrad   dgrad * act'(.) (autograd of ReLU etc.)
//   EpiStore     plain alpha*acc (+ beta*old): split-K wgrad partials, classifier dgrads
//
// Two entry points per functor:
//   apply<NV>(row, col, v, red, split)      -- sgemm: transform NV consecutive accumulator columns of one row AND store them;
//   tc_transform(row, col, N, valid, v, aux, red) -- tcgen05: transform 32 columns in registers only.  The engine then rounds to
//       TOut, stages the 32x32 block in shared memory and writes it with one TMA store (coalesced, clipped at the matrix edge);
//       `aux` is the functor's auxiliary 32x32 bf16 tile (kAuxBytes > 0: the forward activation for EpiActGrad, the target x for EpiMse) which the engine fetched by
//       TMA load.  kColSum: the engine also emits the column sums of what was stored (bias gradients); kReduce: per-CTA sum of `red`.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace psvae {

enum : int { ACT_NONE = -1, ACT_RELU = 0, ACT_TANH = 1, ACT_SIGMOID = 2, ACT_LEAKY = 3 };

template <int ACT> __device__ __forceinline__ float act_fwd(float u) {
  if constexpr (ACT == ACT_RELU) return fmaxf(u, 0.f);
  else if constexpr (ACT == ACT_TANH) return tanhf(u);
  else if constexpr (ACT == ACT_SIGMOID) return 1.f / (1.f + expf(-u));
  else if constexpr (ACT == ACT_LEAKY) return u > 0.f ? u : 0.01f * u;
  else return u;
}
// derivative expressed through the POST-activation value a (what the forward pass stored)
template <int ACT> __device__ __forceinline__ float act_grad_from_out(float a) {
  if constexpr (ACT == ACT_RELU) return a > 0.f ? 1.f : 0.f;
  else if constexpr (ACT == ACT_TANH) return 1.f - a * a;
  else if constexpr (ACT == ACT_SIGMOID) return a * (1.f - a);
  else if constexpr (ACT == ACT_LEAKY) return a > 0.f ? 1.f : 0.01f;
  else return 1.f;
}

template <typename TOut_, int ACT>
struct EpiBiasAct {
  using TOut = TOut_;
  static constexpr bool kReduce = false, kColSum = false, kSplit = false;
  static constexpr bool kBias = true, kReluPack = (ACT == ACT_RELU) && sizeof(TOut_) == 2;
  static constexpr int kAuxBytes = 0;
  const float* bias;   // [N] or nullptr
  TOut* out;
  int64_t ldo;
  float* red_out;      // unused
  uint32_t* mask;      // tcgen05 engine, optional: bit i of mask[(col/32) * mask_ld + row] = (output[row][col + i] > 0) -- the ReLU
  int64_t mask_ld;     //   derivative the backward pass needs, 1 bit per element instead of re-reading the bf16 activation
  template <int NV>
  __device__ __forceinline__ void apply(int64_t row, int col, float (&v)[NV], float& red, int split) const {
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = act_fwd<ACT>(v[i] + (bias ? __ldg(bias + col + i) : 0.f));
    store_vec<NV>(out + row * ldo + col, v);
  }
  __device__ __forceinline__ uint32_t tc_pre(int64_t row, int col, bool valid) const { return 0u; }
  // The engine has already added the bias (kBias: it loads the block's 32 bias values while the TMEM read is in flight).
  // kReluPack (bf16 output + ReLU): v leaves as the PRE-activation; the engine's cvt.rn.relu.bf16x2 clamps while it packs, and the mask
  // comes from sign bits gathered with funnel shifts (one ALU op per element instead of FMNMX + FSETP + SEL + IADD3).
  __device__ __forceinline__ void tc_transform(int64_t row, int col, int N, bool valid, float (&v)[32], const float (&aux)[32], uint32_t pre,
                                               float& red) const {
    if constexpr (kReluPack) {
      if (mask) {
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          uint32_t b = 0;
#pragma unroll
          for (int i = 6; i >= 0; i -= 2) {
            float n0, n1;
            ptx::sub2(n0, n1, 0.f, 0.f, v[8 * k + i], v[8 * k + i + 1]);      // sign bit set  <=>  v > 0  (exact, also for +-0); one FADD2 per pair
            b = __funnelshift_l(__float_as_uint(n1), b, 1);
            b = __funnelshift_l(__float_as_uint(n0), b, 1);
          }
          w[k] = b;
        }
        const uint32_t bits = w[0] | (w[1] << 8) | (w[2] << 16) | (w[3] << 24);
        if (valid) mask[(int64_t)(col >> 5) * mask_ld + row] = bits;      // lanes = consecutive rows: one coalesced 128-byte store per warp
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = act_fwd<ACT>(v[i]);
      if (ACT == ACT_RELU && mask) {
        uint32_t bits = 0;
#pragma unroll
        for (int i = 0; i < 32; ++i) bits |= (v[i] > 0.f ? 1u : 0u) << i;
        if (valid) mask[(int64_t)(col >> 5) * mask_ld + row] = bits;
      }
    }
  }
};

// CS: the tcgen05 engine also emits the column sums of the stored gradient (= the bias gradient of the last decoder layer)
// TX: type of the reconstruction target (float: the caller's fp32 batch; bf16: a batch that arrived in bf16, psvae_b200.h PSVAE_X_BF16)
template <typename TOut_, bool CS = false, typename TX = float>
struct EpiMse {
  using TOut = TOut_;
  static constexpr bool kReduce = true, kColSum = CS, kSplit = false;
  static constexpr bool kBias = true, kReluPack = false;
  static constexpr int kAuxBytes = 1024 * (int)sizeof(TX);      // tcgen05 engine: the target tile x[32 rows][32 cols] arrives by TMA (4 KB fp32 / 2 KB bf16)
  __host__ const void* aux_ptr() const { return x; }
  __host__ int64_t aux_ld() const { return ldx; }
  const float* bias;   // [N]
  const TX* x;         // [M, ldx] target
  int64_t ldx;
  float* x_hat;        // optional fp32 output [M, ldxh]
  int64_t ldxh;
  TOut* out;           // gradient output (x_hat - x) * scale   (may be nullptr for sgemm when no gradients are wanted)
  int64_t ldo;
  float scale;
  float* red_out;      // one slot per CTA: sum of squared differences
  float* colsum;       // CS: [4 * CTAs][N] partial column sums of the gradient, or (colsum_atomic) the [N] bias gradient itself
  int colsum_atomic;
  template <int NV>
  __device__ __forceinline__ void apply(int64_t row, int col, float (&v)[NV], float& red, int split) const {
    float xv[NV];
    load_vec<NV>(x + row * ldx + col, xv);
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] += __ldg(bias + col + i);
    if (x_hat) store_vec<NV>(x_hat + row * ldxh + col, v);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float d = v[i] - xv[i];
      red = fmaf(d, d, red);
      v[i] = d * scale;
    }
    if (out) store_vec<NV>(out + row * ldo + col, v);
  }
  __device__ __forceinline__ uint32_t tc_pre(int64_t row, int col, bool valid) const { return 0u; }
  // aux = the x tile (fp32, fetched by TMA; zero outside the matrix); x_hat (optional) is written straight to global memory
  __device__ __forceinline__ void tc_transform(int64_t row, int col, int N, bool valid, float (&v)[32], const float (&aux)[32], uint32_t pre,
                                               float& red) const {
    if (valid && col + 32 <= N) {
      if (x_hat) store_vec<32>(x_hat + row * ldxh + col, v);
      float r0 = 0.f, r1 = 0.f;
#pragma unroll
      for (int i = 0; i < 32; i += 2) {      // packed pairs: FADD2 / FFMA2 / FMUL2
        float d0, d1;
        ptx::sub2(d0, d1, v[i], v[i + 1], aux[i], aux[i + 1]);
        ptx::fma2(r0, r1, d0, d1, d0, d1);
        ptx::scale2(d0, d1, scale);
        v[i] = d0; v[i + 1] = d1;
      }
      red += r0 + r1;
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        float o = 0.f;
        if (valid && col + i < N) {
          const float h = v[i];
          if (x_hat) x_hat[row * ldxh + col + i] = h;
          const float d = h - aux[i];
          red = fmaf(d, d, red);
          o = d * scale;
        }
        v[i] = o;
      }
    }
  }
};

// CS: also emit the column sums of the stored gradient (= the bias gradient of the layer below)
template <typename TAct, typename TOut_, int ACT, bool CS = false>
struct EpiActGrad {
  using TOut = TOut_;
  static constexpr bool kReduce = false, kColSum = CS, kSplit = false;
  static constexpr bool kBias = false, kReluPack = false;
  static constexpr int kAuxBytes = 0;
  const TAct* act;     // sgemm engine: forward activation (post-activation) [M, lda]
  int64_t lda;
  const uint32_t* mask;   // tcgen05 engine: the bit mask EpiBiasAct wrote in the forward pass, [N/32][mask_ld]
  int64_t mask_ld;
  TOut* out;
  int64_t ldo;
  float beta;          // sgemm only: out = acc * act'(.) + beta * out   (sum over classifier heads)
  float* red_out;
  float* colsum;       // CS: [4 * CTAs][N] partial column sums of the output, or (colsum_atomic) the [N] bias gradient itself
  int colsum_atomic;
  template <int NV>
  __device__ __forceinline__ void apply(int64_t row, int col, float (&v)[NV], float& red, int split) const {
    float a[NV];
    load_vec<NV>(act + row * lda + col, a);
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] *= act_grad_from_out<ACT>(a[i]);
    if (beta != 0.f) {
      float o[NV];
      load_vec<NV>(out + row * ldo + col, o);
#pragma unroll
      for (int i = 0; i < NV; ++i) v[i] = fmaf(beta, o[i], v[i]);
    }
    store_vec<NV>(out + row * ldo + col, v);
  }
  // issued for every block of the tile BEFORE the accumulator is awaited: the (coalesced) mask loads hide behind the MMAs
  __device__ __forceinline__ uint32_t tc_pre(int64_t row, int col, bool valid) const {
    return valid ? __ldg(mask + (int64_t)(col >> 5) * mask_ld + row) : 0u;
  }
  __device__ __forceinline__ void tc_transform(int64_t row, int col, int N, bool valid, float (&v)[32], const float (&aux)[32], uint32_t pre,
                                               float& red) const {
    static_assert(ACT == ACT_RELU, "the bit mask encodes the ReLU derivative");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = (pre >> i) & 1u ? v[i] : 0.f;
  }
};

struct EpiStore {
  using TOut = float;
  static constexpr bool kReduce = false, kColSum = false, kSplit = true;
  static constexpr bool kBias = false, kReluPack = false;
  static constexpr int kAuxBytes = 0;
  float* out;
  int64_t ldo;
  int64_t split_stride;  // elements between split-K partials
  float alpha, beta;     // beta is honoured by the sgemm engine only
  float* red_out;
  int reduce_add;        // tcgen05 engine only: accumulate into `out` ([M][N], no split slots) with TMA reduce-add instead of storing
  template <int NV>
  __device__ __forceinline__ void apply(int64_t row, int col, float (&v)[NV], float& red, int split) const {
    float* p = out + (int64_t)split * split_stride + row * ldo + col;
    if (beta != 0.f) {
      float o[NV];
      load_vec<NV>(p, o);
#pragma unroll
      for (int i = 0; i < NV; ++i) v[i] = fmaf(alpha, v[i], beta * o[i]);
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) v[i] *= alpha;
    }
    store_vec<NV>(p, v);
  }
  __device__ __forceinline__ uint32_t tc_pre(int64_t row, int col, bool valid) const { return 0u; }
  __device__ __forceinline__ void tc_transform(int64_t row, int col, int N, bool valid, float (&v)[32], const float (&aux)[32], uint32_t pre,
                                               float& red) const {
    if (alpha != 1.f) {
#pragma unroll
      for (int i = 0; i < 32; i += 2) ptx::scale2(v[i], v[i + 1], alpha);
    }
  }
};

// Fused encoder head (option "fused_head", tcgen05 engine only; see gemm_tc.cuh, kLat): ONE kernel computes mu = he[:, :H] W_mu^T and
// log_sigma = he[:, H:] W_sigma^T into one 128-column accumulator tile laid out [mu 0-63 | ls 0-63] (one 64-column MMA per encoder and k-step), and its epilogue
// does what clf_fused_kernel<REPARAM> does today -- biases, eps (Philox or injected), z = mu + sigma eps, sigma eps / 2, the KL partial sum,
// the linear-head classifier on mu, cross entropy, accuracy, d loss / d logits -- with a row's mu AND log_sigma in one thread's registers
// (model.py:54-57, lightning.py:73-83,115-117).  Outputs: mu / log_sigma (fp32) and z / sigma eps / 2 (TZ) through TMA stores, d loss / d logits
// rows for the backward (latent_bwd_clf_kernel), one (kl, nll, acc) partial per CTA.  Single classifier head with <= 4 classes, or none.
// DEV_OFF: the Philox offset is *offset_dev (device step counters), read by the epilogue warps after their accumulator-ready wait (only the
// producer passes griddepcontrol.wait; the epilogue is ordered behind it by the mbarrier chain, so by then what earlier kernels wrote is visible)
template <typename TZ, bool DEV_OFF = false>
struct EpiLatent {
  using TOut = float;
  static constexpr bool kReduce = false, kColSum = false, kSplit = false;
  static constexpr bool kBias = false, kReluPack = false;
  static constexpr int kAuxBytes = 0;
  static constexpr bool kLatent = true;
  float* out;            // mu [M][L]; log_sigma is the second slice of the 3D output map
  int64_t ldo;
  const float* bias;     // [2L]: mu biases, then log_sigma biases
  TZ* z;                 // z [M][L]; sigma eps / 2 is the second slice of the 3D aux map
  const float* eps;      // optional injected noise [M][L]
  uint64_t seed, offset;
  int64_t first_quad;    // global index of this shard's first Philox block (row0 * L / 4)
  int L;
  int nc;                // classes of the (single) linear head on mu; 0: no classifier
  const float* clf_w;    // [nc][L]
  const float* clf_b;    // [nc]
  const int64_t* y;      // [M]
  float gscale;          // clf_weight / B
  float* g_rows;         // [M][8] d loss / d logits (nullptr: no gradients wanted)
  float* kl_part;        // [CTAs]
  float* nll_part;       // [CTAs]
  float* acc_part;       // [CTAs]
  const uint64_t* offset_dev;   // DEV_OFF only
  // read where the noise is drawn: after the accumulator-ready wait
  __device__ __forceinline__ uint64_t rng_offset() const {
    if constexpr (DEV_OFF) return *offset_dev;
    else return offset;
  }
  // the generic epilogue loop is never entered for this functor (the kernel's kLat branch takes every tile); these keep it compilable
  __device__ __forceinline__ uint32_t tc_pre(int64_t, int, bool) const { return 0u; }
  __device__ __forceinline__ void tc_transform(int64_t, int, int, bool, float (&)[32], const float (&)[32], uint32_t, float&) const {}
};

}  // namespace psvae
