// Element-wise / reduction kernels of the hot path (everything that is not a GEMM):
//   adam_kernel            torch.optim.Adam single-tensor update (torch/optim/adam.py:416-547) over the flat buffer; one template
//                          <DC, EX, CLIP> for the device-counter, amsgrad / maximize and clipped forms
//   grad_norm_kernel       global L2 norm + clip coefficient of clip_grad_norm_ (adam_kernel<DC, EX, CLIP_NORM> applies it)
//   philox_*_kernel        torch.randn / randn_like replacement (model.py:57, inference.py:23,73,95)
//   cast_bf16_kernel       fp32 -> bf16 operand copies
//   latent_fwd_kernel      sigma = exp(.5 ls); z = mu + sigma*eps; KL partial sums  (model.py:56-57, lightning.py:115-117)
//   latent_bwd_kernel      dmu, dls from dz (SURVEY 3.5)
//   ce_kernel              F.cross_entropy + Accuracy + dlogits (lightning.py:79-80)
//   colsum / reduce        bias gradients, split-K partial sums (deterministic two-stage)
//   row_normalize_kernel   F.normalize(x_hat, p=2, dim=1) (model.py:60-61,67-68)
//   finalize_losses_kernel total = recon + kl_w*kl + clf_w*clf (lightning.py:119-124)
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace psvae {

// ---------------------------------------------------------------- Adam
// HBM-bound: 16 B read (p,g,m,v) + 12 B written per parameter (+2 B bf16 shadow).  One float4 per thread per
// iteration, grid-stride, grid = multiple of the SM count.
struct AdamArgs {
  float lr_step;      // lr / (1 - beta1^t)          (torch: step_size)
  float bc2_sqrt;     // sqrt(1 - beta2^t)
  float beta1, beta2, one_minus_beta1, one_minus_beta2, eps, weight_decay, grad_scale;
};

// Gradient clipping inside the update (torch.nn.utils.clip_grad_norm_ / clip_grad_value_ as Lightning calls them before optimizer.step()),
// before weight decay is added and before maximize negates.  CLIP_NORM: g_eff = g * fp32(grad_scale * coef), coef = min(max_norm /
// (total_norm + 1e-6), 1) read from device memory (grad_norm_kernel) -- folded into grad_scale, so that the update is the unclipped
// kernel's code with another scale (a separate multiply lets the compiler contract the moment updates differently, and coef = 1 would
// then not reproduce the unclipped step bit for bit).  CLIP_VALUE: clamp(g * grad_scale, -v, v); NaN passes through as in torch.clamp.
enum { CLIP_NONE = 0, CLIP_NORM = 1, CLIP_VALUE = 2 };
template <int CLIP>
__device__ __forceinline__ float clip_grad(float g, float c) {
  if constexpr (CLIP == CLIP_VALUE) return g < -c ? -c : (g > c ? c : g);
  return g;
}

template <int CLIP = CLIP_NONE>
__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, const AdamArgs& a, float clip = 0.f) {
  g *= a.grad_scale;
  g = clip_grad<CLIP>(g, clip);
  if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
  m = m + (g - m) * a.one_minus_beta1;                    // exp_avg.lerp_(grad, 1-beta1)
  v = v * a.beta2 + a.one_minus_beta2 * g * g;            // mul_(beta2).addcmul_(g, g, 1-beta2)
  const float denom = sqrtf(v) / a.bc2_sqrt + a.eps;
  p = p - a.lr_step * (m / denom);                        // addcdiv_(m, denom, value=-step_size)
}
// amsgrad (torch/optim/adam.py: max_exp_avg_sqs = maximum(max_exp_avg_sqs, exp_avg_sq); denom from the maximum) / maximize (grad = -grad)
template <int CLIP = CLIP_NONE>
__device__ __forceinline__ void adam_one_ex(float& p, float g, float& m, float& v, float& vmax, const AdamArgs& a, bool amsgrad, bool maximize,
                                            float clip = 0.f) {
  g *= a.grad_scale;
  g = clip_grad<CLIP>(g, clip);
  if (maximize) g = -g;
  if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
  m = m + (g - m) * a.one_minus_beta1;
  v = v * a.beta2 + a.one_minus_beta2 * g * g;
  float vd = v;
  if (amsgrad) { vmax = fmaxf(vmax, v); vd = vmax; }
  const float denom = sqrtf(vd) / a.bc2_sqrt + a.eps;
  p = p - a.lr_step * (m / denom);
}
// the general form: one element per thread and trip (these configurations are not on any benchmarked path)
template <int CLIP = CLIP_NONE>
__device__ __forceinline__ void adam_ex_pass(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                             float* __restrict__ vmax, int64_t n, const AdamArgs& a, int amsgrad, int maximize, bf16* __restrict__ shadow,
                                             float clip = 0.f) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float pp = p[i], mm = m[i], vv = v[i], vx = amsgrad ? vmax[i] : 0.f;
    adam_one_ex<CLIP>(pp, g[i], mm, vv, vx, a, amsgrad != 0, maximize != 0, clip);
    p[i] = pp; m[i] = mm; v[i] = vv;
    if (amsgrad) vmax[i] = vx;
    if (shadow) shadow[i] = __float2bfloat16_rn(pp);
  }
}

template <int CLIP = CLIP_NONE>
__device__ __forceinline__ void adam_pass(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
                                          const AdamArgs& a, bf16* __restrict__ shadow, float clip = 0.f) {
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = __ldg(reinterpret_cast<const float4*>(g) + i);
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    adam_one<CLIP>(pp.x, gg.x, mm.x, vv.x, a, clip);
    adam_one<CLIP>(pp.y, gg.y, mm.y, vv.y, a, clip);
    adam_one<CLIP>(pp.z, gg.z, mm.z, vv.z, a, clip);
    adam_one<CLIP>(pp.w, gg.w, mm.w, vv.w, a, clip);
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
    if (shadow) {
      uint2 u;
      u.x = pack_bf16x2(pp.x, pp.y);
      u.y = pack_bf16x2(pp.z, pp.w);
      reinterpret_cast<uint2*>(shadow)[i] = u;
    }
  }
  // tail (n not a multiple of 4)
  const int64_t t = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) {
    float pp = p[t], mm = m[t], vv = v[t];
    adam_one<CLIP>(pp, g[t], mm, vv, a, clip);
    p[t] = pp; m[t] = mm; v[t] = vv;
    if (shadow) shadow[t] = __float2bfloat16_rn(pp);
  }
}

// The one Adam update kernel.  EX: the amsgrad / maximize form (one element per thread and trip), else float4 (16-byte aligned buffers).
// DC, the device-counter form (CUDA-graph replay): t = *step_done + 1 and lr = *lr come from device memory, read after the grid dependency
// (the previous step's counter advance and a host write of the block are complete by then).  `a` arrives with lr_step / bc2_sqrt unset; they
// are formed here in fp64 exactly as the host forms them for the other form, each rounded to fp32 once.  CLIP_NORM reads coef = *clip_coef
// after the grid dependency (grad_norm_kernel wrote it) and runs the unclipped pass with grad_scale * coef; CLIP_VALUE clamps at clip_value.
// The shared-memory prologue exists only where it is needed: <false, *, CLIP_NONE> is the bare pass.
template <bool DC, bool EX, int CLIP>
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                                   float* __restrict__ vmax, int64_t n, AdamArgs a, double beta1, double beta2,
                                                   const double* __restrict__ lr, const int64_t* __restrict__ step_done, int amsgrad, int maximize,
                                                   bf16* __restrict__ shadow, const float* __restrict__ clip_coef, float clip_value) {
  PSVAE_GRID_DEP();
  if constexpr (DC || CLIP != CLIP_NONE) {
    __shared__ float s_lr_step, s_bc2_sqrt, s_clip;
    if (threadIdx.x == 0) {
      if constexpr (DC) {
        const double t = (double)(*step_done + 1);
        const double bc1 = 1.0 - pow(beta1, t);
        const double bc2 = 1.0 - pow(beta2, t);
        s_lr_step = (float)(*lr / bc1);
        s_bc2_sqrt = (float)sqrt(bc2);
      }
      if constexpr (CLIP != CLIP_NONE) s_clip = CLIP == CLIP_NORM ? a.grad_scale * *clip_coef : clip_value;
    }
    __syncthreads();
    if constexpr (DC) {
      a.lr_step = s_lr_step;
      a.bc2_sqrt = s_bc2_sqrt;
    }
    if constexpr (CLIP == CLIP_NORM) a.grad_scale = s_clip;
    if constexpr (CLIP == CLIP_VALUE) {
      if constexpr (EX) adam_ex_pass<CLIP>(p, g, m, v, vmax, n, a, amsgrad, maximize, shadow, s_clip);
      else adam_pass<CLIP>(p, g, m, v, n, a, shadow, s_clip);
      return;
    }
  }
  if constexpr (EX) adam_ex_pass(p, g, m, v, vmax, n, a, amsgrad, maximize, shadow);
  else adam_pass(p, g, m, v, n, a, shadow);
}

// Global L2 norm of g * scale over a list of [a, b) spans of the flat gradient buffer, and the clip coefficient of
// torch.nn.utils.clip_grad_norm_: coef = min(max_norm / (total_norm + 1e-6), 1) in fp32.  Each thread sums its squares in fp64 in a fixed
// order (grid-stride over the spans), the block reduces in a fixed tree and stores one fp64 partial; the last block to finish (ticket)
// adds the partials in index order.  The grid is GRAD_NORM_BLOCKS whatever the device, so the result is bit-identical from run to run.
// The last block resets the ticket to zero: the kernel can be replayed from a CUDA graph.
constexpr int GRAD_NORM_MAX_SPANS = 16;
constexpr int GRAD_NORM_BLOCKS = 296;
struct GradNormSpans {
  int64_t a[GRAD_NORM_MAX_SPANS], b[GRAD_NORM_MAX_SPANS];
  int n;
};
__device__ __forceinline__ double block_sum_f64(double t, double* sm) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) sm[warp] = t;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0) {
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sm[w];
  }
  return s;        // valid in thread 0
}
__global__ void __launch_bounds__(256) grad_norm_kernel(const float* __restrict__ g, GradNormSpans sp, float scale, float max_norm,
                                                        double* __restrict__ part, unsigned* __restrict__ ticket, float* __restrict__ total_norm,
                                                        float* __restrict__ coef) {
  PSVAE_GRID_DEP();
  __shared__ double sm[8];
  __shared__ bool s_last;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double t = 0.0;
  for (int s = 0; s < sp.n; ++s)
    for (int64_t i = sp.a[s] + tid; i < sp.b[s]; i += stride) {
      const double x = (double)(__ldg(g + i) * scale);
      t = fma(x, x, t);
    }
  const double bs = block_sum_f64(t, sm);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = bs;
    __threadfence();
    s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double u = 0.0;
  for (int j = threadIdx.x; j < (int)gridDim.x; j += blockDim.x) u += __ldcg(part + j);
  __syncthreads();          // sm is reused
  const double tot = block_sum_f64(u, sm);
  if (threadIdx.x == 0) {
    const float tn = (float)sqrt(tot);
    *total_norm = tn;
    *coef = fminf(max_norm / (tn + 1e-6f), 1.0f);
    *ticket = 0u;
  }
}

// grads[i] += part[i]: the accumulating train step adds the gradient of this micro-batch (computed into a scratch buffer exactly as the
// non-accumulating step computes it) to what the buffer holds -- one fp32 addition per element
__global__ void __launch_bounds__(256) grad_accumulate_kernel(float* __restrict__ grads, const float* __restrict__ part, int64_t n) {
  PSVAE_GRID_DEP();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t n4 = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 a = reinterpret_cast<float4*>(grads)[i];
    const float4 b = __ldg(reinterpret_cast<const float4*>(part) + i);
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    reinterpret_cast<float4*>(grads)[i] = a;
  }
  const int64_t t = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) grads[t] += part[t];
}

// rng_offset += d_rng, adam_step += d_step: the end of a device-counter micro-batch that does (d_step = 1) or does not (d_step = 0) step the
// optimiser (every reader of the block has finished: it is the last launch)
__global__ void step_counters_advance_by_kernel(uint64_t* __restrict__ rng_offset, int64_t* __restrict__ adam_step, uint64_t d_rng, int64_t d_step) {
  PSVAE_GRID_DEP();
  *rng_offset += d_rng;
  *adam_step += d_step;
}

// ---------------------------------------------------------------- Philox
__global__ void __launch_bounds__(256) philox_u32_kernel(uint32_t* __restrict__ out, int64_t n, uint64_t seed, uint64_t offset, int64_t first) {
  PSVAE_GRID_DEP();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t q_first = first >> 2, q_last = (first + n - 1) >> 2;
  for (int64_t q = q_first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q <= q_last; q += stride) {
    const uint4 r = philox4x32_10((uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)offset, (uint32_t)(offset >> 32), (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t e = (q << 2) + j - first;
      if (e >= 0 && e < n) out[e] = w[j];
    }
  }
}

// [n_rows, n_cols] normals, element index g = (row0 + r) * n_cols + c  (n_cols % 4 == 0)
template <typename T>
__global__ void __launch_bounds__(256) philox_normal_kernel(T* __restrict__ out, int64_t n_elems, uint64_t seed, uint64_t offset, int64_t first_elem) {
  PSVAE_GRID_DEP();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nq = n_elems >> 2;
  const uint64_t q0 = (uint64_t)first_elem >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += stride) {
    const float4 z = philox_normal4(q0 + (uint64_t)i, seed, offset);
    float v[4] = {z.x, z.y, z.z, z.w};
    store_vec<4>(out + (i << 2), v);
  }
}

// ---------------------------------------------------------------- casts
// zero_buf (optional): `zero_n` floats (a multiple of 4) cleared by the same pass -- the train step's gradient buffer, which the
// backward kernels then accumulate into; a separate memset node would also break the programmatic-launch chain between the optimiser
// pass of the previous step and this kernel
__global__ void __launch_bounds__(256) cast_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, int64_t n, float* __restrict__ zero_buf,
                                                        int64_t zero_n) {
  PSVAE_GRID_DEP();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (zero_buf) {
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (zero_n >> 2); i += stride) reinterpret_cast<float4*>(zero_buf)[i] = z4;
  }
  const int64_t n8 = n >> 3;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    float v[8];
    load_vec<8>(in + (i << 3), v);
    store_vec<8>(out + (i << 3), v);
  }
  const int64_t t = (n8 << 3) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = __float2bfloat16_rn(in[t]);
}

// ---------------------------------------------------------------- batch gather out of an HBM-resident embedding store
// dst[i][:] = src[idx[i]][:] for rows of `vec_per_row` 16-byte vectors (a 256-d bf16 row = 32 vectors = one warp-wide 512-byte read):
// the DataLoader's collate (ps_vae/data/cv.py:73-76 + default_collate) when the packed store lives in HBM.  An index outside [0, src_rows)
// yields a zero row.  HBM-bound: rows are >= 256 B, so every sector fetched is used.
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint4* __restrict__ src, int64_t src_rows, int vec_per_row, const int64_t* __restrict__ idx,
                                                          int64_t n, uint4* __restrict__ dst) {
  PSVAE_GRID_DEP();
  const int64_t total = n * vec_per_row;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t r = i / vec_per_row;
    const int v = (int)(i - r * vec_per_row);
    const int64_t s = __ldg(idx + r);
    uint4 val = make_uint4(0u, 0u, 0u, 0u);
    if (s >= 0 && s < src_rows) val = __ldg(src + s * vec_per_row + v);
    dst[i] = val;
  }
}

// ---------------------------------------------------------------- latent forward / backward
// Thread = 4 consecutive latent elements (= one Philox block).  KL partial: one slot per block.
// DEV_OFF: the Philox offset is *offset_dev (device step counters, read after the grid dependency) instead of `offset`
template <typename TAct, bool DEV_OFF = false>
__global__ void __launch_bounds__(256) latent_fwd_kernel(const float* __restrict__ mu, const float* __restrict__ ls, const float* __restrict__ eps,
                                                         uint64_t seed, uint64_t offset, int64_t first_elem, int64_t n_elems,
                                                         TAct* __restrict__ z, float* __restrict__ z_f32, float* __restrict__ kl_partials,
                                                         TAct* __restrict__ hs, const uint64_t* __restrict__ offset_dev) {
  // hs (optional): sigma * eps / 2 = d z / d log_sigma, stashed for the backward pass (which then needs neither eps nor exp(ls / 2))
  PSVAE_GRID_DEP();
  if constexpr (DEV_OFF) offset = *offset_dev;
  __shared__ float scratch[32];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nq = n_elems >> 2;
  float kl = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += stride) {
    float m[4], l[4], e[4], zz[4], hh[4];
    load_vec<4>(mu + (i << 2), m);
    load_vec<4>(ls + (i << 2), l);
    if (eps) {
      load_vec<4>(eps + (i << 2), e);
    } else {
      const float4 t = philox_normal4(((uint64_t)first_elem >> 2) + (uint64_t)i, seed, offset);
      e[0] = t.x; e[1] = t.y; e[2] = t.z; e[3] = t.w;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float sigma = expf(0.5f * l[j]);
      zz[j] = fmaf(sigma, e[j], m[j]);
      hh[j] = 0.5f * sigma * e[j];
      kl += 1.f + l[j] - m[j] * m[j] - sigma * sigma;          // exp(ls) = sigma^2: one exponential per element
    }
    if (z) store_vec<4>(z + (i << 2), zz);
    if (z_f32) store_vec<4>(z_f32 + (i << 2), zz);
    if (hs) store_vec<4>(hs + (i << 2), hh);
  }
  const float s = block_sum(kl, scratch);
  if (threadIdx.x == 0 && kl_partials) kl_partials[blockIdx.x] = s;
}

// dmu = dz + (kl_w/B) mu + dmu_clf ;  dls = dz * (eps * 0.5 sigma) + (kl_w/2B)(exp(ls) - 1); hs = eps * 0.5 sigma from the forward pass
template <typename TAct>
__global__ void __launch_bounds__(256) latent_bwd_kernel(const float* __restrict__ dz, const float* __restrict__ mu, const float* __restrict__ ls,
                                                         const TAct* __restrict__ hs, int64_t n_elems, const float* __restrict__ dmu_clf, float kl_over_b,
                                                         TAct* __restrict__ dmu, TAct* __restrict__ dls, int qpr, int64_t ld_d,
                                                         const float* __restrict__ dls_ext) {
  // dmu_clf / dls_ext (optional, [rows][L] fp32): gradients reaching mu / log_sigma from outside the VAE -- the latent classifier, or a caller's own loss
  // dmu / dls are [rows][L] views with row stride ld_d (the two halves of one [rows][2L] buffer); qpr = L / 4
  PSVAE_GRID_DEP();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nq = n_elems >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += stride) {
    float g[4], m[4], l[4], e[4], c[4] = {0.f, 0.f, 0.f, 0.f}, om[4], ol[4];
    load_vec<4>(dz + (i << 2), g);
    load_vec<4>(mu + (i << 2), m);
    load_vec<4>(ls + (i << 2), l);
    if (dmu_clf) load_vec<4>(dmu_clf + (i << 2), c);
    load_vec<4>(hs + (i << 2), e);
    float x4[4] = {0.f, 0.f, 0.f, 0.f};
    if (dls_ext) load_vec<4>(dls_ext + (i << 2), x4);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      om[j] = g[j] + kl_over_b * m[j] + c[j];
      ol[j] = fmaf(g[j], e[j], 0.5f * kl_over_b * expm1f(l[j])) + x4[j];   // expm1: no cancellation for ls ~ 0
    }
    const int64_t o = (int64_t)((uint32_t)i / (uint32_t)qpr) * ld_d + (((uint32_t)i % (uint32_t)qpr) << 2);
    store_vec<4>(dmu + o, om);
    store_vec<4>(dls + o, ol);
  }
}

// ---------------------------------------------------------------- cross entropy (one thread per row)
// logits [rows, C] fp32 -> in place: dlogits = (softmax - onehot) * gscale ; partial sums of NLL and of (argmax == y)
__global__ void __launch_bounds__(256) ce_kernel(float* __restrict__ logits, const int64_t* __restrict__ y, int64_t rows, int C, float gscale,
                                                 int write_grad, float* __restrict__ nll_partials, float* __restrict__ acc_partials) {
  PSVAE_GRID_DEP();
  __shared__ float scratch[32];
  float nll = 0.f, correct = 0.f;
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < rows) {
    float* lg = logits + r * C;
    float mx = lg[0];
    int arg = 0;
    for (int c = 1; c < C; ++c)
      if (lg[c] > mx) { mx = lg[c]; arg = c; }      // first maximum, like torch.argmax
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(lg[c] - mx);
    const float lse = logf(se);
    // a label outside [0, C) (utils.map_cv_*_to_label returns -1 for unknown metadata; torch's cross_entropy raises): no out-of-bounds
    // read, and the loss is poisoned with NaN instead of a plausible-looking value
    const int64_t ty = y[r];
    const bool bad = ty < 0 || ty >= (int64_t)C;
    const int t = bad ? 0 : (int)ty;
    nll = bad ? __int_as_float(0x7fc00000) : -(lg[t] - mx - lse);
    correct = (!bad && arg == t) ? 1.f : 0.f;
    if (write_grad) {
      for (int c = 0; c < C; ++c) {
        const float p = expf(lg[c] - mx - lse);
        lg[c] = (p - (c == t ? 1.f : 0.f)) * gscale;
      }
    }
  }
  const float s1 = block_sum(nll, scratch);
  const float s2 = block_sum(correct, scratch);
  if (threadIdx.x == 0) {
    nll_partials[blockIdx.x] = s1;
    acc_partials[blockIdx.x] = s2;
  }
}

// ---------------------------------------------------------------- column sums (bias gradients)
// partials[chunk][col] = sum over the chunk's rows of in[row, col];  block = 32 cols x 8 row-lanes
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ in, int64_t ld, int64_t rows, int N, int64_t rows_per_chunk, float* __restrict__ partials) {
  PSVAE_GRID_DEP();
  __shared__ float sm[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk, r1 = min(rows, r0 + rows_per_chunk);
  float s = 0.f;
  if (col < N)
    for (int64_t r = r0 + ty; r < r1; r += 8) s += to_f32<T>(in[r * ld + col]);
  sm[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && col < N) {
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) t += sm[j][tx];
    partials[(int64_t)blockIdx.y * N + col] = t;
  }
}

// out[i] = scale * sum_s partials[s][i]   (fixed order: deterministic)
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ partials, int64_t n, int S, int64_t stride_s, float scale, float* __restrict__ out) {
  PSVAE_GRID_DEP();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float t = 0.f;
  for (int s = 0; s < S; ++s) t += partials[(int64_t)s * stride_s + i];
  out[i] = t * scale;
}

// out[i] = sum_s partials[s][i] for S >= 32 partial rows and few columns: block = 32 columns x 32 row lanes; row lane y sums rows
// y, y+32, ... in order, then the 32 lane sums are added in a fixed order (deterministic)
__global__ void __launch_bounds__(1024) reduce_tall_kernel(const float* __restrict__ partials, int n, int S, int64_t stride_s, float* __restrict__ out) {
  PSVAE_GRID_DEP();
  __shared__ float sm[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  float t0 = 0.f, t1 = 0.f;
  if (col < n) {
    int s = ty;
    for (; s + 32 < S; s += 64) {
      t0 += partials[(int64_t)s * stride_s + col];
      t1 += partials[(int64_t)(s + 32) * stride_s + col];
    }
    if (s < S) t0 += partials[(int64_t)s * stride_s + col];
  }
  sm[ty][tx] = t0 + t1;
  __syncthreads();
  if (ty == 0 && col < n) {
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) t += sm[j][tx];
    out[col] = t;
  }
}

// ---------------------------------------------------------------- F.normalize(p=2, dim=1): one warp per row
__global__ void __launch_bounds__(256) row_normalize_kernel(float* __restrict__ x, int64_t rows, int D) {
  PSVAE_GRID_DEP();
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  float* p = x + r * D;
  float ss = 0.f;
  for (int c = lane; c < D; c += 32) ss = fmaf(p[c], p[c], ss);
  ss = warp_sum(ss);
  const float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);
  for (int c = lane; c < D; c += 32) p[c] *= inv;
}

// ---------------------------------------------------------------- loss scalars
struct LossPartials {
  const float* sse; int n_sse;           // sum of squared reconstruction errors
  const float* kl; int n_kl;             // sum over elements of (1 + ls - mu^2 - e^ls)
  const float* nll[4]; const float* acc[4]; int n_ce; int n_heads;
  int ce_stride;                         // elements between consecutive nll / acc partials (1, or the per-block record length of the fused classifier pass)
  float recon_scale;                     // 1 / (B * D * 10) for MSE/10, 1 / B for the cosine loss
  float inv_b;                           // 1 / B
  float kl_w, clf_w;
  const float* cons_nll; const float* cons_acc; int n_cons;     // consistency classifier on x_hat (lightning.py:100-108); n_cons = 0: none
  float cons_w;
};

// The 12 sums (sse, kl, 4 x nll, 4 x acc, consistency nll / acc) as 24 warp tasks: task t = (job t & 15, half t >> 4) adds the even / odd
// 32-element chunks of its job's partials, each lane its strided elements in order, then the fixed shuffle tree -- the result depends only on
// the partials, not on timing or on how many warps share the tasks (32 in finalize_losses_kernel, 8 in the block that latent_bwd_clf8_kernel
// lends to it).  part: 32 floats of shared memory.
__device__ __forceinline__ void finalize_losses_block(const LossPartials& lp, float* __restrict__ losses, float* part, int n_warps) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int t = warp; t < 32; t += n_warps) {
    const int job = t & 15, half = t >> 4;
    const float* p = nullptr;
    int n = 0, stride = 1;
    if (job == 0) { p = lp.sse; n = lp.n_sse; }
    else if (job == 1) { p = lp.kl; n = lp.n_kl; }
    else if (job < 6) { if (job - 2 < lp.n_heads) { p = lp.nll[job - 2]; n = lp.n_ce; stride = lp.ce_stride; } }
    else if (job < 10) { if (job - 6 < lp.n_heads) { p = lp.acc[job - 6]; n = lp.n_ce; stride = lp.ce_stride; } }
    else if (job == 10) { p = lp.cons_nll; n = lp.n_cons; }
    else if (job == 11) { p = lp.cons_acc; n = lp.n_cons; }
    float v = 0.f;
    if (p)
      for (int i = half * 32 + lane; i < n; i += 64) v += p[(int64_t)i * stride];
    v = warp_sum(v);
    if (lane == 0) part[t] = v;
  }
  __syncthreads();
  auto total = [&](int j) { return part[j] + part[j + 16]; };
  const float sse = total(0), kls = total(1);
  float nll[4], acc[4];
  for (int h = 0; h < 4; ++h) { nll[h] = total(2 + h); acc[h] = total(6 + h); }
  const float cons_nll = total(10), cons_acc = total(11);
  if (threadIdx.x == 0) {
    const float recon = sse * lp.recon_scale;
    const float kl = -0.5f * kls * lp.inv_b;
    float clf = 0.f;
    for (int h = 0; h < lp.n_heads; ++h) clf += nll[h] * lp.inv_b;
    if (lp.n_heads > 0) clf /= (float)lp.n_heads;
    for (int i = 0; i < 16; ++i) losses[i] = 0.f;
    const float cons = cons_nll * lp.inv_b;
    losses[0] = recon + lp.kl_w * kl + lp.clf_w * clf + (lp.n_cons > 0 ? lp.cons_w * cons : 0.f);
    losses[1] = recon;
    losses[2] = kl;
    losses[3] = clf;
    for (int h = 0; h < lp.n_heads; ++h) {
      losses[4 + h] = nll[h] * lp.inv_b;
      losses[8 + h] = acc[h] * lp.inv_b;
    }
    if (lp.n_cons > 0) {
      losses[12] = cons;
      losses[13] = cons_acc * lp.inv_b;
    }
  }
}

__global__ void __launch_bounds__(1024) finalize_losses_kernel(LossPartials lp, float* __restrict__ losses) {
  PSVAE_GRID_DEP();
  __shared__ float part[32];
  finalize_losses_block(lp, losses, part, 32);
}

}  // namespace psvae

namespace psvae {

// ---------------------------------------------------------------- reconstruction tail, general form
// One warp per row, used when normalize_decoder (model.py:60-61) or use_cos_loss (lightning.py:110-111) is on
// (the plain MSE case is fused into the last decoder GEMM, EpiMse).  u = decoder output before normalisation.
//   x_hat = normalize ? u / max(|u|, 1e-12) : u
//   cos   : loss_row = 1 - <x_hat,x> / sqrt((|x_hat|^2+1e-12)(|x|^2+1e-12)) ; d/dx_hat as in F.cosine_embedding_loss
//   mse   : loss_row = sum (x_hat-x)^2 ; d/dx_hat = (x_hat-x) * gscale
//   du    = normalize ? (dxh - x_hat <x_hat,dxh>) / den : dxh
// gx (optional, [rows][D] fp32): a further d loss / d x_hat added to dxh before the normalisation backward -- the gradient of the
// consistency classifier's cross entropy (lightning.py:100-108).  x == nullptr: only x_hat is written.
template <typename TAct>
__global__ void __launch_bounds__(256) recon_rows_kernel(const float* __restrict__ u, const float* __restrict__ x, int64_t rows, int D, int normalize,
                                                         int use_cos, float gscale, float* __restrict__ x_hat, TAct* __restrict__ du,
                                                         float* __restrict__ loss_partials, const float* __restrict__ gx) {
  PSVAE_GRID_DEP();
  __shared__ float scratch[32];
  const int lane = threadIdx.x & 31;
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  float loss = 0.f;
  if (r < rows) {
    const float* ur = u + r * D;
    const float* xr = x ? x + r * D : nullptr;
    float inv_den = 1.f;
    if (normalize) {
      float ss = 0.f;
      for (int c = lane; c < D; c += 32) ss = fmaf(ur[c], ur[c], ss);
      ss = warp_sum(ss);
      inv_den = 1.f / fmaxf(sqrtf(ss), 1e-12f);
    }
    if (x_hat)
      for (int c = lane; c < D; c += 32) x_hat[r * D + c] = ur[c] * inv_den;
    if (!xr && gx && du) {
      // no reconstruction term: only an incoming d loss / d x_hat (a caller's own loss on the outputs of VAEModel.forward) goes back
      float hd = 0.f;
      if (normalize) {
        for (int c = lane; c < D; c += 32) hd = fmaf(ur[c] * inv_den, gx[r * D + c], hd);
        hd = warp_sum(hd);
      }
      for (int c = lane; c < D; c += 32) {
        float g = gx[r * D + c];
        if (normalize) g = (g - ur[c] * inv_den * hd) * inv_den;
        du[r * D + c] = from_f32<TAct>(g);
      }
    }
    if (xr) {
      float dot = 0.f, m1 = 0.f, m2 = 0.f, sse = 0.f;
      for (int c = lane; c < D; c += 32) {
        const float h = ur[c] * inv_den, xv = xr[c];
        dot = fmaf(h, xv, dot); m1 = fmaf(h, h, m1); m2 = fmaf(xv, xv, m2);
        const float d = h - xv;
        sse = fmaf(d, d, sse);
      }
      dot = warp_sum(dot); m1 = warp_sum(m1); m2 = warp_sum(m2); sse = warp_sum(sse);
      float cosv = 0.f, inv_dn = 0.f, c_over_m1 = 0.f;
      if (use_cos) {
        m1 += 1e-12f; m2 += 1e-12f;
        inv_dn = 1.f / sqrtf(m1 * m2);
        cosv = dot * inv_dn;
        c_over_m1 = cosv / m1;
        loss = 1.f - cosv;
      } else {
        loss = sse;
      }
      if (du) {
        // <x_hat, dxh> for the normalisation backward
        float hd = 0.f;
        if (normalize) {
          for (int c = lane; c < D; c += 32) {
            const float h = ur[c] * inv_den, xv = xr[c];
            float g = use_cos ? -(xv * inv_dn - c_over_m1 * h) * gscale : (h - xv) * gscale;
            if (gx) g += gx[r * D + c];
            hd = fmaf(h, g, hd);
          }
          hd = warp_sum(hd);
        }
        for (int c = lane; c < D; c += 32) {
          const float h = ur[c] * inv_den, xv = xr[c];
          float g = use_cos ? -(xv * inv_dn - c_over_m1 * h) * gscale : (h - xv) * gscale;
          if (gx) g += gx[r * D + c];
          if (normalize) g = (g - h * hd) * inv_den;
          du[r * D + c] = from_f32<TAct>(g);
        }
      }
    }
  }
  if (loss_partials) {
    const float s = block_sum(lane == 0 ? loss : 0.f, scratch);
    if (threadIdx.x == 0) loss_partials[blockIdx.x] = s;
  }
}

// fp32 [rows][cols] -> TAct (same shape, contiguous): z handed to psvae_decode
template <typename TAct>
__global__ void __launch_bounds__(256) convert_kernel(const float* __restrict__ in, TAct* __restrict__ out, int64_t n) {
  PSVAE_GRID_DEP();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = from_f32<TAct>(in[i]);
}

}  // namespace psvae

namespace psvae {

// ---------------------------------------------------------------- fused latent classifier (no trunk: Linear(L, C) heads)
// lightning.py:73-83 + its backward in one pass over mu: logits, log-softmax, NLL, accuracy, dlogits, dmu_clf = sum_h dlogits_h W_h,
// and per-block partial sums of dW_h = dlogits_h^T mu, db_h = colsum(dlogits_h).  One warp per row, lane l owns latent dims
// [l*LPL, (l+1)*LPL).  C is 2..3 per head: far below any tensor-core tile, and the whole thing is one read of mu.
constexpr int CLF_MAXC = 8;     // classes summed over all heads
struct ClfFusedArgs {
  int n_heads, total_classes;
  int head_classes[4], head_off[4];
  int64_t w_off[4], b_off[4];
  float gscale;                 // clf_w / (B * n_heads)
  int write_grad;
  // fast (non-deterministic) mode: the blocks add their dW / db / nll / acc partials straight into the zeroed gradient buffer / sums[8]
  // with atomics and the finish kernel is not launched
  int atomic_out;
  float* grads;
  float* sums;
  // option "clf_grad_in_bwd" (fast mode): only d loss / d logits leaves this pass, as g_rows[B][CLF_MAXC]; d loss / d mu and the classifier's
  // own weight / bias gradients are then formed by the latent backward kernel, which streams mu anyway (no [B][L] dmu buffer round trip)
  float* g_rows;
};
// REPARAM: the same pass over mu also does the reparameterisation (model.py:56-57) and the KL partial sums (lightning.py:115-117):
// z = mu + exp(ls/2) * eps with eps from `eps` or the counter-based Philox stream (counter = global quad index), one read of ls, z written once
struct ReparamArgs {
  const float* ls;
  const float* eps;             // optional injected noise [B][L]
  uint64_t seed, offset;
  int64_t first_quad;           // global index of this shard's first group of 4 latent elements (row0 * L / 4)
  void* z;                      // [B][L] TZ
  float* kl_part;               // one slot per block
  void* hs;                     // optional [B][L] TZ: sigma * eps / 2, stashed for the backward pass
  const uint64_t* offset_dev;   // clf_fused_kernel<..., DEV_OFF = true>: the Philox offset lives here (device step counters)
};
__host__ __device__ __forceinline__ int clf_part_len(int L) { return 8 + CLF_MAXC * L + CLF_MAXC; }   // nll[4] acc[4] dW[8][L] db[8]

constexpr int CLF_TILE = 128;   // rows per block pass (= threads per block): small tiles, 4-5 blocks resident per SM -- the phases of one block
                                // (load, row pass, gradient pass) are serial, so latency is hidden across blocks
constexpr int CLF_ACCW = 4;     // dW elements a thread may own (total_classes * L <= CLF_ACCW * CLF_TILE)
static inline size_t clf_fused_smem_bytes(int L) { return ((size_t)CLF_TILE * (L + 4) + (size_t)CLF_TILE * CLF_MAXC + (size_t)CLF_MAXC * L + CLF_MAXC) * sizeof(float); }

// A block stages a tile of 256 rows of mu in shared memory (read once from HBM, coalesced); then
//   phase 2: thread = row: logits, log-softmax, NLL / accuracy, dlogits -> smem;
//   phase 3: dmu_clf[row][k] = sum_c dlogits[row][c] W[c][k] written coalesced; thread = (class, latent dim): dW[c][k] += sum_rows dlogits[row][c] mu[row][k].
// L is a template parameter (16/32/64/128) so that the row/column index arithmetic is shifts and everything moves as float4; class
// loops run over the classes that exist (2..3 per head), not over the CLF_MAXC slots.
// GROWS (option "clf_grad_in_bwd"): only g_rows leaves the pass; phase 3 and the classifier-gradient tail are compiled out
// DEV_OFF: the Philox offset is *rp.offset_dev, read after the grid dependency
template <int L, typename TZ, bool REPARAM, bool GROWS = false, bool DEV_OFF = false>
__global__ void __launch_bounds__(CLF_TILE) clf_fused_kernel(const float* __restrict__ params, const float* __restrict__ mu, const int64_t* __restrict__ y,
                                                             int64_t B, ClfFusedArgs a, float* __restrict__ dmu_clf, float* __restrict__ part, ReparamArgs rp) {
  PSVAE_GRID_DEP();
  if constexpr (DEV_OFF) rp.offset = *rp.offset_dev;
  float kl = 0.f;
  extern __shared__ __align__(16) float clf_smem[];
  __shared__ float scratch[32];
  constexpr int ldm = L + 4;                            // 16-byte aligned rows; row-per-lane float4 reads are conflict-free per quarter warp
  constexpr int QPR = L / 4;
  float* mu_s = clf_smem;                               // [256][L+4]
  float* g_s = mu_s + CLF_TILE * ldm;                   // [256][8]
  float* W_s = g_s + CLF_TILE * CLF_MAXC;               // [8][L]
  float* b_s = W_s + CLF_MAXC * L;                      // [8]
  const int t = threadIdx.x;
  const int PART = clf_part_len(L);
  const int nc = a.total_classes;
  for (int i = t; i < CLF_MAXC * L; i += CLF_TILE) W_s[i] = 0.f;
  if (t < CLF_MAXC) b_s[t] = 0.f;
  __syncthreads();
  for (int h = 0; h < a.n_heads; ++h) {
    for (int i = t; i < a.head_classes[h] * L; i += CLF_TILE) W_s[a.head_off[h] * L + i] = params[a.w_off[h] + i];
    if (t < a.head_classes[h]) b_s[a.head_off[h] + t] = params[a.b_off[h] + t];
  }
  float nll[4] = {0.f, 0.f, 0.f, 0.f}, acc[4] = {0.f, 0.f, 0.f, 0.f};
  float accW[CLF_ACCW] = {0.f, 0.f, 0.f, 0.f}, accb = 0.f;
  const int n_out = nc * L;                             // dW elements; thread t owns t and t + 256 ...
  const int n_parts = (n_out <= CLF_TILE / 2) ? CLF_TILE / n_out : 1;   // ... or, when there are few, (element, row range) pairs
  const int rows_per_part = CLF_TILE / n_parts;
  const int64_t tiles = (B + CLF_TILE - 1) / CLF_TILE;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t row0 = tile * CLF_TILE;
    __syncthreads();                                    // previous pass is done with the tile buffers (and W_s is loaded)
    {
      // phase 1: thread t owns quads t, t + CLF_TILE, ... of the tile (QPR of them).  The loop is kept ROLLED (two quads per trip, the
      // next trip's mu / log_sigma loads issued before this trip's arithmetic): fully unrolled, 16 copies of Philox + Box-Muller were
      // 64 KB of code and the warps mostly waited for instruction fetch (ncu: no_instruction was the top stall reason).
      auto load_q = [&](int j, float4& mv, float4& lv) {
        const int i = j * CLF_TILE + t;
        mv = make_float4(0.f, 0.f, 0.f, 0.f);
        lv = mv;
        if (row0 + i / QPR < B) {
          mv = __ldg(reinterpret_cast<const float4*>(mu + (row0 + i / QPR) * L + 4 * (i % QPR)));
          if constexpr (REPARAM) lv = __ldg(reinterpret_cast<const float4*>(rp.ls + (row0 + i / QPR) * L + 4 * (i % QPR)));
        }
      };
      auto do_q = [&](int j, const float4& mv, const float4& lv) {
        const int i = j * CLF_TILE + t;
        if constexpr (REPARAM) {
          if (row0 + i / QPR < B) {
            const int64_t el = (row0 + i / QPR) * L + 4 * (i % QPR);
            float4 e;
            if (rp.eps) e = __ldg(reinterpret_cast<const float4*>(rp.eps + el));
            else e = philox_normal4((uint64_t)rp.first_quad + (uint64_t)(el >> 2), rp.seed, rp.offset);
            const float m[4] = {mv.x, mv.y, mv.z, mv.w}, l[4] = {lv.x, lv.y, lv.z, lv.w}, ee[4] = {e.x, e.y, e.z, e.w};
            float zz[4], hh[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float sigma = expf(0.5f * l[q]);
              zz[q] = fmaf(sigma, ee[q], m[q]);
              hh[q] = 0.5f * sigma * ee[q];
              kl += 1.f + l[q] - m[q] * m[q] - sigma * sigma;      // exp(ls) = sigma^2: one exponential per element
            }
            store_vec<4>(static_cast<TZ*>(rp.z) + el, zz);
            if (rp.hs) store_vec<4>(static_cast<TZ*>(rp.hs) + el, hh);
          }
        }
        *reinterpret_cast<float4*>(mu_s + (i / QPR) * ldm + 4 * (i % QPR)) = mv;
      };
      static_assert(QPR % 2 == 0, "two quads per trip");
      float4 m0, l0, m1, l1;
      load_q(0, m0, l0);
      load_q(1, m1, l1);
#pragma unroll 1
      for (int j = 0; j < QPR; j += 2) {
        float4 nm0 = m0, nl0 = l0, nm1 = m1, nl1 = l1;
        if (j + 2 < QPR) {
          load_q(j + 2, nm0, nl0);
          load_q(j + 3, nm1, nl1);
        }
        do_q(j, m0, l0);
        do_q(j + 1, m1, l1);
        m0 = nm0; l0 = nl0; m1 = nm1; l1 = nl1;
      }
    }
    __syncthreads();
    {   // phase 2: one row per thread
      const int64_t r = row0 + t;
      float g[CLF_MAXC];
#pragma unroll
      for (int c = 0; c < CLF_MAXC; ++c) g[c] = 0.f;
      if (r < B) {
        float logit[CLF_MAXC];
#pragma unroll
        for (int c = 0; c < CLF_MAXC; ++c) logit[c] = b_s[c];
        const float* m = mu_s + t * ldm;
#pragma unroll 4
        for (int k = 0; k < L; k += 4) {
          const float4 mv = *reinterpret_cast<const float4*>(m + k);
#pragma unroll
          for (int c = 0; c < CLF_MAXC; ++c)
            if (c < nc) {
              const float4 w = *reinterpret_cast<const float4*>(W_s + c * L + k);
              logit[c] = fmaf(mv.x, w.x, logit[c]); logit[c] = fmaf(mv.y, w.y, logit[c]);
              logit[c] = fmaf(mv.z, w.z, logit[c]); logit[c] = fmaf(mv.w, w.w, logit[c]);
            }
        }
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          if (h < a.n_heads) {
            const int c0 = a.head_off[h], C = a.head_classes[h];
            const int64_t ty = y[(int64_t)h * B + r];
            const int tgt = (ty < 0 || ty >= (int64_t)C) ? -1 : (int)ty;
            float mx = -INFINITY, lt = (tgt < 0) ? __int_as_float(0x7fc00000) : 0.f;      // label out of range: NaN loss (see ce_kernel)
            int arg = 0;
#pragma unroll
            for (int c = 0; c < CLF_MAXC; ++c)
              if (c >= c0 && c < c0 + C) {
                if (logit[c] > mx) { mx = logit[c]; arg = c - c0; }        // first maximum, like torch.argmax
                if (c - c0 == tgt) lt = logit[c];
              }
            float se = 0.f;
#pragma unroll
            for (int c = 0; c < CLF_MAXC; ++c)
              if (c >= c0 && c < c0 + C) se += expf(logit[c] - mx);
            const float lse = logf(se);
            nll[h] += -(lt - mx - lse);
            acc[h] += (arg == tgt) ? 1.f : 0.f;
#pragma unroll
            for (int c = 0; c < CLF_MAXC; ++c)
              if (c >= c0 && c < c0 + C) g[c] = (expf(logit[c] - mx - lse) - ((c - c0) == tgt ? 1.f : 0.f)) * a.gscale;
          }
        }
      }
      *reinterpret_cast<float4*>(g_s + t * CLF_MAXC) = make_float4(g[0], g[1], g[2], g[3]);
      *reinterpret_cast<float4*>(g_s + t * CLF_MAXC + 4) = make_float4(g[4], g[5], g[6], g[7]);
      if constexpr (GROWS) {
        if (a.write_grad && r < B) {
          *reinterpret_cast<float4*>(a.g_rows + r * CLF_MAXC) = make_float4(g[0], g[1], g[2], g[3]);
          *reinterpret_cast<float4*>(a.g_rows + r * CLF_MAXC + 4) = make_float4(g[4], g[5], g[6], g[7]);
        }
      }
    }
    __syncthreads();
    if (a.write_grad && !GROWS) {
      if (dmu_clf) {
        for (int i = t; i < CLF_TILE * QPR; i += CLF_TILE) {      // thread = (row, 4 latent dims): one 16-byte coalesced store
          const int r = i / QPR, k = 4 * (i % QPR);
          if (row0 + r < B) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int c = 0; c < CLF_MAXC; ++c)
              if (c < nc) {
                const float gc = g_s[r * CLF_MAXC + c];
                const float4 w = *reinterpret_cast<const float4*>(W_s + c * L + k);
                v.x = fmaf(gc, w.x, v.x); v.y = fmaf(gc, w.y, v.y); v.z = fmaf(gc, w.z, v.z); v.w = fmaf(gc, w.w, v.w);
              }
            *reinterpret_cast<float4*>(dmu_clf + (row0 + r) * L + k) = v;
          }
        }
      }
      if (n_parts > 1) {
        // few classes: every thread owns one dW element and one of n_parts row ranges of the tile (summed in a fixed order at the end)
        const int o = t % n_out, part_i = t / n_out;
        if (part_i < n_parts) {
          const int c = o / L, k = o % L, r0 = part_i * rows_per_part;
          float v = 0.f;
#pragma unroll 4
          for (int r = r0; r < r0 + rows_per_part; ++r) v = fmaf(g_s[r * CLF_MAXC + c], mu_s[r * ldm + k], v);
          accW[0] += v;
        }
      } else {
#pragma unroll
        for (int j = 0; j < CLF_ACCW; ++j) {
          const int o = t + j * CLF_TILE;
          if (o < n_out) {
            const int c = o / L, k = o % L;
            float v = 0.f;
#pragma unroll 4
            for (int r = 0; r < CLF_TILE; ++r) v = fmaf(g_s[r * CLF_MAXC + c], mu_s[r * ldm + k], v);
            accW[j] += v;
          }
        }
      }
      if (t < nc) {
        float v = 0.f;
        for (int r = 0; r < CLF_TILE; ++r) v += g_s[r * CLF_MAXC + t];
        accb += v;
      }
    }
  }
  if constexpr (REPARAM) {
    const float ks = block_sum(kl, scratch);
    if (t == 0) rp.kl_part[blockIdx.x] = ks;
  }
  // where one accumulated dW / db element goes in the flat gradient buffer (atomic_out)
  auto grad_slot = [&](int c, int k) -> float* {
    for (int h = 0; h < a.n_heads; ++h)
      if (c >= a.head_off[h] && c < a.head_off[h] + a.head_classes[h])
        return k >= 0 ? a.grads + a.w_off[h] + (int64_t)(c - a.head_off[h]) * L + k : a.grads + a.b_off[h] + (c - a.head_off[h]);
    return nullptr;
  };
  if (a.atomic_out) {
    for (int h = 0; h < a.n_heads; ++h) {
      const float s1 = block_sum(nll[h], scratch);
      const float s2 = block_sum(acc[h], scratch);
      if (t == 0) { part[(int64_t)blockIdx.x * PART + h] = s1; part[(int64_t)blockIdx.x * PART + 4 + h] = s2; }   // losses stay order-fixed: summed by finalize_losses
    }
    if (!a.write_grad || GROWS) return;
    if (n_parts > 1) {
      __syncthreads();
      float* comb = clf_smem;
      if (t < n_parts * n_out) comb[(t / n_out) * n_out + t % n_out] = accW[0];
      __syncthreads();
      if (t < n_out) {
        float v = 0.f;
        for (int p = 0; p < n_parts; ++p) v += comb[p * n_out + t];
        atomicAdd(grad_slot(t / L, t % L), v);
      }
    } else {
#pragma unroll
      for (int j = 0; j < CLF_ACCW; ++j) {
        const int o = t + j * CLF_TILE;
        if (o < n_out) atomicAdd(grad_slot(o / L, o % L), accW[j]);
      }
    }
    if (t < nc) atomicAdd(grad_slot(t, -1), accb);
    return;
  }
  float* mine = part + (int64_t)blockIdx.x * PART;
  for (int h = 0; h < 4; ++h) {
    const float s1 = block_sum(nll[h], scratch);
    const float s2 = block_sum(acc[h], scratch);
    if (t == 0) { mine[h] = s1; mine[4 + h] = s2; }
  }
  for (int o = t; o < CLF_MAXC * L; o += CLF_TILE) mine[8 + o] = 0.f;
  if (n_parts > 1) {
    __syncthreads();                           // the tile buffers are free now: reuse them to combine the row-range partials
    float* comb = clf_smem;                    // [n_parts][n_out] <= 256 floats
    if (t < n_parts * n_out) comb[(t / n_out) * n_out + t % n_out] = accW[0];
    __syncthreads();
    if (t < n_out) {
      float v = 0.f;
      for (int p = 0; p < n_parts; ++p) v += comb[p * n_out + t];
      mine[8 + t] = v;
    }
  } else {
#pragma unroll
    for (int j = 0; j < CLF_ACCW; ++j) {
      const int o = t + j * CLF_TILE;
      if (o < n_out) mine[8 + o] = accW[j];    // same thread wrote the zero above: program order
    }
  }
  if (t < CLF_MAXC) mine[8 + CLF_MAXC * L + t] = (t < nc) ? accb : 0.f;
}

// sum the per-block partials in block order (32 row lanes, fixed-order tree) and scatter: nll/acc sums -> sums[8], dW/db -> the flat gradient buffer
__global__ void __launch_bounds__(1024) clf_fused_finish_kernel(const float* __restrict__ part, int blocks, int L, ClfFusedArgs a, float* __restrict__ sums,
                                                                float* __restrict__ grads) {
  PSVAE_GRID_DEP();
  __shared__ float sm[32][33];
  const int PART = clf_part_len(L);
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + tx;
  float t = 0.f;
  if (i < PART)
    for (int b = ty; b < blocks; b += 32) t += part[(int64_t)b * PART + i];
  sm[ty][tx] = t;
  __syncthreads();
  if (ty != 0 || i >= PART) return;
  t = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j) t += sm[j][tx];
  if (i < 8) { sums[i] = t; return; }
  if (!a.write_grad || !grads) return;
  int c, k = -1;
  if (i < 8 + CLF_MAXC * L) { c = (i - 8) / L; k = (i - 8) % L; } else { c = i - 8 - CLF_MAXC * L; }
  for (int h = 0; h < a.n_heads; ++h)
    if (c >= a.head_off[h] && c < a.head_off[h] + a.head_classes[h]) {
      const int cc = c - a.head_off[h];
      if (k >= 0) grads[a.w_off[h] + (int64_t)cc * L + k] = t;
      else grads[a.b_off[h] + cc] = t;
    }
}

// ---------------------------------------------------------------- latent backward with fused bias gradients
// As latent_bwd_kernel, plus the column sums of dmu and dls (= bias gradients of the encoders' last Linear): every thread always
// owns the same 4 latent columns (the grid stride is a multiple of L/4), so it sums them privately; block partials [blocks][2L].
template <typename TAct>
__global__ void __launch_bounds__(256) latent_bwd_cs_kernel(const float* __restrict__ dz, const float* __restrict__ mu, const float* __restrict__ ls,
                                                            const TAct* __restrict__ hs, int64_t n_elems, int L, const float* __restrict__ dmu_clf, float kl_over_b,
                                                            TAct* __restrict__ dmu, TAct* __restrict__ dls, float* __restrict__ partials,
                                                            float* __restrict__ bias_grad, int64_t ld_d, const float* __restrict__ dls_ext) {
  // dmu / dls: [rows][L] views with row stride ld_d (the two halves of one [rows][2L] buffer)
  // bias_grad != nullptr (fast mode): the block's 2L column sums are added straight into the zeroed [mu | sigma] bias gradient with atomics;
  // otherwise one partial row per block for the ordered reduce
  PSVAE_GRID_DEP();
  extern __shared__ float lb_smem[];        // [256][8]
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nq = n_elems >> 2;
  float sm_[4] = {0.f, 0.f, 0.f, 0.f}, sl_[4] = {0.f, 0.f, 0.f, 0.f};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += stride) {
    float g[4], m[4], l[4], e[4], c[4] = {0.f, 0.f, 0.f, 0.f}, om[4], ol[4];
    load_vec<4>(dz + (i << 2), g);
    load_vec<4>(mu + (i << 2), m);
    load_vec<4>(ls + (i << 2), l);
    if (dmu_clf) load_vec<4>(dmu_clf + (i << 2), c);
    load_vec<4>(hs + (i << 2), e);
    float x4[4] = {0.f, 0.f, 0.f, 0.f};
    if (dls_ext) load_vec<4>(dls_ext + (i << 2), x4);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      om[j] = g[j] + kl_over_b * m[j] + c[j];
      ol[j] = fmaf(g[j], e[j], 0.5f * kl_over_b * expm1f(l[j])) + x4[j];
      sm_[j] += om[j];
      sl_[j] += ol[j];
    }
    const uint32_t qpr_ = (uint32_t)L >> 2;
    const int64_t o = (int64_t)((uint32_t)i / qpr_) * ld_d + (((uint32_t)i % qpr_) << 2);
    store_vec<4>(dmu + o, om);
    store_vec<4>(dls + o, ol);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) { lb_smem[threadIdx.x * 8 + j] = sm_[j]; lb_smem[threadIdx.x * 8 + 4 + j] = sl_[j]; }
  __syncthreads();
  const int qpr = L >> 2;                   // quads per row; 256 % qpr == 0 (host-checked)
  if ((int)threadIdx.x < 2 * L) {
    const int which = threadIdx.x / L, col = threadIdx.x % L, quad = col >> 2, j = col & 3;
    float t = 0.f;
    for (int th = quad; th < 256; th += qpr) t += lb_smem[th * 8 + which * 4 + j];
    if (bias_grad) atomicAdd(bias_grad + threadIdx.x, t);
    else partials[(int64_t)blockIdx.x * 2 * L + threadIdx.x] = t;
  }
}

// ---------------------------------------------------------------- latent backward + the linear-head classifier's backward from d loss / d logits
// latent_bwd_cs_kernel plus (option "clf_grad_in_bwd", fast mode): g_rows[B][CLF_MAXC] = d loss / d logits of the fused classifier pass;
//   dmu_clf[r][k] = sum_c g[r][c] W[c][k]      (formed in registers: the thread's 4 columns of W are loaded once)
//   dW[c][k]     += sum_r g[r][c] mu[r][k]     (private partial per thread, block-reduced like the bias sums, then atomics)
//   db[c]        += sum_r g[r][c]
// NC = classes summed over all heads (2..CLF_MAXC): registers scale with it.
struct ClfBwdArgs {
  int n_heads, total_classes;
  int head_classes[4], head_off[4];
  int64_t w_off[4], b_off[4];
  const float* params;
  float* grads;
  const float* g_rows;
};
template <typename TAct, int NC>
__global__ void __launch_bounds__(256, 3) latent_bwd_clf_kernel(const float* __restrict__ dz, const float* __restrict__ mu, const float* __restrict__ ls,
                                                             const TAct* __restrict__ hs, int64_t n_elems, int L, float kl_over_b, TAct* __restrict__ dmu,
                                                             TAct* __restrict__ dls, float* __restrict__ bias_grad, int64_t ld_d, ClfBwdArgs ca) {
  PSVAE_GRID_DEP();
  extern __shared__ float lb_smem[];        // [256][8]
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nq = n_elems >> 2;
  const uint32_t qpr_ = (uint32_t)L >> 2;   // quads per row; the grid stride is a multiple of it: a thread keeps its 4 columns
  const int col4 = (int)(((uint32_t)blockIdx.x * blockDim.x + threadIdx.x) % qpr_) << 2;
  const int nc = ca.total_classes;
  auto head_of = [&](int cc) {
    int h = 0;
    for (int i = 0; i < ca.n_heads; ++i)
      if (cc >= ca.head_off[i] && cc < ca.head_off[i] + ca.head_classes[i]) h = i;
    return h;
  };
  float Wc[NC][4], accW[NC][4], accb[NC];
#pragma unroll
  for (int cc = 0; cc < NC; ++cc) {
    accb[cc] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) { Wc[cc][j] = 0.f; accW[cc][j] = 0.f; }
    if (cc < nc) {
      const int h = head_of(cc);
      load_vec<4>(ca.params + ca.w_off[h] + (int64_t)(cc - ca.head_off[h]) * L + col4, Wc[cc]);
    }
  }
  float sm_[4] = {0.f, 0.f, 0.f, 0.f}, sl_[4] = {0.f, 0.f, 0.f, 0.f};
  // Two quads per trip, every load of both issued before any arithmetic (the kernel is latency-bound: ~7 trips per thread, 5 dependent-free
  // loads each); d loss / d logits comes in as one or two float4 straight into registers (an indexed local array cost a stack frame)
  struct Quad { float4 g, m, l, e, ga, gb; int64_t row; uint32_t q; bool on; };
  auto load_quad = [&](int64_t i) {
    Quad t;
    t.on = i < nq;
    t.g = t.m = t.l = t.e = t.ga = t.gb = make_float4(0.f, 0.f, 0.f, 0.f);
    t.row = 0; t.q = 0;
    if (t.on) {
      t.g = __ldg(reinterpret_cast<const float4*>(dz) + i);
      t.m = __ldg(reinterpret_cast<const float4*>(mu) + i);
      t.l = __ldg(reinterpret_cast<const float4*>(ls) + i);
      float hv[4];
      load_vec<4>(hs + (i << 2), hv);
      t.e = make_float4(hv[0], hv[1], hv[2], hv[3]);
      t.row = (int64_t)((uint32_t)i / qpr_);
      t.q = (uint32_t)i % qpr_;
      t.ga = __ldg(reinterpret_cast<const float4*>(ca.g_rows + t.row * CLF_MAXC));
      if (NC > 4) t.gb = __ldg(reinterpret_cast<const float4*>(ca.g_rows + t.row * CLF_MAXC + 4));
    }
    return t;
  };
  auto do_quad = [&](const Quad& t) {
    if (!t.on) return;
    const float g[4] = {t.g.x, t.g.y, t.g.z, t.g.w}, m[4] = {t.m.x, t.m.y, t.m.z, t.m.w}, l[4] = {t.l.x, t.l.y, t.l.z, t.l.w}, e[4] = {t.e.x, t.e.y, t.e.z, t.e.w};
    const float gr[8] = {t.ga.x, t.ga.y, t.ga.z, t.ga.w, t.gb.x, t.gb.y, t.gb.z, t.gb.w};
    float c[4] = {0.f, 0.f, 0.f, 0.f}, om[4], ol[4];
    const bool first_quad = t.q == 0;
#pragma unroll
    for (int cc = 0; cc < NC; ++cc) {
      if (cc < nc) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          c[j] = fmaf(gr[cc], Wc[cc][j], c[j]);
          accW[cc][j] = fmaf(gr[cc], m[j], accW[cc][j]);
        }
        if (first_quad) accb[cc] += gr[cc];
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      om[j] = g[j] + kl_over_b * m[j] + c[j];
      ol[j] = fmaf(g[j], e[j], 0.5f * kl_over_b * expm1f(l[j]));
      sm_[j] += om[j];
      sl_[j] += ol[j];
    }
    const int64_t o = t.row * ld_d + (t.q << 2);
    store_vec<4>(dmu + o, om);
    store_vec<4>(dls + o, ol);
  };
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += 2 * stride) {
    const Quad a0 = load_quad(i);
    const Quad a1 = load_quad(i + stride);
    do_quad(a0);
    do_quad(a1);
  }
  const int qpr = L >> 2;
  // bias gradients of the encoders' last Linear: as latent_bwd_cs_kernel (atomics into the zeroed [mu | sigma] bias gradient)
#pragma unroll
  for (int j = 0; j < 4; ++j) { lb_smem[threadIdx.x * 8 + j] = sm_[j]; lb_smem[threadIdx.x * 8 + 4 + j] = sl_[j]; }
  __syncthreads();
  if ((int)threadIdx.x < 2 * L) {
    const int which = threadIdx.x / L, col = threadIdx.x % L, quad = col >> 2, j = col & 3;
    float t = 0.f;
    for (int th = quad; th < 256; th += qpr) t += lb_smem[th * 8 + which * 4 + j];
    atomicAdd(bias_grad + threadIdx.x, t);
  }
  // the classifier's own gradients, one class at a time through the same staging array
#pragma unroll
  for (int cc = 0; cc < NC; ++cc) {
    if (cc < nc) {            // block-uniform
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 4; ++j) lb_smem[threadIdx.x * 8 + j] = accW[cc][j];
      lb_smem[threadIdx.x * 8 + 4] = accb[cc];
      __syncthreads();
      const int h = head_of(cc), lc = cc - ca.head_off[h];
      if ((int)threadIdx.x < L) {
        const int col = threadIdx.x, quad = col >> 2, j = col & 3;
        float t = 0.f;
        for (int th = quad; th < 256; th += qpr) t += lb_smem[th * 8 + j];
        atomicAdd(ca.grads + ca.w_off[h] + (int64_t)lc * L + col, t);
      } else if ((int)threadIdx.x == L) {
        float t = 0.f;
        for (int th = 0; th < 256; ++th) t += lb_smem[th * 8 + 4];      // only the threads that own a row's first quad added to it
        atomicAdd(ca.grads + ca.b_off[h] + lc, t);
      }
    }
  }
}

// The classifier's own gradients from g_rows alone (classifier-only train step, fast mode, fused encoder head): the fused head leaves
// d loss / d logits per row in g_rows, and with the VAE frozen there is no latent backward to fold them into.
//   dW[c][k] += sum_r g[r][c] mu[r][k],   db[c] += sum_r g[r][c]
// Same thread layout and block reduction as latent_bwd_clf_kernel (a thread keeps its 4 columns; 256 % (L / 4) == 0), atomics into the
// zeroed classifier span.  One read of mu and g_rows.
template <int NC>
__global__ void __launch_bounds__(256) clf_rows_wgrad_kernel(const float* __restrict__ mu, int64_t n_elems, int L, ClfBwdArgs ca) {
  PSVAE_GRID_DEP();
  __shared__ float lb_smem[256 * 8];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nq = n_elems >> 2;
  const uint32_t qpr_ = (uint32_t)L >> 2;
  const int nc = ca.total_classes;
  float accW[NC][4], accb[NC];
#pragma unroll
  for (int cc = 0; cc < NC; ++cc) {
    accb[cc] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) accW[cc][j] = 0.f;
  }
#pragma unroll 4
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += stride) {
    const float4 m = __ldg(reinterpret_cast<const float4*>(mu) + i);
    const int64_t row = (int64_t)((uint32_t)i / qpr_);
    const float4 ga = __ldg(reinterpret_cast<const float4*>(ca.g_rows + row * CLF_MAXC));
    float4 gb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (NC > 4) gb = __ldg(reinterpret_cast<const float4*>(ca.g_rows + row * CLF_MAXC + 4));
    const float gr[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
    const float mv[4] = {m.x, m.y, m.z, m.w};
    const bool first_quad = ((uint32_t)i % qpr_) == 0;
#pragma unroll
    for (int cc = 0; cc < NC; ++cc) {
      if (cc < nc) {
#pragma unroll
        for (int j = 0; j < 4; ++j) accW[cc][j] = fmaf(gr[cc], mv[j], accW[cc][j]);
        if (first_quad) accb[cc] += gr[cc];
      }
    }
  }
  const int qpr = L >> 2;
  for (int cc = 0; cc < NC; ++cc) {
    if (cc < nc) {            // block-uniform
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 4; ++j) lb_smem[threadIdx.x * 8 + j] = accW[cc][j];
      lb_smem[threadIdx.x * 8 + 4] = accb[cc];
      __syncthreads();
      int h = 0;
      for (int i = 0; i < ca.n_heads; ++i)
        if (cc >= ca.head_off[i] && cc < ca.head_off[i] + ca.head_classes[i]) h = i;
      const int lc = cc - ca.head_off[h];
      if ((int)threadIdx.x < L) {
        const int col = threadIdx.x, quad = col >> 2, j = col & 3;
        float t = 0.f;
        for (int th = quad; th < 256; th += qpr) t += lb_smem[th * 8 + j];
        atomicAdd(ca.grads + ca.w_off[h] + (int64_t)lc * L + col, t);
      } else if ((int)threadIdx.x == L) {
        float t = 0.f;
        for (int th = 0; th < 256; ++th) t += lb_smem[th * 8 + 4];      // only the threads that own a row's first quad added to it
        atomicAdd(ca.grads + ca.b_off[h] + lc, t);
      }
    }
  }
}

// The same pass for the tcgen05 mode's common shape (bf16 sigma eps / 2 and outputs, L % 8 == 0, at most 4 classes in total): one thread owns
// EIGHT consecutive latent columns of a row per trip and two rows are in flight (16 independent 16-byte loads per thread before the first use;
// 128 registers at two blocks per SM).  The 4-column form above ran at 2.3 TB/s with spills at its 80-register cap
// (profiles/r02_ncu_full_step_v20.csv: 26.7 us for 77 MB); d loss / d logits of a row arrives as one float4.
template <int NC>
__global__ void __launch_bounds__(256, 2) latent_bwd_clf8_kernel(const float* __restrict__ dz, const float* __restrict__ mu, const float* __restrict__ ls,
                                                                  const bf16* __restrict__ hs, int64_t rows, int L, float kl_over_b, bf16* __restrict__ dmu,
                                                                  bf16* __restrict__ dls, float* __restrict__ bias_grad, int64_t ld_d, ClfBwdArgs ca,
                                                                  LossPartials lp, float* __restrict__ losses) {
  PSVAE_GRID_DEP();
  static_assert(NC >= 1 && NC <= 4, "one float4 of d loss / d logits per row");
  extern __shared__ float lb_smem[];        // [256][8]
  // losses != nullptr: the LAST block of the grid turns the forward pass's loss partials into the 16 loss scalars (what finalize_losses_kernel
  // does as a launch of its own between the forward and the backward pass: one launch boundary less on the step's critical path)
  const int n_blocks = (int)gridDim.x - (losses ? 1 : 0);
  if (losses && (int)blockIdx.x == n_blocks) {
    finalize_losses_block(lp, losses, lb_smem, 8);
    return;
  }
  const int tpr = L >> 3;                   // threads per row
  const int rpb = 256 / tpr;                // rows per block and trip
  const int cgp = (int)threadIdx.x % tpr, col8 = cgp << 3, rin = (int)threadIdx.x / tpr;
  const int nc = ca.total_classes;
  auto head_of = [&](int cc) {
    int h = 0;
    for (int i = 0; i < ca.n_heads; ++i)
      if (cc >= ca.head_off[i] && cc < ca.head_off[i] + ca.head_classes[i]) h = i;
    return h;
  };
  // the classifier weights live in shared memory behind the reduction array ([NC][L] floats, read back as two 16-byte loads per class and trip:
  // 16 fewer live registers than a private copy)
  float* const Wsh = lb_smem + 256 * 8;
  for (int i = threadIdx.x; i < NC * L; i += 256) {
    const int cc = i / L, k = i % L;
    float wv = 0.f;
    if (cc < nc) {
      const int h = head_of(cc);
      wv = ca.params[ca.w_off[h] + (int64_t)(cc - ca.head_off[h]) * L + k];
    }
    Wsh[i] = wv;
  }
  __syncthreads();
  float accW[NC][8], accb[NC];
#pragma unroll
  for (int cc = 0; cc < NC; ++cc) {
    accb[cc] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) accW[cc][j] = 0.f;
  }
  float sm_[8], sl_[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) sm_[j] = sl_[j] = 0.f;
  struct Oct { float4 g0, g1, m0, m1, l0, l1, gr; uint4 e; };
  auto load_oct = [&](int64_t row, Oct& t) {
    const int64_t o = row * L + col8;
    t.g0 = __ldg(reinterpret_cast<const float4*>(dz + o));
    t.g1 = __ldg(reinterpret_cast<const float4*>(dz + o) + 1);
    t.m0 = __ldg(reinterpret_cast<const float4*>(mu + o));
    t.m1 = __ldg(reinterpret_cast<const float4*>(mu + o) + 1);
    t.l0 = __ldg(reinterpret_cast<const float4*>(ls + o));
    t.l1 = __ldg(reinterpret_cast<const float4*>(ls + o) + 1);
    t.e = __ldg(reinterpret_cast<const uint4*>(hs + o));
    t.gr = __ldg(reinterpret_cast<const float4*>(ca.g_rows + row * CLF_MAXC));
  };
  auto do_oct = [&](int64_t row, const Oct& t) {
    const float g[8] = {t.g0.x, t.g0.y, t.g0.z, t.g0.w, t.g1.x, t.g1.y, t.g1.z, t.g1.w};
    const float m[8] = {t.m0.x, t.m0.y, t.m0.z, t.m0.w, t.m1.x, t.m1.y, t.m1.z, t.m1.w};
    const float l[8] = {t.l0.x, t.l0.y, t.l0.z, t.l0.w, t.l1.x, t.l1.y, t.l1.z, t.l1.w};
    const uint32_t ew[4] = {t.e.x, t.e.y, t.e.z, t.e.w};
    const float gr[4] = {t.gr.x, t.gr.y, t.gr.z, t.gr.w};
    float c[8], om[8], ol[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) c[j] = 0.f;
#pragma unroll
    for (int cc = 0; cc < NC; ++cc) {
      if (cc < nc) {
        const float4 w0 = *reinterpret_cast<const float4*>(Wsh + cc * L + col8), w1 = *reinterpret_cast<const float4*>(Wsh + cc * L + col8 + 4);
        const float wc[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          c[j] = fmaf(gr[cc], wc[j], c[j]);
          accW[cc][j] = fmaf(gr[cc], m[j], accW[cc][j]);
        }
        if (cgp == 0) accb[cc] += gr[cc];
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float e = __uint_as_float((j & 1) ? (ew[j >> 1] & 0xFFFF0000u) : (ew[j >> 1] << 16));
      om[j] = g[j] + kl_over_b * m[j] + c[j];
      ol[j] = fmaf(g[j], e, 0.5f * kl_over_b * expm1f(l[j]));
      sm_[j] += om[j];
      sl_[j] += ol[j];
    }
    uint4 um, ul;
    um.x = pack_bf16x2(om[0], om[1]); um.y = pack_bf16x2(om[2], om[3]); um.z = pack_bf16x2(om[4], om[5]); um.w = pack_bf16x2(om[6], om[7]);
    ul.x = pack_bf16x2(ol[0], ol[1]); ul.y = pack_bf16x2(ol[2], ol[3]); ul.z = pack_bf16x2(ol[4], ol[5]); ul.w = pack_bf16x2(ol[6], ol[7]);
    *reinterpret_cast<uint4*>(dmu + row * ld_d + col8) = um;
    *reinterpret_cast<uint4*>(dls + row * ld_d + col8) = ul;
  };
  // software pipeline: the NEXT row's eight 16-byte loads are issued before the current row's arithmetic (expm1f, 2 NC x 8 FMAs, packing), so
  // that memory requests are in flight all the time -- with both rows loaded and then both computed the kernel alternated between the two
  const int64_t step = (int64_t)n_blocks * rpb;
  int64_t r = (int64_t)blockIdx.x * rpb + rin;
  if (r < rows) {
    Oct cur, nxt;
    load_oct(r, cur);
    for (; r < rows; r += step) {
      const bool more = r + step < rows;
      if (more) load_oct(r + step, nxt);
      do_oct(r, cur);
      if (more) cur = nxt;
    }
  }
  // bias gradients of the encoders' last Linear ([mu | sigma], atomics into the zeroed gradient): the tpr-strided threads own the same 8 columns
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; ++j) lb_smem[threadIdx.x * 8 + j] = which ? sl_[j] : sm_[j];
    __syncthreads();
    if ((int)threadIdx.x < L) {
      const int col = threadIdx.x, grp = col >> 3, j = col & 7;
      float t = 0.f;
      for (int th = grp; th < 256; th += tpr) t += lb_smem[th * 8 + j];
      atomicAdd(bias_grad + which * L + col, t);
    }
  }
  // the classifier's own gradients, one class at a time through the same staging array
#pragma unroll
  for (int cc = 0; cc < NC; ++cc) {
    if (cc < nc) {            // block-uniform
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 8; ++j) lb_smem[threadIdx.x * 8 + j] = accW[cc][j];
      __syncthreads();
      const int h = head_of(cc), lc = cc - ca.head_off[h];
      if ((int)threadIdx.x < L) {
        const int col = threadIdx.x, grp = col >> 3, j = col & 7;
        float t = 0.f;
        for (int th = grp; th < 256; th += tpr) t += lb_smem[th * 8 + j];
        atomicAdd(ca.grads + ca.w_off[h] + (int64_t)lc * L + col, t);
      }
      __syncthreads();
      if (cgp == 0) lb_smem[rin] = accb[cc];
      __syncthreads();
      if (threadIdx.x == 0) {
        float t = 0.f;
        for (int th = 0; th < rpb; ++th) t += lb_smem[th];
        atomicAdd(ca.grads + ca.b_off[h] + lc, t);
      }
    }
  }
}

}  // namespace psvae
